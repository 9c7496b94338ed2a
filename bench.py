#!/usr/bin/env python
"""bench.py — the reference's headline benchmark (caf_rust/benches/caf_bench.rs:150-168: one 400 x 8192
fp64 CAF surface + find_peak on the chirp_0 pair) on B200, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg1|cfg2]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path over one surface: FFT(s1) once, the fused row kernel over all doppler
rows, find_peak -- ONE kernel launch.  At N > 1 every rank owns its own s0/s1 pairs (pairs sharded, no data-path
collective: "scaling": "weak").  `value` is device-resident throughput (inputs already in HBM): W warm-up steps, then
exactly K steps between two barriers with one CUDA event pair on the launching stream, max over ranks.  L2 is kept cold
by the working set (the steps rotate over 320 seeded pairs and 8 surface buffers = 252 MB > the 126 MB L2); round 1's
method (L2 flushed before every step, one event pair per step) is reported beside it as `flushed_per_step`.
`e2e` is the reference-facing call sequence through the C ABI with pageable HOST inputs: CafSurface::caf_surface +
find_peak as the Rust shim binds them (device-resident surface object with lazy rows -- CafSurfaceRow's fields are private
upstream -- so what crosses PCIe per step is 134 KB in and find_peak's answer out); `e2e_surface_to_host` is the same call
with the whole 26 MB surface delivered to host memory.
The same run also measures the SHARDED path at every N (`sharded`: config 3 with its doppler rows sharded over the ranks
+ the library's NCCL peak exchange, strong scaling; a config-4 slice with pairs sharded + gather) and, at N = 1, compact
config-2 and config-5-row blocks.

--impl reference times the reference's CPU algorithm (oracle port of CafRustFFTThreadpool, all host
cores) on the same workload; the Rust crate itself cannot be compiled in this image (DESIGN.md).

--dump-outputs DIR writes what the timed path returned in its last timed step (rank 0) as DIR/<name>.npy, float64
(float32 for cfg2's surface and row peak values): surface, row_peak_value, row_peak_index and peak.  The inputs are seeded, so two
builds run with the same arguments can be compared array for array.  The bench writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the bench writes nothing into the tree: it imports modules the build never does (scripts/bench_stream,
# caf_cookoff_b200.generate / .dist), whose bytecode caches would otherwise be created next to them
sys.dont_write_bytecode = True

FS = 48000
L = 4096
N = 2 * L
# BASELINE.md section 1: the reference's published figure for exactly this metric (one 400 x 8192 fp64 surface +
# find_peak, README.md:36, rust RustFFT + threadpool on an R9-3900X, 12C/24T): 28 ms = 117.0 Mcell/s.  Other hardware.
PUBLISHED_CELLS_PER_S = 400 * N / 28e-3
PUBLISHED_NOTE = "BASELINE.md: rust RustFFT + threadpool, 28 ms per surface on an R9-3900X (README.md:36)"
# ONE workload string for both arms (the driver compares them): BASELINE config 1
WORKLOAD_CFG1 = ("cfg1: 400 doppler x 8192 delay fp64 CAF surface + peak per step per GPU, utils/generate.py seed-0 pairs "
                 "(rank r uses chirp_r), fs=48000")
WORKLOAD_CFG2 = WORKLOAD_CFG1.replace("cfg1", "cfg2").replace("fp64", "complex64/float32")


_JSON_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner on the first
    communicator), so fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, surface, row_peak_val, row_peak_idx, peak):
    """The outputs of one step as the caller receives them: the D x 2L surface, every row's peak value and delay index,
    and find_peak's answer as [value, freq_hz, doppler_idx, delay_idx].  Indices are stored as float64 (exact below 2^53)."""
    arrays = {"surface": np.asarray(surface), "row_peak_value": np.asarray(row_peak_val),
              "row_peak_index": np.asarray(row_peak_idx).astype(np.float64),
              "peak": np.asarray(peak, dtype=np.float64)}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def algorithmic_flops(d: int, n: int) -> float:
    """SURVEY.md section 8(d): per row 10 N log2 N + 15 N; plus 5 N log2 N once per pair for FFT(s1)."""
    lg = np.log2(n)
    return d * (10.0 * n * lg + 15.0 * n) + 5.0 * n * lg


def planted_answer(index: int):
    """(lag in samples, doppler offset in Hz) the generator planted into fixture `index`: it is in the file name
    (generate.py:68), e.g. chirp_0_T+202samp_F+69.25Hz.c64."""
    import re
    data = os.path.join(ROOT, "tests", "golden", "data")
    index %= 10
    name = sorted(f for f in os.listdir(data) if f.startswith(f"chirp_{index}_T"))[0]
    m = re.match(r"chirp_\d+_T([+-]\d+)samp_F([+-][0-9.]+)Hz\.c64", name)
    return int(m.group(1)), float(m.group(2))


def peak_is_planted(index: int, freq_hz: float, delay: int, grid_step_hz: float = 0.5) -> bool:
    """The timed call's answer must be the pair's planted lag, on a doppler bin next to the planted offset; for the
    README pair (index 0) it must be the known answer of the 0.5 Hz bench grid, (69.0 Hz, 202)."""
    lag, fo = planted_answer(index)
    if index % 10 == 0 and (freq_hz, delay) != (69.0, 202):
        return False
    return delay == lag and abs(freq_hz - fo) <= grid_step_hz


def load_pair(index: int):
    """s0/s1 of the reference benchmark (chirp_0) or, for other ranks, the next pairs of the same seed-0
    stream — read from the committed fixtures, which the seeded generator port reproduces bit-exactly."""
    from caf_cookoff_b200 import read_file_c64
    data = os.path.join(ROOT, "tests", "golden", "data")
    index %= 10
    names = sorted(f for f in os.listdir(data) if f.startswith(f"chirp_{index}_T"))
    needle = read_file_c64(os.path.join(data, f"chirp_{index}_raw.c64"))
    hay = read_file_c64(os.path.join(data, names[0]))
    hay = np.resize(hay[: needle.size], needle.size) if hay.size >= needle.size else np.concatenate(
        [hay, np.zeros(needle.size - hay.size, dtype=hay.dtype)])   # caf_bench.rs:28 haystack.resize
    return needle, hay


class ClockSampler:
    """nvidia-smi style clock / throttle-reason sampling during the timed region (NVML)."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # NVML missing: report that, do not invent clocks
            self.nv, self.err = None, repr(e)

    _NAMES = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
              0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def sample(self):
        if not self.nv:
            return
        try:
            self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.dev, self.nv.NVML_CLOCK_SM)))
            r = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.dev))
            for bit, name in self._NAMES.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def start(self):
        def loop():
            while not self._stop.is_set():
                self.sample()
                time.sleep(0.002)
        self._thr = threading.Thread(target=loop, daemon=True)
        self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": getattr(self, "err", "nvml")}
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def bind_to_gpu_cpus(index: int):
    """One process per GPU: run (and first-touch the pinned host buffers) on the CPUs NVML reports as local to this
    GPU, so the 26 MB D2H copy of every e2e step does not cross the socket interconnect.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def committed_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the row kernel, per launch, from the newest committed
    `ncu --set full` capture (profiles/rNN_traffic.json, written by scripts/summarize_ncu.py)."""
    try:
        pdir = os.path.join(ROOT, "profiles")
        names = sorted(n for n in os.listdir(pdir) if n.endswith("_traffic.json"))
        return json.load(open(os.path.join(pdir, names[-1]))).get("dram_bytes_per_launch") if names else None
    except Exception:
        return None


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def cpu_baseline_run(needle, hay, freqs, budget_s: float, threads: int):
    """The oracle port of CafRustFFTThreadpool (mod.rs:391-461) on this box's host cores."""
    from oracle import oracle as O
    O.caf_surface(needle, hay, freqs[:8], FS, threads=threads, want_surface=True)   # warm (page-in, plan)
    times = []
    t_end = time.perf_counter() + budget_s
    while True:
        t0 = time.perf_counter()
        surf, pidx, pval = O.caf_surface(needle, hay, freqs, FS, threads=threads, want_surface=True)
        O.find_peak(freqs, pidx, pval)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() >= t_end and len(times) >= 3:
            break
    return float(np.median(times)), len(times)


# ------------------------------------------------------------------------------------------------------------------
# The other BASELINE configs, measured in the same run (compact blocks of the JSON line).  Every block checks the peak
# it timed: a wrong answer marks the block "check_ok": false and the run exits non-zero after printing the line.
# ------------------------------------------------------------------------------------------------------------------
class Ctx:
    pass


def _timed(ctx, step, k, warm):
    """One CUDA event pair around k back-to-back steps (working sets here are far larger than L2), max over ranks."""
    import torch
    import torch.distributed as dist
    for _ in range(warm):
        step()
    if ctx.world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(ctx.stream)
    for _ in range(k):
        step()
    e1.record(ctx.stream)
    if ctx.world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / k], dtype=torch.float64, device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def _row_flops(n):
    return 10.0 * n * np.log2(n) + 15.0 * n


def block_cfg3_sharded(ctx, d_total=4096, l=32768, steps=5):
    """BASELINE config 3 (4096 doppler x 65536 delay fp64 surface + peak), STRONG scaling: the doppler rows are sharded
    across the ranks (mod.rs:185,283: rows are independent), each rank runs its block with caf_b200_sharded_f64_dev --
    local rows, find_peak packed in the kernel, ONE ncclAllGather of 32 B per rank over the library-owned communicator,
    device-side resolve -- all inside the timed step, no host synchronisation.  At N > 1 rank 0 also times the
    unsharded job alone in the same run, so efficiency_vs_n1 needs no second process."""
    import tempfile
    import torch
    import torch.distributed as dist
    from caf_cookoff_b200 import generate as G, dist as cdist
    lib, h, dev = ctx.lib, ctx.h, ctx.dev
    pr = G.pair(0, seed=0, chirp_length=l)
    needle, hay = G.as_inputs(pr)
    freqs = np.linspace(-100.0, 100.0, d_total, endpoint=False)
    id_path = os.path.join(tempfile.gettempdir(), "caf_bench_nccl_id_%s_%s" % (
        os.environ.get("MASTER_PORT", "0"), os.environ.get("TORCHELASTIC_RUN_ID", str(os.getpid()))))
    comm = cdist.Comm(h, ctx.world, ctx.rank, id_path)
    lo, hi = comm.shard(d_total)
    d_loc = hi - lo
    nd = torch.from_numpy(needle).to(dev); hd = torch.from_numpy(hay).to(dev)
    fd = torch.from_numpy(freqs[lo:hi].copy()).to(dev)
    surf = torch.empty((max(d_loc, 1), 2 * l), dtype=torch.float64, device=dev)
    rv = torch.empty(max(d_loc, 1), dtype=torch.float64, device=dev); ri = torch.empty(max(d_loc, 1), dtype=torch.int64, device=dev)
    outp = torch.zeros(4, dtype=torch.int64, device=dev)
    launches0 = h.launch_count

    def step():
        comm.sharded_dev(nd.data_ptr(), hd.data_ptr(), l, fd.data_ptr(), d_loc, lo, FS, outp.data_ptr(),
                         surface_local_dev=surf.data_ptr(), row_val_dev=rv.data_ptr(), row_idx_dev=ri.data_ptr())

    ms = _timed(ctx, step, steps, 2)
    launches = (h.launch_count - launches0) // (steps + 2)
    o = outp.cpu().numpy()
    got = (float(o.view(np.float64)[0]), float(o.view(np.float64)[1]), int(o[2]), int(o[3]))   # value, freq, row, delay
    remote_err = comm.remote_error()
    p2p = comm.uses_p2p()
    # ---- the unsharded answer (and, at N > 1, the N = 1 time) on rank 0 --------------------------------------------
    n1_ms, ref = ms, got
    if ctx.world > 1:
        ref_t = torch.zeros(4, dtype=torch.int64, device=dev)
        t1 = torch.zeros(1, dtype=torch.float64, device=dev)
        if ctx.rank == 0:
            fall = torch.from_numpy(freqs).to(dev)
            surf1 = torch.empty((d_total, 2 * l), dtype=torch.float64, device=dev)
            rv1 = torch.empty(d_total, dtype=torch.float64, device=dev); ri1 = torch.empty(d_total, dtype=torch.int64, device=dev)

            def step1():
                rc = lib.caf_b200_batch_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 1, l, fall.data_ptr(), d_total, FS,
                                                surf1.data_ptr(), rv1.data_ptr(), ri1.data_ptr(), ref_t.data_ptr())
                if rc != 0:
                    raise RuntimeError(lib.caf_b200_last_error().decode())
            step1(); torch.cuda.synchronize()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(ctx.stream)
            for _ in range(3):
                step1()
            e1.record(ctx.stream); torch.cuda.synchronize()
            t1[0] = e0.elapsed_time(e1) / 3
            del surf1
        dist.broadcast(ref_t, 0); dist.broadcast(t1, 0)
        r = ref_t.cpu().numpy()
        ref = (float(r.view(np.float64)[0]), float(r.view(np.float64)[1]), int(r[2]), int(r[3]))
        n1_ms = float(t1.item())
    ok = (got == ref) and (got[3] == pr.lag) and not remote_err      # every rank: global peak == unsharded answer, on the planted lag
    okt = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
    if ctx.world > 1:
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    comm.close()
    n = 2 * l
    fl = d_total * _row_flops(n)
    surf_bytes = d_total * n * 8
    return {
        "workload": f"cfg3: {d_total} doppler x {n} delay fp64 surface + peak, doppler rows sharded x{ctx.world} "
                    f"(caf_b200_sharded_f64_dev: local rows + packed find_peak + the 32 B/rank exchange inside the step: "
                    + ("ONE kernel per rank posting into every peer's mailbox over NVLink peer memory and resolving)" if p2p
                       else "ncclAllGather + device resolve)" if ctx.world > 1 else "world of one)"),
        "peak_exchange": "p2p_mailbox_kernel" if p2p else "nccl_allgather",
        "scaling": "strong", "ms_per_step": ms, "cells_per_s": d_total * n / (ms * 1e-3), "steps": steps,
        "rows_per_gpu": d_loc, "launches_per_step": int(launches),
        "n1_ms_same_run": n1_ms, "efficiency_vs_n1": n1_ms / (ctx.world * ms),
        "roofline": {"bound": "fp64", "achieved": fl / (ms * 1e-3) / 1e12, "peak": ctx.world * ctx.tf64, "unit": "TFLOP/s",
                     "frac": fl / (ms * 1e-3) / 1e12 / (ctx.world * ctx.tf64) if ctx.tf64 else None,
                     "hbm_frac_surface_write": surf_bytes / (ms * 1e-3) / 1e9 / (ctx.world * ctx.hbm_peak)},
        "peak": {"value": got[0], "freq_hz": got[1], "doppler_idx": got[2], "delay_idx": got[3], "planted_lag": pr.lag,
                 "planted_foffset_hz": pr.foffset_hz},
        "check_ok": bool(int(okt.item())),
    }


def block_cfg4_slice(ctx, pairs_per_gpu=592, steps=2):
    """A slice of BASELINE config 4 (4096 independent pairs of 400 x 8192, pairs sharded, peaks only): 592 pairs per GPU
    = 4 whole pairs per SM, so this is also the row kernel's STEADY STATE (1600 rows per CTA).  One
    dist.gather_pair_peaks_dev (all_gather of 32 B per pair, device to device) inside the step.  Pair j = seed-0 fixture j mod 10: every copy
    must return its fixture's known answer."""
    import torch
    from caf_cookoff_b200 import bench_shifts, read_file_c64, dist as cdist
    lib, h, dev = ctx.lib, ctx.h, ctx.dev
    data = os.path.join(ROOT, "tests", "golden", "data")
    names = sorted(os.listdir(data))
    ns = np.stack([read_file_c64(os.path.join(data, f"chirp_{i}_raw.c64")) for i in range(10)])
    hs = np.stack([read_file_c64(os.path.join(data, [n for n in names if n.startswith(f"chirp_{i}_T")][0]))[:L] for i in range(10)])
    p_total = pairs_per_gpu * ctx.world
    lo, hi = cdist.shard_bounds(p_total, ctx.world, ctx.rank)
    idx = np.arange(lo, hi) % 10
    freqs = bench_shifts(); d = freqs.size
    nd = torch.from_numpy(ns[idx]).to(dev); hd = torch.from_numpy(hs[idx]).to(dev); fd = torch.from_numpy(freqs).to(dev)
    pk = torch.zeros((hi - lo, 4), dtype=torch.int64, device=dev)
    res = {}

    def step():
        rc = lib.caf_b200_batch_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), hi - lo, L, fd.data_ptr(), d, FS,
                                        None, None, None, pk.data_ptr())
        if rc != 0:
            raise RuntimeError(lib.caf_b200_last_error().decode())
        res["all"] = cdist.gather_pair_peaks_dev(pk, p_total)      # one all_gather_into_tensor on the device, stream-ordered

    ms = _timed(ctx, step, steps, 1)
    allw = res["all"]
    allw = allw.cpu().numpy() if hasattr(allw, "cpu") else np.asarray(allw)
    allw = allw.view(np.uint64).reshape(-1, 4)
    # known answers of the ten fixtures on the 0.5 Hz bench grid: the first copy of each fixture is the reference for
    # the rest (bit-exact), and fixture 0 must be the README answer (69.0 Hz, delay 202)
    ok = allw.shape[0] == p_total
    for j in range(min(p_total, allw.shape[0])):
        ok = ok and bool((allw[j] == allw[j % 10]).all())
    f0 = float(allw[0, 1:2].view(np.float64)[0]); d0 = int(allw[0, 3])
    ok = ok and (f0, d0) == (69.0, 202)
    fl = p_total * d * _row_flops(N)
    return {
        "workload": f"cfg4 slice: {p_total} independent pairs of 400 x 8192 fp64, pairs sharded x{ctx.world} ({pairs_per_gpu} per GPU), "
                    "peaks only, one all_gather of 32 B per pair inside the step",
        "scaling": "weak", "ms_per_step": ms, "cells_per_s": p_total * d * N / (ms * 1e-3), "steps": steps,
        "us_per_row_per_sm": ms * 1e3 / (pairs_per_gpu * d / ctx.sm_count),
        "roofline": {"bound": "fp64", "achieved": fl / (ms * 1e-3) / 1e12, "peak": ctx.world * ctx.tf64, "unit": "TFLOP/s",
                     "frac": fl / (ms * 1e-3) / 1e12 / (ctx.world * ctx.tf64) if ctx.tf64 else None,
                     "note": "row kernel in steady state (1600 rows per CTA): the per-launch costs of the single surface are amortised"},
        "first_peaks": [[float(allw[i, 1:2].view(np.float64)[0]), int(allw[i, 3])] for i in range(min(3, allw.shape[0]))],
        "check_ok": bool(ok),
    }


def block_cfg2(ctx, steps=40):
    """BASELINE config 2: the 400 x 8192 surface in complex64 / float32, device-resident, timed the way the headline is
    (the steps rotate over 320 seeded pairs and 16 surface buffers -- 231 MB, larger than L2 -- one event pair around the
    back-to-back launches, every pair's peak checked against its planted lag), with round 1's figure (L2 flushed before
    every step, one event pair per step) beside it.  The chirp_0 pair is checked against the fp64 answer."""
    import torch
    from caf_cookoff_b200 import bench_shifts
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import bench_stream
    lib, h, dev = ctx.lib, ctx.h, ctx.dev
    needle, hay = load_pair(0)
    freqs = bench_shifts(); d = freqs.size
    nd = torch.from_numpy(needle.astype(np.complex64)).to(dev); hd = torch.from_numpy(hay.astype(np.complex64)).to(dev)
    fd = torch.from_numpy(freqs).to(dev)
    surf = torch.empty((d, N), dtype=torch.float32, device=dev); rv = torch.empty(d, dtype=torch.float32, device=dev)
    ri = torch.empty(d, dtype=torch.int64, device=dev); pk = torch.zeros(4, dtype=torch.int64, device=dev)

    def step():
        rc = lib.caf_b200_batch_f32_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 1, L, fd.data_ptr(), d, FS,
                                        surf.data_ptr(), rv.data_ptr(), ri.data_ptr(), pk.data_ptr())
        if rc != 0:
            raise RuntimeError(lib.caf_b200_last_error().decode())
    ts = []
    for i in range(steps + 5):
        ctx.flush.zero_()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(ctx.stream); step(); e1.record(ctx.stream)
        torch.cuda.synchronize()
        if i >= 5:
            ts.append(e0.elapsed_time(e1))
    ms_flushed = float(np.mean(ts))
    p = pk.cpu().numpy()
    got = (float(p.view(np.float64)[1]), int(p.view(np.uint64)[3]))
    del surf
    rot = bench_stream.measure(lib, h, ctx.stream, dev, pairs=320, surfaces=16, steps=200, warmup=40, f32=True)
    ser = bench_stream.measure(lib, h, ctx.stream, dev, pairs=320, surfaces=16, steps=200, warmup=40, f32=True, overlap=False)
    ms = rot["us_per_surface"] * 1e-3
    fl = d * _row_flops(N)
    return {"workload": "cfg2: 400 doppler x 8192 delay CAF surface + peak in complex64/float32, working set larger than L2 "
                        "(320 seeded pairs, 16 surface buffers), one event pair around 200 back-to-back launches, independent launches overlap",
            "ms_per_step": ms, "cells_per_s": d * N / (ms * 1e-3), "steps": rot["steps"],
            "working_set_mb": rot["working_set_mb"], "pairs_checked": rot["pairs_checked"], "peaks_off": rot["peaks_off"],
            "roofline": {"bound": "fp32", "achieved": fl / (ms * 1e-3) / 1e12, "peak": ctx.tf32, "unit": "TFLOP/s",
                         "frac": fl / (ms * 1e-3) / 1e12 / ctx.tf32 if ctx.tf32 else None},
            "launches_serialised": {"ms_per_step": ser["us_per_surface"] * 1e-3, "frac": ser["frac"], "peaks_off": ser["peaks_off"],
                                    "method": "the same rotation with caf_b200_set_overlap(0)"},
            "flushed_per_step": {"ms_per_step": ms_flushed, "frac": fl / (ms_flushed * 1e-3) / 1e12 / ctx.tf32 if ctx.tf32 else None,
                                 "method": "L2 flushed (256 MiB overwrite) before every step, one CUDA event pair per step (round 1's figure)"},
            "peak": list(got), "check_ok": got == (69.0, 202) and not rot["peaks_off"] and not ser["peaks_off"]}


def block_cfg5_rows(ctx, rows=296, l=1 << 19, steps=2):
    """Rows of BASELINE config 5 (2^20 delay cells, peak only -- the surface is never materialised): `rows` doppler rows
    on this GPU.  The full config is 16 384 such rows over 8 GPUs = 2048 per GPU; time scales with the row count."""
    import torch
    from caf_cookoff_b200 import generate as G
    lib, h, dev = ctx.lib, ctx.h, ctx.dev
    pr = G.pair(0, seed=0, chirp_length=l)
    needle, hay = G.as_inputs(pr)
    # the rows are a slice of the full config's grid (16 384 shifts over [-100, 100) Hz, 0.0122 Hz apart) around the planted
    # offset: 2^19 samples integrate coherently over 10.9 s, so the main lobe is only ~0.09 Hz wide
    full = np.linspace(-100.0, 100.0, 16384, endpoint=False)
    c0 = int(np.argmin(np.abs(full - pr.foffset_hz)))
    r0 = min(max(c0 - rows // 2, 0), full.size - rows)
    freqs = full[r0:r0 + rows].copy()
    nd = torch.from_numpy(needle).to(dev); hd = torch.from_numpy(hay).to(dev); fd = torch.from_numpy(freqs).to(dev)
    pk = torch.zeros(4, dtype=torch.int64, device=dev)

    def step():
        rc = lib.caf_b200_batch_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 1, l, fd.data_ptr(), rows, FS,
                                        None, None, None, pk.data_ptr())
        if rc != 0:
            raise RuntimeError(lib.caf_b200_last_error().decode())
    world = ctx.world
    ctx.world = 1                       # every rank runs its own rows; no cross-rank step in this block
    try:
        ms = _timed(ctx, step, steps, 1)
    finally:
        ctx.world = world
    p = pk.cpu().numpy()
    got = (float(p.view(np.float64)[1]), int(p.view(np.uint64)[3]))
    n = 2 * l
    fl = rows * _row_flops(n)
    # scratch traffic of the three passes (spread2 writes, core reads + writes, gather2 reads one row of n complex128 each)
    moved = rows * 4.0 * n * 16
    return {"workload": f"cfg5 rows: {rows} doppler x {n} delay fp64, peak only (surface never materialised), one GPU",
            "ms_per_step": ms, "us_per_row": ms * 1e3 / rows, "cells_per_s": rows * n / (ms * 1e-3), "steps": steps,
            "roofline": {"bound": "fp64", "achieved": fl / (ms * 1e-3) / 1e12, "peak": ctx.tf64, "unit": "TFLOP/s",
                         "frac": fl / (ms * 1e-3) / 1e12 / ctx.tf64 if ctx.tf64 else None,
                         "hbm_frac_scratch_traffic": moved / (ms * 1e-3) / 1e9 / ctx.hbm_peak,
                         "scratch_bytes_per_row": 4.0 * n * 16, "algorithmic_bytes_per_row": 0},
            "peak": list(got), "planted_lag": pr.lag, "planted_foffset_hz": pr.foffset_hz,
            "check_ok": got[1] == pr.lag and abs(got[0] - pr.foffset_hz) <= 0.1}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    needle, hay = load_pair(0)
    from caf_cookoff_b200 import bench_shifts
    freqs = bench_shifts()
    from oracle import oracle as O
    for _ in range(max(args.warmup, 1)):
        O.caf_surface(needle, hay, freqs, FS, threads=threads, want_surface=True)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        surf, pidx, pval = O.caf_surface(needle, hay, freqs, FS, threads=threads, want_surface=True)
        pk = O.find_peak(freqs, pidx, pval)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        row = int(np.argmax(pval))         # find_peak's strict `>` keeps the first row holding the maximum
        dump_outputs(args.dump_outputs, surf, pval, pidx, [pval[row], pk[0], row, pk[1]])
    med = float(np.median(times))          # the same statistic the GPU arm's cpu_baseline reports
    cells = freqs.size * N
    value = cells / med
    line = {
        "impl": "reference", "metric": "CAF cells/s (400x8192 fp64 surface + peak)", "value": value, "unit": "cells/s",
        "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * med,
        "ms_per_step_mean": 1e3 * float(np.mean(times)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": value / PUBLISHED_CELLS_PER_S,
        "vs_baseline_note": PUBLISHED_NOTE, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD_CFG1},
        "check": {"peak_freq_hz": float(pk[0]), "peak_delay": int(pk[1]), "check_ok": (float(pk[0]), int(pk[1])) == (69.0, 202)},
        "cpu_baseline": {"value": value, "unit": "cells/s", "cores": threads, "kind": "port",
                         "sample": f"{len(times)} whole 400x8192 surfaces (median), oracle port of CafRustFFTThreadpool (3 FFTs/row), {threads} threads"},
        "e2e": {"value": value, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_b200(args):
    import torch
    import torch.distributed as dist
    from caf_cookoff_b200 import Handle, _lib, bench_shifts

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: torch.cuda.is_available() is False and there is no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_cpus(local)       # pinned staging buffers then live on the socket the GPU hangs off
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    f32 = args.workload == "cfg2"
    cdt, rdt = (np.complex64, np.float32) if f32 else (np.complex128, np.float64)
    tcdt, trdt = (torch.complex64, torch.float32) if f32 else (torch.complex128, torch.float64)
    sfx = "f32" if f32 else "f64"

    needle, hay = load_pair(rank)
    freqs = bench_shifts()
    D = freqs.size
    stream = torch.cuda.Stream(device=dev)     # every kernel, copy and event of this bench lives on this stream
    torch.cuda.set_stream(stream)
    h = Handle(local, stream=stream.cuda_stream)

    # ---- device-resident inputs / outputs -----------------------------------------------------------
    needle_d = torch.from_numpy(needle.astype(cdt)).to(dev)
    hay_d = torch.from_numpy(hay.astype(cdt)).to(dev)
    freqs_d = torch.from_numpy(freqs).to(dev)
    surf_d = torch.empty((D, N), dtype=trdt, device=dev)
    rv_d = torch.empty(D, dtype=trdt, device=dev)
    ri_d = torch.empty(D, dtype=torch.int64, device=dev)
    pk_d = torch.zeros(4, dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 2 x the 126 MB L2
    dev_fn = getattr(lib, f"caf_b200_batch_{sfx}_dev")

    def step_dev():
        rc = dev_fn(h.raw, needle_d.data_ptr(), hay_d.data_ptr(), 1, L, freqs_d.data_ptr(), D, FS,
                    surf_d.data_ptr(), rv_d.data_ptr(), ri_d.data_ptr(), pk_d.data_ptr())
        if rc != 0:
            raise RuntimeError(lib.caf_b200_last_error().decode())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_pass(step, k):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        for s0, s1 in evs:
            flush.zero_()
            s0.record(stream)
            step()
            s1.record(stream)
        return evs

    # ---- the timed region (the contract's base form: W warm-up steps, then EXACTLY K steps between two barriers +
    #      synchronise, one CUDA event pair on the launching stream, max over ranks).  L2 is kept cold by the WORKING SET,
    #      not by a flush: the steps rotate over `n_pairs` distinct seeded s0/s1 pairs (utils/generate.py port; pair 0 of
    #      rank 0 is the README's chirp_0 pair) and `n_surf` surface buffers of 26.2 MB -- 320 pairs + 8 surfaces = 252 MB
    #      against the 126 MB L2 -- so nothing a step reads or writes (twiddle tables and code aside) was left in L2 by an
    #      earlier step.  Every pair that ran is checked against the lag / offset the generator planted.
    #      (Round 1 flushed L2 before every step and gave each step its own event pair; that charges every ~41 us kernel the
    #      ~6 us ANY kernel pays between two events after a 256 MiB memset.  That figure is still measured: `flushed_per_step`.)
    from caf_cookoff_b200 import generate as G
    n_pairs, n_surf = 320, 8
    needles_np = np.empty((n_pairs, L), dtype=cdt); hays_np = np.empty((n_pairs, L), dtype=cdt)
    planted = []
    i_ = 0
    seed_ = 32 * rank                                   # ten pairs per seed; every rank draws its own seeds
    while i_ < n_pairs:
        for p_ in G.pairs(seed=seed_, count=min(10, n_pairs - i_)):
            n__, h__ = G.as_inputs(p_)
            needles_np[i_], hays_np[i_] = n__.astype(cdt), h__[:L].astype(cdt)
            planted.append((p_.lag, p_.foffset_hz))
            i_ += 1
        seed_ += 1
    nd_all = torch.from_numpy(needles_np).to(dev); hd_all = torch.from_numpy(hays_np).to(dev)
    surfs = [surf_d] + [torch.empty((D, N), dtype=trdt, device=dev) for _ in range(n_surf - 1)]
    rv_all = torch.empty((n_pairs, D), dtype=trdt, device=dev)
    ri_all = torch.empty((n_pairs, D), dtype=torch.int64, device=dev)
    pk_all = torch.zeros((n_pairs, 4), dtype=torch.int64, device=dev)

    def step_rot(k):
        i = k % n_pairs
        rc = dev_fn(h.raw, nd_all[i].data_ptr(), hd_all[i].data_ptr(), 1, L, freqs_d.data_ptr(), D, FS,
                    surfs[k % n_surf].data_ptr(), rv_all[i].data_ptr(), ri_all[i].data_ptr(), pk_all[i].data_ptr())
        if rc != 0:
            raise RuntimeError(lib.caf_b200_last_error().decode())

    # consecutive steps touch disjoint buffers and nothing else is enqueued between them, which is what the library's
    # overlap switch asks of a caller: a launch may then start on the SMs its predecessor has already left (the same
    # rotation with the launches serialised is timed right after the headline: `launches_serialised`)
    lib.caf_b200_set_overlap(h.raw, 4)
    warm = max(args.warmup, 3)
    for k in range(warm):
        step_rot(k)
    barrier()
    sampler = ClockSampler(local)
    launches0 = h.launch_count
    sampler.start()
    barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(warm, warm + args.steps):
        step_rot(k)
    e1.record(stream)
    sampler.sample()
    barrier()
    sampler.stop()
    launches = h.launch_count - launches0
    if args.dump_outputs and rank == 0:
        k_last = warm + args.steps - 1          # its surface buffer is not written again before this copy
        i_last = k_last % n_pairs
        pk_last = pk_all[i_last].cpu().numpy()
        dump_outputs(args.dump_outputs, surfs[k_last % n_surf].cpu().numpy(), rv_all[i_last].cpu().numpy(),
                     ri_all[i_last].cpu().numpy(), [pk_last.view(np.float64)[0], pk_last.view(np.float64)[1],
                                                    pk_last.view(np.uint64)[2], pk_last.view(np.uint64)[3]])
    total_ms = float(e0.elapsed_time(e1))
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    cells_step = D * N
    value = world * cells_step * args.steps / (total_ms_max * 1e-3)
    step_ms = total_ms_max / args.steps
    # the same K steps with every launch waiting for the one before it (round 2's figure before the overlap existed)
    lib.caf_b200_set_overlap(h.raw, 0)
    for k in range(warm):
        step_rot(k)
    barrier()
    s0_ = torch.cuda.Event(enable_timing=True); s1_ = torch.cuda.Event(enable_timing=True)
    s0_.record(stream)
    for k in range(warm, warm + args.steps):
        step_rot(k)
    s1_.record(stream)
    barrier()
    ts_ = torch.tensor([float(s0_.elapsed_time(s1_))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ts_, op=dist.ReduceOp.MAX)
    serial_ms = float(ts_.item()) / args.steps

    # correctness of what was just timed (asserted below: a wrong peak marks the line check_ok = false and the process
    # exits non-zero): every pair that ran sits on its planted lag, on a doppler bin next to the planted offset; the
    # README pair (rank 0, pair 0) gives its known answer on the 0.5 Hz grid, (69.0 Hz, 202)
    w_ = pk_all.cpu().numpy()
    ran = sorted({k % n_pairs for k in range(warm + args.steps)})
    off = []
    for i in ran:
        f_ = float(w_[i].view(np.float64)[1]); lag_ = int(w_[i].view(np.uint64)[3])
        if lag_ != planted[i][0] % N or abs(f_ - planted[i][1]) > 0.5:
            off.append((i, f_, lag_))
    peak_freq = float(w_[0].view(np.float64)[1]); peak_delay = int(w_[0].view(np.uint64)[3])
    checks = {"device": not off and (rank != 0 or (peak_freq, peak_delay) == (69.0, 202))}

    # ---- the round-1 figure beside it: L2 flushed (256 MiB overwrite) before every step, one event pair per step ----
    fl_steps = min(args.steps, 200)
    for _ in range(3):
        flush.zero_(); step_dev()
    barrier()
    evs = timed_pass(step_dev, fl_steps)
    barrier()
    per_step = np.array([a.elapsed_time(b) for a, b in evs])   # ms
    t = torch.tensor([float(per_step.sum())], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    flushed_ms = float(t.item()) / fl_steps
    pk = pk_d.cpu().numpy()
    checks["device_flushed"] = peak_is_planted(rank, float(pk.view(np.float64)[1]), int(pk.view(np.uint64)[3]))

    # ---- roofline pass: the row kernel alone, same flush regimen, CUDA events inside the library ----------
    lib.caf_b200_set_profiling(h.raw, 1)
    rows_ms, spec_ms, peak_ms = [], [], []
    a_, b_, c_ = C.c_float(), C.c_float(), C.c_float()
    for _ in range(min(max(args.steps, 10), 200)):
        flush.zero_()
        step_dev()
        lib.caf_b200_last_kernel_ms(h.raw, C.byref(a_), C.byref(b_), C.byref(c_))
        spec_ms.append(a_.value); rows_ms.append(b_.value); peak_ms.append(c_.value)
    lib.caf_b200_set_profiling(h.raw, 0)
    rows_flushed_ms = float(np.mean(rows_ms))
    # the dominant kernel's average launch duration over the TIMED REGION: the region holds nothing but K launches of it
    # (one fused launch per step), so it is the region's time / K on this rank
    rows_avg_ms = total_ms / args.steps
    tf = C.c_double()
    lib.caf_b200_probe_fma_tflops(h.raw, 0 if f32 else 1, C.byref(tf))
    row_flops = D * (10.0 * N * np.log2(N) + 15.0 * N)
    achieved_tf = row_flops / (rows_avg_ms * 1e-3) / 1e12
    mp = measured_peaks()
    hbm_peak = (mp or {}).get("hbm_gbs", 6650.0)
    surf_bytes = D * N * np.dtype(rdt).itemsize
    roofline = {
        "bound": "fp64" if not f32 else "fp32", "kernel": f"caf_rows_kernel<{'float' if f32 else 'double'}, kSurface>",
        "achieved": achieved_tf, "peak": tf.value, "unit": "TFLOP/s", "frac": achieved_tf / tf.value if tf.value else None,
        "peak_source": "in-run FMA-pipe probe (caf_b200_probe_fma_tflops); MEASURED_PEAKS.json has no fp64/fp32 entry",
        "flops_per_launch": row_flops, "kernel_ms": rows_avg_ms,
        "traffic": committed_traffic() if not f32 else None,
        "traffic_note": "DRAM bytes per launch from the committed ncu capture; the 26.2 MB surface is written back from the 126 MB L2 after the kernel ends",
        "hbm": {"achieved": surf_bytes / (rows_avg_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": surf_bytes / (rows_avg_ms * 1e-3) / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json (measured)" if mp else "fallback 6650 GB/s"},
        "step_share": {"spectrum_ms": 0.0, "rows_ms": rows_avg_ms, "peak_ms": 0.0,
                       "note": "one fused launch per step: FFT(s1), the rows and find_peak are the same kernel"},
        "kernel_ms_note": "the timed region holds K launches of this kernel and nothing else: kernel_ms = region / K.  Consecutive launches "
                          "overlap (about four share the GPU, caf_b200_set_overlap(4)), so this is a launch's SHARE of the region, not its latency; "
                          "launches_serialised is the same figure with every launch waiting for the one before it",
        "launches_serialised": {"kernel_ms": serial_ms, "frac": row_flops / (serial_ms * 1e-3) / 1e12 / tf.value if tf.value else None},
        "flushed_per_step": {"kernel_ms": rows_flushed_ms, "frac": row_flops / (rows_flushed_ms * 1e-3) / 1e12 / tf.value if tf.value else None,
                             "note": "the same kernel timed alone by CUDA events inside the library, L2 flushed before every launch (round 1's figure)"},
    }
    # the other roofline the north star names: shared memory.  A row moves every value of its two pipelines through the
    # exchange fabric 4 times each way plus the radix-2 mailbox: 72 stores and 72 loads of one complex value per thread
    # (DESIGN.md section 3); nominal peak 128 B/clk per SM at the SM clock.
    try:
        sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
        sm_hz = 1e6 * float(sampler.max_mhz or (mp or {}).get("sm_max_mhz", 1965.0))
        smem_bytes_row = 512 * 144 * (8 if f32 else 16)
        smem_achieved = D * smem_bytes_row / (rows_avg_ms * 1e-3) / 1e12
        smem_peak = sm_count * 128.0 * sm_hz / 1e12
        roofline["smem"] = {"achieved": smem_achieved, "peak": smem_peak, "unit": "TB/s", "frac": smem_achieved / smem_peak,
                            "bytes_per_row": smem_bytes_row,
                            "note": "nominal 128 B/clk/SM; measured LDS.128 runs at 64 B/clk, STS.128 at 112 (scripts/micro/mio_cost.cu)"}
    except Exception as e:      # never let the extra figure break the bench line
        roofline["smem"] = {"error": repr(e)}

    # ---- e2e: the host-pointer C ABI, H2D + D2H inside the timed region.  The caller's three inputs sit back to back in
    #      ONE pinned block from caf_b200_host_alloc (needle | haystack | freqs).  The surface call (pipelined D2H) moves it
    #      with a single DMA (three small H2D copies cost ~6 us each on B200); the peak-only and drop-in calls issue NO copy:
    #      the row kernel's own CTAs read the block across PCIe while they set up (RowArgs::pull_*, CAF_B200_PULL=0 restores
    #      the DMA).  `*_pageable` repeats the calls with plain pageable numpy buffers -- what a caller that knows nothing
    #      about pinned memory (the Rust shim's Vecs, std::vector) pays: one memcpy into the library's pinned block first. -----
    csz = np.dtype(cdt).itemsize
    blk = C.c_void_p()
    if lib.caf_b200_host_alloc(C.byref(blk), 2 * L * csz + D * 8) != 0:
        raise RuntimeError(lib.caf_b200_last_error().decode())
    raw_blk = (C.c_ubyte * (2 * L * csz + D * 8)).from_address(blk.value)
    needle_h = np.frombuffer(raw_blk, dtype=cdt, count=L, offset=0); needle_h[:] = needle.astype(cdt)
    hay_h = np.frombuffer(raw_blk, dtype=cdt, count=L, offset=L * csz); hay_h[:] = hay.astype(cdt)
    freqs_h = np.frombuffer(raw_blk, dtype=np.float64, count=D, offset=2 * L * csz); freqs_h[:] = freqs
    surf_h = torch.empty((D, N), dtype=trdt).pin_memory()
    rv_h = torch.empty(D, dtype=trdt).pin_memory()
    ri_h = torch.empty(D, dtype=torch.int64).pin_memory()
    host_fn = getattr(lib, f"caf_b200_surface_{sfx}")
    peak_fn = getattr(lib, f"caf_b200_peak_{sfx}")
    e2e_steps = min(args.steps, 200)
    h2d = 2 * L * csz + D * 8
    d2h = surf_h.numel() * surf_h.element_size() + rv_h.numel() * rv_h.element_size() + ri_h.numel() * 8 + 32

    def time_host(step):
        # A host call is synchronous: what its caller pays is wall-clock time.  The event pair around a call only measures
        # that if the GPU is IDLE when the call begins -- with the L2 flush still running, the call's host-side work (staging
        # memcpy, launch) would hide behind it and the events would read ~10 us less than the caller waits (as rounds 1 and
        # early 2 did).  So: flush, SYNCHRONISE, then event / call / event.  The plain wall clock per call of an unflushed
        # loop is reported beside it.
        for _ in range(3):
            step()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(e2e_steps)]
        wall_flushed = 0.0
        for s0, s1 in evs:
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            s0.record(stream)
            step()
            s1.record(stream)
            wall_flushed += time.perf_counter() - t0
        barrier()
        tt = torch.tensor([float(sum(a.elapsed_time(b) for a, b in evs))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            step()
        wall_loop = time.perf_counter() - t0
        time_host.last_wall_unflushed_ms = 1e3 * wall_loop / e2e_steps
        return float(tt.item()) / e2e_steps, 1e3 * wall_flushed / e2e_steps

    def surface_call(n_, h_, f_, s_, rv_, ri_, pk_):
        def step():
            rc = host_fn(h.raw, n_.ctypes.data, h_.ctypes.data, L, f_.ctypes.data, D, FS, s_, rv_, ri_, C.cast(C.byref(pk_), C.c_void_p))
            if rc != 0:
                raise RuntimeError(lib.caf_b200_last_error().decode())
        return step

    def peak_call(n_, h_, f_, pk_):
        def step():
            rc = peak_fn(h.raw, n_.ctypes.data, h_.ctypes.data, L, f_.ctypes.data, D, FS, C.cast(C.byref(pk_), C.c_void_p))
            if rc != 0:
                raise RuntimeError(lib.caf_b200_last_error().decode())
        return step

    pk_h = _lib.Peak()
    ms, wall_ms = time_host(surface_call(needle_h, hay_h, freqs_h, surf_h.data_ptr(), rv_h.data_ptr(), ri_h.data_ptr(), pk_h))
    e2e = {"value": world * cells_step / (ms * 1e-3), "unit": "cells/s", "ms_per_step": ms, "steps": e2e_steps,
           "wall_ms_per_step": wall_ms, "wall_ms_per_step_unflushed_loop": time_host.last_wall_unflushed_ms,
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "host_buffers": "pinned: inputs in one caf_b200_host_alloc block (one H2D), outputs in pinned memory",
           "peak": [pk_h.freq_hz, int(pk_h.delay_idx)]}
    checks["e2e_surface_to_host"] = peak_is_planted(rank, pk_h.freq_hz, int(pk_h.delay_idx)) and float(surf_h[int(pk_h.doppler_idx), int(pk_h.delay_idx)]) == pk_h.value

    # the same call without the surface crossing PCIe: caf_b200_peak_* (what caf_bench.rs's closure observes:
    # find_peak(caf_surface(..)) returns (freq, delay); CafSurfaceRow's fields are private, mod.rs:17-22)
    pk2 = _lib.Peak()
    ms, wall_ms = time_host(peak_call(needle_h, hay_h, freqs_h, pk2))
    e2e_peak = {"value": world * cells_step / (ms * 1e-3), "unit": "cells/s", "ms_per_step": ms,
                "wall_ms_per_step": wall_ms, "wall_ms_per_step_unflushed_loop": time_host.last_wall_unflushed_ms,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 32 + 4, "peak": [pk2.freq_hz, int(pk2.delay_idx)],
                "note": "host inputs in (one pinned block, read across PCIe by the kernel's own CTAs: no H2D DMA in front of the launch), "
                        "(freq, delay) out: the surface stays on the GPU (caf_b200_peak_*); the kernel stores the peak into pinned "
                        "host memory and the host spins on a sequence word next to it"}
    checks["e2e_peak_only"] = peak_is_planted(rank, pk2.freq_hz, int(pk2.delay_idx))

    # pageable host memory on both sides (numpy arrays): the drop-in caller's cost
    n_pg, h_pg, f_pg = needle.astype(cdt).copy(), hay.astype(cdt).copy(), freqs.copy()
    surf_pg = np.empty((D, N), dtype=rdt); rv_pg = np.empty(D, dtype=rdt); ri_pg = np.empty(D, dtype=np.uint64)
    pk3, pk4 = _lib.Peak(), _lib.Peak()
    ms, _ = time_host(surface_call(n_pg, h_pg, f_pg, surf_pg.ctypes.data, rv_pg.ctypes.data, ri_pg.ctypes.data, pk3))
    e2e_pageable = {"value": world * cells_step / (ms * 1e-3), "unit": "cells/s", "ms_per_step": ms,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "peak": [pk3.freq_hz, int(pk3.delay_idx)],
                    "host_buffers": "pageable numpy arrays for inputs AND outputs (std::vector / Vec<Complex64> callers)"}
    checks["e2e_surface_to_host_pageable"] = peak_is_planted(rank, pk3.freq_hz, int(pk3.delay_idx)) and float(surf_pg[int(pk3.doppler_idx), int(pk3.delay_idx)]) == pk3.value
    ms, wall_ms = time_host(peak_call(n_pg, h_pg, f_pg, pk4))
    e2e_peak_pageable = {"value": world * cells_step / (ms * 1e-3), "unit": "cells/s", "ms_per_step": ms,
                         "wall_ms_per_step": wall_ms, "wall_ms_per_step_unflushed_loop": time_host.last_wall_unflushed_ms,
                         "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 32 + 4, "peak": [pk4.freq_hz, int(pk4.delay_idx)],
                         "host_buffers": "pageable numpy inputs (one memcpy into the library's pinned block, which the kernel reads across PCIe itself)"}
    checks["e2e_peak_only_pageable"] = peak_is_planted(rank, pk4.freq_hz, int(pk4.delay_idx))
    # what the reference-facing call sequence costs now: CafSurface::caf_surface + find_peak as the Rust shim / the C++
    # mirror issue it (caf_b200_surface_create + _find_peak + _destroy, pageable Vec inputs): the rows stay on the GPU
    # behind CafSurfaceRow (its fields are private upstream), nothing but find_peak's answer crosses PCIe
    so = C.c_void_p(); pk5 = _lib.Peak()
    create_fn = getattr(lib, f"caf_b200_surface_create_{sfx}")

    def step_dropin():
        rc = create_fn(h.raw, n_pg.ctypes.data, h_pg.ctypes.data, L, f_pg.ctypes.data, D, FS, C.byref(so))
        if rc != 0:
            raise RuntimeError(lib.caf_b200_last_error().decode())
        lib.caf_b200_surface_find_peak(so, C.byref(pk5))
        lib.caf_b200_surface_destroy(so)
    ms, wall_ms = time_host(step_dropin)
    e2e_dropin = {"value": world * cells_step / (ms * 1e-3), "unit": "cells/s", "ms_per_step": ms,
                  "wall_ms_per_step": wall_ms, "wall_ms_per_step_unflushed_loop": time_host.last_wall_unflushed_ms,
                  "timing": "L2 flushed, GPU idle (synchronised) when the call begins, one CUDA event pair around the call; wall clock beside it",
                  "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 32 + 4, "peak": [pk5.freq_hz, int(pk5.delay_idx)],
                  "note": "caf_surface + find_peak as rust/src/caf/mod.rs and include/caf_b200.hpp issue them: device-resident "
                          "surface object with lazy rows (caf_bench.rs:163-167's closure); pageable inputs, one memcpy into the library's pinned "
                          "block, which the kernel reads across PCIe itself; the peak comes back through pinned memory"}
    checks["e2e"] = peak_is_planted(rank, pk5.freq_hz, int(pk5.delay_idx))
    del needle_h, hay_h, freqs_h, raw_blk
    lib.caf_b200_host_free(blk)

    # ---- the other BASELINE configs in the same run: the SHARDED path at every N (cfg3 rows sharded + NCCL peak
    #      exchange, strong scaling; a cfg4 slice, pairs sharded + gather), and at N = 1 compact cfg2 / cfg5-row blocks ----
    ctx = Ctx()
    ctx.lib, ctx.h, ctx.stream, ctx.dev, ctx.rank, ctx.world, ctx.flush = lib, h, stream, dev, rank, world, flush
    ctx.sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    ctx.hbm_peak = hbm_peak
    if f32:
        ctx.tf32 = tf.value
        t64 = C.c_double(); lib.caf_b200_probe_fma_tflops(h.raw, 1, C.byref(t64)); ctx.tf64 = t64.value
    else:
        ctx.tf64 = tf.value
        t32 = C.c_double(); lib.caf_b200_probe_fma_tflops(h.raw, 0, C.byref(t32)); ctx.tf32 = t32.value
    del surf_h, surfs
    sharded, extra = {}, {}

    def run_block(store, key, fn):
        try:
            store[key] = fn(ctx)
        except BaseException as e:          # a block must never take the headline line down with it
            store[key] = {"error": repr(e), "check_ok": False}
        torch.cuda.synchronize()

    if not args.no_blocks:
        run_block(sharded, "cfg3", block_cfg3_sharded)
        run_block(sharded, "cfg4_slice", block_cfg4_slice)
        if world == 1:
            run_block(extra, "cfg2" if not f32 else "cfg1_fp64_skipped", block_cfg2 if not f32 else (lambda c: {"check_ok": True}))
            run_block(extra, "cfg5_rows", block_cfg5_rows)
    for k_, v_ in list(sharded.items()) + list(extra.items()):
        checks[k_] = bool(v_.get("check_ok", False))

    # ---- CPU baseline beside it (rank 0, N = 1 only) ----------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)          # the CPU baseline gets every host core again
        cores = len(all_cpus) or 1
        med, reps = cpu_baseline_run(needle, hay, freqs, args.cpu_budget_s, cores)
        cpu = {"value": cells_step / med, "unit": "cells/s", "ms_per_surface": med * 1e3, "cores": cores, "kind": "port",
               "sample": f"{reps} whole 400x8192 surfaces (median), oracle port of CafRustFFTThreadpool, {cores} threads"}

    if rank == 0:
        line = {
            "metric": "CAF cells/s (400x8192 %s surface + peak)" % ("fp32" if f32 else "fp64"),
            "value": value, "unit": "cells/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": step_ms, "ms_per_surface": step_ms,
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None if f32 else value / PUBLISHED_CELLS_PER_S,
            "vs_baseline_note": "no published complex64 figure" if f32 else PUBLISHED_NOTE,
            "dtype": "f32" if f32 else "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD_CFG2 if f32 else WORKLOAD_CFG1,
                       "doppler_rows": D, "delay_cells": N, "pairs_per_step_per_gpu": 1,
                       "l2": "working set larger than L2: the steps rotate over 320 seeded pairs and 8 surface buffers (252 MB); one CUDA "
                             "event pair around the K back-to-back steps (flushed_per_step = round 1's method, beside it)",
                       "launch_overlap": "caf_b200_set_overlap(4): a step touches no buffer of the seven steps before it, so its launch does "
                                         "not wait for the previous grid and uses a quarter of the SMs -- about four steps share the GPU at any "
                                         "time, each CTA carries 10-11 rows instead of 2-3 (a single surface then takes ~110 us from launch to "
                                         "completion); launches_serialised = the same rotation with overlap off (every launch waits, one CTA per SM)",
                       "pairs_in_rotation": n_pairs, "surface_buffers": n_surf,
                       "parallelism": f"pairs sharded x{world}, no data-path collective",
                       "host_cpus_bound_to_gpu": numa},
            # `e2e`: the reference-facing call sequence of the benchmark (caf_bench.rs:163-167: find_peak(caf_surface(..))) as the
            # Rust shim / C++ mirror issue it, pageable host inputs in, find_peak's answer out.  The same call with the whole
            # 26 MB surface delivered to host memory is `e2e_surface_to_host` (pinned) / `e2e_surface_to_host_pageable`.
            "e2e": e2e_dropin, "e2e_surface_to_host": e2e, "e2e_surface_to_host_pageable": e2e_pageable,
            "e2e_peak_only": e2e_peak, "e2e_peak_only_pageable": e2e_peak_pageable, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "flushed_per_step": {"ms_per_step": flushed_ms, "cells_per_s": world * cells_step / (flushed_ms * 1e-3), "steps": fl_steps,
                                 "method": "L2 flushed (256 MiB overwrite) before every step, one CUDA event pair per step, summed"},
            "launches_serialised": {"ms_per_step": serial_ms, "cells_per_s": world * cells_step / (serial_ms * 1e-3), "steps": args.steps,
                                    "method": "the headline's rotation with caf_b200_set_overlap(0): every launch waits for the one before it"},
            "sharded": sharded, **extra,
            "clocks": sampler.summary(),
            "check": {"peak_freq_hz": peak_freq, "peak_delay": peak_delay, "checks": checks},
            "check_ok": all(checks.values()),
            "flushed_step_ms_min_med_max": [float(per_step.min()), float(np.median(per_step)), float(per_step.max())],
            "pairs_checked": len(ran), "peaks_off": off[:5],
        }
        emit(line)
    ok_t = torch.tensor([1 if all(checks.values()) else 0], dtype=torch.int32, device=dev)
    if world > 1:
        dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
        dist.destroy_process_group()
    if not int(ok_t.item()):
        sys.stderr.write("bench.py: a timed call returned a wrong peak: %r\n" % (checks,))
        raise SystemExit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--workload", choices=["cfg1", "cfg2"], default="cfg1")
    ap.add_argument("--cpu-budget-s", type=float, default=3.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-blocks", action="store_true", help="skip the cfg2/cfg3/cfg4/cfg5 blocks (development)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
