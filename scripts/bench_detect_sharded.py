"""Detection on row-sharded config-3 surfaces (caf_b200_detect_*rows_*_dev, the merges and the exchange; DESIGN.md
section 12).

    python scripts/bench_detect_sharded.py [--out FILE] [--iters N] [--k K]
    python -m torch.distributed.run --nproc-per-node G scripts/bench_detect_sharded.py --dist [--out FILE]

One GPU (default): a config-3-sized f64 surface of seeded uniform noise (4096 x 65 536, 2.1 GB, the surface of
scripts/bench_detect_cfar.py) and the block rank 3 of 8 would hold (rows 1536 ... 2047 plus the halo: 2 rows for
detect, 6 for the CFAR detectors at guard 2 x 2, training 4 x 16, k_max 16).  CUDA events around back-to-back launches on
the handle's stream time each detector on the whole surface and on the block, in the same run, and the merge kernels
over the eight ranks' lists.  Each sharded answer is also checked against the whole-surface one.  Then, with a host clock
around work that ends in a synchronise, one rank's compute step (the halo'd block's rows by caf_b200_batch_f64_dev, then
block detection) beside the whole surface and whole detection (config 3: l = 32 768, d = 4096, seeded inputs).

--dist (one process per GPU under torchrun): the step "halo'd sharded surface + block detection + exchange" over the
library's communicator (Comm.detect_sharded's work, timed from issue to the exchange's return), the maximum over
ranks.  Prints one JSON object (also written to --out) with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_detect import card, time_launches   # noqa: E402

L3, D3 = 32768, 4096       # config 3
GR, GD, TR, TC = 2, 2, 4, 16


def inputs(torch, dev):
    rng = np.random.default_rng(3)
    needle = np.hanning(L3) * (rng.standard_normal(L3) + 1j * rng.standard_normal(L3))
    hay = np.concatenate([np.zeros(500), needle])[:L3] * np.exp(2j * np.pi * 21.0 * np.arange(L3) / 48000)
    hay = hay + 0.1 * (rng.standard_normal(L3) + 1j * rng.standard_normal(L3))
    freqs = np.linspace(-200.0, 200.0, D3)
    return (torch.from_numpy(needle).to(dev), torch.from_numpy(hay).to(dev), torch.from_numpy(freqs).to(dev))


def windows(api):
    N = api.cfar_train_cells(GR, GD, TR, TC)
    rank = (3 * N + 3) // 4
    return {"detect": {}, "cfar": {"scale": api.cfar_scale(1e-6, N)},
            "cfar_os": {"rank": rank, "scale": api.cfar_os_scale(1e-6, N, rank)}}


def one_gpu(a, res):
    import torch
    from caf_cookoff_b200 import _lib, api
    from caf_cookoff_b200.dist import shard_bounds
    dev = torch.device("cuda", 0)
    h = api.Handle(0, stream=torch.cuda.current_stream().cuda_stream)
    K, world, me = a.k, 8, 3
    win = windows(api)
    g = torch.Generator(device=dev).manual_seed(3)
    big = torch.rand((D3, 2 * L3), dtype=torch.float64, device=dev, generator=g)
    f3 = torch.linspace(-100.0, 100.0, D3, dtype=torch.float64, device=dev)
    n = 2 * L3

    def call(det, surf_ptr, d, f_ptr, out, cnt, rows=None):
        kw = dict(guard_doppler=GR, guard_delay=GD, handle=h)
        if det != "detect":
            kw.update(train_doppler=TR, train_delay=TC, **win[det])
        if rows is None:
            fn = {"detect": api.detect_dev, "cfar": api.detect_cfar_dev, "cfar_os": api.detect_cfar_os_dev}[det]
            fn(surf_ptr, 1, d, n, f_ptr, K, out.data_ptr(), cnt.data_ptr(), **kw)
        else:
            fn = {"detect": api.detect_rows_dev, "cfar": api.detect_cfar_rows_dev,
                  "cfar_os": api.detect_cfar_os_rows_dev}[det]
            fn(surf_ptr, d, n, f_ptr, *rows, D3, K, out.data_ptr(), cnt.data_ptr(), **kw)

    def block(det, r):
        lo, hi = shard_bounds(D3, world, r)
        H = api.halo_rows(det, GR, 0 if det == "detect" else TR)
        b_lo, b_hi = max(lo - H, 0), min(hi + H, D3)
        return (big[b_lo].data_ptr(), b_hi - b_lo, f3[b_lo:].data_ptr(), (lo - b_lo, hi - b_lo, b_lo))

    for det in ("detect", "cfar", "cfar_os"):
        w = 6 if det == "detect" else 8
        out = torch.empty((K, w), dtype=torch.float64, device=dev)
        cnt = torch.empty(1, dtype=torch.int64, device=dev)
        lists = torch.empty((world, K, w), dtype=torch.float64, device=dev)
        counts = torch.empty(world, dtype=torch.int64, device=dev)
        merged = torch.empty((K, w), dtype=torch.float64, device=dev)
        mcnt = torch.empty(1, dtype=torch.int64, device=dev)
        n_it = max(10, a.iters // 10)
        us_whole = time_launches(lambda i: call(det, big.data_ptr(), D3, f3.data_ptr(), out, cnt), n_it, torch)
        p, d_buf, fp, rows = block(det, me)
        us_block = time_launches(lambda i: call(det, p, d_buf, fp, lists[me], counts[me:me + 1], rows), a.iters, torch)
        for r in range(world):
            p, d_buf, fp, rows = block(det, r)
            call(det, p, d_buf, fp, lists[r], counts[r:r + 1], rows)

        def mrg(i):
            if det == "detect":
                api.detect_merge_dev(lists.data_ptr(), counts.data_ptr(), world, K, merged.data_ptr(), mcnt.data_ptr(),
                                     handle=h)
            else:
                api.cfar_merge_dev(lists.data_ptr(), counts.data_ptr(), world, K, merged.data_ptr(), mcnt.data_ptr(),
                                   handle=h)
        us_merge = time_launches(mrg, a.iters, torch)
        call(det, big.data_ptr(), D3, f3.data_ptr(), out, cnt)
        torch.cuda.synchronize()
        same = torch.equal(out.view(torch.int64), merged.view(torch.int64)) and int(cnt[0]) == int(mcnt[0])   # bits
        assert same, det + ": the world-8 merge differs from the whole-surface call"
        res["cfg3_f64_" + det] = {"whole_us": round(us_whole, 2), "block_rank3_of_8_us": round(us_block, 2),
                                  "block_rows": d_buf, "ratio_block_to_whole": round(us_block / us_whole, 4),
                                  "merge_world8_us": round(us_merge, 2), "count": int(cnt[0]),
                                  "merged_equals_whole": same}
    del big

    # one rank's compute step beside the whole surface, host clock around work that ends in a synchronise
    nd, hd, fd = inputs(torch, dev)
    lib = _lib.load()
    whole_s = torch.empty((D3, n), dtype=torch.float64, device=dev)
    lo, hi = shard_bounds(D3, world, me)

    def step(det, rows_lo, rows_hi, surf):
        H = api.halo_rows(det, GR, 0 if det == "detect" else TR)
        b_lo, b_hi = max(rows_lo - H, 0), min(rows_hi + H, D3)
        assert lib.caf_b200_batch_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 1, L3, fd[b_lo:].data_ptr(), b_hi - b_lo,
                                          48000, surf.data_ptr(), None, None, None) == 0
        out = torch.empty((K, 8), dtype=torch.float64, device=dev)
        cnt = torch.empty(1, dtype=torch.int64, device=dev)
        if (rows_lo, rows_hi) == (0, D3):
            call(det, surf.data_ptr(), D3, fd.data_ptr(), out, cnt)
        else:
            call(det, surf.data_ptr(), b_hi - b_lo, fd[b_lo:].data_ptr(), out, cnt, (rows_lo - b_lo, rows_hi - b_lo, b_lo))

    def host_ms(fn, reps):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps * 1e3

    for det in ("detect", "cfar", "cfar_os"):
        ms_whole = host_ms(lambda: step(det, 0, D3, whole_s), 5)
        ms_rank = host_ms(lambda: step(det, lo, hi, whole_s), 20)
        res["cfg3_step_" + det] = {"whole_surface_and_detection_ms": round(ms_whole, 3),
                                   "rank3_of_8_block_surface_and_detection_ms": round(ms_rank, 3),
                                   "ratio": round(ms_rank / ms_whole, 4)}
    h.close()


def distributed(a, res):
    import torch
    import torch.distributed as tdist
    from caf_cookoff_b200 import api
    from caf_cookoff_b200.dist import Comm
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    tdist.init_process_group("nccl", device_id=dev)
    h = api.Handle(local)
    id_path = os.path.join(tempfile.gettempdir(), "caf_bench_sharded_%s_%s" % (
        os.environ.get("MASTER_PORT", "0"), os.environ.get("TORCHELASTIC_RUN_ID", "x")))
    comm = Comm(h, world, rank, id_path)
    nd, hd, fd = inputs(torch, dev)
    win = windows(api)
    res["world"] = world
    for det in ("detect", "cfar", "cfar_os"):
        kw = dict(guard_doppler=GR, guard_delay=GD)
        if det != "detect":
            kw.update(train_doppler=TR, train_delay=TC, **win[det])
        times = []
        for i in range(a.reps + 2):
            tdist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            comm.detect_sharded(det, nd, hd, fd, 48000, a.k, **kw)
            times.append(time.perf_counter() - t0)
        ms = torch.tensor([sorted(times[2:])[len(times[2:]) // 2] * 1e3], dtype=torch.float64, device=dev)
        tdist.all_reduce(ms, op=tdist.ReduceOp.MAX)
        res["cfg3_sharded_step_" + det] = {"median_ms_max_over_ranks": round(float(ms[0]), 3), "reps": a.reps}
    comm.close()
    h.close()
    tdist.destroy_process_group()
    return rank


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_bench_detect_sharded.json"))
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--dist", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    res = {"card": card(), "k_max": a.k, "guard_doppler": GR, "guard_delay": GD, "train_doppler": TR, "train_delay": TC}
    rank = 0
    if a.dist:
        rank = distributed(a, res)
    else:
        one_gpu(a, res)
    if rank == 0:
        line = json.dumps(res)
        print(line)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
