"""Throughput and memory of non-coherent integration (caf_b200_integrate_*_dev) against the compute floor and against the
workaround it replaces, measured in the same run.

    python scripts/bench_integrate.py [--out FILE] [--reps N] [--budgets MB,MB,...] [--no-bench]

Per shape, alternated over --reps rounds (median reported), CUDA events around back-to-back calls after a warm-up:
  - integrate: caf_b200_integrate_*_dev of K segment pairs, surface + row peaks + peak, once per chunk budget
    (CAF_B200_INTEGRATE_MB, read at handle creation: one handle per budget, all on the same stream);
  - floor: caf_b200_batch_*_dev of the same K pairs, peak only (surface NULL): the row compute without any surface traffic;
  - workaround: caf_b200_batch_*_dev writing the whole [K][d][2l] stack, then a sequential torch sum in double.
Shapes: the config-1 grid (400 rows x 8192 cells) in f64 and f32 at K = 16 and 64, and the config-3 row length (4096 rows x
65 536 cells) at K = 4 in f64.  Inputs are seeded noise; every surface is larger than the 126 MB L2 or is rewritten
between reads.  Device memory: torch.cuda.mem_get_info before and after the first integrate call on a fresh handle (the
handle's grow-only workspace) per shape and budget, and the stack the workaround needs.  Times are per segment.
Unless --no-bench, the default bench.py line is run in the same call and its JSON line is included.  Prints one JSON
object (also written to --out) with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_detect import card   # noqa: E402


def make_handle(api, stream, mb):
    old = os.environ.get("CAF_B200_INTEGRATE_MB")
    if mb is None:
        os.environ.pop("CAF_B200_INTEGRATE_MB", None)
    else:
        os.environ["CAF_B200_INTEGRATE_MB"] = str(mb)
    try:
        return api.Handle(0, stream=stream.cuda_stream)
    finally:
        if old is None:
            os.environ.pop("CAF_B200_INTEGRATE_MB", None)
        else:
            os.environ["CAF_B200_INTEGRATE_MB"] = old


def timed(fn, iters, torch):
    s = torch.cuda.current_stream()
    fn()
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(iters):
        fn()
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters        # us per call


def run_shape(torch, api, lib, stream, name, f32, k, l, d, budgets, reps, iters):
    dev = torch.device("cuda", 0)
    n = 2 * l
    rng = np.random.default_rng(k * 1000 + l)
    cdt = np.complex64 if f32 else np.complex128
    tdt = torch.float32 if f32 else torch.float64
    esz = 4 if f32 else 8
    needles = torch.from_numpy(((rng.standard_normal((k, l)) + 1j * rng.standard_normal((k, l))) / np.sqrt(2)).astype(cdt)).to(dev)
    hays = torch.from_numpy(((rng.standard_normal((k, l)) + 1j * rng.standard_normal((k, l))) / np.sqrt(2)).astype(cdt)).to(dev)
    step = 200.0 / d
    freqs = torch.tensor([-100.0 + step * i for i in range(d)], dtype=torch.float64, device=dev)
    S = torch.empty((d, n), dtype=torch.float64, device=dev)
    rv = torch.empty(d, dtype=torch.float64, device=dev)
    ri = torch.empty(d, dtype=torch.int64, device=dev)
    pk = torch.empty(4, dtype=torch.int64, device=dev)
    peaks = torch.empty((k, 4), dtype=torch.int64, device=dev)
    sfx = "f32" if f32 else "f64"
    integ = getattr(lib, "caf_b200_integrate_%s_dev" % sfx)
    batch = getattr(lib, "caf_b200_batch_%s_dev" % sfx)
    seg_bytes = esz * d * n
    res = {"shape": name, "precision": sfx, "k": k, "rows": d, "cells": n, "segment_mb": seg_bytes / 2 ** 20}

    handles, memory = {}, {}
    for mb in budgets:
        free0 = torch.cuda.mem_get_info(dev)[0]
        h = make_handle(api, stream, mb)
        assert integ(h.raw, needles.data_ptr(), hays.data_ptr(), k, l, freqs.data_ptr(), d, 48000, S.data_ptr(),
                     rv.data_ptr(), ri.data_ptr(), pk.data_ptr()) == 0
        torch.cuda.synchronize()
        free1 = torch.cuda.mem_get_info(dev)[0]
        chunk = max(1, min(k, ((mb if mb is not None else 256) << 20) // seg_bytes))
        label = "default" if mb is None else "%dMB" % mb
        handles[label] = (h, chunk)
        memory[label] = {"chunk_segments": chunk, "workspace_mb": (free0 - free1) / 2 ** 20}
    res["memory"] = memory
    res["workaround_stack_mb"] = k * seg_bytes / 2 ** 20
    ref = S.clone()

    methods = {}
    for label, (h, _) in handles.items():
        methods["integrate_" + label] = (lambda h=h: integ(h.raw, needles.data_ptr(), hays.data_ptr(), k, l, freqs.data_ptr(),
                                                           d, 48000, S.data_ptr(), rv.data_ptr(), ri.data_ptr(),
                                                           pk.data_ptr()))
    hb = next(iter(handles.values()))[0]
    methods["floor_peak_only"] = lambda: batch(hb.raw, needles.data_ptr(), hays.data_ptr(), k, l, freqs.data_ptr(), d,
                                               48000, None, None, None, peaks.data_ptr())
    stack = None
    free = torch.cuda.mem_get_info(dev)[0]
    if k * seg_bytes < 0.6 * free:
        stack = torch.empty((k, d, n), dtype=tdt, device=dev)
        acc = torch.empty((d, n), dtype=torch.float64, device=dev)

        def workaround():
            batch(hb.raw, needles.data_ptr(), hays.data_ptr(), k, l, freqs.data_ptr(), d, 48000, stack.data_ptr(), None,
                  None, None)
            acc.zero_()
            for i in range(k):
                acc.add_(stack[i])
        methods["workaround_stack_sum"] = workaround
    times = {m: [] for m in methods}
    for _ in range(reps):
        for m, fn in methods.items():
            times[m].append(timed(fn, iters, torch) / k)
    torch.cuda.synchronize()
    res["us_per_segment"] = {m: statistics.median(v) for m, v in times.items()}
    res["us_per_segment_spread"] = {m: [min(v), max(v)] for m, v in times.items()}
    floor = res["us_per_segment"]["floor_peak_only"]
    res["over_floor"] = {m: v / floor for m, v in res["us_per_segment"].items()}
    if stack is not None:
        res["workaround_equal_bits"] = bool(torch.equal(acc, ref))
    res["repeat_equal_bits"] = bool(torch.equal(S, ref))
    for h, _ in handles.values():
        h.close()
    del stack
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_bench_integrate.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--budgets", default="50,200,800,1600")
    ap.add_argument("--no-bench", action="store_true")
    a = ap.parse_args()
    import torch
    from caf_cookoff_b200 import _lib, api
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    lib = _lib.load()
    stream = torch.cuda.current_stream()
    budgets = [None] + [int(x) for x in a.budgets.split(",") if x]
    out = {"card": card(), "budgets_mb": a.budgets, "shapes": []}
    for f32, k in ((False, 16), (False, 64), (True, 16), (True, 64)):
        out["shapes"].append(run_shape(torch, api, lib, stream, "config-1 grid", f32, k, 4096, 400, budgets, a.reps, 10))
        print(json.dumps(out["shapes"][-1]), file=sys.stderr, flush=True)
    out["shapes"].append(run_shape(torch, api, lib, stream, "config-3 rows", False, 4, 32768, 4096, [None, 8192], 3, 2))
    print(json.dumps(out["shapes"][-1]), file=sys.stderr, flush=True)
    if not a.no_bench:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "200", "--warmup", "20"],
                           capture_output=True, text=True, cwd=ROOT)
        lines = [x for x in r.stdout.splitlines() if x.startswith("{")]
        out["bench_py"] = json.loads(lines[-1]) if lines else {"error": r.stderr[-2000:]}
    out["card_after"] = card()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
