"""Throughput of detection (caf_b200_detect_*_dev, caf_b200_surface_detect) against the HBM floor.

    python scripts/bench_detect.py [--out FILE] [--iters N] [--k K] [--guard-doppler R] [--guard-delay C]

Measures, with CUDA events around many back-to-back launches on the handle's stream:
  - detect_f64_dev / detect_f32_dev over config-1 surfaces (400 x 8192, the bench grid), 8 in f64 and 16 in f32 so that
    either rotation holds 210 MB, more than the 126 MB L2: each launch reads a surface that has left the L2;
  - one config-3-sized surface (4096 x 65 536 f64, 2.1 GB; filled with seeded noise, which has far more local maxima
    than a CAF, so the candidate lists are the longest they get);
and with a host clock, caf_b200_surface_detect end to end (a synchronous call) on a config-1 surface object.
Bytes are the surface bytes each launch must read once; the floor is those bytes at --hbm-tbs (6.5 TB/s measured).
Prints one JSON object (also written to --out) with the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:    # the measurement still stands; say why the card is unnamed
        return {"error": repr(e)}


def time_launches(launch, n_iter, torch):
    s = torch.cuda.current_stream()
    for i in range(8):
        launch(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for i in range(n_iter):
        launch(i)
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n_iter      # us per launch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=400)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--guard-doppler", type=int, default=2)
    ap.add_argument("--guard-delay", type=int, default=2)
    ap.add_argument("--hbm-tbs", type=float, default=6.5)
    a = ap.parse_args()
    import torch
    from caf_cookoff_b200 import _lib, api, bench_shifts
    from oracle import oracle as O
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()
    h = api.Handle(0, stream=stream.cuda_stream)
    lib = _lib.load()
    data = os.path.join(ROOT, "tests", "golden", "data")
    cases = json.load(open(os.path.join(ROOT, "tests", "golden", "known_answers.json")))["cases"]
    L, D = 4096, 400
    shifts = bench_shifts()
    fd = torch.from_numpy(shifts).to(dev)
    K, gr, gd = a.k, a.guard_doppler, a.guard_delay
    res = {"card": card(), "k_max": K, "guard_doppler": gr, "guard_delay": gd, "hbm_tbs_floor": a.hbm_tbs,
           "iters": a.iters}

    def pairs(cdt, count):
        out = []
        for c in (cases * 2)[:count]:
            nd = O.read_file_c64(os.path.join(data, "chirp_%d_raw.c64" % c["chirp"]))
            hy = O.read_file_c64(os.path.join(data, c["haystack"]))[:L]
            out.append((torch.from_numpy(nd.astype(cdt)).to(dev), torch.from_numpy(hy.astype(cdt)).to(dev)))
        return out

    for name, cdt, tdt, f32 in (("f64", np.complex128, torch.float64, False), ("f32", np.complex64, torch.float32, True)):
        ns = 16 if f32 else 8
        surfs = [torch.empty((D, 2 * L), dtype=tdt, device=dev) for _ in range(ns)]
        fn = lib.caf_b200_batch_f32_dev if f32 else lib.caf_b200_batch_f64_dev
        for s_, (nd, hy) in zip(surfs, pairs(cdt, ns)):
            assert fn(h.raw, nd.data_ptr(), hy.data_ptr(), 1, L, fd.data_ptr(), D, 48000, s_.data_ptr(), None, None, None) == 0
        out = torch.empty((ns, K, 6), dtype=torch.float64, device=dev)
        cnt = torch.empty(ns, dtype=torch.int64, device=dev)

        def launch(i):
            j = i % ns
            api.detect_dev(surfs[j].data_ptr(), 1, D, 2 * L, fd.data_ptr(), K, out[j].data_ptr(), cnt[j].data_ptr(),
                           guard_doppler=gr, guard_delay=gd, f32=f32, handle=h)
        us = time_launches(launch, a.iters, torch)
        nbytes = surfs[0].numel() * surfs[0].element_size()
        floor = nbytes / (a.hbm_tbs * 1e12) * 1e6
        res["cfg1_dev_" + name] = {"us_per_surface": round(us, 3), "surfaces_rotated": ns, "bytes": nbytes, "tb_per_s": round(nbytes / us / 1e6, 3),
                                   "hbm_floor_us": round(floor, 3), "share_of_floor": round(floor / us, 3),
                                   "counts": [int(x) for x in cnt.cpu()]}
        del surfs

    # config-3-sized surface: 4096 x 65536 f64
    g = torch.Generator(device=dev).manual_seed(3)
    big = torch.rand((4096, 65536), dtype=torch.float64, device=dev, generator=g)
    f3 = torch.linspace(-100.0, 100.0, 4096, dtype=torch.float64, device=dev)
    out = torch.empty((1, K, 6), dtype=torch.float64, device=dev)
    cnt = torch.empty(1, dtype=torch.int64, device=dev)

    def launch3(i):
        api.detect_dev(big.data_ptr(), 1, 4096, 65536, f3.data_ptr(), K, out.data_ptr(), cnt.data_ptr(),
                       guard_doppler=gr, guard_delay=gd, handle=h)
    us = time_launches(launch3, max(20, a.iters // 10), torch)
    nbytes = big.numel() * 8
    floor = nbytes / (a.hbm_tbs * 1e12) * 1e6
    res["cfg3_dev_f64"] = {"us_per_surface": round(us, 3), "bytes": nbytes, "tb_per_s": round(nbytes / us / 1e6, 3),
                           "hbm_floor_us": round(floor, 3), "share_of_floor": round(floor / us, 3), "count": int(cnt[0])}
    del big

    # host call on a surface object (config 1, chirp_0)
    nd = O.read_file_c64(os.path.join(data, "chirp_0_raw.c64"))
    hy = O.read_file_c64(os.path.join(data, cases[0]["haystack"]))[:L]
    s = api.DeviceSurface(nd, hy, shifts, 48000, handle=h)
    for _ in range(10):
        s.detect(K, gr, gd)
    n_host = max(50, a.iters // 4)
    t0 = time.perf_counter()
    for _ in range(n_host):
        dets = s.detect(K, gr, gd)
    res["cfg1_surface_detect_host_us"] = round((time.perf_counter() - t0) / n_host * 1e6, 2)
    res["cfg1_detection0"] = {"lag_samples": dets[0].lag_samples, "freq_hz_interp": dets[0].freq_hz_interp,
                              "delay_idx": int(dets[0].delay_idx), "freq_hz": dets[0].freq_hz}
    s.close()
    h.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
