"""Throughput of OS-CFAR detection (caf_b200_detect_cfar_os_*_dev, caf_b200_surface_detect_cfar_os) beside CA-CFAR and
detect, measured in the same run on the same surfaces, and of the OS noise map.

    python scripts/bench_detect_cfar_os.py [--out FILE] [--iters N] [--k K] [--guard-doppler R] [--guard-delay C]
                                           [--train-doppler A] [--train-delay B] [--rank K] [--pfa P]

Defaults: k_max 16, guard 2 x 2, training 4 x 16 (N = 456), rank ceil(3N / 4) = 342, Pfa 1e-6 (CA's scale from
cfar_scale, OS's from cfar_os_scale).  The surfaces and the method are scripts/bench_detect_cfar.py's: CUDA events
around many back-to-back launches on the handle's stream, over
  - config-1 surfaces (400 x 8192, the bench grid), 8 rotated in f64 and 16 in f32 (either rotation holds 210 MB, more
    than the 126 MB L2);
  - one config-3-sized f64 surface of seeded noise (4096 x 65 536, 2.1 GB);
and a host clock around caf_b200_surface_detect / _cfar / _cfar_os end to end on a config-1 surface object.
OS's two steps are split by a second OS run at a scale no candidate passes (1e300): it counts every candidate and
selects for none, so it is the counting step alone; the rest of OS's time is the selection of the qualifying ones.
The OS dense map is timed on config-1 f64 surfaces.  Prints one JSON object (also written to --out) with the card's name
and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bench_detect import card, time_launches   # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bench_cfar_os.json"))
    ap.add_argument("--iters", type=int, default=400)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--guard-doppler", type=int, default=2)
    ap.add_argument("--guard-delay", type=int, default=2)
    ap.add_argument("--train-doppler", type=int, default=4)
    ap.add_argument("--train-delay", type=int, default=16)
    ap.add_argument("--rank", type=int, default=None)
    ap.add_argument("--pfa", type=float, default=1e-6)
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
    K, gr, gd, tr, tc = a.k, a.guard_doppler, a.guard_delay, a.train_doppler, a.train_delay
    N = api.cfar_train_cells(gr, gd, tr, tc)
    rank = a.rank or (3 * N + 3) // 4
    scale_ca = api.cfar_scale(a.pfa, N)
    scale_os = api.cfar_os_scale(a.pfa, N, rank)
    res = {"card": card(), "k_max": K, "guard_doppler": gr, "guard_delay": gd, "train_doppler": tr, "train_delay": tc,
           "train_cells": N, "rank": rank, "pfa": a.pfa, "scale_ca": scale_ca, "scale_os": scale_os, "iters": a.iters}

    def pairs(cdt, count):
        out = []
        for c in (cases * 2)[:count]:
            nd = O.read_file_c64(os.path.join(data, "chirp_%d_raw.c64" % c["chirp"]))
            hy = O.read_file_c64(os.path.join(data, c["haystack"]))[:L]
            out.append((torch.from_numpy(nd.astype(cdt)).to(dev), torch.from_numpy(hy.astype(cdt)).to(dev)))
        return out

    def three(surf_of, d, n, f, ns, f32, n_iter, tag):
        """detect, CA, OS and OS counting only on the same surfaces, in one run"""
        out = torch.empty((ns, K, 6), dtype=torch.float64, device=dev)
        outc = torch.empty((ns, K, 8), dtype=torch.float64, device=dev)
        cnt = torch.empty(ns, dtype=torch.int64, device=dev)
        cntc = torch.empty(ns, dtype=torch.int64, device=dev)
        cnto = torch.empty(ns, dtype=torch.int64, device=dev)

        def det(i):
            j = i % ns
            api.detect_dev(surf_of(j), 1, d, n, f.data_ptr(), K, out[j].data_ptr(), cnt[j].data_ptr(),
                           guard_doppler=gr, guard_delay=gd, f32=f32, handle=h)

        def ca(i):
            j = i % ns
            api.detect_cfar_dev(surf_of(j), 1, d, n, f.data_ptr(), K, outc[j].data_ptr(), cntc[j].data_ptr(),
                                scale=scale_ca, guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc,
                                f32=f32, handle=h)

        def os_(scale, counts):
            def launch(i):
                j = i % ns
                api.detect_cfar_os_dev(surf_of(j), 1, d, n, f.data_ptr(), K, outc[j].data_ptr(), counts[j].data_ptr(),
                                       rank=rank, scale=scale, guard_doppler=gr, guard_delay=gd, train_doppler=tr,
                                       train_delay=tc, f32=f32, handle=h)
            return launch
        us_d = time_launches(det, n_iter, torch)
        us_c = time_launches(ca, n_iter, torch)
        us_o = time_launches(os_(scale_os, cnto), n_iter, torch)
        us_n = time_launches(os_(1e300, cntc), n_iter, torch)
        assert int(cntc.sum()) == 0
        res[tag + "_detect"] = {"us_per_surface": round(us_d, 3)}
        res[tag + "_detect_cfar"] = {"us_per_surface": round(us_c, 3), "ratio_to_detect": round(us_c / us_d, 3)}
        res[tag + "_detect_cfar_os"] = {"us_per_surface": round(us_o, 3), "ratio_to_ca": round(us_o / us_c, 3),
                                        "ratio_to_detect": round(us_o / us_d, 3), "counts": [int(x) for x in cnto.cpu()]}
        res[tag + "_detect_cfar_os_count_only"] = {"us_per_surface": round(us_n, 3), "ratio_to_ca": round(us_n / us_c, 3)}

    for name, cdt, tdt, f32 in (("f64", np.complex128, torch.float64, False), ("f32", np.complex64, torch.float32, True)):
        ns = 16 if f32 else 8
        surfs = [torch.empty((D, 2 * L), dtype=tdt, device=dev) for _ in range(ns)]
        fn = lib.caf_b200_batch_f32_dev if f32 else lib.caf_b200_batch_f64_dev
        for s_, (nd, hy) in zip(surfs, pairs(cdt, ns)):
            assert fn(h.raw, nd.data_ptr(), hy.data_ptr(), 1, L, fd.data_ptr(), D, 48000, s_.data_ptr(), None, None, None) == 0
        three(lambda j: surfs[j].data_ptr(), D, 2 * L, fd, ns, f32, a.iters, "cfg1_" + name)
        if not f32:
            noise = torch.empty((D, 2 * L), dtype=torch.float64, device=dev)

            def nmap(i):
                api.cfar_os_noise_dev(surfs[i % ns].data_ptr(), 1, D, 2 * L, noise.data_ptr(), rank=rank,
                                      guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc, handle=h)
            res["cfg1_os_noise_map_f64"] = {"us_per_surface": round(time_launches(nmap, 20, torch), 3)}
            del noise
        del surfs

    # config-3-sized surface of noise: 4096 x 65536 f64
    g = torch.Generator(device=dev).manual_seed(3)
    big = torch.rand((4096, 65536), dtype=torch.float64, device=dev, generator=g)
    f3 = torch.linspace(-100.0, 100.0, 4096, dtype=torch.float64, device=dev)
    three(lambda j: big.data_ptr(), 4096, 65536, f3, 1, False, max(20, a.iters // 10), "cfg3_f64")
    del big

    # host calls on a surface object (config 1, chirp_0)
    nd = O.read_file_c64(os.path.join(data, "chirp_0_raw.c64"))
    hy = O.read_file_c64(os.path.join(data, cases[0]["haystack"]))[:L]
    s = api.DeviceSurface(nd, hy, shifts, 48000, handle=h)
    n_host = max(50, a.iters // 4)
    for label, call in (("cfg1_surface_detect_host_us", lambda: s.detect(K, gr, gd)),
                        ("cfg1_surface_detect_cfar_host_us", lambda: s.detect_cfar(K, gr, gd, tr, tc, scale_ca)),
                        ("cfg1_surface_detect_cfar_os_host_us", lambda: s.detect_cfar_os(K, gr, gd, tr, tc, rank, scale_os))):
        for _ in range(10):
            call()
        t0 = time.perf_counter()
        for _ in range(n_host):
            call()
        res[label] = round((time.perf_counter() - t0) / n_host * 1e6, 2)
    s.close()
    h.close()
    res["goal_os_le_2x_ca_cfg1_f64"] = res["cfg1_f64_detect_cfar_os"]["ratio_to_ca"] <= 2.0
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
