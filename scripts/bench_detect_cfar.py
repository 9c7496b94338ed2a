"""Throughput of CFAR detection (caf_b200_detect_cfar_*_dev, caf_b200_surface_detect_cfar) and the noise map
(caf_b200_cfar_noise_*_dev), beside detect measured in the same run, against the HBM floor.

    python scripts/bench_detect_cfar.py [--out FILE] [--iters N] [--k K] [--guard-doppler R] [--guard-delay C]
                                        [--train-doppler A] [--train-delay B] [--pfa P]

Defaults: k_max 16, guard 2 x 2, training 4 x 16, scale = cfar_scale(1e-6, N).  With CUDA events around many
back-to-back launches on the handle's stream:
  - detect and detect_cfar over config-1 surfaces (400 x 8192, the bench grid), 8 rotated in f64 and 16 in f32 so that
    either rotation holds 210 MB, more than the 126 MB L2;
  - both on one config-3-sized f64 surface of seeded noise (4096 x 65 536, 2.1 GB: far more local maxima than a CAF);
  - the dense noise map of config-1 f64 surfaces (reads the surface, writes 8 bytes per cell);
and with a host clock, caf_b200_surface_detect and caf_b200_surface_detect_cfar end to end on a config-1 surface object.
Each time stands beside the HBM floor of its bytes at --hbm-tbs (6.5 TB/s measured).  Prints one JSON object (also
written to --out) with the card's name and power limit read in the same run.
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_bench_cfar.json"))
    ap.add_argument("--iters", type=int, default=400)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--guard-doppler", type=int, default=2)
    ap.add_argument("--guard-delay", type=int, default=2)
    ap.add_argument("--train-doppler", type=int, default=4)
    ap.add_argument("--train-delay", type=int, default=16)
    ap.add_argument("--pfa", type=float, default=1e-6)
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
    K, gr, gd, tr, tc = a.k, a.guard_doppler, a.guard_delay, a.train_doppler, a.train_delay
    N = api.cfar_train_cells(gr, gd, tr, tc)
    scale = api.cfar_scale(a.pfa, N)
    res = {"card": card(), "k_max": K, "guard_doppler": gr, "guard_delay": gd, "train_doppler": tr, "train_delay": tc,
           "train_cells": N, "pfa": a.pfa, "scale": scale, "hbm_tbs_floor": a.hbm_tbs, "iters": a.iters}

    def pairs(cdt, count):
        out = []
        for c in (cases * 2)[:count]:
            nd = O.read_file_c64(os.path.join(data, "chirp_%d_raw.c64" % c["chirp"]))
            hy = O.read_file_c64(os.path.join(data, c["haystack"]))[:L]
            out.append((torch.from_numpy(nd.astype(cdt)).to(dev), torch.from_numpy(hy.astype(cdt)).to(dev)))
        return out

    def entry(us, nbytes, **extra):
        floor = nbytes / (a.hbm_tbs * 1e12) * 1e6
        return dict({"us_per_surface": round(us, 3), "bytes": nbytes, "tb_per_s": round(nbytes / us / 1e6, 3),
                     "hbm_floor_us": round(floor, 3), "share_of_floor": round(floor / us, 3)}, **extra)

    for name, cdt, tdt, f32 in (("f64", np.complex128, torch.float64, False), ("f32", np.complex64, torch.float32, True)):
        ns = 16 if f32 else 8
        surfs = [torch.empty((D, 2 * L), dtype=tdt, device=dev) for _ in range(ns)]
        fn = lib.caf_b200_batch_f32_dev if f32 else lib.caf_b200_batch_f64_dev
        for s_, (nd, hy) in zip(surfs, pairs(cdt, ns)):
            assert fn(h.raw, nd.data_ptr(), hy.data_ptr(), 1, L, fd.data_ptr(), D, 48000, s_.data_ptr(), None, None, None) == 0
        nbytes = surfs[0].numel() * surfs[0].element_size()
        out = torch.empty((ns, K, 6), dtype=torch.float64, device=dev)
        outc = torch.empty((ns, K, 8), dtype=torch.float64, device=dev)
        cnt = torch.empty(ns, dtype=torch.int64, device=dev)
        cntc = torch.empty(ns, dtype=torch.int64, device=dev)

        def det(i):
            j = i % ns
            api.detect_dev(surfs[j].data_ptr(), 1, D, 2 * L, fd.data_ptr(), K, out[j].data_ptr(), cnt[j].data_ptr(),
                           guard_doppler=gr, guard_delay=gd, f32=f32, handle=h)

        def cfar(i):
            j = i % ns
            api.detect_cfar_dev(surfs[j].data_ptr(), 1, D, 2 * L, fd.data_ptr(), K, outc[j].data_ptr(), cntc[j].data_ptr(),
                                scale=scale, guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc, f32=f32,
                                handle=h)
        us_d = time_launches(det, a.iters, torch)
        us_c = time_launches(cfar, a.iters, torch)
        res["cfg1_detect_" + name] = entry(us_d, nbytes, surfaces_rotated=ns, counts=[int(x) for x in cnt.cpu()])
        res["cfg1_detect_cfar_" + name] = entry(us_c, nbytes, surfaces_rotated=ns, counts=[int(x) for x in cntc.cpu()],
                                                ratio_to_detect=round(us_c / us_d, 3))
        if not f32:
            noise = torch.empty((D, 2 * L), dtype=torch.float64, device=dev)

            def nmap(i):
                api.cfar_noise_dev(surfs[i % ns].data_ptr(), 1, D, 2 * L, noise.data_ptr(), guard_doppler=gr,
                                   guard_delay=gd, train_doppler=tr, train_delay=tc, handle=h)
            us_m = time_launches(nmap, max(40, a.iters // 10), torch)
            res["cfg1_noise_map_f64"] = entry(us_m, nbytes + noise.numel() * 8)
            del noise
        del surfs

    # config-3-sized surface of noise: 4096 x 65536 f64
    g = torch.Generator(device=dev).manual_seed(3)
    big = torch.rand((4096, 65536), dtype=torch.float64, device=dev, generator=g)
    f3 = torch.linspace(-100.0, 100.0, 4096, dtype=torch.float64, device=dev)
    out = torch.empty((1, K, 6), dtype=torch.float64, device=dev)
    outc = torch.empty((1, K, 8), dtype=torch.float64, device=dev)
    cnt = torch.empty(1, dtype=torch.int64, device=dev)
    cntc = torch.empty(1, dtype=torch.int64, device=dev)

    def det3(i):
        api.detect_dev(big.data_ptr(), 1, 4096, 65536, f3.data_ptr(), K, out.data_ptr(), cnt.data_ptr(),
                       guard_doppler=gr, guard_delay=gd, handle=h)

    def cfar3(i):
        api.detect_cfar_dev(big.data_ptr(), 1, 4096, 65536, f3.data_ptr(), K, outc.data_ptr(), cntc.data_ptr(),
                            scale=scale, guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc, handle=h)
    n3 = max(20, a.iters // 10)
    us_d = time_launches(det3, n3, torch)
    us_c = time_launches(cfar3, n3, torch)
    nbytes = big.numel() * 8
    res["cfg3_detect_f64"] = entry(us_d, nbytes, count=int(cnt[0]))
    res["cfg3_detect_cfar_f64"] = entry(us_c, nbytes, count=int(cntc[0]), ratio_to_detect=round(us_c / us_d, 3))
    del big

    # host calls on a surface object (config 1, chirp_0)
    nd = O.read_file_c64(os.path.join(data, "chirp_0_raw.c64"))
    hy = O.read_file_c64(os.path.join(data, cases[0]["haystack"]))[:L]
    s = api.DeviceSurface(nd, hy, shifts, 48000, handle=h)
    n_host = max(50, a.iters // 4)
    for label, call in (("cfg1_surface_detect_host_us", lambda: s.detect(K, gr, gd)),
                        ("cfg1_surface_detect_cfar_host_us", lambda: s.detect_cfar(K, gr, gd, tr, tc, scale))):
        for _ in range(10):
            call()
        t0 = time.perf_counter()
        for _ in range(n_host):
            dets = call()
        res[label] = round((time.perf_counter() - t0) / n_host * 1e6, 2)
    res["cfg1_cfar_detections"] = [{"delay_idx": int(x.delay_idx), "freq_hz": x.freq_hz, "snr_db": round(10 * np.log10(x.value / x.noise), 2),
                                    "train_cells": int(x.train_cells)} for x in dets]
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
