"""Non-coherent integration of CAF surfaces over K segments on the GPU (caf_b200_integrate_*_dev,
caf_b200_surface_create_integrated_*, DeviceSurface.integrate), include/caf_b200.h and DESIGN.md section 13: the sum is the
batch path's surfaces added in double in ascending k, bit for bit, and a weak emitter that one segment's CFAR misses
clears the threshold of the sum."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from caf_cookoff_b200 import _lib, api, bench_shifts
from conftest import DATA, FS, ROOT, rel_max

pytestmark = pytest.mark.gpu

CFAR_REC = np.dtype([("value", "f8"), ("freq_hz", "f8"), ("doppler_idx", "u8"), ("delay_idx", "u8"),
                     ("lag_samples", "f8"), ("freq_hz_interp", "f8"), ("noise", "f8"), ("train_cells", "u8")])
DET_REC = np.dtype([("value", "f8"), ("freq_hz", "f8"), ("doppler_idx", "u8"), ("delay_idx", "u8"),
                    ("lag_samples", "f8"), ("freq_hz_interp", "f8")])
VARIANTS = [api._Variant, api._Variant32]
VIDS = ["f64", "f32"]


def cuda():
    import torch
    return torch, torch.device("cuda", 0)


def to_dev(x):
    torch, dev = cuda()
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def handle_with_budget(mb):
    """a handle whose integration chunks hold at most `mb` MB of segment surfaces (read at creation)"""
    old = os.environ.get("CAF_B200_INTEGRATE_MB")
    os.environ["CAF_B200_INTEGRATE_MB"] = str(mb)
    try:
        return api.Handle(0)
    finally:
        if old is None:
            del os.environ["CAF_B200_INTEGRATE_MB"]
        else:
            os.environ["CAF_B200_INTEGRATE_MB"] = old


def pairs(k, l, seed, variant=api._Variant, lag=None, freq=None, amp=0.3):
    """k random segment pairs [k, l] of the variant's dtype, each haystack holding its needle delayed and shifted"""
    rng = np.random.default_rng(seed)
    needles = (rng.standard_normal((k, l)) + 1j * rng.standard_normal((k, l))) / np.sqrt(2)
    hays = (rng.standard_normal((k, l)) + 1j * rng.standard_normal((k, l))) / np.sqrt(2)
    lag = l // 7 if lag is None else lag
    freq = 21.5 if freq is None else freq
    x = np.concatenate([np.zeros((k, lag)), needles[:, :l - lag]], axis=1)
    hays = hays + amp * x * np.exp(2j * np.pi * freq * np.arange(l) / FS)
    return needles.astype(variant.cdt), hays.astype(variant.cdt)


def batch_stack(needles, hays, freqs, variant):
    """[k][d][2l] surfaces of caf_b200_batch_*_dev, in the variant's precision"""
    torch, dev = cuda()
    k, l = needles.shape
    d = len(freqs)
    nd, hd, fd = to_dev(needles), to_dev(hays), to_dev(np.asarray(freqs, dtype=np.float64))
    out = torch.empty((k, d, 2 * l), dtype=torch.float64 if variant is api._Variant else torch.float32, device=dev)
    fn = getattr(_lib.load(), "caf_b200_batch_%s_dev" % variant.sfx)
    assert fn(api.default_handle().raw, nd.data_ptr(), hd.data_ptr(), k, l, fd.data_ptr(), d, FS, out.data_ptr(),
              None, None, None) == 0
    torch.cuda.synchronize()
    return out.cpu().numpy()


def sequential_sum(stack):
    """the contract's order: +0.0, then s_0, s_1, ... added one at a time in double (not np.sum, which is pairwise)"""
    acc = np.zeros(stack.shape[1:], dtype=np.float64)
    for s in stack:
        acc += s.astype(np.float64)
    return acc


def row_peaks(S):
    """mod.rs:141-153: the first cell holding each row's maximum (0 for an all-zero row)"""
    idx = np.argmax(S, axis=1) if S.shape[1] else np.zeros(S.shape[0], dtype=np.int64)
    return S[np.arange(S.shape[0]), idx], idx.astype(np.uint64)


def find_peak(freqs, pval, pidx):
    """mod.rs:31-42 with the library's dummy row: (value, freq, doppler_idx, delay_idx)"""
    best = (0.0, 0.0, (1 << 64) - 1, 0)
    for r, v in enumerate(pval):
        if v > best[0]:
            best = (float(v), float(freqs[r]), r, int(pidx[r]))
    return best


def integrate(needles, hays, freqs, variant, handle=None, rows=True, peak=True):
    """caf_b200_integrate_*_dev -> (S [d][2l] float64, row_peak_val, row_peak_idx, peak tuple)"""
    torch, dev = cuda()
    k, l = needles.shape
    d = len(freqs)
    nd, hd, fd = to_dev(needles), to_dev(hays), to_dev(np.asarray(freqs, dtype=np.float64))
    S = torch.full((d, 2 * l), -7.0, dtype=torch.float64, device=dev)     # the first chunk must not read it
    rv = torch.full((max(d, 1),), -1.0, dtype=torch.float64, device=dev)
    ri = torch.full((max(d, 1),), -1, dtype=torch.int64, device=dev)
    pk = torch.zeros(4, dtype=torch.int64, device=dev)
    api.integrate_dev(nd.data_ptr(), hd.data_ptr(), k, l, fd.data_ptr(), d, FS, S.data_ptr(),
                      rv.data_ptr() if rows else 0, ri.data_ptr() if rows else 0, pk.data_ptr() if peak else 0,
                      f32=variant is api._Variant32, handle=handle)
    torch.cuda.synchronize()
    p = pk.cpu().numpy()
    ptuple = (float(p[0:1].view(np.float64)[0]), float(p[1:2].view(np.float64)[0]), int(p[2:3].view(np.uint64)[0]),
              int(p[3:4].view(np.uint64)[0]))
    return S.cpu().numpy(), rv.cpu().numpy()[:d], ri.cpu().numpy().view(np.uint64)[:d], ptuple


def same_bits(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape
    assert np.array_equal(a.view(np.uint64), b.view(np.uint64))


def same_peak(got, want):
    assert np.float64(got[0]).view(np.uint64) == np.float64(want[0]).view(np.uint64)
    assert got[1:] == want[1:]


# ---- 1. bit identity with the batch path -----------------------------------------------------------------------------
CASES = [   # (l, rows, k, chunk budget in MB or None for the default)
    (4096, 64, 11, 8),       # 4 MB f64 / 2 MB f32 segments: chunks of 2 (f64) / 4 (f32), the last one partial
    (4096, 64, 11, None),    # the same sum in one chunk
    (1000, 37, 5, None),     # a length that is not a power of two: two blocks per 2000-cell row
    (300, 9, 4, 1),          # one block per row; a 1 MB budget still takes two segments (f32: all four)
    (32768, 3, 3, None),     # long rows (the four-step path): 64 blocks per row
]


@pytest.mark.parametrize("variant", VARIANTS, ids=VIDS)
@pytest.mark.parametrize("l,d,k,mb", CASES)
def test_sum_of_batch_surfaces_bit_for_bit(variant, l, d, k, mb):
    freqs = bench_shifts()[150:150 + d]
    needles, hays = pairs(k, l, seed=l + d + k, variant=variant, freq=freqs[d // 2])
    want = sequential_sum(batch_stack(needles, hays, freqs, variant))
    wv, wi = row_peaks(want)
    h = handle_with_budget(mb) if mb else None
    S, rv, ri, pk = integrate(needles, hays, freqs, variant, handle=h)
    same_bits(S, want)
    same_bits(rv, wv)
    assert np.array_equal(ri, wi)
    same_peak(pk, find_peak(freqs, wv, wi))
    assert pk[0] > 0.0 and pk[3] == l // 7
    # row peaks without the peak, the peak without row peaks, and neither: the surface is the same
    for rows, peak in ((True, False), (False, True), (False, False)):
        S2, rv2, ri2, pk2 = integrate(needles, hays, freqs, variant, handle=h, rows=rows, peak=peak)
        same_bits(S2, want)
        if rows:
            same_bits(rv2, wv)
        if peak:
            same_peak(pk2, find_peak(freqs, wv, wi))
    if h is not None:
        h.close()


@pytest.mark.parametrize("variant", VARIANTS, ids=VIDS)
def test_one_segment_is_the_widened_surface(variant):
    torch, dev = cuda()
    freqs = bench_shifts()
    needles, hays = pairs(1, 4096, seed=5, variant=variant)
    nd, hd, fd = to_dev(needles), to_dev(hays), to_dev(freqs)
    T = torch.float64 if variant is api._Variant else torch.float32
    s1 = torch.empty((400, 8192), dtype=T, device=dev)
    rv1 = torch.empty(400, dtype=T, device=dev)
    ri1 = torch.empty(400, dtype=torch.int64, device=dev)
    pk1 = torch.zeros(4, dtype=torch.int64, device=dev)
    fn = getattr(_lib.load(), "caf_b200_batch_%s_dev" % variant.sfx)
    assert fn(api.default_handle().raw, nd.data_ptr(), hd.data_ptr(), 1, 4096, fd.data_ptr(), 400, FS, s1.data_ptr(),
              rv1.data_ptr(), ri1.data_ptr(), pk1.data_ptr()) == 0
    torch.cuda.synchronize()
    S, rv, ri, pk = integrate(needles, hays, freqs, variant)
    same_bits(S, s1.cpu().numpy().astype(np.float64))
    same_bits(rv, rv1.cpu().numpy().astype(np.float64))
    assert np.array_equal(ri, ri1.cpu().numpy().view(np.uint64))
    p1 = pk1.cpu().numpy()
    assert pk == (float(p1[0:1].view(np.float64)[0]), float(p1[1:2].view(np.float64)[0]), int(p1[2:3].view(np.uint64)[0]),
                  int(p1[3:4].view(np.uint64)[0]))


def test_empty_shapes_behave_as_the_batch_calls():
    torch, dev = cuda()
    freqs = bench_shifts()[:5]
    # l == 0: rows of peak 0.0 at cell 0, find_peak's dummy row
    S, rv, ri, pk = integrate(np.zeros((3, 0), np.complex128), np.zeros((3, 0), np.complex128), freqs, api._Variant)
    assert S.shape == (5, 0) and np.all(rv == 0.0) and np.all(ri == 0)
    assert pk == (0.0, 0.0, (1 << 64) - 1, 0)
    # d == 0
    needles, hays = pairs(2, 64, seed=3)
    S, rv, ri, pk = integrate(needles, hays, np.zeros(0), api._Variant)
    assert S.shape == (0, 128) and pk == (0.0, 0.0, (1 << 64) - 1, 0)
    s = api.DeviceSurface.integrate(np.zeros((2, 0)), np.zeros((2, 0)), freqs, FS)
    assert s.shape == (5, 0) and s.find_peak().doppler_idx == (1 << 64) - 1
    s.close()


# ---- 2. against the oracle -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant,tol", [(api._Variant, 1e-9), (api._Variant32, 1e-4)], ids=VIDS)
def test_golden_chirp_segments_against_the_oracle(variant, tol):
    from oracle import oracle as O
    needle = O.read_file_c64(os.path.join(DATA, "chirp_0_raw.c64"))
    hay = O.read_file_c64(os.path.join(DATA, "chirp_0_T+202samp_F+69.25Hz.c64"))[: needle.size]
    k = 4
    l = needle.size // k
    freqs = O.gen_float_shifts(40.0, 100.0, 0.5)
    want = np.zeros((freqs.size, 2 * l))
    for i in range(k):
        surf, _, _ = O.caf_surface(needle[i * l:(i + 1) * l], hay[i * l:(i + 1) * l], freqs, FS)
        want += surf
    S, rv, ri, pk = integrate(needle[:k * l].reshape(k, l).astype(variant.cdt), hay[:k * l].reshape(k, l).astype(variant.cdt),
                              freqs, variant)
    assert rel_max(S, want) <= tol
    assert pk[3] == 202 and abs(pk[1] - 69.25) <= 5.0         # Doppler is flat over a 1024-sample segment, delay is not


# ---- 3. sub-grids and the row-sharded detectors ----------------------------------------------------------------------
def test_sub_grids_and_sharded_cfar_on_the_sum():
    """The integrated surface of grid rows [a, b) is rows [a, b) of the whole sum; detect_cfar_rows_dev on integrated
    blocks with their halo, merged over 2 and 3 ranks on one GPU, equals detect_cfar_dev on the whole sum byte for byte."""
    torch, dev = cuda()
    freqs = bench_shifts()
    d, l, k = freqs.size, 4096, 4
    needles, hays = pairs(k, l, seed=77, amp=0.05)
    S, _, _, _ = integrate(needles, hays, freqs, api._Variant)
    for a, b in ((0, 400), (37, 161), (399, 400), (0, 1), (200, 233)):
        Sab, _, _, _ = integrate(needles, hays, freqs[a:b], api._Variant)
        same_bits(Sab, S[a:b])
    gr, gd, tr, tc, k_max = 2, 2, 4, 16, 32
    scale = 2.5
    H = api.halo_rows("cfar", gr, tr)
    Sd, fd = to_dev(S), to_dev(freqs)
    out = torch.zeros((k_max, 8), dtype=torch.float64, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    api.detect_cfar_dev(Sd.data_ptr(), 1, d, 2 * l, fd.data_ptr(), k_max, out.data_ptr(), cnt.data_ptr(), scale=scale,
                        guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc)
    torch.cuda.synchronize()
    want, want_cnt = out.cpu().numpy().tobytes(), int(cnt.item())
    assert want_cnt >= 2
    nd, hd = to_dev(needles), to_dev(hays)
    keep = []                # the blocks live on the library's stream until the merge has run
    for world in (2, 3):
        lists = torch.zeros((world, k_max, 8), dtype=torch.float64, device=dev)
        counts = torch.zeros(world, dtype=torch.int64, device=dev)
        for rank in range(world):
            lo, hi = d * rank // world, d * (rank + 1) // world
            off, end = max(lo - H, 0), min(hi + H, d)
            blk = torch.full((end - off, 2 * l), -7.0, dtype=torch.float64, device=dev)
            fb = to_dev(freqs[off:end])
            keep.append((blk, fb))
            api.integrate_dev(nd.data_ptr(), hd.data_ptr(), k, l, fb.data_ptr(), end - off, FS, blk.data_ptr())
            api.detect_cfar_rows_dev(blk.data_ptr(), end - off, 2 * l, fb.data_ptr(), lo - off, hi - off, off, d, k_max,
                                     lists[rank].data_ptr(), counts[rank:rank + 1].data_ptr(), scale=scale,
                                     guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc)
        mo = torch.zeros((k_max, 8), dtype=torch.float64, device=dev)
        mc = torch.zeros(1, dtype=torch.int64, device=dev)
        api.cfar_merge_dev(lists.data_ptr(), counts.data_ptr(), world, k_max, mo.data_ptr(), mc.data_ptr())
        torch.cuda.synchronize()
        assert int(mc.item()) == want_cnt
        assert mo.cpu().numpy().tobytes() == want


# ---- 4. the reason for the feature -----------------------------------------------------------------------------------
SCENE_L, SCENE_LAG, SCENE_FREQ, SCENE_K = 4096, 202, 69.0, 64
SCENE_AMP = 0.03
PG = (32, 2, 0, 64)          # guard_doppler, guard_delay, train_doppler, train_delay (test_gpu_cfar's planted scene)


def scene(k=SCENE_K, amp=SCENE_AMP, emitter=True, seed=1):
    """k segments of one weak emitter: a clean (Hann-windowed complex Gaussian) needle per segment and a haystack holding it
    at lag 202, +69 Hz, amplitude amp, under unit-power complex noise drawn independently per segment."""
    rng = np.random.default_rng(seed)
    n = np.arange(SCENE_L)
    needles = np.hanning(SCENE_L) * (rng.standard_normal((k, SCENE_L)) + 1j * rng.standard_normal((k, SCENE_L))) / np.sqrt(2)
    hays = (rng.standard_normal((k, SCENE_L)) + 1j * rng.standard_normal((k, SCENE_L))) / np.sqrt(2)
    if emitter:
        x = np.concatenate([np.zeros((k, SCENE_LAG)), needles[:, :SCENE_L - SCENE_LAG]], axis=1)
        hays = hays + amp * x * np.exp(2j * np.pi * SCENE_FREQ * n / FS)
    return needles, hays


def snr_margins(S, scale, shifts, skip=None):
    """(the best value over noise at the emitter's delay within 2.5 Hz of its Doppler, the best local maximum's elsewhere),
    both in dB above scale; skip = a detected (row, cell) left out of the second"""
    from oracle import cfar as F
    from oracle.detect import local_maxima
    gr, gd, tr, tc = PG
    noise, _ = F.noise_map(S, gr, gd, tr, tc)
    near = np.flatnonzero(np.abs(shifts - SCENE_FREQ) <= 2.5)
    em = 10 * np.log10(np.max(S[near, SCENE_LAG] / noise[near, SCENE_LAG]) / scale)
    lm = local_maxima(S, gr, gd)
    if skip is not None:
        lm[skip] = False
    with np.errstate(invalid="ignore"):
        other = np.nanmax(np.where(lm, S / noise, np.nan))
    return em, 10 * np.log10(other / scale)


@pytest.mark.parametrize("variant", VARIANTS, ids=VIDS)
def test_integration_finds_the_emitter_one_segment_misses(variant):
    """One weak emitter, post-correlation SNR about 5 dB per segment (amplitude chosen with a numpy restatement first).  At Pfa 1e-6 (N = 8320 training cells) one
    segment's CFAR does not report it: its best cell is SCENE_MISS_DB or more under that threshold.  The sum of 64 segments
    with cfar_scale(1e-6, N, looks=64) reports it at its delay, within 2.5 Hz of its Doppler, and nothing else: it clears
    the threshold by SCENE_HIT_DB or more and every other local maximum stays SCENE_REST_DB or more under it.  The 64
    segments without the emitter give an empty list, their best local maximum SCENE_NOISE_DB or more under the threshold.
    The inputs are seeded, so the margins are fixed (the measured values are beside the constants); f32 rounding moves
    them by ~1e-6 dB.  The seed matters: on 3 of 8 seeds tried, the noise alone put one local maximum 0.06 to 0.14 dB
    over the Gamma(64) threshold somewhere on the 400 x 8192 surface -- the model's Pfa is that of the threshold test on
    independent cells, and a CAF's cells are neither independent nor of one noise power across the delay axis."""
    gr, gd, tr, tc = PG
    N = api.cfar_train_cells(gr, gd, tr, tc)
    shifts = bench_shifts()
    needles, hays = scene()
    one = api.DeviceSurface(needles[0], hays[0], shifts, FS, variant=variant)
    assert one.detect_cfar(8, gr, gd, tr, tc) == []
    em1, _ = snr_margins(one.fetch_rows().astype(np.float64), api.cfar_scale(1e-6, N), shifts)
    one.close()
    s = api.DeviceSurface.integrate(needles.astype(variant.cdt), hays.astype(variant.cdt), shifts, FS, variant=variant)
    assert s.looks == SCENE_K
    scale = api.cfar_scale(1e-6, N, looks=SCENE_K)
    dets = s.detect_cfar(8, gr, gd, tr, tc)
    S = s.fetch_rows()
    em, rest = snr_margins(S, scale, shifts, skip=(int(dets[0].doppler_idx), int(dets[0].delay_idx)) if dets else None)
    print("integration scene %s: one segment %.2f dB, sum %.2f dB, rest %.2f dB" % (variant.sfx, em1, em, rest))
    assert len(dets) == 1, [(x.doppler_idx, x.delay_idx, x.value / x.noise / scale) for x in dets]
    x = dets[0]
    assert int(x.delay_idx) == SCENE_LAG and abs(x.freq_hz - SCENE_FREQ) <= 2.5 and abs(x.freq_hz_interp - SCENE_FREQ) <= 2.5
    assert record_bytes(s.detect_cfar(8, gr, gd, tr, tc, scale)) == record_bytes(dets)       # the default is looks=64
    assert em1 <= -SCENE_MISS_DB and em >= SCENE_HIT_DB and rest <= -SCENE_REST_DB, (em1, em, rest)
    s.close()
    needles, hays = scene(emitter=False)
    s = api.DeviceSurface.integrate(needles.astype(variant.cdt), hays.astype(variant.cdt), shifts, FS, variant=variant)
    assert s.detect_cfar(8, gr, gd, tr, tc) == []
    _, rest0 = snr_margins(s.fetch_rows(), scale, shifts)
    print("integration scene %s: noise only, best local maximum %.2f dB" % (variant.sfx, rest0))
    assert rest0 <= -SCENE_NOISE_DB, rest0
    s.close()


# margins measured on a B200 (f64 and f32 alike): one segment -2.18 dB, the sum +1.83 dB, the rest -0.19 dB, noise only
# -0.19 dB.  Segment 0's noise happens to add to the emitter's cell: a typical segment sits ~6 dB under.
SCENE_MISS_DB = 1.0
SCENE_HIT_DB = 1.0
SCENE_REST_DB = 0.01
SCENE_NOISE_DB = 0.01


# ---- 5. the surface object -------------------------------------------------------------------------------------------
def record_bytes(recs):
    return b"".join(bytes(r) for r in recs)


@pytest.mark.parametrize("variant", VARIANTS, ids=VIDS)
def test_surface_object_matches_the_dev_path(variant):
    torch, dev = cuda()
    lib = _lib.load()
    freqs = bench_shifts()
    k, l = 6, 4096
    needles, hays = pairs(k, l, seed=31, variant=variant, amp=0.08)
    S, rv, ri, pk = integrate(needles, hays, freqs, variant)
    s = api.DeviceSurface.integrate(needles, hays, freqs, FS, variant=variant)
    assert s.looks == k and s.shape == (400, 2 * l)
    p = s.find_peak()
    assert (p.value, p.freq_hz, p.doppler_idx, p.delay_idx) == pk
    fr, pv, pi = np.zeros(400), np.zeros(400), np.zeros(400, dtype=np.uint64)
    assert lib.caf_b200_surface_row_peaks(s.raw, api._ptr(fr), api._ptr(pv), api._ptr(pi)) == 0
    same_bits(fr, freqs)
    same_bits(pv, rv)
    assert np.array_equal(pi, ri)
    rows = s.fetch_rows()
    assert rows.dtype == np.float64
    same_bits(rows, S)
    same_bits(s.fetch_rows(17, 5), S[17:22])
    Sd, fd = to_dev(S), to_dev(freqs)
    gr, gd, tr, tc = 2, 2, 4, 16
    N = api.cfar_train_cells(gr, gd, tr, tc)
    # detect
    out = torch.zeros((16, 6), dtype=torch.float64, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    api.detect_dev(Sd.data_ptr(), 1, 400, 2 * l, fd.data_ptr(), 16, out.data_ptr(), cnt.data_ptr(), guard_doppler=gr,
                   guard_delay=gd)
    torch.cuda.synchronize()
    got = s.detect(16, gr, gd)
    assert len(got) == int(cnt.item()) and record_bytes(got) == out.cpu().numpy()[:len(got)].tobytes()
    # CA-CFAR: the default scale is the Gamma(k) one
    scale = api.cfar_scale(1e-6, N, looks=k)
    out = torch.zeros((16, 8), dtype=torch.float64, device=dev)
    api.detect_cfar_dev(Sd.data_ptr(), 1, 400, 2 * l, fd.data_ptr(), 16, out.data_ptr(), cnt.data_ptr(), scale=scale,
                        guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc)
    torch.cuda.synchronize()
    got = s.detect_cfar(16, gr, gd, tr, tc)
    assert len(got) == int(cnt.item()) >= 1
    assert record_bytes(got) == out.cpu().numpy()[:len(got)].tobytes()
    assert record_bytes(s.detect_cfar(16, gr, gd, tr, tc, scale)) == record_bytes(got)
    # OS-CFAR: no looks model, so an explicit scale is required
    with pytest.raises(ValueError):
        s.detect_cfar_os(16, gr, gd, tr, tc)
    rank = (3 * N + 3) // 4
    api.detect_cfar_os_dev(Sd.data_ptr(), 1, 400, 2 * l, fd.data_ptr(), 16, out.data_ptr(), cnt.data_ptr(), rank=rank,
                           scale=3.0, guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc)
    torch.cuda.synchronize()
    got = s.detect_cfar_os(16, gr, gd, tr, tc, rank=rank, scale=3.0)
    assert len(got) == int(cnt.item()) >= 1
    assert record_bytes(got) == out.cpu().numpy()[:len(got)].tobytes()
    s.close()
    one = api.DeviceSurface(needles[0], hays[0], freqs, FS, variant=variant)
    assert one.looks == 1 and one.fetch_rows(0, 1).dtype == variant.rdt
    one.close()


# ---- 6. errors -------------------------------------------------------------------------------------------------------
def test_error_codes_write_nothing():
    torch, dev = cuda()
    lib = _lib.load()
    h = api.default_handle()
    freqs = bench_shifts()[:16]
    needles, hays = pairs(3, 256, seed=9)
    nd, hd, fd = to_dev(needles), to_dev(hays), to_dev(freqs)
    S = torch.full((16, 512), 3.25, dtype=torch.float64, device=dev)
    rv = torch.full((16,), 3.25, dtype=torch.float64, device=dev)
    ri = torch.full((16,), 12345, dtype=torch.int64, device=dev)
    pk = torch.full((4,), 777, dtype=torch.int64, device=dev)
    f64 = lib.caf_b200_integrate_f64_dev

    def call(fn=f64, k=3, l=256, n=nd.data_ptr(), y=hd.data_ptr(), f=fd.data_ptr(), d=16, fs=FS, s=S.data_ptr(), hh=None):
        return fn(h.raw if hh is None else hh, n, y, k, l, f, d, fs, s, rv.data_ptr(), ri.data_ptr(), pk.data_ptr())

    assert call(k=0) == -1
    assert call(n=None) == -1
    assert call(y=None) == -1
    assert call(f=None) == -1
    assert call(s=None) == -1
    assert call(fs=0) == -1
    assert call(hh=C.c_void_p(0)) == -1
    assert call(l=(1 << 19) + 1, k=1) == -3
    assert call(fn=lib.caf_b200_integrate_f32_dev, k=0) == -1
    assert call(fn=lib.caf_b200_integrate_f32_dev, l=(1 << 19) + 1, k=1) == -3
    torch.cuda.synchronize()
    assert torch.all(S == 3.25) and torch.all(rv == 3.25) and torch.all(ri == 12345) and torch.all(pk == 777)
    out = C.c_void_p(12345)
    n64, h64 = needles.copy(), hays.copy()
    assert lib.caf_b200_surface_create_integrated_f64(h.raw, api._ptr(n64), api._ptr(h64), 0, 256, api._ptr(freqs), 16,
                                                      FS, C.byref(out)) == -1
    assert not out.value
    assert lib.caf_b200_surface_create_integrated_f64(h.raw, api._ptr(n64), api._ptr(h64), 3, 256, api._ptr(freqs), 16,
                                                      0, C.byref(out)) == -1
    assert lib.caf_b200_surface_create_integrated_f64(h.raw, api._ptr(n64), api._ptr(h64), 1, (1 << 19) + 1,
                                                      api._ptr(freqs), 16, FS, C.byref(out)) == -3
    with pytest.raises(api.CafError):
        api.DeviceSurface.integrate(needles[:0], hays[:0], freqs, FS)


# ---- 7. order and repeatability --------------------------------------------------------------------------------------
def test_integrate_between_overlapped_surface_launches():
    """Overlap mode 4 with rotated outputs: integrate calls (chunked, so each internal batch launch rewrites the scratch the
    previous sum read) placed between single-pair surface launches leave every surface, peak and sum bit-identical to the
    serialised run."""
    torch, dev = cuda()
    stream = torch.cuda.Stream(device=dev)
    lib = _lib.load()
    old = os.environ.get("CAF_B200_INTEGRATE_MB")
    os.environ["CAF_B200_INTEGRATE_MB"] = "26"      # one 400 x 8192 f64 segment per chunk
    try:
        h = api.Handle(0, stream=stream.cuda_stream)
    finally:
        if old is None:
            del os.environ["CAF_B200_INTEGRATE_MB"]
        else:
            os.environ["CAF_B200_INTEGRATE_MB"] = old
    L = 4096
    freqs = bench_shifts()
    needles, hays = pairs(3, L, seed=41, amp=0.2)
    nd, hd, fd = to_dev(needles), to_dev(hays), to_dev(freqs)
    K, NB = 12, 9

    def run(overlap, with_integrate):
        lib.caf_b200_set_overlap(h.raw, overlap)
        surfs = [torch.zeros((400, 2 * L), dtype=torch.float64, device=dev) for _ in range(NB)]
        pk = torch.zeros((K, 4), dtype=torch.int64, device=dev)
        sums = [torch.zeros((400, 2 * L), dtype=torch.float64, device=dev) for _ in range(4)]
        ipk = torch.zeros((4, 4), dtype=torch.int64, device=dev)
        with torch.cuda.stream(stream):
            for i in range(K):
                j = i % 3
                assert lib.caf_b200_batch_f64_dev(h.raw, nd[j].data_ptr(), hd[j].data_ptr(), 1, L, fd.data_ptr(), 400, FS,
                                                  surfs[i % NB].data_ptr(), None, None, pk[i].data_ptr()) == 0
                if with_integrate and i % 3 == 1:
                    q = i // 3
                    assert lib.caf_b200_integrate_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 3, L, fd.data_ptr(), 400, FS,
                                                          sums[q].data_ptr(), None, None, ipk[q].data_ptr()) == 0
        torch.cuda.synchronize()
        return [x.cpu().numpy() for x in surfs], pk.cpu().numpy(), [x.cpu().numpy() for x in sums], ipk.cpu().numpy()

    want = run(0, False)
    got = run(4, True)
    for a, b in zip(want[0], got[0]):
        same_bits(a, b)
    assert np.array_equal(want[1], got[1])
    ref = sequential_sum(batch_stack(needles, hays, freqs, api._Variant))
    for q in range(4):
        same_bits(got[2][q], ref)
        assert np.array_equal(got[3][q], got[3][0])
    lib.caf_b200_set_overlap(h.raw, 0)
    h.close()


def test_repeated_calls_and_a_second_handle_give_the_same_bits():
    freqs = bench_shifts()
    for variant in VARIANTS:
        needles, hays = pairs(5, 4096, seed=13, variant=variant)
        first = integrate(needles, hays, freqs, variant)
        h2 = api.Handle(0)
        for hh in (None, h2, None, h2):
            again = integrate(needles, hays, freqs, variant, handle=hh)
            same_bits(again[0], first[0])
            same_bits(again[1], first[1])
            assert np.array_equal(again[2], first[2]) and again[3] == first[3]
        h2.close()


# ---- 8. CLI and C++ --------------------------------------------------------------------------------------------------
def _cli(tmp_path):
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "caf_cli")
    subprocess.check_call([shutil.which("g++"), "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tools", "caf_cli.cpp"), "-o", exe, "-L", so_dir, "-lcaf_b200",
                           f"-Wl,-rpath,{so_dir}"])
    return exe


def test_cli_segments(tmp_path):
    """--segments 1 prints what the program prints without it; --segments K --detect / --cfar-db print the report and the
    detections of DeviceSurface.integrate over the same K windows."""
    from oracle import oracle as O
    exe = _cli(tmp_path)
    a = os.path.join(DATA, "chirp_0_raw.c64")
    b = os.path.join(DATA, "chirp_0_T+202samp_F+69.25Hz.c64")
    for extra in ([], ["--detect", "4"], ["--detect", "4", "--cfar-db", "12"]):
        plain = subprocess.run([exe, a, b] + extra, capture_output=True, timeout=120)
        seg1 = subprocess.run([exe, a, b, "--segments", "1"] + extra, capture_output=True, timeout=120)
        assert plain.returncode == 0 and seg1.returncode == 0
        assert seg1.stdout == plain.stdout and seg1.stderr == plain.stderr
    k = 8
    needles, hays = scene(k=k, amp=0.06)
    na, ha = str(tmp_path / "needle.c64"), str(tmp_path / "hay.c64")
    for path, x in ((na, needles.ravel()), (ha, np.concatenate([hays.ravel(), hays[0, :100]]))):   # a tail to drop
        np.stack([x.real, x.imag], axis=1).astype("<f4").tofile(path)
    n32 = O.read_file_c64(na).reshape(k, SCENE_L)
    h32 = O.read_file_c64(ha)[:k * SCENE_L].reshape(k, SCENE_L)
    shifts = O.gen_float_shifts(-100.0, 100.0, 0.5)
    s = api.DeviceSurface.integrate(n32, h32, shifts, FS)
    pk = s.find_peak()
    head = "Frequency offset: %.1fHz\nTime offset: %d samples (%.3fms)\n" % (pk.freq_hz, pk.delay_idx,
                                                                              pk.delay_idx / (FS / 1e3))
    res = subprocess.run([exe, na, ha, "--segments", str(k)], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    assert res.stdout == head
    res = subprocess.run([exe, na, ha, "--segments", str(k), "--detect", "5"], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    dets = s.detect(5, 1, 1)
    want = head + "".join("Detection %d: %.4fHz (grid %.2fHz), %.3f samples (cell %d), %.2f dB below the first\n" % (
        i, x.freq_hz_interp, x.freq_hz, x.lag_samples, x.delay_idx, 10 * np.log10(dets[0].value / x.value))
        for i, x in enumerate(dets))
    assert res.stdout == want
    assert len(dets) == 5 and dets[0].delay_idx == SCENE_LAG
    db = 6.0
    res = subprocess.run([exe, na, ha, "--segments", str(k), "--detect", "8", "--guard-doppler", "32", "--guard-delay", "2",
                          "--train-doppler", "0", "--train-delay", "64", "--cfar-db", "%.1f" % db], capture_output=True,
                         text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    cd = s.detect_cfar(8, 32, 2, 0, 64, 10 ** (db / 10))
    assert len(cd) >= 1 and cd[0].delay_idx == SCENE_LAG
    want = head + "".join("Detection %d: %.4fHz (grid %.2fHz), %.3f samples (cell %d), %.2f dB below the first, %.2f dB "
                          "above the noise\n" % (i, x.freq_hz_interp, x.freq_hz, x.lag_samples, x.delay_idx,
                                                 10 * np.log10(cd[0].value / x.value), 10 * np.log10(x.value / x.noise))
                          for i, x in enumerate(cd))
    assert res.stdout == want
    s.close()
    bad = subprocess.run([exe, na, ha, "--segments", "2", "--layout", "go"], capture_output=True, text=True, timeout=120)
    assert bad.returncode == 2


def test_cpp_integrate_refuses_other_threads(tmp_path):
    """The C++ factory's surface belongs to the creating thread's handle, as caf_surface's does."""
    src = tmp_path / "owner.cpp"
    src.write_text(r'''
#include <cmath>
#include <cstdio>
#include <thread>
#include "caf_b200.hpp"
int main() {
    const std::size_t k = 3, l = 256;
    std::vector<caf::Complex64> x(k * l), y(k * l);
    for (std::size_t i = 0; i < k * l; ++i) x[i] = {std::sin(0.37 * i * i), std::cos(1.3 * i + 0.011 * i * i)};
    for (std::size_t s = 0; s < k; ++s)
        for (std::size_t i = 0; i < l; ++i) y[s * l + i] = x[s * l + (i + l - 6) % l];      // each segment delayed by 6
    const auto rows = caf::CafB200::integrate(x, y, k, {-1.0, 0.0, 1.0}, 48000);
    const auto [f, idx] = caf::CafB200::find_peak(rows);
    const auto here = caf::CafB200::detect_cfar(rows, 3, 1, 1, 0, 16, 10.0);
    bool refused = false;
    std::thread t([&] { try { caf::CafB200::detect_cfar(rows, 3, 1, 1, 0, 16, 10.0); } catch (const caf::Panic&) { refused = true; } });
    t.join();
    std::printf("%zu %d %zu %g %zu\n", here.size(), refused ? 1 : 0, idx, f, rows[1].xcor_mag().size());
    return 0;
}
''')
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "owner")
    subprocess.check_call([shutil.which("g++"), "-std=c++17", "-O2", "-pthread", "-I", os.path.join(ROOT, "include"), str(src),
                           "-o", exe, "-L", so_dir, "-lcaf_b200", f"-Wl,-rpath,{so_dir}"])
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    n, refused, idx, f, cells = res.stdout.split()
    assert int(n) >= 1 and refused == "1" and int(idx) == 6 and float(f) == 0.0 and int(cells) == 512
