"""CA-CFAR detection and the noise map on the GPU (caf_b200_surface_detect_cfar, caf_b200_detect_cfar_*_dev,
caf_b200_cfar_noise_*_dev) against oracle/cfar.py, bit for bit (include/caf_b200.h, DESIGN.md section 10)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from caf_cookoff_b200 import _lib, api, bench_shifts
from conftest import FS
from oracle import cfar as F

pytestmark = pytest.mark.gpu

REC = np.dtype([("value", "f8"), ("freq_hz", "f8"), ("doppler_idx", "u8"), ("delay_idx", "u8"),
                ("lag_samples", "f8"), ("freq_hz_interp", "f8"), ("noise", "f8"), ("train_cells", "u8")])


def bits(x):
    return np.float64(x).view(np.uint64)


def key(rec):
    """a record with every double as its bit pattern: equal keys are equal bits"""
    return tuple(int(bits(x)) if isinstance(x, float) else int(x) for x in rec)


def as_tuples(recs):
    return [(float(x["value"]), float(x["freq_hz"]), int(x["doppler_idx"]), int(x["delay_idx"]), float(x["lag_samples"]),
             float(x["freq_hz_interp"]), float(x["noise"]), int(x["train_cells"])) for x in recs]


def of_structs(dets):
    return [(x.value, x.freq_hz, x.doppler_idx, x.delay_idx, x.lag_samples, x.freq_hz_interp, x.noise, x.train_cells)
            for x in dets]


def same(got, want):
    assert [key(x) for x in got] == [key(x) for x in want]


def run_dev(S, freqs, k_max, gr, gd, tr, tc, scale, handle=None):
    """S [p][d][n] numpy (float64 or float32) -> (records [p][k_max] as tuples, counts [p]) through detect_cfar_*_dev"""
    import torch
    dev = torch.device("cuda", 0)
    p, d, n = S.shape
    ts = torch.from_numpy(np.ascontiguousarray(S)).to(dev)
    tf = torch.from_numpy(np.ascontiguousarray(freqs, dtype=np.float64)).to(dev)
    out = torch.zeros((p, k_max, 8), dtype=torch.float64, device=dev)
    cnt = torch.full((p,), -1, dtype=torch.int64, device=dev)
    api.detect_cfar_dev(ts.data_ptr(), p, d, n, tf.data_ptr(), k_max, out.data_ptr(), cnt.data_ptr(), scale=scale,
                        guard_doppler=gr, guard_delay=gd, train_doppler=tr, train_delay=tc, f32=S.dtype == np.float32,
                        handle=handle)
    torch.cuda.synchronize()
    recs = out.cpu().numpy().view(REC).reshape(p, k_max)
    return [as_tuples(recs[i]) for i in range(p)], [int(c) for c in cnt.cpu().numpy()]


def run_map(S, gr, gd, tr, tc, handle=None):
    import torch
    dev = torch.device("cuda", 0)
    p, d, n = S.shape
    ts = torch.from_numpy(np.ascontiguousarray(S)).to(dev)
    out = torch.zeros((p, d, n), dtype=torch.float64, device=dev)
    api.cfar_noise_dev(ts.data_ptr(), p, d, n, out.data_ptr(), guard_doppler=gr, guard_delay=gd, train_doppler=tr,
                       train_delay=tc, f32=S.dtype == np.float32, handle=handle)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def map_equal(got, want):
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got[~nan].view(np.uint64), want[~nan].view(np.uint64))


def check_against_reference(S, freqs, k_max, gr, gd, tr, tc, scale):
    got, cnt = run_dev(S, freqs, k_max, gr, gd, tr, tc, scale)
    noise = run_map(S, gr, gd, tr, tc)
    for i in range(S.shape[0]):
        want = F.detect_cfar(S[i], freqs, k_max, gr, gd, tr, tc, scale)
        assert cnt[i] == len(want)
        same(got[i], F.padded(want, k_max))
        for x in got[i][:cnt[i]]:
            assert bits(x[6]) == bits(noise[i, x[2], x[3]])          # a record's noise is the map's cell
    return got, cnt


MAP_CASES = [  # (p, d, n, gr, gd, tr, tc)
    (3, 9, 300, 1, 1, 2, 16), (1, 40, 600, 2, 3, 30, 253), (2, 37, 520, 0, 0, 32, 256), (1, 5, 9, 0, 1, 1, 3),
    (2, 70, 1000, 2, 2, 4, 16), (1, 1, 64, 0, 2, 0, 5),
]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("case", MAP_CASES)
def test_dense_map_matches_reference_bit_for_bit(case, dtype):
    p, d, n, gr, gd, tr, tc = case
    rng = np.random.default_rng(hash(case) % 1000)
    S = (rng.random((p, d, n)) ** 3 * 1e3).astype(dtype)
    S[rng.random(S.shape) < 0.03] = np.nan
    got = run_map(S, gr, gd, tr, tc)
    for i in range(p):
        map_equal(got[i], F.noise_map(S[i], gr, gd, tr, tc)[0])


SHAPES = [  # (p, d, n, gr, gd, tr, tc, k_max)
    (3, 1, 300, 0, 0, 0, 5, 7), (3, 2, 517, 1, 1, 1, 4, 16), (2, 37, 1000, 2, 3, 4, 16, 64), (1, 37, 600, 2, 3, 30, 253, 3),
    (1, 37, 1000, 0, 0, 0, 1, 1024), (4, 2, 9, 1, 1, 0, 3, 3), (1, 40, 520, 5, 40, 10, 20, 1024), (2, 20, 257, 32, 1, 0, 2, 1),
    (1, 70, 700, 0, 0, 32, 256, 5), (2, 33, 800, 2, 2, 30, 36, 40),
]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("shape", SHAPES)
def test_tie_heavy_surfaces_match_reference(shape, dtype):
    p, d, n, gr, gd, tr, tc, k_max = shape
    rng = np.random.default_rng(hash(shape) % 1000)
    S = rng.integers(0, 5, size=(p, d, n)).astype(dtype)
    S[rng.random(S.shape) < 0.02] = np.nan
    freqs = np.cumsum(rng.random(d) + 0.05) - 3.0
    for scale in (0.9, 1.6):
        got, _ = check_against_reference(S, freqs, k_max, gr, gd, tr, tc, scale)
        one = [run_dev(S[i:i + 1], freqs, k_max, gr, gd, tr, tc, scale)[0][0] for i in range(p)]
        assert [[key(x) for x in g] for g in got] == [[key(x) for x in o] for o in one]   # a batch equals its pairs


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_many_candidates_repeatable_and_handle_independent(dtype):
    """Noise with a low scale: many qualifying maxima per tile, the per-tile cut and the pair floor at k_max up to 1024;
    the same bits on every call and from a second handle.  The windows give tiles of 16, 8, 4 and 1 rows."""
    rng = np.random.default_rng(5)
    S = (rng.random((2, 100, 4100)) ** 3).astype(dtype)
    freqs = np.linspace(-50.0, 50.0, 100)
    other = api.Handle(0)
    for k_max, gr, gd, tr, tc, scale in ((1024, 1, 1, 2, 16, 1.0), (200, 0, 0, 1, 1, 2.0), (33, 4, 17, 8, 40, 3.0),
                                         (16, 2, 2, 4, 16, 1.5), (8, 2, 2, 30, 36, 1.5)):
        got, _ = check_against_reference(S, freqs, k_max, gr, gd, tr, tc, scale)
        for _ in range(2):
            assert run_dev(S, freqs, k_max, gr, gd, tr, tc, scale)[0] == got
        assert run_dev(S, freqs, k_max, gr, gd, tr, tc, scale, handle=other)[0] == got
    other.close()


def test_spike_surface():
    """A spike 1e12 above an exponential floor: the cells around it keep an accurate noise estimate (no running sum), the
    spike is detected, and its neighbours' lists match the reference bit for bit."""
    rng = np.random.default_rng(3)
    S = rng.exponential(1.0, size=(1, 64, 2000))
    S[0, 30, 1000] = 1e12
    freqs = np.arange(64.0)
    got, cnt = check_against_reference(S, freqs, 32, 1, 2, 3, 9, api.cfar_scale(1e-6, api.cfar_train_cells(1, 2, 3, 9)))
    assert cnt[0] >= 1 and (got[0][0][2], got[0][0][3]) == (30, 1000)
    noise = run_map(S, 1, 2, 3, 9)[0]
    assert 0.8 < noise[30, 1000] < 1.25                       # the spike is in its own guard block
    assert noise[30, 1005] > 1e9                              # ... and in its neighbours' training cells


def planted(sigma=None, emitters=True):
    """The four emitters of test_gpu_detect.planted (or none) under complex noise of std PLANTED_SIGMA per component."""
    sigma = PLANTED_SIGMA if sigma is None else sigma
    rng = np.random.default_rng(7)
    N = 4096
    needle = np.hanning(N) * (rng.standard_normal(N) + 1j * rng.standard_normal(N)) / np.sqrt(2)
    hay = np.zeros(N, dtype=np.complex128)
    ems = [(202, 69.0, 1.0), (57, -31.5, 0.5), (140, 12.0, 0.25), (90, -80.25, 0.15)]
    for lag, f, a in (ems if emitters else []):
        x = np.concatenate([np.zeros(lag), needle])[:N]
        hay += a * x * np.exp(2j * np.pi * f * np.arange(N) / FS)
    hay += sigma * (rng.standard_normal(N) + 1j * rng.standard_normal(N))
    return needle, hay, ems


# the planted scene: noise, guard and training region (see test_cfar_finds_exactly_the_four_emitters)
PLANTED_SIGMA = 0.1
PG = (32, 2, 0, 64)          # guard_doppler, guard_delay, train_doppler, train_delay


@pytest.mark.parametrize("variant", [api._Variant, api._Variant32], ids=["f64", "f32"])
def test_cfar_finds_exactly_the_four_emitters(variant):
    """detect's ranking cannot say how many emitters there are: it returns k_max local maxima on the emitters' pair and on
    a noise-only pair alike.  CFAR at Pfa 1e-6 returns the four emitters and nothing else, and nothing on the noise-only
    pair.  The weakest emitter clears the threshold by >= 3 dB.  The strongest other local maximum stays under it by only
    >= 0.3 dB (0.38 dB measured with the emitters, 0.54 without), and no seed does much better: at Pfa 1e-6, ~1e-3 of the
    cells of noise exceed half the threshold, and a 400 x 8192 surface has ~1e5 independent ones.  The inputs are seeded,
    so the margin is fixed; f32 rounding moves it by ~1e-7."""
    gr, gd, tr, tc = PG
    scale = api.cfar_scale(1e-6, api.cfar_train_cells(gr, gd, tr, tc))
    shifts = bench_shifts()
    needle, hay, ems = planted()
    s = api.DeviceSurface(needle, hay, shifts, FS, variant=variant)
    dets = s.detect_cfar(8, gr, gd, tr, tc, scale)
    assert len(dets) == 4
    for x, (lag, f, _) in zip(dets, ems):
        assert x.lag_samples == pytest.approx(lag, abs=0.5) and int(x.delay_idx) == lag
        assert abs(x.freq_hz - f) <= 2.5 and abs(x.freq_hz_interp - f) <= 2.5
    S = s.fetch_rows()
    same(of_structs(dets), F.detect_cfar(S, shifts, 8, gr, gd, tr, tc, scale))
    # margins: the weakest emitter's SNR over scale, and scale over the best non-emitter local maximum, both >= 3 dB
    noise, _ = F.noise_map(S, gr, gd, tr, tc)
    snr_em = min(x.value / x.noise for x in dets)
    from oracle.detect import local_maxima
    lm = local_maxima(S, gr, gd)
    for x in dets:
        lm[x.doppler_idx, x.delay_idx] = False
    with np.errstate(invalid="ignore"):
        snr_other = np.nanmax(np.where(lm, S.astype(np.float64) / noise, np.nan))
    assert 10 * np.log10(snr_em / scale) >= 3.0
    assert 10 * np.log10(scale / snr_other) >= 0.3
    assert len(s.detect(8, gr, gd)) == 8                                   # rank alone: 8 asked, 8 returned
    s.close()

    needle, hay, _ = planted(emitters=False)
    s = api.DeviceSurface(needle, hay, shifts, FS, variant=variant)
    assert s.detect_cfar(8, gr, gd, tr, tc, scale) == []
    assert len(s.detect(8, gr, gd)) == 8                                   # ... with nothing there
    S = s.fetch_rows()
    noise, _ = F.noise_map(S, gr, gd, tr, tc)
    with np.errstate(invalid="ignore"):
        snr_noise = np.nanmax(np.where(local_maxima(S, gr, gd), S.astype(np.float64) / noise, np.nan))
    assert 10 * np.log10(scale / snr_noise) >= 0.3
    s.close()


@pytest.mark.parametrize("variant", [api._Variant, api._Variant32], ids=["f64", "f32"])
def test_real_surfaces_match_reference(variant):
    """Config-1 CAF surfaces (400 x 8192) and long rows (l = 8192): lists bit for bit at two windows and scales."""
    needle, hay, _ = planted()
    s = api.DeviceSurface(needle, hay, bench_shifts(), FS, variant=variant)
    S = s.fetch_rows()
    for gr, gd, tr, tc, k_max, scale in ((2, 2, 4, 16, 16, 5.0), (1, 1, 2, 16, 64, 3.0), (3, 20, 6, 100, 16, 8.0)):
        same(of_structs(s.detect_cfar(k_max, gr, gd, tr, tc, scale)), F.detect_cfar(S, bench_shifts(), k_max, gr, gd, tr, tc, scale))
    s.close()
    rng = np.random.default_rng(11)
    L = 8192
    needle = rng.standard_normal(L) + 1j * rng.standard_normal(L)
    hay = np.roll(needle, 300) * np.exp(2j * np.pi * 20.0 * np.arange(L) / FS) + 0.5 * (rng.standard_normal(L) + 1j * rng.standard_normal(L))
    freqs = np.linspace(0.0, 40.0, 16)
    s = api.DeviceSurface(needle, hay, freqs, FS, variant=variant)
    assert s.shape == (16, 2 * L)
    S = s.fetch_rows()
    dets = s.detect_cfar(100, 1, 2, 2, 16, 4.0)
    same(of_structs(dets), F.detect_cfar(S, freqs, 100, 1, 2, 2, 16, 4.0))
    assert dets[0].delay_idx == 300
    s.close()


def test_error_codes():
    import torch
    lib = _lib.load()
    h = api.Handle(0)
    needle, hay, _ = planted()
    shifts = np.linspace(-5, 5, 11)
    s = api.DeviceSurface(needle[:64], hay[:64], shifts, FS, handle=h)           # 11 x 128
    out = (_lib.CfarDetection * 1025)()
    C.memset(out, 0x5a, C.sizeof(out))
    before = bytes(out)
    cnt = C.c_size_t(77)
    for args in ((0, 1, 1, 2, 16, 10.0), (1025, 1, 1, 2, 16, 10.0), (4, 1, 1, 32, 16, 10.0), (4, 33, 1, 0, 16, 10.0),
                 (4, 1, 1, 2, 256, 10.0), (4, 1, 257, 2, 0, 10.0), (4, 1, 1, 0, 0, 10.0), (4, 1, 1, 2, 63, 10.0),
                 (4, 1, 1, 2, 16, 0.0), (4, 1, 1, 2, 16, -1.0), (4, 1, 1, 2, 16, float("inf")), (4, 1, 1, 2, 16, float("nan"))):
        assert lib.caf_b200_surface_detect_cfar(s.raw, *args, out, C.byref(cnt)) == -1, args
        assert cnt.value == 77 and bytes(out) == before
    assert lib.caf_b200_surface_detect_cfar(s.raw, 4, 1, 1, 2, 62, 10.0, out, C.byref(cnt)) == 0       # 2 * 63 + 1 <= 128
    assert lib.caf_b200_surface_detect_cfar(s.raw, 4, 1, 1, 2, 16, 10.0, None, C.byref(cnt)) == -1
    assert lib.caf_b200_surface_detect_cfar(s.raw, 4, 1, 1, 2, 16, 10.0, out, None) == -1
    dev = torch.device("cuda", 0)
    S = torch.rand((1, 4, 16), dtype=torch.float64, device=dev)
    f = torch.zeros(4, dtype=torch.float64, device=dev)
    o = torch.full((1, 4, 8), 3.0, dtype=torch.float64, device=dev)
    c = torch.full((1,), 9, dtype=torch.int64, device=dev)
    nz = torch.full((1, 4, 16), 3.0, dtype=torch.float64, device=dev)
    P = lambda t: t.data_ptr()
    assert lib.caf_b200_detect_cfar_f64_dev(h.raw, P(S), 1, 4, 16, P(f), 4, 1, 1, 0, 7, 2.0, P(o), P(c)) == -1    # 2C + 1 > n
    assert lib.caf_b200_detect_cfar_f64_dev(h.raw, None, 1, 4, 16, P(f), 4, 1, 1, 0, 2, 2.0, P(o), P(c)) == -1
    assert lib.caf_b200_detect_cfar_f64_dev(h.raw, P(S), 1, 4, 16, None, 4, 1, 1, 0, 2, 2.0, P(o), P(c)) == -1
    assert lib.caf_b200_detect_cfar_f64_dev(h.raw, P(S), 1, 4, 16, P(f), 4, 1, 1, 0, 2, 2.0, None, P(c)) == -1
    assert lib.caf_b200_detect_cfar_f64_dev(h.raw, P(S), 1, 4, 16, P(f), 4, 1, 1, 0, 2, 2.0, P(o), None) == -1
    assert lib.caf_b200_cfar_noise_f64_dev(h.raw, P(S), 1, 4, 16, 1, 1, 0, 7, P(nz)) == -1
    assert lib.caf_b200_cfar_noise_f64_dev(h.raw, P(S), 1, 4, 16, 1, 1, 0, 0, P(nz)) == -1
    assert lib.caf_b200_cfar_noise_f64_dev(h.raw, P(S), 1, 4, 16, 30, 1, 3, 1, P(nz)) == -1
    assert lib.caf_b200_cfar_noise_f32_dev(h.raw, P(S), 1, 4, 16, 1, 1, 0, 2, None) == -1
    torch.cuda.synchronize()
    assert bool((o == 3.0).all()) and int(c[0]) == 9 and bool((nz == 3.0).all())
    # empty shapes: count 0, every slot "none"
    assert lib.caf_b200_detect_cfar_f64_dev(h.raw, P(S), 1, 0, 16, P(f), 4, 1, 1, 0, 2, 2.0, P(o), P(c)) == 0
    torch.cuda.synchronize()
    assert int(c[0]) == 0 and as_tuples(o.cpu().numpy().view(REC).reshape(4)) == [F.NONE] * 4
    # a surface whose handle is gone
    h.close()
    assert lib.caf_b200_surface_detect_cfar(s.raw, 4, 1, 1, 2, 16, 10.0, out, C.byref(cnt)) == -1
    assert "handle" in lib.caf_b200_last_error().decode()
    s.close()


def test_overlap_detect_cfar_between_surface_launches():
    """With overlap mode 4 and rotated outputs, detect_cfar calls between surface launches leave every surface and peak
    bit-identical to the serialised run, raise the launch count by two each, and give the reference's list."""
    import torch
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    lib = _lib.load()
    h = api.Handle(0, stream=stream.cuda_stream)
    L = 4096
    needle, hay, _ = planted()
    nd = torch.from_numpy(needle).to(dev)
    hd = torch.from_numpy(hay).to(dev)
    shifts = bench_shifts()
    fd = torch.from_numpy(shifts).to(dev)
    K, NB = 12, 9

    def run(overlap, with_detect):
        lib.caf_b200_set_overlap(h.raw, overlap)
        surfs = [torch.zeros((400, 2 * L), dtype=torch.float64, device=dev) for _ in range(NB)]
        rv = torch.zeros((K, 400), dtype=torch.float64, device=dev); ri = torch.zeros((K, 400), dtype=torch.int64, device=dev)
        pk = torch.zeros((K, 4), dtype=torch.int64, device=dev)
        out = torch.zeros((K, 8, 8), dtype=torch.float64, device=dev); cnt = torch.zeros(K, dtype=torch.int64, device=dev)
        with torch.cuda.stream(stream):
            for k in range(K):
                sb = k % NB
                assert lib.caf_b200_batch_f64_dev(h.raw, nd.data_ptr(), hd.data_ptr(), 1, L, fd.data_ptr(), 400, FS,
                                                  surfs[sb].data_ptr(), rv[k].data_ptr(), ri[k].data_ptr(), pk[k].data_ptr()) == 0
                if with_detect and k % 3 == 1:
                    before = h.launch_count
                    assert lib.caf_b200_detect_cfar_f64_dev(h.raw, surfs[sb].data_ptr(), 1, 400, 2 * L, fd.data_ptr(), 8, 2, 2,
                                                            4, 16, 5.0, out[k].data_ptr(), cnt[k].data_ptr()) == 0
                    assert h.launch_count == before + 2
        torch.cuda.synchronize()
        return [x.cpu().numpy() for x in surfs], rv.cpu().numpy(), ri.cpu().numpy(), pk.cpu().numpy(), out.cpu().numpy(), cnt.cpu().numpy()

    want = run(0, False)
    got = run(4, True)
    for a, b in zip(want[0], got[0]):
        assert np.array_equal(a, b)
    for i in (1, 2, 3):
        assert np.array_equal(want[i], got[i])
    ref = F.detect_cfar(want[0][1], shifts, 8, 2, 2, 4, 16, 5.0)
    for k in range(1, K, 3):
        same(as_tuples(got[4][k].view(REC).reshape(8))[:int(got[5][k])], ref)
    lib.caf_b200_set_overlap(h.raw, 0)
    h.close()


def test_two_handles_alternate_large_and_small_windows():
    """The tile kernel's shared-memory allowance belongs to the device: a handle that ran small windows must not take it
    away from another handle's one-row tile that stages a ~200 KB training region, nor from the largest windows."""
    rng = np.random.default_rng(21)
    S64 = (rng.random((1, 70, 700)) ** 3)
    S32 = S64.astype(np.float32)
    freqs = np.linspace(-10.0, 10.0, 70)
    a, b = api.Handle(0), api.Handle(0)
    for S in (S64, S32, S64):
        for h, w in ((a, (2, 2, 30, 36)), (b, (1, 1, 0, 1)), (a, (0, 0, 32, 256)), (b, (0, 0, 1, 0)), (a, (2, 2, 30, 36)),
                     (b, (31, 255, 1, 1)), (a, (1, 1, 2, 16))):
            got, cnt = run_dev(S, freqs, 8, *w, 1.5, handle=h)
            want = F.detect_cfar(S[0], freqs, 8, *w, 1.5)
            assert cnt[0] == len(want)
            same(got[0], F.padded(want, 8))
    a.close()
    b.close()


def _cli(tmp_path):
    import shutil
    import subprocess
    from conftest import ROOT
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "caf_cli")
    subprocess.check_call([shutil.which("g++"), "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tools", "caf_cli.cpp"), "-o", exe, "-L", so_dir, "-lcaf_b200",
                           f"-Wl,-rpath,{so_dir}"])
    return exe


def test_cli_cfar_prints_exactly_the_four_emitters(tmp_path):
    """--detect 8 --cfar-db X: the two main.rs lines, then the four emitters and no more; on the noise-only pair only the
    two lines; without --cfar-db the output is the plain report."""
    import subprocess
    exe = _cli(tmp_path)
    gr, gd, tr, tc = PG
    db = 10 * np.log10(api.cfar_scale(1e-6, api.cfar_train_cells(gr, gd, tr, tc)))
    win = ["--guard-doppler", str(gr), "--guard-delay", str(gd)]
    cf = ["--cfar-db", "%.6f" % db, "--train-doppler", str(tr), "--train-delay", str(tc)]
    for emitters in (True, False):
        needle, hay, ems = planted(emitters=emitters)
        a, b = str(tmp_path / "needle.c64"), str(tmp_path / "hay.c64")
        for path, x in ((a, needle), (b, hay)):
            np.stack([x.real, x.imag], axis=1).astype("<f4").tofile(path)
        plain = subprocess.run([exe, a, b], capture_output=True, text=True, timeout=120)
        assert plain.returncode == 0 and plain.stdout.count("\n") == 2, plain.stderr
        res = subprocess.run([exe, a, b, "--detect", "8"] + win + cf, capture_output=True, text=True, timeout=120)
        assert res.returncode == 0, res.stderr
        assert res.stdout.startswith(plain.stdout)
        lines = res.stdout.splitlines()[2:]
        if not emitters:
            assert lines == []
            continue
        assert len(lines) == 4
        for line, (lag, f, _) in zip(lines, ems):
            m = re.match(r"Detection \d: (\S+)Hz \(grid (\S+)Hz\), (\S+) samples \(cell (\d+)\), (\S+) dB below the first, "
                         r"(\S+) dB above the noise$", line)
            assert m and int(m.group(4)) == lag and abs(float(m.group(1)) - f) <= 2.5, line
            assert float(m.group(6)) > db + 3.0, line
        ranked = subprocess.run([exe, a, b, "--detect", "8"] + win, capture_output=True, text=True, timeout=120)
        assert ranked.returncode == 0 and len(ranked.stdout.splitlines()) == 10 and "noise" not in ranked.stdout


def test_cpp_detect_cfar_refuses_other_threads(tmp_path):
    """caf_b200_surface_detect_cfar runs on the surface's handle: the C++ mirror refuses other threads."""
    import shutil
    import subprocess
    from conftest import ROOT
    src = tmp_path / "owner.cpp"
    src.write_text(r'''
#include <cmath>
#include <cstdio>
#include <thread>
#include "caf_b200.hpp"
int main() {
    std::vector<caf::Complex64> x(256), y(256);
    for (int i = 0; i < 256; ++i) x[i] = {std::sin(0.37 * i * i), std::cos(1.3 * i + 0.011 * i * i)};
    for (int i = 0; i < 256; ++i) y[i] = x[(i + 250) % 256];      // delayed by 6 samples
    const auto rows = caf::CafB200::caf_surface(x, y, {-1.0, 0.0, 1.0}, 48000);
    const auto here = caf::CafB200::detect_cfar(rows, 3, 1, 1, 0, 16, 10.0);
    bool refused = false;
    std::thread t([&] { try { caf::CafB200::detect_cfar(rows, 3, 1, 1, 0, 16, 10.0); } catch (const caf::Panic&) { refused = true; } });
    t.join();
    std::printf("%zu %d %llu %llu\n", here.size(), refused ? 1 : 0, (unsigned long long)here[0].delay_idx,
                (unsigned long long)here[0].train_cells);
    return 0;
}
''')
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "owner")
    subprocess.check_call([shutil.which("g++"), "-std=c++17", "-O2", "-pthread", "-I", os.path.join(ROOT, "include"), str(src),
                           "-o", exe, "-L", so_dir, "-lcaf_b200", f"-Wl,-rpath,{so_dir}"])
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    n, refused, k, m = res.stdout.split()
    assert int(n) >= 1 and refused == "1" and int(k) == 6 and int(m) == 3 * 32   # 3 rows x (2 x 16) side cells
