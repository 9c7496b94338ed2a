"""The OS-CFAR contract (include/caf_b200.h, caf_b200_surface_detect_cfar_os) on the CPU: oracle/cfar_os.py's vectorised
map and detector against a per-cell loop, the threshold helper cfar_os_scale, a masked-emitter scene where CA-CFAR misses
the weak emitter and OS-CFAR finds it, and the argument checks that need no device."""
import ctypes as C
import math

import numpy as np
import pytest

from caf_cookoff_b200 import _lib, api, bench_shifts
from oracle import cfar as F
from oracle import cfar_os as O

FS = 48000


def same_bits(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64).view(np.uint64), np.asarray(b, dtype=np.float64).view(np.uint64))


def brute_map(S, gr, gd, tr, tc, rank):
    d, n = S.shape
    noise = np.empty((d, n))
    m = np.empty((d, n), dtype=np.int64)
    for r in range(d):
        for k in range(n):
            noise[r, k], m[r, k] = O.noise_os_brute(S, r, k, gr, gd, tr, tc, rank)
    return noise, m


CASES = [  # (d, n, gr, gd, tr, tc)
    (1, 9, 0, 1, 0, 3),        # d = 1: only the cell's own row; 2C + 1 = n
    (2, 11, 1, 1, 1, 2),       # every row an edge row
    (5, 13, 1, 2, 2, 0),       # tc = 0
    (6, 17, 2, 1, 0, 3),       # tr = 0: only the guard rows' side segments
    (7, 15, 0, 0, 3, 7),       # the window wraps the whole row
    (9, 21, 1, 1, 2, 4),
    (4, 10, 3, 4, 1, 0),       # many m = 0 cells once NaN is added
]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("case", CASES)
def test_vectorised_reference_equals_per_cell_loop(case, dtype):
    """Tie-heavy integers with NaN, -0.0 and +inf cells at ranks 1, ceil(N/2), ceil(3N/4) and N: the map is the per-cell
    order statistic bit for bit, edge rows use k_m = ceil(rank m / N), and the detector's list is the per-cell loop's."""
    d, n, gr, gd, tr, tc = case
    N = F.train_cells(gr, gd, tr, tc)
    rng = np.random.default_rng(hash(case) % 991)
    for trial in range(4):
        S = rng.integers(-1, 6, size=(d, n)).astype(dtype)
        S[S == -1] = -0.0
        S[rng.random(S.shape) < 0.03] = np.inf
        S[rng.random(S.shape) < (0.05 if trial < 2 else 0.4)] = np.nan
        if trial == 3:
            S[:, : n // 2] = np.nan
        f = np.cumsum(rng.random(d) + 0.1)
        for rank in sorted({1, (N + 1) // 2, (3 * N + 3) // 4, N}):
            noise, m = O.os_noise_map(S, gr, gd, tr, tc, rank)
            bn, bm = brute_map(S, gr, gd, tr, tc, rank)
            assert np.array_equal(m, bm)
            assert same_bits(noise, bn)
            assert np.array_equal(m, F.noise_map(S, gr, gd, tr, tc)[1])          # CA's training cells
            assert np.all(np.isnan(noise[m == 0])) and not np.any(np.isnan(noise[m > 0]))
            assert not np.any(np.signbit(noise[m > 0]))                         # -0.0 counts as +0.0
            for scale in (0.5, 1.0, 2.0):
                for k_max in (1, 50):
                    got = O.detect_cfar_os(S, f, k_max, gr, gd, tr, tc, rank, scale)
                    assert got == O.detect_cfar_os_brute(S, f, k_max, gr, gd, tr, tc, rank, scale)
                    for x in got:
                        assert x[7] > 0 and x[0] > scale * x[6]
                        assert same_bits(x[6], noise[x[2], x[3]]) and x[7] == m[x[2], x[3]]


def test_hand_computed_order_statistics():
    S = np.ones((5, 12))
    S[2, 6] = 9.0
    S[0, 6] = 3.0                                          # a training cell of (2, 6)
    S[4, 3:10] = 5.0                                       # a whole training row of (2, 6)
    gr, gd, tr, tc = 1, 1, 1, 2                            # N = 35 - 9 = 26
    N = 26
    # (2, 6): 26 cells: 18 ones, the 3, seven 5s
    for rank, want in ((1, 1.0), (18, 1.0), (19, 3.0), (20, 5.0), (26, 5.0)):
        noise, m = O.os_noise_map(S, gr, gd, tr, tc, rank)
        assert m[2, 6] == N and noise[2, 6] == want, rank
    # (0, 6): rows 0..2 clipped, m = 15: k_m = ceil(20 * 15 / 26) = 12 of [3 (own row is guard), ...]
    noise, m = O.os_noise_map(S, gr, gd, tr, tc, 20)
    assert m[0, 6] == 15 and O.rank_of(20, 15, N) == 12
    vals = sorted(x for row in F.cell_training(S, 0, 6, gr, gd, tr, tc) for x in row)
    assert noise[0, 6] == vals[11]
    got = O.detect_cfar_os(S, np.arange(5.0), 8, gr, gd, tr, tc, 19, 2.9)
    assert (got[0][2], got[0][3], got[0][6], got[0][7]) == (2, 6, 3.0, 26)     # 9 > 2.9 x 3
    got = O.detect_cfar_os(S, np.arange(5.0), 8, gr, gd, tr, tc, 19, 3.0)
    assert (2, 6) not in [(x[2], x[3]) for x in got]                          # 9 == 3 x 3 is not above


def test_m_zero_never_qualifies():
    S = np.full((3, 9), np.nan)
    S[1, 4] = 10.0
    noise, m = O.os_noise_map(S, 1, 1, 1, 2, 5)
    assert m[1, 4] == 0 and math.isnan(noise[1, 4])
    assert O.detect_cfar_os(S, [0.0, 1.0, 2.0], 4, 1, 1, 1, 2, 5, 1e-300) == []
    S[0, 1] = 1.0                                           # one training cell: k_m = ceil(5 / N) = 1
    got = O.detect_cfar_os(S, [0.0, 1.0, 2.0], 4, 1, 1, 1, 2, 5, 2.0)
    assert [(x[2], x[3], x[6], x[7]) for x in got] == [(1, 4, 1.0, 1)]


def test_a_strong_cell_in_the_training_region_does_not_move_the_estimate():
    """CA's mean rises with one spike among the training cells; the 3N/4-th order statistic does not."""
    rng = np.random.default_rng(4)
    S = rng.exponential(1.0, size=(30, 200))
    gr, gd, tr, tc = 1, 1, 2, 8
    N = F.train_cells(gr, gd, tr, tc)
    rank = (3 * N + 3) // 4
    before = O.os_noise_map(S, gr, gd, tr, tc, rank)[0][15, 100]
    ca_before = F.noise_map(S, gr, gd, tr, tc)[0][15, 100]
    S[13, 105] = 1e6
    after = O.os_noise_map(S, gr, gd, tr, tc, rank)[0][15, 100]
    ca_after = F.noise_map(S, gr, gd, tr, tc)[0][15, 100]
    assert ca_after > 1e3 * ca_before
    assert abs(after - before) <= 0.2 * before


def test_cfar_os_scale_rank_one_is_closed_form():
    for pfa, n in ((1e-6, 456), (1e-3, 46), (0.25, 3), (0.5, 1)):
        assert api.cfar_os_scale(pfa, n, 1) == pytest.approx(n * (1.0 / pfa - 1.0), rel=1e-12)


def test_cfar_os_scale_solves_the_product_and_is_monotone():
    N = 456
    prev = math.inf
    for k in (1, 2, 10, 100, 342, 455, 456):
        a = api.cfar_os_scale(1e-6, N, k)
        p = math.exp(sum(math.log((N - i) / (N - i + a)) for i in range(k)))
        assert p == pytest.approx(1e-6, rel=1e-9)
        assert a < prev                                    # a higher rank needs a lower factor
        prev = a
    assert api.cfar_os_scale(1e-6, N, 342) == pytest.approx(10.23, abs=0.01)
    for k in (1, 342):
        assert api.cfar_os_scale(1e-3, N, k) < api.cfar_os_scale(1e-6, N, k) < api.cfar_os_scale(1e-9, N, k)
    for bad in ((0.0, 10, 1), (1.0, 10, 1), (1e-3, 0, 1), (1e-3, 10, 0), (1e-3, 10, 11)):
        with pytest.raises(ValueError):
            api.cfar_os_scale(*bad)


def test_cfar_os_scale_calibration():
    """On i.i.d. exponential cells the interior exceedance rate of v > alpha x noise is Pfa = 1e-3 to within 15 %
    (400 x 8192 cells, ~3.2e6 interior tests, ~3200 expected exceedances: 1 sigma = 1.8 %)."""
    rng = np.random.default_rng(2025)
    S = rng.exponential(1.0, size=(400, 8192))
    gr, gd, tr, tc = 1, 1, 1, 4
    N = F.train_cells(gr, gd, tr, tc)
    assert N == 5 * 11 - 9
    rank = (3 * N + 3) // 4
    pfa = 1e-3
    alpha = api.cfar_os_scale(pfa, N, rank)
    R = gr + tr
    rr, kk = np.divmod(np.arange(R * 8192, (400 - R) * 8192, dtype=np.int64), 8192)
    noise, m = O.os_noise_at(S, rr, kk, gr, gd, tr, tc, rank)
    assert np.all(m == N)
    frac = float(np.mean(S[rr, kk] > alpha * noise))
    assert abs(frac - pfa) <= 0.15 * pfa, frac


def planted_scene(ems, seed, sigma=0.1, n=4096):
    """test_gpu_cfar.planted's generator with chosen emitters (lag, Hz, amplitude): a Hann-windowed noise needle, the
    haystack its delayed, Doppler-shifted copies under complex noise of std sigma per component."""
    rng = np.random.default_rng(seed)
    needle = np.hanning(n) * (rng.standard_normal(n) + 1j * rng.standard_normal(n)) / np.sqrt(2)
    hay = np.zeros(n, dtype=np.complex128)
    for lag, f, a in ems:
        x = np.concatenate([np.zeros(lag), needle])[:n]
        hay += a * x * np.exp(2j * np.pi * f * np.arange(n) / FS)
    hay += sigma * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return needle, hay


def margins_db(recs, scale):
    """delay cell -> the best margin over the threshold of a detection there, in dB"""
    out = {}
    for x in recs:
        out[x[3]] = max(out.get(x[3], -np.inf), 10 * np.log10(x[0] / (scale * x[6])))
    return out


def test_masked_emitter_scene():
    """Strong (202, 69 Hz, 1.0) and weak (230, 69 Hz, 0.15) emitters, the bench grid cut to 40 ... 100 Hz.  With the
    training region in delay only (guard 32 x 2, training 0 x 64), the strong emitter's lobe sits in the weak one's
    training cells: CA-CFAR misses it, OS-CFAR finds it with +4.9 dB (seeded: the margins are fixed).  At the default
    4 x 16 window the strong emitter's own Doppler lobe caps CA's margin at +6.1 dB; OS's is +21.5 dB."""
    from oracle import np_oracle
    freqs = bench_shifts()
    freqs = freqs[(freqs >= 40.0) & (freqs < 100.0)]
    needle, hay = planted_scene([(202, 69.0, 1.0), (230, 69.0, 0.15)], 7)
    S = np_oracle.caf_surface(needle, hay, freqs, FS)[0]
    strong, weak = 202, 230

    w = (32, 2, 0, 64)
    N = F.train_cells(*w)
    rank = (3 * N + 3) // 4
    a_ca, a_os = api.cfar_scale(1e-6, N), api.cfar_os_scale(1e-6, N, rank)
    ca = margins_db(F.detect_cfar(S, freqs, 16, *w, a_ca), a_ca)
    os_ = margins_db(O.detect_cfar_os(S, freqs, 16, *w, rank, a_os), a_os)
    assert strong in ca and ca[strong] > 20.0
    assert weak not in ca
    assert strong in os_ and os_[strong] > 20.0
    assert weak in os_ and os_[weak] > 4.0

    w = (2, 2, 4, 16)
    N = F.train_cells(*w)
    rank = (3 * N + 3) // 4
    assert (N, rank) == (456, 342)
    a_ca, a_os = api.cfar_scale(1e-6, N), api.cfar_os_scale(1e-6, N, rank)
    ca = margins_db(F.detect_cfar(S, freqs, 16, *w, a_ca), a_ca)
    os_ = margins_db(O.detect_cfar_os(S, freqs, 16, *w, rank, a_os), a_os)
    assert ca[strong] < 7.0 and os_[strong] > 15.0


def test_record_layout_and_symbols():
    for name in ("caf_b200_surface_detect_cfar_os", "caf_b200_detect_cfar_os_f64_dev", "caf_b200_detect_cfar_os_f32_dev",
                 "caf_b200_cfar_os_noise_f64_dev", "caf_b200_cfar_os_noise_f32_dev"):
        assert name in _lib.SYMBOLS


def test_null_surface_and_null_handle_are_rejected():
    lib = _lib.load()
    out = (_lib.CfarDetection * 4)()
    C.memset(out, 0x5a, C.sizeof(out))
    before = bytes(out)
    cnt = C.c_size_t(123)
    assert lib.caf_b200_surface_detect_cfar_os(None, 4, 1, 1, 2, 16, 10, 10.0, out, C.byref(cnt)) == -1
    assert cnt.value == 123 and bytes(out) == before
    for fn in (lib.caf_b200_detect_cfar_os_f64_dev, lib.caf_b200_detect_cfar_os_f32_dev):
        assert fn(None, None, 1, 4, 64, None, 4, 1, 1, 2, 16, 10, 10.0, None, None) == -1
    for fn in (lib.caf_b200_cfar_os_noise_f64_dev, lib.caf_b200_cfar_os_noise_f32_dev):
        assert fn(None, None, 1, 4, 64, 1, 1, 2, 16, 10, None) == -1
    assert "handle" in lib.caf_b200_last_error().decode()


def test_cli_rejects_bad_cfar_rank(tmp_path):
    """tools/caf_cli: --cfar-rank without --cfar-db, zero, or not a number exit with 2 before any GPU work."""
    import os
    import shutil
    import subprocess
    from conftest import ROOT
    gxx = shutil.which("g++")
    assert gxx, "g++ is required for the CLI"
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "caf_cli")
    subprocess.check_call([gxx, "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tools", "caf_cli.cpp"),
                           "-o", exe, "-L", so_dir, "-lcaf_b200", f"-Wl,-rpath,{so_dir}"])
    for bad in (["--detect", "4", "--cfar-rank", "3"], ["--detect", "4", "--cfar-db", "13", "--cfar-rank", "0"],
                ["--detect", "4", "--cfar-db", "13", "--cfar-rank", "x"], ["--cfar-db", "13", "--cfar-rank", "3"]):
        res = subprocess.run([exe, "a.c64", "b.c64"] + bad, capture_output=True, text=True)
        assert res.returncode == 2 and "caf_cli:" in res.stderr, (bad, res.returncode, res.stderr)
