"""The CA-CFAR contract (include/caf_b200.h, caf_b200_surface_detect_cfar) on the CPU: oracle/cfar.py's vectorised map and
detector against a per-cell loop in the contract's summation order, the accuracy of that order next to a huge peak, the
calibration of cfar_scale, and the argument checks that need no device."""
import ctypes as C
import math

import numpy as np
import pytest

from caf_cookoff_b200 import _lib, api
from oracle import cfar as F


def brute_map(S, gr, gd, tr, tc):
    d, n = S.shape
    noise = np.empty((d, n))
    m = np.empty((d, n), dtype=np.int64)
    for r in range(d):
        for k in range(n):
            noise[r, k], m[r, k] = F.noise_brute(S, r, k, gr, gd, tr, tc)
    return noise, m


def same_bits(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64).view(np.uint64), np.asarray(b, dtype=np.float64).view(np.uint64))


CASES = [  # (d, n, gr, gd, tr, tc)
    (1, 9, 0, 1, 0, 3),        # d = 1: no training rows beyond the cell's own; 2C + 1 = n
    (2, 11, 1, 1, 1, 2),       # d = 2: every row an edge row
    (5, 13, 1, 2, 2, 0),       # tc = 0: guard rows contribute nothing
    (6, 17, 2, 1, 0, 3),       # tr = 0: only the guard rows' side segments
    (7, 15, 0, 0, 3, 7),       # 2C + 1 = n, the window wraps the whole row
    (9, 21, 1, 1, 2, 4),
    (4, 10, 3, 4, 1, 0),       # the guard block covers whole rows: many cells with m = 0 once NaN is added
]


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("case", CASES)
def test_vectorised_reference_equals_per_cell_loop(case, dtype):
    """Tie-heavy integers with NaN cells: the map is the per-cell sum bit for bit, and so is the detector's list."""
    d, n, gr, gd, tr, tc = case
    rng = np.random.default_rng(hash(case) % 997)
    for trial in range(4):
        S = rng.integers(0, 6, size=(d, n)).astype(dtype)
        S[rng.random(S.shape) < (0.05 if trial < 2 else 0.4)] = np.nan
        if trial == 3:
            S[:, : n // 2] = np.nan            # whole training regions NaN: m = 0 cells
        f = np.cumsum(rng.random(d) + 0.1)
        noise, m = F.noise_map(S, gr, gd, tr, tc)
        bn, bm = brute_map(S, gr, gd, tr, tc)
        assert np.array_equal(m, bm)
        assert same_bits(noise, bn)
        assert np.all(np.isnan(noise[m == 0])) and not np.any(np.isnan(noise[m > 0]))
        for scale in (0.5, 1.0, 1.7):
            for k_max in (1, 3, 50):
                got = F.detect_cfar(S, f, k_max, gr, gd, tr, tc, scale)
                want = F.detect_cfar_brute(S, f, k_max, gr, gd, tr, tc, scale)
                assert got == want
                for x in got:
                    assert x[7] > 0 and x[0] > scale * x[6]
                    assert same_bits(x[6], noise[x[2], x[3]]) and x[7] == m[x[2], x[3]]


def test_m_zero_never_qualifies():
    """A peak whose every training cell is NaN has noise NaN, m = 0, and is not a detection at any scale."""
    S = np.full((3, 9), np.nan)
    S[1, 4] = 10.0
    noise, m = F.noise_map(S, 1, 1, 1, 2)
    assert m[1, 4] == 0 and math.isnan(noise[1, 4])
    assert F.detect_cfar(S, [0.0, 1.0, 2.0], 4, 1, 1, 1, 2, 1e-300) == []
    S[0, 1] = 1.0                                           # one training cell (row 0, j = -3): now it qualifies
    got = F.detect_cfar(S, [0.0, 1.0, 2.0], 4, 1, 1, 1, 2, 2.0)
    assert [(x[2], x[3], x[6], x[7]) for x in got] == [(1, 4, 1.0, 1)]


def test_hand_computed_noise_and_detection():
    S = np.ones((5, 12))
    S[2, 6] = 9.0
    S[2, 7] = 4.0                                          # in the guard: not training
    S[0, 6] = 3.0                                          # training (row r - 2)
    noise, m = F.noise_map(S, 1, 1, 1, 2)
    # R = 2, C = 3: rows 0..4 x cells 3..9, without guard rows 1..3 x cells 5..7: 35 - 9 = 26 cells, 25 ones and the 3
    assert m[2, 6] == 26 and noise[2, 6] == 28.0 / 26.0
    # (0, 6): rows 0..2 (clipped); row 2 is a training row holding the 9 and the 4: 4 + 4 + 18 over 15 cells
    assert m[0, 6] == 15 and noise[0, 6] == 26.0 / 15.0
    got = F.detect_cfar(S, np.arange(5.0), 8, 1, 1, 1, 2, 8.0)
    assert [(x[2], x[3], x[7]) for x in got] == [(2, 6, 26)]   # 9 > 8 x 1.077; 3 is not above 8 x 1.733, nor 1 above 8 x ~1
    assert F.detect_cfar(S, np.arange(5.0), 8, 1, 1, 1, 2, 9.0 / (28.0 / 26.0) * (1 + 1e-9)) == []


def test_noise_is_accurate_next_to_a_huge_spike():
    """Non-negative terms summed in order: within (m + 1) 2^-53 relative of the exactly rounded mean of the same cells,
    including cells whose training region holds a spike 1e12 above the floor (a running sum would lose the floor)."""
    rng = np.random.default_rng(3)
    S = rng.exponential(1.0, size=(24, 160))
    S[12, 80] = 1e12
    gr, gd, tr, tc = 1, 2, 3, 9
    noise, m = F.noise_map(S, gr, gd, tr, tc)
    for r in range(6, 19):
        for k in list(range(60, 101)) + [0, 159]:
            rows = F.cell_training(S, r, k, gr, gd, tr, tc)
            cells = [x for row in rows for x in row]
            exact = math.fsum(cells) / len(cells)
            assert m[r, k] == len(cells)
            assert abs(noise[r, k] - exact) <= (m[r, k] + 1) * 2.0 ** -53 * exact, (r, k)
    far = noise[12, 10]
    assert abs(far - 1.0) < 0.2                               # the spike is outside this cell's region


def test_cfar_scale_calibration():
    """cfar_scale(Pfa, N) on i.i.d. exponential cells: the fraction of interior-row cells above alpha x their noise is
    Pfa to within 15 % (400 x 8192 cells, ~2.7e6 interior tests, ~2700 expected exceedances: 1 sigma = 2 %)."""
    rng = np.random.default_rng(2024)
    S = rng.exponential(1.0, size=(400, 8192))
    gr, gd, tr, tc = 1, 1, 2, 16
    N = api.cfar_train_cells(gr, gd, tr, tc)
    assert N == F.train_cells(gr, gd, tr, tc) == 7 * 35 - 9
    pfa = 1e-3
    alpha = api.cfar_scale(pfa, N)
    assert alpha == F.scale_for_pfa(pfa, N)
    assert abs((1.0 + alpha / N) ** -N - pfa) < 1e-15
    noise, m = F.noise_map(S, gr, gd, tr, tc)
    R = gr + tr
    inner = slice(R, 400 - R)
    assert np.all(m[inner] == N)
    frac = float(np.mean(S[inner] > alpha * noise[inner]))
    assert abs(frac - pfa) <= 0.15 * pfa, frac


def test_cfar_scale_arguments():
    assert api.cfar_train_cells(0, 0, 0, 1) == 2
    assert api.cfar_scale(0.5, 1) == pytest.approx(1.0)    # one cell: P(v > a u) = 1 / (1 + a)
    for bad in ((0.0, 10), (1.0, 10), (-1e-3, 10), (1e-3, 0)):
        with pytest.raises(ValueError):
            api.cfar_scale(*bad)


def test_cfar_record_layout():
    assert C.sizeof(_lib.CfarDetection) == 64
    assert [f[0] for f in _lib.CfarDetection._fields_][:6] == [f[0] for f in _lib.Detection._fields_]
    assert [f[0] for f in _lib.CfarDetection._fields_][6:] == ["noise", "train_cells"]


def test_null_surface_and_null_handle_are_rejected():
    lib = _lib.load()
    out = (_lib.CfarDetection * 4)()
    cnt = C.c_size_t(123)
    assert lib.caf_b200_surface_detect_cfar(None, 4, 1, 1, 2, 16, 10.0, out, C.byref(cnt)) == -1
    assert cnt.value == 123
    for fn in (lib.caf_b200_detect_cfar_f64_dev, lib.caf_b200_detect_cfar_f32_dev):
        assert fn(None, None, 1, 4, 64, None, 4, 1, 1, 2, 16, 10.0, None, None) == -1
    for fn in (lib.caf_b200_cfar_noise_f64_dev, lib.caf_b200_cfar_noise_f32_dev):
        assert fn(None, None, 1, 4, 64, 1, 1, 2, 16, None) == -1
    assert "handle" in lib.caf_b200_last_error().decode()


def test_cli_rejects_bad_cfar_arguments(tmp_path):
    """tools/caf_cli: --cfar-db without --detect, with --min-db, not a number, or --train-* out of range / without
    --cfar-db exit with 2 before any GPU work."""
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
    for bad in (["--cfar-db", "13"], ["--detect", "4", "--cfar-db", "13", "--min-db", "3"], ["--detect", "4", "--cfar-db", "x"],
                ["--detect", "4", "--cfar-db", "inf"], ["--detect", "4", "--cfar-db", "13", "--train-doppler", "33"],
                ["--detect", "4", "--cfar-db", "13", "--train-delay", "-1"], ["--detect", "4", "--train-delay", "8"]):
        res = subprocess.run([exe, "a.c64", "b.c64"] + bad, capture_output=True, text=True)
        assert res.returncode == 2 and "caf_cli:" in res.stderr, (bad, res.returncode, res.stderr)
