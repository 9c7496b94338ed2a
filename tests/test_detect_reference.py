"""The detection contract (include/caf_b200.h, caf_b200_surface_detect) on the CPU: oracle/detect.py against a per-cell
loop, crafted cases whose answer is known by hand, and the argument checks that need no device."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

from caf_cookoff_b200 import _lib
from conftest import GOLDEN, load_case
from oracle import detect as D

UMAX = (1 << 64) - 1


@pytest.mark.parametrize("seed", range(6))
def test_vectorised_reference_equals_per_cell_loop(seed):
    """Small integer values: ties everywhere, so the equal-value rule decides most cells."""
    rng = np.random.default_rng(seed)
    for _ in range(60):
        d, n = int(rng.integers(1, 7)), int(rng.integers(1, 14))
        gd, gr = int(rng.integers(0, (n - 1) // 2 + 1)), int(rng.integers(0, 4))
        S = rng.integers(0, 4, size=(d, n)).astype(np.float64)
        if rng.random() < 0.3:
            S[rng.random((d, n)) < 0.2] = np.nan
        f = np.cumsum(rng.random(d) + 0.1)
        k_max, ratio = int(rng.integers(1, 20)), float(rng.choice([0.0, 0.4, 1.0]))
        assert D.detect(S, f, k_max, gr, gd, ratio) == D.detect_brute(S, f, k_max, gr, gd, ratio)


def test_plateau_is_one_detection_at_its_first_cell():
    S = np.zeros((3, 10))
    S[1, 3:6] = 5.0
    S[0, 4] = 5.0
    got = D.detect(S, [0.0, 1.0, 2.0], 8, 1, 1)
    assert [(x[2], x[3]) for x in got] == [(0, 4)]          # flat 4 comes before 13, 14, 15
    got = D.detect(S, [0.0, 1.0, 2.0], 8, 0, 1)             # rows apart: one per row
    assert [(x[2], x[3]) for x in got] == [(0, 4), (1, 3)]


def test_plateau_across_the_delay_wrap():
    S = np.zeros((1, 12))
    S[0, [11, 0, 1]] = 2.0
    got = D.detect(S, [5.0], 4, 0, 1)
    assert [(x[2], x[3]) for x in got] == [(0, 0)]          # the lowest flat index of the plateau, though it wraps
    got = D.detect(S, [5.0], 4, 0, 0)
    assert [(x[2], x[3]) for x in got] == [(0, 0), (0, 1), (0, 11)]


def test_equal_peaks_in_different_rows_order_by_flat_index():
    S = np.zeros((5, 16))
    S[3, 2] = S[1, 9] = S[4, 12] = 7.0
    got = D.detect(S, np.arange(5.0), 8, 1, 1)
    assert [(x[2], x[3]) for x in got] == [(1, 9), (3, 2), (4, 12)]
    got = D.detect(S, np.arange(5.0), 8, 1, 8)              # (4, 12) now sees (3, 2)'s equal value at a lower index
    assert [(x[2], x[3]) for x in got] == [(1, 9), (3, 2)]


def test_nan_never_detected_and_never_blocks():
    S = np.zeros((3, 8))
    S[1, 4] = 3.0
    S[1, 5] = np.nan
    S[0, 4] = np.nan
    got = D.detect(S, [0.0, 1.0, 2.0], 8, 1, 1)
    assert [(x[2], x[3]) for x in got] == [(1, 4)]
    assert got[0][4] == -4.0                                # NaN neighbour: no delay fit (cell 4 of 8 is lag -4)
    assert D.detect(np.full((2, 5), np.nan), [0.0, 1.0], 4, 1, 1) == []


def test_edge_rows_single_row_and_small_n():
    S = np.array([[0.0, 1.0, 3.0, 2.0], [0.0, 0.0, 1.0, 0.0], [4.0, 0.0, 0.0, 1.0]])
    got = D.detect(S, [10.0, 20.0, 40.0], 8, 1, 1)
    assert [(x[2], x[3]) for x in got] == [(2, 0), (0, 2)]
    for x in got:
        assert x[5] == x[1]                                 # first / last row: no Doppler fit
    one = D.detect(S[:1], [7.0], 8, 5, 1)                   # d = 1: a guard beyond the rows is clipped
    assert [(x[2], x[3]) for x in one] == [(0, 2)] and one[0][5] == 7.0
    two = D.detect(np.array([[1.0, 2.0]]), [0.0], 4, 0, 0)  # n = 2: no delay fit; cell 1 is lag -1
    assert [(x[3], x[4]) for x in two] == [(1, -1.0), (0, 0.0)]


def test_k_max_truncates_then_min_ratio_drops():
    S = np.zeros((1, 40))
    S[0, [2, 10, 18, 26, 34]] = [1.0, 9.0, 5.0, 0.5, 2.0]
    got = D.detect(S, [0.0], 3, 0, 1)
    assert [x[0] for x in got] == [9.0, 5.0, 2.0]
    got = D.detect(S, [0.0], 5, 0, 1, min_ratio=2.0 / 9.0)
    assert [x[0] for x in got] == [9.0, 5.0, 2.0]           # 2 >= 9 * 2/9 stays; 1 and 0.5 go
    got = D.detect(S, [0.0], 5, 0, 1, min_ratio=1.0)
    assert [x[0] for x in got] == [9.0]
    assert D.padded(got, 3) == [got[0], D.NONE, D.NONE] and D.NONE[2] == UMAX


def test_exact_parabola_recovers_the_offset():
    """Samples of a downward parabola: the fit returns its vertex to rounding, in delay and in a non-uniform grid."""
    n, k0, dk = 64, 60, 0.3137
    ks = np.arange(n, dtype=float)
    S = np.zeros((5, n))
    r0, dr = 2, -0.2719
    for r in range(5):
        S[r] = 100.0 - (ks - (k0 + dk)) ** 2 - 3.0 * (r - (r0 + dr)) ** 2
    S[S < 0] = 0.0
    f = np.array([-3.0, -1.0, 0.5, 2.0, 6.0])
    x = D.detect(S, f, 1, 1, 2)[0]
    assert (x[2], x[3]) == (r0, k0)
    assert abs(x[4] - (k0 - n + dk)) <= 1e-12 * n           # cell 60 of 64 is lag -4
    assert abs(x[5] - (f[r0] + dr * (f[r0] - f[r0 - 1]))) <= 1e-12 * 6.0


def test_fixture_refinement_is_sub_cell():
    """The oracle surfaces of the ten fixtures on their test.rs grids, guard 1 x 1: the refined detection 0 lands within
    0.01 Hz of the offset in the file name and 0.01 sample of the planted lag (it is within 0.004 of both)."""
    from oracle import np_oracle as N
    cases = json.load(open(os.path.join(GOLDEN, "known_answers.json")))["cases"]
    seen = set()
    for case in cases:
        if case["haystack"] in seen:
            continue
        seen.add(case["haystack"])
        needle, hay, shifts = load_case(case)
        S, pidx, pval = N.caf_surface(needle, hay, shifts, 48000)
        m = re.search(r"T\+(\d+)samp_F([+-][\d.]+)Hz", case["haystack"])
        x = D.detect(S, shifts, 4, 1, 1)[0]
        assert (x[3], x[1]) == (int(pidx[x[2]]), float(shifts[int(np.argmax(pval))]))   # == find_peak
        assert abs(x[4] - int(m.group(1))) <= 0.01, case["haystack"]
        assert abs(x[5] - float(m.group(2))) <= 0.01, case["haystack"]
    assert len(seen) == 10


def test_detection_record_layout():
    assert C.sizeof(_lib.Detection) == 48
    assert [f[0] for f in _lib.Detection._fields_][:4] == [f[0] for f in _lib.Peak._fields_]


def test_null_surface_and_null_handle_are_rejected():
    lib = _lib.load()
    out = (_lib.Detection * 4)()
    cnt = C.c_size_t(123)
    assert lib.caf_b200_surface_detect(None, 4, 1, 1, 0.0, out, C.byref(cnt)) == -1
    assert cnt.value == 123
    assert lib.caf_b200_detect_f64_dev(None, None, 1, 4, 8, None, 4, 1, 1, 0.0, None, None) == -1
    assert lib.caf_b200_detect_f32_dev(None, None, 1, 4, 8, None, 4, 1, 1, 0.0, None, None) == -1


def test_cli_rejects_bad_detection_arguments(tmp_path):
    """tools/caf_cli: --detect / --guard-* / --min-db that are not numbers in range exit with 2 before any GPU work."""
    import shutil
    import subprocess
    from conftest import ROOT
    gxx = shutil.which("g++")
    assert gxx, "g++ is required for the CLI"
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = str(tmp_path / "caf_cli")
    subprocess.check_call([gxx, "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tools", "caf_cli.cpp"),
                           "-o", exe, "-L", so_dir, "-lcaf_b200", f"-Wl,-rpath,{so_dir}"])
    for bad in (["--detect", "abc"], ["--detect", "-1"], ["--detect", "0"], ["--detect", "1025"], ["--detect", "4x"],
                ["--detect", "4", "--guard-doppler", "33"], ["--detect", "4", "--guard-delay", "-2"],
                ["--detect", "4", "--min-db", "x"], ["--detect", "4", "--min-db", "-3"]):
        res = subprocess.run([exe, "a.c64", "b.c64"] + bad, capture_output=True, text=True)
        assert res.returncode == 2 and "caf_cli:" in res.stderr, (bad, res.returncode, res.stderr)
