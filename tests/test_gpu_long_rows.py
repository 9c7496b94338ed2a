"""GPU parity for rows longer than 8192 delay cells (BASELINE config 3: 65 536 cells) — the four-step path.

Checker: the C oracle for power-of-two lengths, its numpy/pocketfft twin for the others (the C oracle's fallback for
non-power-of-two transforms is an O(n^2) long-double DFT, too slow at these sizes)."""
import numpy as np
import pytest

import caf_cookoff_b200 as caf
from caf_cookoff_b200 import api, generate as G
from conftest import FS, rel_max
from oracle import oracle as O
from surface_checks import (assert_indices_match_oracle, assert_peak_is_find_peak, assert_peak_matches_oracle,
                            assert_row_peaks_are_cells, oracle_surface, tol_of)

pytestmark = pytest.mark.gpu


def _pair(l, seed=0):
    p = G.pair(0, seed=seed, chirp_length=l)
    return G.as_inputs(p)


def _with_f32(values):
    """(value, variant) cases: complex128 under the value's own id, complex64 under "<value>-f32"."""
    return [pytest.param(v, var, id=str(v) if var is api._Variant else f"{v}-f32")
            for var in (api._Variant, api._Variant32) for v in values]


BASE = np.array([-50.0, 0.0, 12.5, 68.0, 69.25, 70.5])


# Every row class (one level: top radix 2, 4, 8, 16; two levels: 2, 4, 8) at a ragged l and at l = N/2, where every
# cell is an output cell and the gathers skip the remap into the 2l-cell layout.
@pytest.mark.parametrize("l,variant", _with_f32([4097, 5000, 8192, 10000, 16384, 20001, 32768, 40000, 65536, 65537,
                                                  100000, 131072, 200000, 262144, 300001, 524288]))
def test_long_rows_match_oracle(l, variant):
    """Surface, row peaks and peak against the oracle, on a grid that also holds a NaN shift (an all-NaN row that keeps
    (0, 0.0) and never wins) and an alias of the 69.25 Hz row (f + fs, which must give that row)."""
    needle, hay = _pair(l)
    tol, exact = tol_of(variant), variant.rdt == np.float64
    shifts = np.concatenate([BASE, [np.nan, BASE[4] + FS]])
    nan_row, fin = 6, [0, 1, 2, 3, 4, 5, 7]
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS, variant=variant)
    o = oracle_surface(needle, hay, BASE, FS)
    # the oracle on the kernel's grid: row 7 is row 4, the NaN row holds what find_peak sees there
    rows = [0, 1, 2, 3, 4, 5, 0, 4]
    osurf, opidx, opval = o[0][rows], np.asarray(o[1])[rows], np.asarray(o[2])[rows]
    osurf[nan_row], opidx[nan_row], opval[nan_row] = np.nan, 0, 0.0
    assert surf.shape == (8, 2 * l) and surf.dtype == variant.rdt
    assert np.isnan(surf[nan_row]).all() and (int(pidx[nan_row]), float(pval[nan_row])) == (0, 0.0)
    assert rel_max(surf[fin].astype(np.float64), osurf[fin]) <= tol
    assert rel_max(surf[7], surf[4]) <= tol
    assert_indices_match_oracle(pidx, osurf, opidx, fin, tol, exact)
    assert_row_peaks_are_cells(surf, pidx, pval, fin)
    assert_peak_is_find_peak(pk, shifts, pidx, pval)
    assert_peak_matches_oracle(pk, opidx, opval, tol, exact)
    # peak only: the surface is never materialised, the row peaks and the peak are the same bits
    _, pidx2, pval2, pk2 = caf.surface_arrays(needle, hay, shifts, FS, variant=variant, want_surface=False)
    assert np.array_equal(pidx2, pidx) and np.array_equal(pval2, pval)
    assert (pk2.value, pk2.freq_hz, pk2.doppler_idx, pk2.delay_idx) == (pk.value, pk.freq_hz, pk.doppler_idx, pk.delay_idx)


def test_config3_miniature_and_peak_only():
    """4096 doppler x 65536 delay is config 3; here 96 rows of the same row length."""
    needle, hay = _pair(32768)
    shifts = np.linspace(-100.0, 100.0, 96, endpoint=False)
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS)
    osurf, opidx, opval = O.caf_surface(needle, hay, shifts, FS)
    assert rel_max(surf, osurf) <= 1e-9
    assert np.array_equal(pidx, opidx)
    assert (pk.freq_hz, int(pk.delay_idx)) == O.find_peak(shifts, opidx, opval)
    # peak-only entry (surface never materialised) agrees
    _, pidx2, pval2, pk2 = caf.surface_arrays(needle, hay, shifts, FS, want_surface=False)
    assert np.array_equal(pidx2, pidx) and np.array_equal(pval2, pval)
    assert (pk2.freq_hz, pk2.delay_idx, pk2.doppler_idx) == (pk.freq_hz, pk.delay_idx, pk.doppler_idx)


def test_long_row_delay_and_doppler_properties():
    """The generator puts s1 `lag` samples and `foffset` Hz away from s0: the peak must land there."""
    p = G.pair(0, seed=3, chirp_length=65536)
    needle, hay = G.as_inputs(p)
    step = 0.5
    f0 = round(p.foffset_hz / step) * step
    shifts = np.array([f0 - step, f0, f0 + step])
    _, _, _, pk = caf.surface_arrays(needle, hay, shifts, FS, want_surface=False)
    assert int(pk.delay_idx) == p.lag
    assert pk.freq_hz == f0


def test_config5_row_length_peak_only():
    """BASELINE config 5 row length (2^20 delay cells), peak only: the surface is never materialised."""
    p = G.pair(0, seed=1, chirp_length=1 << 19)
    needle, hay = G.as_inputs(p)
    step = 0.25
    f0 = round(p.foffset_hz / step) * step
    shifts = np.array([f0 - step, f0, f0 + step, f0 + 2 * step])
    _, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS, want_surface=False)
    _, opidx, opval = O.caf_surface(needle, hay, shifts, FS, want_surface=False)
    assert np.array_equal(pidx, opidx)
    assert rel_max(pval, opval) <= 1e-9
    assert (pk.freq_hz, int(pk.delay_idx)) == O.find_peak(shifts, opidx, opval)
    assert abs(int(pk.delay_idx) - p.lag) <= 16     # the chirp's delay-doppler ridge moves the peak a few samples


def test_too_long_is_unsupported():
    z = np.zeros((1 << 19) + 1, dtype=complex)
    with pytest.raises(caf.CafError) as e:
        caf.surface_arrays(z, z, [0.0], FS)
    assert e.value.status == -3


@pytest.mark.parametrize("l,variant", _with_f32([8192, 131072]))
def test_long_rows_beyond_nyquist_and_non_finite_doppler(l, variant):
    """The long-row kernels have their own phasor (caf_large_spread_top / caf_large_spread2): shifts beyond fs/2 alias,
    a NaN or infinite shift poisons its row and never wins (mod.rs:55-60, 148-151) — one- and two-level rows."""
    needle, hay = _pair(l)
    tol, exact = tol_of(variant), variant.rdt == np.float64
    shifts = np.array([69.25, 69.25 + FS, np.nan, 69.25 - 2 * FS, np.inf, FS / 2.0])
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS, variant=variant)
    osurf, opidx, opval = O.caf_surface(needle, hay, shifts, FS)
    for r in (2, 4):
        assert np.isnan(osurf[r]).all() and np.isnan(surf[r]).all()
        assert (int(pidx[r]), float(pval[r])) == (0, 0.0) == (int(opidx[r]), float(opval[r]))
    fin = [0, 1, 3, 5]
    assert rel_max(surf[fin].astype(np.float64), osurf[fin]) <= tol
    pk_rows = [0, 1, 3]          # the fs/2 row holds rounding noise only (1e-9 of the maximum): its argmax is not defined
    assert_indices_match_oracle(pidx, osurf, opidx, pk_rows, tol, exact)
    assert_row_peaks_are_cells(surf, pidx, pval, fin)
    assert rel_max(surf[1], surf[0]) <= tol and rel_max(surf[3], surf[0]) <= tol
    assert_peak_is_find_peak(pk, shifts, pidx, pval)
    assert int(pk.doppler_idx) in pk_rows
    if exact:
        assert int(pk.delay_idx) == int(opidx[0])
    _, _, _, pk2 = caf.surface_arrays(needle, hay, shifts, FS, variant=variant, want_surface=False)
    assert (pk2.freq_hz, int(pk2.delay_idx), int(pk2.doppler_idx)) == (pk.freq_hz, int(pk.delay_idx), int(pk.doppler_idx))
