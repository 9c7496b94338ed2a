"""Checks shared by the GPU parity tests: a kernel's row peaks and peak against its own surface (exact, no tolerance)
and against the oracle (the repository's tolerance, and an index rule that fits the precision)."""
import numpy as np

from oracle import np_oracle as NO
from oracle import oracle as O

TOL64 = 1e-9
TOL32 = 1e-4


def tol_of(variant):
    return TOL64 if variant.rdt == np.float64 else TOL32


def oracle_surface(needle, hay, shifts, fs):
    """The C oracle for power-of-two lengths, its numpy/pocketfft twin with the closed-form phasor otherwise (the C
    oracle's transform of other lengths is an O(n^2) long-double DFT, too slow for long rows)."""
    l = len(needle)
    if l & (l - 1) == 0:
        return O.caf_surface(needle, hay, shifts, fs)
    return NO.caf_surface(needle, hay, shifts, fs, direct_phasor=True)


def assert_row_peaks_are_cells(surf, pidx, pval, rows):
    """Each listed row's peak value is, bit for bit, the cell at its reported index, and that index is the first
    maximum of the row the kernel produced (mod.rs:148, strict >)."""
    rows = np.asarray(rows)
    idx = pidx[rows].astype(np.int64)
    assert np.array_equal(pval[rows], surf[rows, idx])
    assert np.array_equal(idx, np.argmax(surf[rows], axis=1))


def assert_peak_is_find_peak(pk, shifts, pidx, pval):
    """The fused peak is find_peak (mod.rs:31-42) over the kernel's own row peaks: the first row holding the maximum."""
    r = int(np.argmax(pval))
    assert pval[r] > 0
    assert (int(pk.doppler_idx), int(pk.delay_idx), pk.freq_hz, pk.value) == \
           (r, int(pidx[r]), float(shifts[r]), float(pval[r]))


def assert_indices_match_oracle(pidx, osurf, opidx, rows, tol, exact):
    """Row argmax against the oracle's on the listed rows (oracle arrays aligned with the kernel's rows).
    exact (fp64): equal on every listed row.  Otherwise (fp32): equal where the oracle's top cell of the row beats the
    row's best cell at any other index by more than 2 tol M, M the largest cell of the oracle surface -- cells closer
    than that may legitimately swap under the tolerance."""
    m = float(np.nanmax(osurf))
    for r in rows:
        o = int(opidx[r])
        if not exact:
            rest = np.delete(osurf[r], o)
            if osurf[r, o] - rest.max() <= 2.0 * tol * m:
                continue
        assert int(pidx[r]) == o, (r, int(pidx[r]), o)


def assert_peak_matches_oracle(pk, opidx, opval, tol, exact):
    """The peak's row is a maximal row of the oracle (exactly for fp64, within 2 tol of the maximum for fp32), and its
    delay is that row's oracle index (fp64; for fp32 the row index rule above covers it).  opval has 0.0 on rows that
    hold no peak (non-finite shifts), as find_peak sees them."""
    r = int(pk.doppler_idx)
    top = float(np.max(opval))
    if exact:
        assert opval[r] == top and int(pk.delay_idx) == int(opidx[r]), (r, float(opval[r]), top)
    else:
        assert opval[r] >= (1.0 - 2.0 * tol) * top, (r, float(opval[r]), top)
