"""Reference CA-CFAR detector for caf_b200_surface_detect_cfar / caf_b200_detect_cfar_*_dev and the noise map of
caf_b200_cfar_noise_*_dev -- TEST INFRASTRUCTURE ONLY.

Numpy restatement of the contract (include/caf_b200.h, DESIGN.md section 10), with R = gr + tr and C = gd + tc:

  training cells of (r, k): rows r' in [r - R, r + R] clipped to [0, d), cells (k + j) mod n for |j| <= C, minus
  |r' - r| <= gr and |j| <= gd; NaN cells are skipped; m = how many remain.
  noise: per row, +0.0 plus its training cells in ascending j, in double; the cell, +0.0 plus the row sums in ascending
  r'; noise = sum / m (NaN when m = 0).  numpy's elementwise double add is IEEE, so `noise_map` (one np.roll per offset,
  accumulated in that order) gives the library's bits.  Adding +0.0 in place of a skipped NaN cell or a clipped row
  leaves every partial sum unchanged (none is -0.0), which is what lets the map be vectorised.
  detection: a local maximum under detect's rule with (gr, gd), m > 0 and v > scale * noise; ordered by value
  descending, then flat index ascending, cut to k_max; refined as in detect.

Records are detect's six fields plus (noise, train_cells).
"""
from __future__ import annotations

import math

import numpy as np

from .detect import local_maxima, refine

NONE = (0.0, 0.0, (1 << 64) - 1, 0, 0.0, 0.0, 0.0, 0)


def train_cells(gr: int, gd: int, tr: int, tc: int) -> int:
    """N = (2R+1)(2C+1) - (2gr+1)(2gd+1): the training cells of an interior cell without NaN."""
    return (2 * (gr + tr) + 1) * (2 * (gd + tc) + 1) - (2 * gr + 1) * (2 * gd + 1)


def scale_for_pfa(pfa: float, n_train: int) -> float:
    """alpha = N (Pfa^(-1/N) - 1): P(v > alpha * mean of N i.i.d. exponential cells) = Pfa for v of the same law."""
    return n_train * (pfa ** (-1.0 / n_train) - 1.0)


def noise_map(S, gr: int, gd: int, tr: int, tc: int):
    """(noise [d, n] float64, m [d, n] int64) of a surface S [d, n]."""
    S = np.asarray(S)
    d, n = S.shape
    v = S.astype(np.float64)
    finite = ~np.isnan(v)
    v0 = np.where(finite, v, 0.0)
    R, C = gr + tr, gd + tc
    # A row sum depends on (r', k) and on whether r' is a guard row of the cell, not on the cell's row otherwise: build
    # both kinds once, full[r', k] over j = -C ... C and side[r', k] over j = -C ... -gd-1, gd+1 ... C, each in ascending j.
    full = np.zeros((d, n))
    side = np.zeros((d, n))
    cfull = np.zeros((d, n), dtype=np.int64)
    cside = np.zeros((d, n), dtype=np.int64)
    for j in range(-C, C + 1):
        u = np.roll(v0, -j, axis=1)                            # u[r', k] = v[r', (k + j) mod n]
        c = np.roll(finite, -j, axis=1)
        full += u
        cfull += c
        if abs(j) > gd:
            side += u
            cside += c
    total = np.zeros((d, n))
    m = np.zeros((d, n), dtype=np.int64)
    for dr in range(-R, R + 1):                                # ascending r' = r + dr
        lo, hi = max(0, -dr), min(d, d - dr)                   # rows r with r + dr inside the surface
        if lo >= hi:
            continue
        guard = abs(dr) <= gr
        total[lo:hi] += (side if guard else full)[lo + dr:hi + dr]
        m[lo:hi] += (cside if guard else cfull)[lo + dr:hi + dr]
    with np.errstate(invalid="ignore", divide="ignore"):
        noise = np.where(m > 0, total / np.maximum(m, 1), np.nan)
    return noise, m


def _finish(S, freqs_hz, rr, kk, noise, m, k_max: int):
    d, n = S.shape
    vals = S[rr, kk].astype(np.float64)
    order = np.lexsort((rr.astype(np.int64) * n + kk, -vals))[:k_max]
    return [refine(S, freqs_hz, int(rr[i]), int(kk[i])) + (float(noise[i]), int(m[i])) for i in order]


def detect_cfar(S, freqs_hz, k_max: int, guard_doppler: int = 1, guard_delay: int = 1, train_doppler: int = 2,
                train_delay: int = 16, scale: float = 1.0):
    S = np.asarray(S)
    if S.size == 0:
        return []
    noise, m = noise_map(S, guard_doppler, guard_delay, train_doppler, train_delay)
    v = S.astype(np.float64)
    with np.errstate(invalid="ignore"):
        ok = local_maxima(S, guard_doppler, guard_delay) & (m > 0) & (v > scale * noise)
    rr, kk = np.nonzero(ok)
    return _finish(S, freqs_hz, rr, kk, noise[rr, kk], m[rr, kk], k_max)


def cell_training(S, r: int, k: int, gr: int, gd: int, tr: int, tc: int):
    """The training cells of (r, k) as a list of rows (ascending r'), each its non-NaN values in ascending j."""
    d, n = S.shape
    R, C = gr + tr, gd + tc
    rows = []
    for r2 in range(max(0, r - R), min(d, r + R + 1)):
        row = []
        for j in range(-C, C + 1):
            if abs(r2 - r) <= gr and abs(j) <= gd:
                continue
            x = float(S[r2, (k + j) % n])
            if not math.isnan(x):
                row.append(x)
        rows.append(row)
    return rows


def noise_brute(S, r: int, k: int, gr: int, gd: int, tr: int, tc: int):
    """(noise, m) of one cell, summed one value at a time in the contract's order."""
    total, m = 0.0, 0
    for row in cell_training(S, r, k, gr, gd, tr, tc):
        s = 0.0
        for x in row:
            s += x
        total += s
        m += len(row)
    return (total / m if m else math.nan), m


def detect_cfar_brute(S, freqs_hz, k_max: int, guard_doppler: int = 1, guard_delay: int = 1, train_doppler: int = 2,
                      train_delay: int = 16, scale: float = 1.0):
    """The contract cell by cell (slow; small surfaces only)."""
    S = np.asarray(S)
    d, n = S.shape
    gr, gd = guard_doppler, guard_delay
    rr, kk, nz, mm = [], [], [], []
    for r in range(d):
        for k in range(n):
            v = float(S[r, k])
            if not v > 0:
                continue
            ok = True
            for r2 in range(max(0, r - gr), min(d, r + gr + 1)):
                for j in range(-gd, gd + 1):
                    k2 = (k + j) % n
                    if (r2, k2) == (r, k):
                        continue
                    u = float(S[r2, k2])
                    if u > v or (u == v and r2 * n + k2 < r * n + k):
                        ok = False
            if not ok:
                continue
            noise, m = noise_brute(S, r, k, gr, gd, train_doppler, train_delay)
            if m > 0 and v > scale * noise:
                rr.append(r)
                kk.append(k)
                nz.append(noise)
                mm.append(m)
    return _finish(S, freqs_hz, np.array(rr, dtype=np.int64), np.array(kk, dtype=np.int64), nz, mm, k_max)


def padded(recs, k_max: int):
    """What the library writes: the records, then "none" up to k_max."""
    return list(recs) + [NONE] * (k_max - len(recs))
