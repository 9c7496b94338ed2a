"""Reference detector for caf_b200_surface_detect / caf_b200_detect_*_dev -- TEST INFRASTRUCTURE ONLY.

Vectorised numpy restatement of the detection contract (include/caf_b200.h, DESIGN.md section 9):

  window of (r, k): rows r' in [r - gr, r + gr] clipped to [0, d), cells (k + j) mod n for |j| <= gd, minus (r, k).
  (r, k) with value v is a local maximum when v > 0, no window cell u > v, and no window cell u == v has a smaller flat
  index r' * n + k'.  NaN cells never qualify and never block.
  Order by value descending, then flat index ascending; keep the first k_max; drop those below min_ratio x the first.
  Refinement in double: 3-point parabola in delay (wrapping, none when n < 3) and in Doppler (interior rows only), each
  offset clamped to +-0.5, zero where a - 2v + b >= 0; freq_hz_interp is piecewise linear in the grid.

`detect` returns a list of records (value, freq_hz, doppler_idx, delay_idx, lag_samples, freq_hz_interp), count long.
`detect_brute` is the same contract as a per-cell loop, for testing `detect` itself.
"""
from __future__ import annotations

import numpy as np

NONE = (0.0, 0.0, (1 << 64) - 1, 0, 0.0, 0.0)


def local_maxima(S, guard_doppler: int, guard_delay: int) -> np.ndarray:
    """Boolean [d, n] mask of the local maxima of S under the window rule."""
    S = np.asarray(S)
    d, n = S.shape
    v = S.astype(np.float64)
    flat = np.arange(d * n, dtype=np.int64).reshape(d, n)
    with np.errstate(invalid="ignore"):
        mask = v > 0                                           # False for NaN
    for dr in range(-guard_doppler, guard_doppler + 1):
        lo, hi = max(0, -dr), min(d, d - dr)                   # rows r with r + dr inside the surface
        if lo >= hi:
            continue
        for j in range(-guard_delay, guard_delay + 1):
            if dr == 0 and j == 0:
                continue
            u = np.roll(v[lo + dr:hi + dr], -j, axis=1)        # u[r, k] = v[r + dr, (k + j) mod n]
            fu = np.roll(flat[lo + dr:hi + dr], -j, axis=1)
            with np.errstate(invalid="ignore"):
                blocked = (u > v[lo:hi]) | ((u == v[lo:hi]) & (fu < flat[lo:hi]))   # NaN compares False
            mask[lo:hi] &= ~blocked
    return mask


def _fit(a: float, v: float, b: float) -> float:
    den = a - 2.0 * v + b
    if not den < 0.0:
        return 0.0
    return min(max(0.5 * (a - b) / den, -0.5), 0.5)


def refine(S, freqs_hz, r: int, k: int):
    """The record of cell (r, k)."""
    d, n = S.shape
    v = float(S[r, k])
    dk = _fit(float(S[r, (k - 1) % n]), v, float(S[r, (k + 1) % n])) if n >= 3 else 0.0
    df = _fit(float(S[r - 1, k]), v, float(S[r + 1, k])) if 0 < r < d - 1 else 0.0
    f = float(freqs_hz[r])
    if df > 0.0:
        fi = f + df * (float(freqs_hz[r + 1]) - f)
    elif df < 0.0:
        fi = f + df * (f - float(freqs_hz[r - 1]))
    else:
        fi = f
    lag = (k if 2 * k < n else k - n) + dk
    return (v, f, int(r), int(k), float(lag), float(fi))


def _finish(S, freqs_hz, rr, kk, k_max: int, min_ratio: float):
    d, n = S.shape
    vals = S[rr, kk].astype(np.float64)
    order = np.lexsort((rr.astype(np.int64) * n + kk, -vals))[:k_max]
    recs = [refine(S, freqs_hz, int(rr[i]), int(kk[i])) for i in order]
    if recs:
        bar = min_ratio * recs[0][0]
        recs = [x for x in recs if not x[0] < bar]
    return recs


def detect(S, freqs_hz, k_max: int, guard_doppler: int = 1, guard_delay: int = 1, min_ratio: float = 0.0):
    S = np.asarray(S)
    if S.size == 0:
        return []
    rr, kk = np.nonzero(local_maxima(S, guard_doppler, guard_delay))
    return _finish(S, freqs_hz, rr, kk, k_max, min_ratio)


def detect_brute(S, freqs_hz, k_max: int, guard_doppler: int = 1, guard_delay: int = 1, min_ratio: float = 0.0):
    """The contract cell by cell (slow; small surfaces only)."""
    S = np.asarray(S)
    d, n = S.shape
    rr, kk = [], []
    for r in range(d):
        for k in range(n):
            v = float(S[r, k])
            if not v > 0:
                continue
            ok = True
            for r2 in range(max(0, r - guard_doppler), min(d, r + guard_doppler + 1)):
                for j in range(-guard_delay, guard_delay + 1):
                    k2 = (k + j) % n
                    if (r2, k2) == (r, k):
                        continue
                    u = float(S[r2, k2])
                    if u > v or (u == v and r2 * n + k2 < r * n + k):
                        ok = False
            if ok:
                rr.append(r)
                kk.append(k)
    return _finish(S, freqs_hz, np.array(rr, dtype=np.int64), np.array(kk, dtype=np.int64), k_max, min_ratio)


def padded(recs, k_max: int):
    """What the library writes: the records, then "none" up to k_max."""
    return list(recs) + [NONE] * (k_max - len(recs))
