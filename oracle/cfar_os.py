"""Reference OS-CFAR detector for caf_b200_surface_detect_cfar_os / caf_b200_detect_cfar_os_*_dev and the noise map of
caf_b200_cfar_os_noise_*_dev -- TEST INFRASTRUCTURE ONLY.

Numpy restatement of the contract (include/caf_b200.h, DESIGN.md section 11).  Training cells, m and N are CA-CFAR's
(oracle/cfar.py); only the noise estimate differs:

  each training value is widened to double and +0.0 is added (-0.0 counts as +0.0); k_m = ceil(rank * m / N) in integers;
  noise = the k_m-th smallest of the m values (NaN when m = 0).  An order statistic is one of the values, so np.sort
  gives the library's bits.
  detection: a local maximum under detect's rule with (gr, gd), m > 0 and v > scale * noise; ordered, cut and refined as
  in CA-CFAR.

Records are CA-CFAR's: detect's six fields plus (noise, train_cells = m).
"""
from __future__ import annotations

import math

import numpy as np

from .cfar import NONE, _finish, cell_training, padded, train_cells  # noqa: F401  (NONE, padded: re-exported)
from .detect import local_maxima


def rank_of(rank: int, m, n_train: int):
    """k_m = ceil(rank * m / N) in integers (m a scalar or an int64 array)."""
    return (rank * np.asarray(m, dtype=np.int64) + n_train - 1) // n_train


def _offsets(gr: int, gd: int, tr: int, tc: int):
    """(dr, j) of the training cells, row-major, without the guard block"""
    R, C = gr + tr, gd + tc
    dr, j = np.meshgrid(np.arange(-R, R + 1), np.arange(-C, C + 1), indexing="ij")
    keep = ~((np.abs(dr) <= gr) & (np.abs(j) <= gd))
    return dr[keep], j[keep]


def os_noise_at(S, rr, kk, gr: int, gd: int, tr: int, tc: int, rank: int, chunk_values: int = 1 << 24):
    """(noise, m) of the cells (rr[i], kk[i]) of a surface S [d, n]: each cell's training values gathered, NaN for a
    clipped row, sorted (NaN last), and the k_m-th taken."""
    S = np.asarray(S)
    d, n = S.shape
    v = S.astype(np.float64) + 0.0
    dr, dj = _offsets(gr, gd, tr, tc)
    N = train_cells(gr, gd, tr, tc)
    rr = np.asarray(rr, dtype=np.int64)
    kk = np.asarray(kk, dtype=np.int64)
    noise = np.full(rr.size, np.nan)
    m = np.zeros(rr.size, dtype=np.int64)
    step = max(1, chunk_values // max(1, dr.size))
    for a in range(0, rr.size, step):
        r2 = rr[a:a + step, None] + dr[None, :]
        k2 = (kk[a:a + step, None] + dj[None, :]) % n
        inside = (r2 >= 0) & (r2 < d)
        vals = np.where(inside, v[np.clip(r2, 0, d - 1), k2], np.nan)
        mm = np.sum(~np.isnan(vals), axis=1)
        vals.sort(axis=1)
        km = rank_of(rank, mm, N)
        got = vals[np.arange(vals.shape[0]), np.maximum(km, 1) - 1]
        noise[a:a + step] = np.where(mm > 0, got, np.nan)
        m[a:a + step] = mm
    return noise, m


def os_noise_map(S, gr: int, gd: int, tr: int, tc: int, rank: int):
    """(noise [d, n] float64, m [d, n] int64) of a surface S [d, n]."""
    S = np.asarray(S)
    d, n = S.shape
    rr, kk = np.divmod(np.arange(d * n, dtype=np.int64), n)
    noise, m = os_noise_at(S, rr, kk, gr, gd, tr, tc, rank)
    return noise.reshape(d, n), m.reshape(d, n)


def detect_cfar_os(S, freqs_hz, k_max: int, guard_doppler: int = 1, guard_delay: int = 1, train_doppler: int = 2,
                   train_delay: int = 16, rank: int = 1, scale: float = 1.0):
    """The noise is computed at the local maxima only, so config-1 surfaces stay quick."""
    S = np.asarray(S)
    if S.size == 0:
        return []
    gr, gd = guard_doppler, guard_delay
    rr, kk = np.nonzero(local_maxima(S, gr, gd))
    noise, m = os_noise_at(S, rr, kk, gr, gd, train_doppler, train_delay, rank)
    v = S[rr, kk].astype(np.float64)
    with np.errstate(invalid="ignore"):
        ok = (m > 0) & (v > scale * noise)
    return _finish(S, freqs_hz, rr[ok], kk[ok], noise[ok], m[ok], k_max)


def noise_os_brute(S, r: int, k: int, gr: int, gd: int, tr: int, tc: int, rank: int):
    """(noise, m) of one cell, one value at a time."""
    vals = sorted(x + 0.0 for row in cell_training(S, r, k, gr, gd, tr, tc) for x in row)
    m = len(vals)
    if m == 0:
        return math.nan, 0
    N = train_cells(gr, gd, tr, tc)
    return vals[(rank * m + N - 1) // N - 1], m


def detect_cfar_os_brute(S, freqs_hz, k_max: int, guard_doppler: int = 1, guard_delay: int = 1, train_doppler: int = 2,
                         train_delay: int = 16, rank: int = 1, scale: float = 1.0):
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
            noise, m = noise_os_brute(S, r, k, gr, gd, train_doppler, train_delay, rank)
            if m > 0 and v > scale * noise:
                rr.append(r)
                kk.append(k)
                nz.append(noise)
                mm.append(m)
    return _finish(S, freqs_hz, np.array(rr, dtype=np.int64), np.array(kk, dtype=np.int64), nz, mm, k_max)
