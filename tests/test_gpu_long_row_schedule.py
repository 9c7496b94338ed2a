"""Host-side scheduling of rows longer than 8192 cells (run_large_dev in caf_b200.cu): rows cut into chunks under a
scratch budget (CAF_B200_CHUNK_MB), chunks capped at 65 535 rows (grid.y), batches of pairs with H = FFT(haystack)/N
rebuilt per pair on a side stream, and pairs alternating on one handle.

Rows are independent and each unit's arithmetic does not depend on which chunk or warp group runs it, so every
schedule must give the same bits: the main checks are exact.  Each call's launch count proves how many chunks ran."""
import numpy as np
import pytest

import caf_cookoff_b200 as caf
from caf_cookoff_b200 import api, generate as G
from conftest import FS, rel_max
from oracle import np_oracle as NO
from surface_checks import (assert_indices_match_oracle, assert_peak_is_find_peak, assert_peak_matches_oracle,
                            assert_row_peaks_are_cells, oracle_surface, tol_of)

pytestmark = pytest.mark.gpu

DEFAULT_CHUNK_MB = 6144


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def chunks(l, d, chunk_mb, variant):
    """Row counts of the chunks run_large_dev cuts d rows of length l into, restated so that any change to the rule is a
    deliberate one: as many rows as fit the budget, then equal chunks rounded up to whole sets of rows (a set gives each
    of the core's 2 x SMs warp groups one 4096-point unit), at most 65 535 rows (grid.y)."""
    n = 16384
    while n < 2 * l:
        n *= 2
    row_bytes = np.dtype(variant.cdt).itemsize * n
    chunk = max(1, (chunk_mb << 20) // row_bytes)
    if chunk < d:
        upr, groups = n // 4096, 2 * _sm_count()
        sets = groups // upr if groups >= upr else 1
        nch = -(-d // chunk)
        chunk = -(-d // nch)
        chunk = -(-chunk // sets) * sets
    chunk = min(max(chunk, 1), d, 65535)
    return [min(chunk, d - off) for off in range(0, d, chunk)]


def launches(p, n_chunks):
    """Per pair: H (spread + core) and three launches per chunk (spread, core, gather); one peak launch per call."""
    return p * (2 + 3 * n_chunks) + 1


@pytest.fixture
def make_handle(monkeypatch):
    """Handles whose long-row scratch budget is `chunk_mb` (None: the default); all are closed after the test."""
    made = []

    def make(chunk_mb=None):
        if chunk_mb is None:
            monkeypatch.delenv("CAF_B200_CHUNK_MB", raising=False)
        else:
            monkeypatch.setenv("CAF_B200_CHUNK_MB", str(chunk_mb))
        made.append(api.Handle(0))
        return made[-1]

    yield make
    for h in made:
        h.close()


def _grid(p, d, step):
    """d shifts around the pair's doppler offset, so that the rows hold a real peak."""
    return round(p.foffset_hz) + step * (np.arange(d) - d // 2)


def _call(h, n_chunks, needle, hay, shifts, variant, want_surface=True):
    before = h.launch_count
    out = caf.surface_arrays(needle, hay, shifts, FS, variant=variant, want_surface=want_surface, handle=h)
    assert h.launch_count - before == launches(1, n_chunks)
    return out


def _same(a, b):
    """Bitwise equal (surface or None, row peak indices, row peak values, peak)."""
    assert (a[0] is None) == (b[0] is None)
    if a[0] is not None and not np.array_equal(a[0], b[0]):
        bad = np.nonzero((a[0] != b[0]).any(axis=1))[0]
        raise AssertionError(f"rows {bad[:8]} ({bad.size}) differ")
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    assert (a[3].value, a[3].freq_hz, a[3].doppler_idx, a[3].delay_idx) == (b[3].value, b[3].freq_hz, b[3].doppler_idx, b[3].delay_idx)


@pytest.mark.parametrize("variant,l,d,chunk_mb,want", [
    pytest.param(api._Variant, 32768, 40, 1, [18, 18, 4], id="f64-65536-full"),
    pytest.param(api._Variant32, 20001, 40, 1, [18, 18, 4], id="f32-65536-ragged"),
    pytest.param(api._Variant32, 100000, 10, 4, [4, 4, 2], id="f32-2^18-two-level"),
    pytest.param(api._Variant, 300001, 5, 16, [1, 1, 1, 1, 1], id="f64-2^20-one-row-chunks"),
])
def test_chunked_rows_give_the_one_chunk_bits(variant, l, d, chunk_mb, want, make_handle):
    """A small budget cuts the rows into several chunks, with a ragged last chunk, and every chunk reuses the gather's
    row tickets and partials (a ticket resets itself when its row is done).  Surface, row peaks and peak are the bits
    of the default budget, which runs one chunk; the first and last row of every chunk match the oracle."""
    p = G.pair(0, seed=2, chirp_length=l)
    needle, hay = G.as_inputs(p)
    shifts = _grid(p, d, 2.5)
    got_chunks = chunks(l, d, chunk_mb, variant)
    if _sm_count() == 148:                            # the chunk sizes listed above are those of a 148-SM B200
        assert got_chunks == want
    assert len(got_chunks) > 1 and chunks(l, d, DEFAULT_CHUNK_MB, variant) == [d]
    one = _call(make_handle(), 1, needle, hay, shifts, variant)
    cut = _call(make_handle(chunk_mb), len(got_chunks), needle, hay, shifts, variant)
    _same(cut, one)
    ends = sorted(set(np.cumsum([0] + got_chunks[:-1]).tolist() + (np.cumsum(got_chunks) - 1).tolist()))
    surf, pidx, pval, pk = cut
    osurf, opidx, opval = oracle_surface(needle, hay, shifts[ends], FS)
    tol, exact = tol_of(variant), variant.rdt == np.float64
    assert rel_max(surf[ends].astype(np.float64), osurf) <= tol
    assert_indices_match_oracle(pidx[ends], osurf, opidx, range(len(ends)), tol, exact)
    assert_row_peaks_are_cells(surf, pidx, pval, range(d))
    assert_peak_is_find_peak(pk, shifts, pidx, pval)


def test_chunk_cap_at_65535_rows(make_handle):
    """A budget that holds every row still runs at most 65 535 rows per chunk (grid.y of the one-level spread and
    gather): 65 537 rows become 65 535 + 2, against two equal chunks on the default budget.  Same row peaks and peak;
    the rows on both sides of the cut match the oracle.  (About 8.6 GB of scratch.)"""
    variant, l, d = api._Variant32, 8192, 65537
    needle, hay = G.as_inputs(G.pair(0, seed=0, chirp_length=l))
    shifts = np.linspace(-100.0, 100.0, d)
    capped, default = chunks(l, d, 9000, variant), chunks(l, d, DEFAULT_CHUNK_MB, variant)
    assert capped == [65535, 2] and len(default) == 2 and default != capped
    a = _call(make_handle(9000), len(capped), needle, hay, shifts, variant, want_surface=False)
    b = _call(make_handle(), len(default), needle, hay, shifts, variant, want_surface=False)
    _same(a, b)
    rows = [0, 65534, 65535, 65536]
    osurf, opidx, opval = NO.caf_surface(needle, hay, shifts[rows], FS, direct_phasor=True)
    _, pidx, pval, pk = a
    tol = tol_of(variant)
    assert rel_max(pval[rows].astype(np.float64), opval) <= tol
    assert_indices_match_oracle(pidx[rows], osurf, opidx, range(4), tol, False)
    assert_peak_is_find_peak(pk, shifts, pidx, pval)


@pytest.mark.parametrize("variant,l,d,chunk_mb", [
    pytest.param(api._Variant, 20001, 40, 1, id="f64-65536"),
    pytest.param(api._Variant32, 100000, 10, 4, id="f32-2^18"),
    pytest.param(api._Variant, 300001, 3, 16, id="f64-2^20"),
])
def test_long_row_batches_match_single_calls_and_oracle(variant, l, d, chunk_mb, make_handle):
    """P = 3 different pairs in one batch: H is rebuilt for every pair into the one buffer the cores read, while the
    main stream still works on the pair before.  Each pair is the bits of its own single call and matches the oracle;
    the same batch on a small budget (pairs x chunks) gives the same bits."""
    P = 3
    ps = list(G.pairs(seed=4, count=P, chirp_length=l))
    ins = [G.as_inputs(p) for p in ps]
    ns, hs = np.stack([x[0] for x in ins]), np.stack([x[1] for x in ins])
    shifts = _grid(ps[0], d, 2.5)
    tol, exact = tol_of(variant), variant.rdt == np.float64
    h = make_handle()
    before = h.launch_count
    batch = caf.batch_arrays(ns, hs, shifts, FS, variant=variant, want_surface=True, handle=h)
    assert h.launch_count - before == launches(P, 1)
    surf, pidx, pval, peaks = batch
    for i in range(P):
        single = _call(h, 1, ns[i], hs[i], shifts, variant)
        _same(single, (surf[i], pidx[i], pval[i], peaks[i]))
        osurf, opidx, opval = oracle_surface(ns[i], hs[i], shifts, FS)
        assert rel_max(surf[i].astype(np.float64), osurf) <= tol
        assert_indices_match_oracle(pidx[i], osurf, opidx, range(d), tol, exact)
        assert_row_peaks_are_cells(surf[i], pidx[i], pval[i], range(d))
        assert_peak_is_find_peak(peaks[i], shifts, pidx[i], pval[i])
        assert_peak_matches_oracle(peaks[i], opidx, opval, tol, exact)
        if exact:
            assert (peaks[i].freq_hz, int(peaks[i].delay_idx)) == NO.find_peak(shifts, opidx, opval)
    cut = chunks(l, d, chunk_mb, variant)
    assert len(cut) > 1
    hs_ = make_handle(chunk_mb)
    before = hs_.launch_count
    got = caf.batch_arrays(ns, hs, shifts, FS, variant=variant, want_surface=True, handle=hs_)
    assert hs_.launch_count - before == launches(P, len(cut))
    assert np.array_equal(got[0], surf) and np.array_equal(got[1], pidx) and np.array_equal(got[2], pval)
    for a, b in zip(got[3], peaks):
        assert (a.value, a.freq_hz, a.doppler_idx, a.delay_idx) == (b.value, b.freq_hz, b.doppler_idx, b.delay_idx)


@pytest.mark.parametrize("l,d", [pytest.param(20001, 12, id="one-level"), pytest.param(100000, 6, id="two-level")])
def test_alternating_long_row_pairs_never_see_a_stale_spectrum(l, d, make_handle):
    """The long-row twin of test_alternating_pairs_never_see_a_stale_haystack_spectrum: H of each call is built on a
    side stream into a buffer the previous call's cores read.  Calls rotate through three pairs on one handle, with
    changing row counts and with and without the surface, starting on fresh handles; every result is the bits of that
    pair's call on a handle of its own."""
    variant = api._Variant
    ps = list(G.pairs(seed=5, count=3, chirp_length=l))
    ins = [G.as_inputs(p) for p in ps]
    shifts = _grid(ps[0], d, 2.5)
    ref = [_call(make_handle(), 1, n, h, shifts, variant) for n, h in ins]
    for fresh in range(2):
        h = make_handle()
        for k in range(12):
            i = (k + fresh) % 3
            dk = d if k % 2 == 0 else d // 2
            want_surface = (k % 3 != 2)
            got = _call(h, 1, ins[i][0], ins[i][1], shifts[:dk], variant, want_surface=want_surface)
            if want_surface:
                assert np.array_equal(got[0], ref[i][0][:dk]), (fresh, k, i)
            assert np.array_equal(got[1], ref[i][1][:dk]) and np.array_equal(got[2], ref[i][2][:dk]), (fresh, k, i)
            assert_peak_is_find_peak(got[3], shifts[:dk], got[1], got[2])
            if dk == d:
                _same((None,) + got[1:], (None,) + ref[i][1:])
