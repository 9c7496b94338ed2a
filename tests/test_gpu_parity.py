"""GPU parity tests (run with `-m gpu` on a B200): the CUDA path, called through the C ABI, against the CPU oracle.

Tolerances (BASELINE.json north_star, with the metric fixed in SURVEY.md section 9 item 8):
  - peak delay and doppler indices: bit exact
  - fp64 surface:  max|gpu - oracle| / max(oracle) <= 1e-9   (measured ~2e-13, which is the reference's own
                   acc *= shift phasor-recursion drift; the GPU evaluates the phasor in closed form)
  - complex64 variant: <= 1e-4 (measured ~5e-7)
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import caf_cookoff_b200 as caf
from caf_cookoff_b200 import _lib, api
from conftest import DATA, FS, load_case, rel_max
from oracle import oracle as O
from surface_checks import (assert_indices_match_oracle, assert_peak_is_find_peak, assert_peak_matches_oracle,
                            assert_row_peaks_are_cells, tol_of)

pytestmark = pytest.mark.gpu

TOL64 = 1e-9
TOL32 = 1e-4

STRATEGIES = [caf.CafRustFFT, caf.CafRustFFTIter, caf.CafRustFFTRayon, caf.CafRustFFTIterRayon,
              caf.CafRustFFTThreads, caf.CafRustFFTThreadpool, caf.CafFFTW]


# ---------------------------------------------------------------------------------------------------------------
# caf_rust/tests/test.rs restated: same files, same grids, same assert_eq! on (freq, samp_idx)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("strategy", STRATEGIES, ids=lambda s: s.__name__)
def test_chirp0_every_strategy(strategy, known_answers):
    """test.rs:15-145 — chirp_0 through all seven strategy structs."""
    needle, hay, shifts = load_case(known_answers[0])
    surface = strategy.caf_surface(needle, hay, shifts, FS)
    freq, samp_idx = strategy.find_peak(surface)
    assert freq == 69.25
    assert samp_idx == 202


@pytest.mark.parametrize("k", range(1, 10))
def test_chirp1_to_9_threads(k, known_answers):
    """test.rs:148-317 — chirps 1..9 through CafRustFFTThreads."""
    case = known_answers[k]
    needle, hay, shifts = load_case(case)
    surface = caf.CafRustFFTThreads.caf_surface(needle, hay, shifts, FS)
    freq, samp_idx = caf.CafRustFFTThreads.find_peak(surface)
    assert freq == case["freq"]
    assert samp_idx == case["samp_idx"]
    # the fused GPU find_peak agrees with the host scan of the rows
    assert (surface.peak.freq_hz, int(surface.peak.delay_idx)) == (freq, samp_idx)


# ---------------------------------------------------------------------------------------------------------------
# surface values, row peaks, peak: GPU vs oracle
# ---------------------------------------------------------------------------------------------------------------
def test_surface_fp64_bench_shape(chirp0):
    """BASELINE config 1: 400 x 8192, complex128 / float64."""
    needle, hay = chirp0
    shifts = caf.bench_shifts()
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS)
    osurf, opidx, opval = O.caf_surface(needle, hay, shifts, FS)
    assert surf.shape == (400, 8192) and surf.dtype == np.float64
    assert rel_max(surf, osurf) <= TOL64
    assert np.array_equal(pidx, opidx)                      # bit exact indices
    assert rel_max(pval, opval) <= TOL64
    assert np.array_equal(pval, surf[np.arange(400), pidx.astype(np.int64)])   # the row peak IS a surface cell
    assert np.array_equal(pidx.astype(np.int64), np.argmax(surf, axis=1))      # ... and the FIRST maximum of its row
    assert (pk.freq_hz, int(pk.delay_idx), int(pk.doppler_idx)) == (69.0, 202, 338)
    assert O.find_peak(shifts, opidx, opval) == (pk.freq_hz, int(pk.delay_idx))
    assert pk.value == pval[338]


def test_surface_fp32_variant(chirp0):
    """BASELINE config 2: complex64 / float32 within 1e-4 of the fp64 oracle; peak indices identical here."""
    needle, hay = chirp0
    shifts = caf.bench_shifts()
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS, variant=api._Variant32)
    osurf, opidx, opval = O.caf_surface(needle, hay, shifts, FS)
    assert surf.dtype == np.float32
    assert rel_max(surf.astype(np.float64), osurf) <= TOL32
    assert (pk.freq_hz, int(pk.delay_idx)) == (69.0, 202)
    assert np.mean(pidx == opidx) > 0.99


def test_peak_only_entry_matches_surface_entry(chirp0):
    needle, hay = chirp0
    shifts = caf.gen_float_shifts(-100.0, 100.0, 0.25)
    assert caf.CafB200.caf_peak(needle, hay, shifts, FS) == (69.25, 202)
    assert caf.CafB200F32.caf_peak(needle, hay, shifts, FS) == (69.25, 202)


def test_host_inputs_in_one_block_scattered_or_adjacent_allocations(chirp0):
    """Small host calls move needle | haystack | freqs with ONE H2D copy: straight from the caller when the three sit
    back to back in one allocation, through the library's pinned staging block otherwise.  Two pinned allocations that
    merely happen to be adjacent must not be copied as one (a DMA may not span allocations): every placement gives the
    same bits."""
    import torch
    from caf_cookoff_b200 import bench_shifts
    needle, hay = chirp0
    freqs = bench_shifts()[:64].copy()
    lib = _lib.load()
    h = api.default_handle()
    L, D = needle.size, freqs.size

    def call(n_ptr, h_ptr, f_ptr):
        surf = np.empty((D, 2 * L)); pk = _lib.Peak()
        rc = lib.caf_b200_surface_f64(h.raw, n_ptr, h_ptr, L, f_ptr, D, FS, surf.ctypes.data, None, None, C.cast(C.byref(pk), C.c_void_p))
        assert rc == 0, lib.caf_b200_last_error()
        pk2 = _lib.Peak()
        assert lib.caf_b200_peak_f64(h.raw, n_ptr, h_ptr, L, f_ptr, D, FS, C.cast(C.byref(pk2), C.c_void_p)) == 0
        assert (pk.value, pk.freq_hz, pk.doppler_idx, pk.delay_idx) == (pk2.value, pk2.freq_hz, pk2.doppler_idx, pk2.delay_idx)
        return surf, (pk.value, pk.freq_hz, int(pk.doppler_idx), int(pk.delay_idx))

    ref = call(needle.ctypes.data, hay.ctypes.data, freqs.ctypes.data)                       # three pageable arrays
    # one pageable block
    blk = np.empty(2 * L * 16 + D * 8, dtype=np.uint8)
    blk[: L * 16] = needle.view(np.uint8); blk[L * 16: 2 * L * 16] = hay.view(np.uint8); blk[2 * L * 16:] = freqs.view(np.uint8)
    got = call(blk.ctypes.data, blk.ctypes.data + L * 16, blk.ctypes.data + 2 * L * 16)
    assert np.array_equal(got[0], ref[0]) and got[1] == ref[1]
    # one pinned block from the library
    pb = C.c_void_p()
    assert lib.caf_b200_host_alloc(C.byref(pb), blk.size) == 0
    C.memmove(pb.value, blk.ctypes.data, blk.size)
    got = call(pb.value, pb.value + L * 16, pb.value + 2 * L * 16)
    assert np.array_equal(got[0], ref[0]) and got[1] == ref[1]
    lib.caf_b200_host_free(pb)
    # separate pinned allocations (torch's caching allocator often hands out adjacent ones)
    tn, th, tf = (torch.from_numpy(x).pin_memory() for x in (needle, hay, freqs))
    got = call(tn.data_ptr(), th.data_ptr(), tf.data_ptr())
    assert np.array_equal(got[0], ref[0]) and got[1] == ref[1]


def test_kernel_side_input_pull_matches_the_copy_path(chirp0, monkeypatch):
    """Small single-pair host calls carry no H2D copy: the grid reads needle | haystack | freqs out of pinned host memory
    itself and meets on a device counter (caf_kernels.cuh, RowArgs::pull_*).  Against a handle created with
    CAF_B200_PULL=0 (cudaMemcpyAsync in front of the kernel) every shape gives the same bits -- grids of 2 ... 148 CTAs,
    blocks that need several rounds per CTA, byte counts that are no multiple of 16, complex64 -- call after call (the
    meeting point is a monotonic counter that has to stay in step with the launches)."""
    from caf_cookoff_b200 import bench_shifts
    needle, hay = chirp0
    monkeypatch.setenv("CAF_B200_PULL", "0")
    h_copy = api.Handle(0)
    monkeypatch.setenv("CAF_B200_PULL", "1")
    h_pull = api.Handle(0)
    shapes = [(4096, bench_shifts()), (4096, bench_shifts()[:2]), (1000, bench_shifts()[:3]), (17, np.linspace(-90, 90, 1777)),
              (4095, bench_shifts()[:149]), (4096, bench_shifts()[:147])]
    for rep in range(3):
        for l, shifts in shapes:
            for variant in (api._Variant, api._Variant32):
                want_surface = (rep == 0)
                a = caf.surface_arrays(needle[:l], hay[:l], shifts, FS, variant=variant, want_surface=want_surface, handle=h_copy)
                b = caf.surface_arrays(needle[:l], hay[:l], shifts, FS, variant=variant, want_surface=want_surface, handle=h_pull)
                if a[0] is not None and not np.array_equal(a[0], b[0]):
                    bad = np.nonzero((a[0] != b[0]).any(axis=1))[0]
                    raise AssertionError(f"l={l} d={shifts.size} {variant.sfx} rep={rep}: rows {bad[:8]} ({bad.size}) differ, "
                                         f"cells {int((a[0] != b[0]).sum())}, first cols {np.nonzero(a[0][bad[0]] != b[0][bad[0]])[0][:8]}")
                assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
                assert (a[3].value, a[3].freq_hz, a[3].doppler_idx, a[3].delay_idx) == (b[3].value, b[3].freq_hz, b[3].doppler_idx, b[3].delay_idx)
    # peak-only calls (the spin-wait path) keep the known answer of the pair
    lib = _lib.load()
    f = bench_shifts()
    for _ in range(20):
        pk = _lib.Peak()
        assert lib.caf_b200_peak_f64(h_pull.raw, needle.ctypes.data, hay.ctypes.data, needle.size, f.ctypes.data, f.size, FS,
                                     C.cast(C.byref(pk), C.c_void_p)) == 0
        assert (pk.freq_hz, int(pk.delay_idx)) == (69.0, 202)
    h_copy.close(); h_pull.close()


def test_alternating_pairs_never_see_a_stale_haystack_spectrum():
    """One pair over many CTAs: CTA 0 / CTA hprod1 publish H = FFT(haystack)/n through L2 and every other CTA picks it up
    behind a release/acquire flag.  A consumer that read the buffer too early would see the PREVIOUS call's H -- invisible
    to any test that repeats one pair.  Alternate different pairs on one handle (and start on fresh handles, whose buffer
    holds no H at all) and hold every surface to the batch kernel's bits (whole pairs per CTA, no hand-over)."""
    from caf_cookoff_b200 import bench_shifts
    from oracle import oracle as O
    cases = [c for c in json.load(open(os.path.join(os.path.dirname(__file__), "golden", "known_answers.json")))["cases"]][:4]
    pairs = []
    for c in cases:
        n = O.read_file_c64(os.path.join(DATA, "chirp_%d_raw.c64" % c["chirp"]))
        pairs.append((n, O.read_file_c64(os.path.join(DATA, c["haystack"]))[: n.size]))
    shifts = bench_shifts()
    ref = caf.batch_arrays(np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs]), shifts, FS, want_surface=True)
    for fresh in range(6):
        h = api.Handle(0)
        for k in range(12):
            i = (k + fresh) % len(pairs)
            want_surface = (k % 3 != 2)
            got = caf.surface_arrays(pairs[i][0], pairs[i][1], shifts if k % 2 == 0 else shifts[:147], FS,
                                     want_surface=want_surface, handle=h)
            d = shifts.size if k % 2 == 0 else 147
            if want_surface: assert np.array_equal(got[0], ref[0][i][:d]), (fresh, k, i)
            assert np.array_equal(got[1], ref[1][i][:d]) and np.array_equal(got[2], ref[2][i][:d]), (fresh, k, i)
        h.close()


def test_device_loader_matches_read_file_c64(tmp_path):
    """caf_b200_load_c64_dev_* (SURVEY section 8 f-2: pinned direct-to-device loader) against the host loader
    (utils.rs:10-35): same samples bit for bit, windows, complex64, error behaviour; and the *_dev entry point fed with the
    loaded samples gives the host call's bits."""
    from caf_cookoff_b200 import bench_shifts
    a, b = os.path.join(DATA, "chirp_0_raw.c64"), os.path.join(DATA, "chirp_0_T+202samp_F+69.25Hz.c64")
    host_a, host_b = caf.read_file_c64(a), caf.read_file_c64(b)
    dev_a = caf.read_file_c64_dev(a)
    assert dev_a.size == host_a.size and np.array_equal(dev_a.to_host(), host_a)
    dev_b = caf.read_file_c64_dev(b, 0, host_a.size)                      # main.rs:15: haystack truncated to the needle
    assert dev_b.size == host_a.size and np.array_equal(dev_b.to_host(), host_b[: host_a.size])
    win = caf.read_file_c64_dev(b, 100, 50)
    assert np.array_equal(win.to_host(), host_b[100:150])
    assert caf.read_file_c64_dev(b, host_b.size + 5, 0).size == 0
    f32 = caf.read_file_c64_dev(a, f32=True)
    assert f32.to_host().dtype == np.complex64 and np.array_equal(f32.to_host(), host_a.astype(np.complex64))
    with pytest.raises(caf.CafError) as ei:
        caf.read_file_c64_dev(str(tmp_path / "missing.c64"))
    assert ei.value.status == -8                                           # CAF_B200_EIO: io::Result Err in the reference
    odd = tmp_path / "odd.c64"; odd.write_bytes(b"\0" * 12)
    with pytest.raises(caf.CafError):
        caf.read_file_c64_dev(str(odd))
    # device-resident inputs through the *_dev entry point
    lib = _lib.load(); h = api.default_handle()
    shifts = bench_shifts(); D = shifts.size
    scratch = C.c_void_p()
    assert lib.caf_b200_dev_alloc(h.raw, D * 8 + 32 + D * 16, C.byref(scratch)) == 0
    assert lib.caf_b200_dev_upload(h.raw, scratch, shifts.ctypes.data, D * 8) == 0
    d_pk, d_rv, d_ri = scratch.value + D * 8, scratch.value + D * 8 + 32, scratch.value + D * 8 + 32 + D * 8
    assert lib.caf_b200_batch_f64_dev(h.raw, dev_a.ptr, dev_b.ptr, 1, dev_a.size, scratch, D, FS, None, d_rv, d_ri, d_pk) == 0
    pk = _lib.Peak(); rv = np.empty(D); ri = np.empty(D, dtype=np.uint64)
    assert lib.caf_b200_dev_download(h.raw, C.byref(pk), d_pk, 32) == 0
    assert lib.caf_b200_dev_download(h.raw, rv.ctypes.data, d_rv, D * 8) == 0 and lib.caf_b200_dev_download(h.raw, ri.ctypes.data, d_ri, D * 8) == 0
    want = caf.surface_arrays(host_a, host_b[: host_a.size], shifts, FS, want_surface=False)
    assert np.array_equal(ri, want[1]) and np.array_equal(rv, want[2])
    assert (pk.value, pk.freq_hz, pk.doppler_idx, pk.delay_idx) == (want[3].value, want[3].freq_hz, want[3].doppler_idx, want[3].delay_idx)
    assert (pk.freq_hz, int(pk.delay_idx)) == (69.0, 202)
    lib.caf_b200_dev_free(scratch)


def test_overlapping_launches_give_the_serialised_bits():
    """caf_b200_set_overlap: a single-pair device launch that directly follows another one and shares no buffer with the
    seven launches before it (where either side writes) does not wait for the grid before it; in modes 2..4 it also
    uses only a half / third / quarter of the SMs so that several launches share the GPU.  Launch-private state (H
    publication buffer and flags, the find_peak ticket) lives in a ring indexed by launch number.  Over a long mixed
    sequence -- rotating pairs, three surface buffers (so every fourth launch aliases and must serialise), grids of
    2 / 7 / 147 CTAs that never overlap, and launches that deliberately reuse their predecessor's outputs -- every row
    peak, every peak and the final content of every surface buffer equals what the same sequence gives with overlap off,
    in every mode."""
    import torch
    from caf_cookoff_b200 import bench_shifts
    from oracle import oracle as O
    cases = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "known_answers.json")))["cases"][:4]
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    lib = _lib.load()
    h = api.Handle(0, stream=stream.cuda_stream)
    L = 4096
    nd, hd = [], []
    for c in cases:
        n = O.read_file_c64(os.path.join(DATA, "chirp_%d_raw.c64" % c["chirp"]))
        nd.append(torch.from_numpy(n).to(dev)); hd.append(torch.from_numpy(O.read_file_c64(os.path.join(DATA, c["haystack"]))[:L].copy()).to(dev))
    shifts = bench_shifts()
    fd = torch.from_numpy(shifts).to(dev)
    K = 72
    plan = []
    for k in range(K):
        d = (400, 147, 7, 300, 148, 2)[k % 6]
        alias_prev = (k % 9 == 5)                      # same surface buffer and peak slot as the launch before: must serialise
        plan.append((k % len(cases), d, alias_prev))

    def run(overlap, nbuf=3):
        lib.caf_b200_set_overlap(h.raw, int(overlap))
        surfs = [torch.zeros((400, 2 * L), dtype=torch.float64, device=dev) for _ in range(nbuf)]
        rv = torch.zeros((K, 400), dtype=torch.float64, device=dev); ri = torch.zeros((K, 400), dtype=torch.int64, device=dev)
        pk = torch.zeros((K, 4), dtype=torch.int64, device=dev)
        with torch.cuda.stream(stream):
            sb, slot = 0, 0
            for k, (pi, d, alias_prev) in enumerate(plan):
                if not alias_prev:
                    sb, slot = (sb + 1) % nbuf, k
                rc = lib.caf_b200_batch_f64_dev(h.raw, nd[pi].data_ptr(), hd[pi].data_ptr(), 1, L, fd.data_ptr(), d, FS,
                                                surfs[sb].data_ptr(), rv[slot].data_ptr(), ri[slot].data_ptr(), pk[slot].data_ptr())
                assert rc == 0, lib.caf_b200_last_error()
        torch.cuda.synchronize()
        return [s_.cpu().numpy() for s_ in surfs], rv.cpu().numpy(), ri.cpu().numpy(), pk.cpu().numpy()

    want = run(0)
    for rep, mode in enumerate((1, 2, 3, 4, 4)):
        got = run(mode)
        for a_, b_ in zip(want[0], got[0]):
            assert np.array_equal(a_, b_), rep
        assert np.array_equal(want[1], got[1]) and np.array_equal(want[2], got[2]) and np.array_equal(want[3], got[3]), rep
    # nine surface buffers: no launch aliases any of the seven before it, the overlap runs as deep as the mode allows
    want9 = run(0, 9)
    for mode in (1, 4, 4):
        got = run(mode, 9)
        for a_, b_ in zip(want9[0], got[0]):
            assert np.array_equal(a_, b_), mode
        assert np.array_equal(want9[1], got[1]) and np.array_equal(want9[2], got[2]) and np.array_equal(want9[3], got[3]), mode
    # and the serialised reference itself is the known answer of each pair on the full grid
    for k, (pi, d, alias_prev) in enumerate(plan):
        if d == 400 and not alias_prev and not (k + 1 < K and plan[k + 1][2]):
            w = want[3][k]
            assert int(w.view(np.uint64)[3]) == cases[pi]["samp_idx"] and abs(float(w.view(np.float64)[1]) - cases[pi]["freq"]) <= 0.5
    lib.caf_b200_set_overlap(h.raw, 0)
    h.close()


def test_stress_bitwise_determinism_over_many_launches(chirp0):
    """compute-sanitizer is closed on this GPU pool (profiles/r02_sanitizer.txt), so the hand-rolled synchronisation of
    the row kernel -- named barriers per warp group, the mailbox mbarrier pair, the cross-CTA H publication flag, the
    last-CTA-done ticket, group 1 folding group 0's candidates -- is held to the strongest black-box property a race
    would break: every one of many launches, over shapes that change the rows per CTA (1, 2-3, dozens) and the pair
    boundaries inside a CTA, returns bit-identical surfaces, row peaks and peaks, equal to the oracle-checked first."""
    from caf_cookoff_b200 import bench_shifts
    needle, hay = chirp0
    for shifts in (bench_shifts(), bench_shifts()[:148], bench_shifts()[:7], np.linspace(-100, 100, 1777, endpoint=False)):
        ref = caf.surface_arrays(needle, hay, shifts, FS)
        for _ in range(25):
            got = caf.surface_arrays(needle, hay, shifts, FS)
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])
            assert (got[3].value, got[3].doppler_idx, got[3].delay_idx) == (ref[3].value, ref[3].doppler_idx, ref[3].delay_idx)
    # batches: pair boundaries fall inside CTAs; peaks only (the fused path) and with surfaces
    ns = np.stack([needle, needle[::-1].copy(), needle * 0.5]); hs = np.stack([hay, hay, hay[::-1].copy()])
    ref = caf.batch_arrays(ns, hs, bench_shifts()[:200], FS, want_surface=True)
    for k in range(15):
        got = caf.batch_arrays(ns, hs, bench_shifts()[:200], FS, want_surface=(k % 2 == 0))
        assert np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])
        assert got[0] is None or np.array_equal(got[0], ref[0])
        assert [(q.value, q.doppler_idx, q.delay_idx) for q in got[3]] == [(q.value, q.doppler_idx, q.delay_idx) for q in ref[3]]


def test_repeated_calls_are_deterministic(chirp0):
    needle, hay = chirp0
    shifts = caf.bench_shifts()
    a = caf.surface_arrays(needle, hay, shifts, FS)
    b = caf.surface_arrays(needle, hay, shifts, FS)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


@pytest.mark.parametrize("l,variant", [pytest.param(l, v, id=str(l) if v is api._Variant else f"{l}-f32")
                                       for v in (api._Variant, api._Variant32) for l in (1, 2, 3, 17, 100, 1000, 2048, 4095, 4096)])
def test_ragged_lengths(l, variant, chirp0):
    """Any input length up to 4096 (the reference plans any n): same 2l-cell layout, same peaks, in both precisions."""
    needle, hay = chirp0
    n, h = needle[:l], hay[:l]
    tol, exact = tol_of(variant), variant.rdt == np.float64
    shifts = np.array([-99.5, -3.25, 0.0, 68.75, 69.25, 70.0])
    surf, pidx, pval, pk = caf.surface_arrays(n, h, shifts, FS, variant=variant)
    osurf, opidx, opval = O.caf_surface(n, h, shifts, FS)
    assert surf.shape == (6, 2 * l) and surf.dtype == variant.rdt
    if osurf.max() > 0:
        assert rel_max(surf.astype(np.float64), osurf) <= tol
    assert_row_peaks_are_cells(surf, pidx, pval, range(6))
    if l >= 100:            # (tiny inputs have near-tied cells; index equality is only meaningful with a real peak)
        assert_indices_match_oracle(pidx, osurf, opidx, range(6), tol, exact)
        assert_peak_is_find_peak(pk, shifts, pidx, pval)
        assert_peak_matches_oracle(pk, opidx, opval, tol, exact)


def test_random_inputs_and_odd_grid():
    rng = np.random.default_rng(2024)
    l = 4096
    needle = rng.normal(size=l) + 1j * rng.normal(size=l)
    hay = np.roll(needle, 37) * np.exp(2j * np.pi * 12.3 * np.arange(l) / FS) + 0.1 * (rng.normal(size=l) + 1j * rng.normal(size=l))
    shifts = np.array([12.3, -7.0, 1e-3, 250.75, 12.25, -12.3, 0.0])      # unsorted, fractional, large
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS)
    osurf, opidx, opval = O.caf_surface(needle, hay, shifts, FS)
    assert rel_max(surf, osurf) <= TOL64
    assert np.array_equal(pidx, opidx)
    assert (pk.freq_hz, int(pk.delay_idx)) == O.find_peak(shifts, opidx, opval) == (12.3, 37)


def test_doppler_beyond_nyquist_and_extreme_sample_rates():
    """`fs` is any u32 and `freq_shift` any f64 (mod.rs:46-65): shifts at and beyond fs/2 alias, fs = 1 and fs = 2^32 - 1
    are legal.  The kernel reduces the phase n*f/fs exactly; the reference rounds 2*pi*f*(1/fs) once and accumulates
    it, so the two drift apart by ~n*eps*|f/fs| -- far inside 1e-9 for the values here."""
    rng = np.random.default_rng(77)
    l = 4096
    needle = rng.normal(size=l) + 1j * rng.normal(size=l)
    hay = np.roll(needle, 37) * np.exp(2j * np.pi * 12.3 * np.arange(l) / FS)
    aliases = [12.3, 12.3 + FS, 12.3 - FS]
    shifts = np.array(aliases + [FS / 2.0, 30000.0, float(FS), -95987.7])
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS)
    osurf, opidx, opval = O.caf_surface(needle, hay, shifts, FS)
    assert rel_max(surf, osurf) <= TOL64
    assert np.array_equal(pidx, opidx)
    assert int(pk.delay_idx) == 37 and pk.freq_hz in aliases + [-95987.7]      # the aliased rows tie to rounding
    assert rel_max(surf[1], surf[0]) <= TOL64 and rel_max(surf[2], surf[0]) <= TOL64
    assert rel_max(surf[5], O.caf_surface(needle, hay, np.array([0.0]), FS)[0][0]) <= TOL64   # f = fs is no shift
    for fs, grid in ((1, [0.0, 0.25, -0.5, 0.125]), (4294967295, [1.0e6, -2.5e8, 3.0e9])):
        x = rng.normal(size=1000) + 1j * rng.normal(size=1000)
        y = np.roll(x, 5) * np.exp(2j * np.pi * grid[1] * np.arange(1000) / fs)
        g = np.array(grid)
        s2, i2, v2, p2 = caf.surface_arrays(x, y, g, fs)
        o2, oi2, ov2 = O.caf_surface(x, y, g, fs)
        assert rel_max(s2, o2) <= TOL64
        assert np.array_equal(i2, oi2)
        assert (p2.freq_hz, int(p2.delay_idx)) == O.find_peak(g, oi2, ov2) == (grid[1], 5)
        assert rel_max(caf.CafB200.apply_freq_shift(x, grid[1], fs), O.apply_freq_shift(x, grid[1], fs)) <= 1e-10


def test_non_finite_doppler_rows_never_win(chirp0):
    """A NaN or infinite `freq_shift` makes the reference's phasor NaN (from_polar, mod.rs:55-60): every cell of that
    row is NaN, no cell passes the strict `>` (mod.rs:148-151), the row keeps (0, 0.0) and find_peak skips it."""
    needle, hay = chirp0
    shifts = np.array([np.nan, 69.0, np.inf, -np.inf, 69.25])
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS)
    osurf, opidx, opval = O.caf_surface(needle, hay, shifts, FS)
    for r in (0, 2, 3):
        assert np.isnan(osurf[r]).all() and (int(opidx[r]), float(opval[r])) == (0, 0.0)
        assert np.isnan(surf[r]).all() and (int(pidx[r]), float(pval[r])) == (0, 0.0)
    for r in (1, 4):
        assert rel_max(surf[r], osurf[r]) <= TOL64 and pidx[r] == opidx[r]
    assert (pk.freq_hz, int(pk.delay_idx), int(pk.doppler_idx)) == (69.25, 202, 4) == O.find_peak(shifts, opidx, opval) + (4,)
    assert caf.CafB200.caf_peak(needle, hay, shifts, FS) == (69.25, 202)
    assert caf.CafB200.caf_peak(needle, hay, np.array([np.nan, np.inf]), FS) == (0.0, 0)     # nothing beats the dummy row


def test_non_finite_and_aliased_doppler_in_complex64_and_in_batches(chirp0):
    """The same two edge cases through the complex64 rows (phase still fp64) and through the batch path, whose
    find_peak is a separate kernel over the row peaks."""
    needle, hay = chirp0
    shifts = np.array([np.nan, 69.0, np.inf, 69.25 + FS, 69.25])
    osurf, opidx, opval = O.caf_surface(needle, hay, shifts, FS)
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS, variant=api._Variant32)
    for r in (0, 2):
        assert np.isnan(surf[r]).all() and (int(pidx[r]), float(pval[r])) == (0, 0.0)
    fin = [1, 3, 4]
    assert rel_max(surf[fin].astype(np.float64), osurf[fin]) <= TOL32
    assert np.array_equal(pidx[fin], opidx[fin])
    assert int(pk.delay_idx) == 202 and pk.freq_hz in (69.25, 69.25 + FS)
    ns, hs = _pairs(3)
    bs, bi, bv, peaks = caf.batch_arrays(ns, hs, shifts, FS, want_surface=True)
    for i in range(3):
        o, oi, ov = O.caf_surface(ns[i], hs[i], shifts, FS)
        assert np.isnan(bs[i][0]).all() and np.isnan(bs[i][2]).all()
        assert rel_max(bs[i][fin], o[fin]) <= TOL64
        assert np.array_equal(bi[i], oi) and bv[i][0] == 0.0 and bv[i][2] == 0.0
        assert int(peaks[i].delay_idx) == O.find_peak(shifts, oi, ov)[1]
        assert int(peaks[i].doppler_idx) in (1, 3, 4)


def test_ties_first_row_wins_and_argmax_is_first_maximum(chirp0):
    """mod.rs:37 keeps the first maximal row (strict >): identical rows are bitwise identical on the GPU, so the
    first of them must win.  mod.rs:148 keeps the first maximal cell of a row: the reported index must be the first
    maximum of the row the kernel itself produced (np.argmax returns the first maximum).  (Cells that are only
    mathematically equal are not a parity criterion: their last bits depend on the FFT factorisation, in the
    reference's two backends as much as here.)"""
    needle, hay = chirp0
    shifts = np.array([69.0, 12.0, 69.0, 69.0, -5.0])
    surf, pidx, pval, pk = caf.surface_arrays(needle, hay, shifts, FS)
    assert np.array_equal(surf[0], surf[2]) and np.array_equal(surf[0], surf[3])
    assert (int(pk.doppler_idx), int(pk.delay_idx), pk.value) == (0, 202, pval[0])
    assert np.array_equal(pidx.astype(np.int64), np.argmax(surf, axis=1))
    # a two-tap haystack produces two cells of (nearly) equal height; whatever their last bits, the index reported
    # must be the first maximum of the produced row
    l = 4096
    n2 = np.zeros(l, dtype=complex); n2[0] = 1.0
    h2 = np.zeros(l, dtype=complex); h2[300] = 2.0; h2[900] = 2.0
    s2, p2, v2, _ = caf.surface_arrays(n2, h2, [0.0, 3.0], FS)
    assert np.array_equal(p2.astype(np.int64), np.argmax(s2, axis=1))
    assert abs(s2[0][300] - 4.0) < 1e-12 and abs(s2[0][900] - 4.0) < 1e-12
    assert set(int(x) for x in p2) <= {300, 900}


def test_all_zero_and_empty_inputs():
    z = np.zeros(4096, dtype=complex)
    surf, pidx, pval, pk = caf.surface_arrays(z, z, [1.0, 2.0], FS)
    assert not surf.any() and list(pidx) == [0, 0] and list(pval) == [0.0, 0.0]
    assert (pk.value, pk.freq_hz, int(pk.delay_idx), int(pk.doppler_idx)) == (0.0, 0.0, 0, api.UINT64_MAX)
    assert caf.CafB200.find_peak(caf.CafB200.caf_surface(z, z, [1.0, 2.0], FS)) == (0.0, 0)
    # no doppler rows: empty surface, find_peak's dummy row
    rows = caf.CafB200.caf_surface(z, z, [], FS)
    assert len(rows) == 0 and caf.CafB200.find_peak(rows) == (0.0, 0)
    # empty signals: empty rows (mod.rs:143-144 defaults), and the iterator variants panic on xcor_mag[0]
    rows = caf.CafRustFFT.caf_surface(z[:0], z[:0], [1.0], FS)
    assert len(rows) == 1 and rows[0].xcor_mag.size == 0 and rows[0].xcor_peak_idx == 0 and rows[0].xcor_peak_val == 0.0
    with pytest.raises(caf.CafPanic):
        caf.CafRustFFTIterRayon.caf_surface(z[:0], z[:0], [1.0], FS)


@pytest.mark.parametrize("l", [1000, 4096, 5000])
def test_nan_sample_never_wins(l):
    """One NaN sample reaches every cell of every row through the transforms.  `val > max` is false for NaN, so each
    row keeps xcor_peak_idx = 0, xcor_peak_val = 0.0 (mod.rs:143-150) and find_peak returns its dummy row
    (mod.rs:32-41) -- on short rows, on ragged lengths and on the long-row kernels alike."""
    rng = np.random.default_rng(l)
    needle = rng.standard_normal(l) + 1j * rng.standard_normal(l)
    hay = rng.standard_normal(l) + 1j * rng.standard_normal(l)
    freqs = np.array([-3.0, 0.0, 7.5])
    for poisoned in ("needle", "haystack"):
        n2, h2 = needle.copy(), hay.copy()
        (n2 if poisoned == "needle" else h2)[l // 3] = complex(np.nan, 0.0)
        surf, pidx, pval, pk = caf.surface_arrays(n2, h2, freqs, FS)
        assert np.isnan(surf).all()
        assert list(pidx) == [0, 0, 0] and list(pval) == [0.0, 0.0, 0.0]
        assert (pk.value, pk.freq_hz, int(pk.delay_idx), int(pk.doppler_idx)) == (0.0, 0.0, 0, api.UINT64_MAX)
        if l == 4096:   # (the oracle's O(n^2) long-double DFT for other lengths is x87 code: minutes on NaN operands)
            osurf, opidx, opval = O.caf_surface(n2, h2, freqs, FS)
            assert np.isnan(osurf).all() and list(opidx) == [0, 0, 0] and list(opval) == [0.0, 0.0, 0.0]
            assert O.find_peak(freqs, opidx, opval) == (0.0, 0)
        assert caf.CafB200.find_peak(caf.CafB200.caf_surface(n2, h2, freqs, FS)) == (0.0, 0)


def test_length_errors_and_unsupported_sizes():
    z = np.zeros(16, dtype=complex)
    with pytest.raises(caf.CafPanic):
        caf.CafB200.caf_surface(z, z[:15], [0.0], FS)
    big = (1 << 19) + 1
    with pytest.raises(caf.CafError) as e:
        caf.Xcor.new(big).run(np.zeros(big, complex), np.zeros(big, complex))
    assert e.value.status == -3      # CAF_B200_EUNSUPPORTED: rows longer than 2^20 cells are not built


# ---------------------------------------------------------------------------------------------------------------
# apply_freq_shift and Xcor
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 7, 4096, 8192, 100000])
def test_apply_freq_shift(n):
    rng = np.random.default_rng(n)
    x = rng.normal(size=n) + 1j * rng.normal(size=n)
    got = caf.CafB200.apply_freq_shift(x, 77.77, FS)          # caf_bench.rs:171-179
    want = O.apply_freq_shift(x, 77.77, FS)
    assert got.shape == want.shape
    if n:
        assert rel_max(got, want) <= (1e-9 if n > 8192 else 1e-11)   # the reference recursion itself drifts ~n*eps
    assert np.array_equal(caf.CafB200.apply_shift(x, 0.0, FS), x)


def test_apply_freq_shift_f32():
    rng = np.random.default_rng(5)
    x = (rng.normal(size=4096) + 1j * rng.normal(size=4096)).astype(np.complex64)
    got = caf.CafB200F32.apply_freq_shift(x, -31.5, FS)
    assert got.dtype == np.complex64
    assert rel_max(got.astype(np.complex128), O.apply_freq_shift(x, -31.5, FS)) <= 1e-6


@pytest.mark.parametrize("n", [4097, 5000, 16384, 20000, 40000, 70001, 140000, 1 << 19])
def test_xcor_any_length(n):
    """Xcor::new(n) plans any n (RustFFT): lengths other than 8192 and <= 4096 go through one row of the long-row kernels
    (complex cells) and a fold of the linear correlation.  Checked against numpy's FFT form of xcor_rustfft.rs:58-76
    (the C oracle's DFT for non-power-of-two n is O(n^2)) and, for the power of two, against the C oracle.  The lengths
    reach every long-row class (top radix 2, 4, 8, 16; two levels 2, 4, 8), in complex128 and complex64."""
    rng = np.random.default_rng(n)
    a = rng.normal(size=n) + 1j * rng.normal(size=n)
    b = rng.normal(size=n) + 1j * rng.normal(size=n)
    want = np.fft.ifft(np.fft.fft(a) * np.conj(np.fft.fft(b)) / n) * n
    got = caf.Xcor.new(n).run(a, b)
    assert got.shape == (n,) and rel_max(got, want) <= 1e-12
    if n == 16384:
        assert rel_max(got, O.xcor(a, b)) <= 1e-12
    got32 = api.XcorF32.new(n).run(a.astype(np.complex64), b.astype(np.complex64))
    assert got32.dtype == np.complex64 and rel_max(got32.astype(np.complex128), want) <= 1e-5


@pytest.mark.parametrize("n", [1, 2, 37, 1000, 4096, 8192])
def test_xcor(n):
    """Xcor::run — circular correlation, 1/n on the product, unnormalised transforms."""
    rng = np.random.default_rng(n + 1)
    a = rng.normal(size=n) + 1j * rng.normal(size=n)
    b = rng.normal(size=n) + 1j * rng.normal(size=n)
    x = caf.Xcor.new(n)
    assert rel_max(x.run(a, b), O.xcor(a, b)) <= 1e-12
    assert rel_max(x.clone().run(b, a), O.xcor(b, a)) <= 1e-12
    a32, b32 = a.astype(np.complex64), b.astype(np.complex64)       # the complex64 twin (kXcorFull / kXcorHalf, float)
    got32 = api.XcorF32.new(n).run(a32, b32)
    assert got32.dtype == np.complex64 and rel_max(got32.astype(np.complex128), O.xcor(a32, b32)) <= 1e-5
    with pytest.raises(caf.CafPanic):
        x.run(a, b[:-1]) if n > 1 else x.run(a, np.zeros(2, complex))


def test_xcor_surface_consistency(chirp0):
    """A surface row is |Xcor::run(haystack_padded, shifted_needle_padded)|^2 (mod.rs:138-147)."""
    needle, hay = chirp0
    f = 69.0
    npad = np.concatenate([needle, np.zeros(4096)]); hpad = np.concatenate([hay, np.zeros(4096)])
    shifted = caf.CafB200.apply_freq_shift(npad, f, FS)
    res = caf.Xcor.new(8192).run(hpad, shifted)
    row = res.real ** 2 + res.imag ** 2
    surf, _, _, _ = caf.surface_arrays(needle, hay, [f], FS)
    assert rel_max(surf[0], row) <= 1e-12


# ---------------------------------------------------------------------------------------------------------------
# batches, sharding, size-independent properties at the full BASELINE size
# ---------------------------------------------------------------------------------------------------------------
def _pairs(k):
    names = sorted(os.listdir(DATA))
    ns, hs = [], []
    for i in range(k):
        ns.append(O.read_file_c64(os.path.join(DATA, f"chirp_{i}_raw.c64")))
        hs.append(O.read_file_c64(os.path.join(DATA, [n for n in names if n.startswith(f"chirp_{i}_T")][0]))[:4096])
    return np.stack(ns), np.stack(hs)


def test_batch_of_pairs_matches_single_calls_and_oracle():
    """BASELINE config 4 in miniature: independent pairs, one shared grid, more pairs than fit one CTA's range; in
    complex128 and complex64."""
    ns, hs = _pairs(10)
    shifts = caf.gen_float_shifts(-100.0, 100.0, 5.0)          # 40 rows
    oracle = [O.caf_surface(ns[i], hs[i], shifts, FS) for i in range(10)]
    for variant in (api._Variant, api._Variant32):
        tol, exact = tol_of(variant), variant.rdt == np.float64
        surf, pidx, pval, peaks = caf.batch_arrays(ns, hs, shifts, FS, variant=variant, want_surface=True)
        assert surf.shape == (10, 40, 8192) and surf.dtype == variant.rdt
        for i in range(10):
            osurf, opidx, opval = oracle[i]
            assert rel_max(surf[i].astype(np.float64), osurf) <= tol
            assert_indices_match_oracle(pidx[i], osurf, opidx, range(40), tol, exact)
            assert_row_peaks_are_cells(surf[i], pidx[i], pval[i], range(40))
            assert_peak_is_find_peak(peaks[i], shifts, pidx[i], pval[i])
            assert_peak_matches_oracle(peaks[i], opidx, opval, tol, exact)
            s1, p1, v1, k1 = caf.surface_arrays(ns[i], hs[i], shifts, FS, variant=variant)
            assert np.array_equal(s1, surf[i]) and np.array_equal(p1, pidx[i])      # batching does not change a bit


def test_many_pairs_peaks_only():
    ns, hs = _pairs(10)
    big_n = np.tile(ns, (40, 1)); big_h = np.tile(hs, (40, 1))   # 400 pairs > 148 CTAs
    shifts = caf.gen_float_shifts(-100.0, 100.0, 12.5)           # 16 rows
    _, pidx, pval, peaks = caf.batch_arrays(big_n, big_h, shifts, FS, want_surface=False)
    for i in range(400):
        assert np.array_equal(pidx[i], pidx[i % 10])
        assert peaks[i].delay_idx == peaks[i % 10].delay_idx and peaks[i].freq_hz == peaks[i % 10].freq_hz


def test_row_sharding_with_packed_peak_resolution(chirp0):
    """SURVEY.md 8(e): doppler rows sharded over ranks + packed maxloc == the unsharded find_peak."""
    needle, hay = chirp0
    shifts = caf.gen_float_shifts(-100.0, 100.0, 0.25)          # 800 rows
    _, _, _, whole = caf.surface_arrays(needle, hay, shifts, FS, want_surface=False)
    for world in (2, 3, 8):
        bounds = [len(shifts) * r // world for r in range(world + 1)]
        words = []
        for r in range(world):
            lo, hi = bounds[r], bounds[r + 1]
            _, _, _, pk = caf.surface_arrays(needle, hay, shifts[lo:hi], FS, want_surface=False)
            words.append(api.peak_pack(pk, lo))
        out = api.peak_resolve(np.stack(words))
        assert (out.value, out.freq_hz, out.doppler_idx, out.delay_idx) == \
               (whole.value, whole.freq_hz, whole.doppler_idx, whole.delay_idx)


def test_property_scaling_and_delay(chirp0):
    """Size-independent properties at the full 400 x 8192 shape: |xcor|^2 scales with |c|^2 of the haystack
    (bit exact for a power of two), and delaying the haystack by d samples moves every row peak by d."""
    needle, hay = chirp0
    shifts = caf.bench_shifts()
    s1, p1, v1, _ = caf.surface_arrays(needle, hay, shifts, FS)
    s2, p2, v2, _ = caf.surface_arrays(needle, 2.0 * hay, shifts, FS)
    assert np.array_equal(s2, 4.0 * s1) and np.array_equal(p1, p2)
    d = 5
    hay_d = np.concatenate([np.zeros(d), hay[:-d]])
    s3, p3, _, pk3 = caf.surface_arrays(needle, hay_d, shifts, FS)
    assert int(pk3.delay_idx) == 202 + d and pk3.freq_hz == 69.0
    core = slice(150, 350)       # rows whose peak is the true correlation peak, away from the truncated tail
    assert np.array_equal(p3[core].astype(np.int64), p1[core].astype(np.int64) + d)


def test_property_doppler_shift_moves_the_peak_row(chirp0):
    """Shifting the haystack by +10 Hz moves the doppler estimate by +10 Hz and leaves the delay alone."""
    needle, hay = chirp0
    shifts = caf.bench_shifts()
    hay10 = hay * np.exp(2j * np.pi * 10.0 * np.arange(hay.size) / FS)
    _, _, _, pk = caf.surface_arrays(needle, hay10, shifts, FS, want_surface=False)
    assert (pk.freq_hz, int(pk.delay_idx)) == (79.0, 202)


def test_native_library_is_what_ran():
    """The handle counts kernel launches: a surface call is exactly one fused launch of the sm_100a kernel."""
    h = caf.default_handle()
    before = h.launch_count
    z = np.ones(4096, dtype=complex)
    caf.surface_arrays(z, z, [0.0, 1.0], FS)
    assert h.launch_count - before == 1
    maps = open("/proc/self/maps").read()
    assert "libcaf_b200.so" in maps
