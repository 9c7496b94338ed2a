"""Detection on row-sharded surfaces (caf_b200_detect_rows_*, caf_b200_detect_cfar_rows_*, caf_b200_detect_cfar_os_rows_*,
caf_b200_detect_merge_dev, caf_b200_cfar_merge_dev; include/caf_b200.h, DESIGN.md section 12), all on one GPU: every
rank's halo'd block is carved from (or computed like) the block a rank would hold, each is searched over its owned rows,
and the merge of the ranks' lists must be the whole-surface call's records and count, byte for byte."""
import ctypes as C

import numpy as np
import pytest

from caf_cookoff_b200 import _lib, api, bench_shifts
from caf_cookoff_b200.dist import _block_detect, shard_bounds
from conftest import FS

pytestmark = pytest.mark.gpu

WORLDS = (1, 2, 3, 8)
DET, CA, OS = "detect", "cfar", "cfar_os"


def dev():
    import torch
    return torch.device("cuda", 0)


def width(det):
    return 6 if det == DET else 8


def whole(det, S, freqs, k_max, w):
    """the one-GPU call on the whole surface S [d][n] (torch): (records bytes, count)"""
    import torch
    d, n = S.shape
    out = torch.full((k_max, width(det)), 7.0, dtype=torch.float64, device=dev())
    cnt = torch.full((1,), -1, dtype=torch.int64, device=dev())
    f32 = S.dtype == torch.float32
    args = (S.data_ptr(), 1, d, n, freqs.data_ptr(), k_max, out.data_ptr(), cnt.data_ptr())
    torch.cuda.synchronize()                  # the library's stream does not wait for torch's
    if det == DET:
        api.detect_dev(*args, guard_doppler=w["gr"], guard_delay=w["gd"], min_ratio=w.get("min_ratio", 0.0), f32=f32)
    elif det == CA:
        api.detect_cfar_dev(*args, scale=w["scale"], guard_doppler=w["gr"], guard_delay=w["gd"], train_doppler=w["tr"],
                            train_delay=w["tc"], f32=f32)
    else:
        api.detect_cfar_os_dev(*args, rank=w["rank"], scale=w["scale"], guard_doppler=w["gr"], guard_delay=w["gd"],
                               train_doppler=w["tr"], train_delay=w["tc"], f32=f32)
    torch.cuda.synchronize()
    return out.cpu().numpy().tobytes(), int(cnt.cpu()[0])


def rows_call(det, blk, freqs_blk, row_lo, row_hi, row_offset, d_global, k_max, w, out, cnt):
    """the block detector on blk [d_buf][n] (torch) into out [k_max][width] and cnt [1]"""
    d_buf, n = blk.shape
    args = (blk.data_ptr(), d_buf, n, freqs_blk.data_ptr(), row_lo, row_hi, row_offset, d_global, k_max, out.data_ptr(),
            cnt.data_ptr())
    f32 = str(blk.dtype) == "torch.float32"
    if det == DET:
        api.detect_rows_dev(*args, guard_doppler=w["gr"], guard_delay=w["gd"], min_ratio=w.get("min_ratio", 0.0), f32=f32)
    elif det == CA:
        api.detect_cfar_rows_dev(*args, scale=w["scale"], guard_doppler=w["gr"], guard_delay=w["gd"],
                                 train_doppler=w["tr"], train_delay=w["tc"], f32=f32)
    else:
        api.detect_cfar_os_rows_dev(*args, rank=w["rank"], scale=w["scale"], guard_doppler=w["gr"], guard_delay=w["gd"],
                                    train_doppler=w["tr"], train_delay=w["tc"], f32=f32)


def halo(det, w):
    return api.halo_rows(det, w["gr"], w.get("tr", 0))


def merge(det, lists, counts, k_max, w):
    import torch
    world = lists.shape[0]
    out = torch.full((k_max, width(det)), 7.0, dtype=torch.float64, device=dev())
    cnt = torch.full((1,), -1, dtype=torch.int64, device=dev())
    torch.cuda.synchronize()
    if det == DET:
        api.detect_merge_dev(lists.data_ptr(), counts.data_ptr(), world, k_max, out.data_ptr(), cnt.data_ptr(),
                             min_ratio=w.get("min_ratio", 0.0))
    else:
        api.cfar_merge_dev(lists.data_ptr(), counts.data_ptr(), world, k_max, out.data_ptr(), cnt.data_ptr())
    torch.cuda.synchronize()
    return out.cpu().numpy().tobytes(), int(cnt.cpu()[0])


def sharded(det, S, freqs, k_max, w, world, ret_ranks=False):
    """every rank's block carved from S with the halo, searched over its owned rows, then merged"""
    import torch
    d = S.shape[0]
    H = halo(det, w)
    lists = torch.full((world, k_max, width(det)), 3.0, dtype=torch.float64, device=dev())
    counts = torch.full((world,), -1, dtype=torch.int64, device=dev())
    torch.cuda.synchronize()
    for r in range(world):
        lo, hi = shard_bounds(d, world, r)
        b_lo, b_hi = max(lo - H, 0), min(hi + H, d)
        rows_call(det, S[b_lo:b_hi], freqs[b_lo:b_hi], lo - b_lo, hi - b_lo, b_lo, d, k_max, w, lists[r], counts[r:r + 1])
    torch.cuda.synchronize()
    res = merge(det, lists, counts, k_max, w)
    return (res, lists, counts) if ret_ranks else res


def check_all_worlds(det, S, freqs, k_max, w, worlds=WORLDS):
    want = whole(det, S, freqs, k_max, w)
    for world in worlds:
        got = sharded(det, S, freqs, k_max, w, world)
        assert got[1] == want[1], (det, world, got[1], want[1])
        assert got[0] == want[0], (det, world, "records differ")
    return want


def windows(det, gr, gd, tr=0, tc=0, scale=None, min_ratio=0.0):
    w = dict(gr=gr, gd=gd, tr=tr, tc=tc, min_ratio=min_ratio)
    if det != DET:
        N = api.cfar_train_cells(gr, gd, tr, tc)
        w["rank"] = (3 * N + 3) // 4
        w["scale"] = (api.cfar_scale(1e-6, N) if det == CA else api.cfar_os_scale(1e-6, N, w["rank"])) if scale is None \
            else scale
    return w


def surface_of(needle, hay, freqs_np, f32):
    """caf_b200_batch_*_dev of one pair over freqs_np: ([d][2l] tensor, freqs tensor)"""
    import torch
    cdt = torch.complex64 if f32 else torch.complex128
    nd = torch.from_numpy(np.asarray(needle)).to(dev(), cdt)
    hd = torch.from_numpy(np.asarray(hay)).to(dev(), cdt)
    fd = torch.from_numpy(np.ascontiguousarray(freqs_np, dtype=np.float64)).to(dev())
    l, d = nd.numel(), fd.numel()
    S = torch.empty((d, 2 * l), dtype=torch.float32 if f32 else torch.float64, device=dev())
    pk = torch.empty(4, dtype=torch.float64, device=dev())
    torch.cuda.synchronize()
    fn = getattr(_lib.load(), "caf_b200_batch_f32_dev" if f32 else "caf_b200_batch_f64_dev")
    assert fn(api.default_handle().raw, nd.data_ptr(), hd.data_ptr(), 1, l, fd.data_ptr(), d, FS, S.data_ptr(), None, None,
              pk.data_ptr()) == 0
    torch.cuda.synchronize()
    return S, fd, nd, hd


def planted(sigma=0.1):
    """the four emitters of the CFAR tests under complex noise"""
    rng = np.random.default_rng(7)
    N = 4096
    needle = np.hanning(N) * (rng.standard_normal(N) + 1j * rng.standard_normal(N)) / np.sqrt(2)
    hay = np.zeros(N, dtype=np.complex128)
    for lag, f, a in [(202, 69.0, 1.0), (57, -31.5, 0.5), (140, 12.0, 0.25), (90, -80.25, 0.15)]:
        x = np.concatenate([np.zeros(lag), needle])[:N]
        hay += a * x * np.exp(2j * np.pi * f * np.arange(N) / FS)
    hay += sigma * (rng.standard_normal(N) + 1j * rng.standard_normal(N))
    return needle, hay


def tensor(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev())


def grid(d):
    return tensor(np.linspace(-100.0, 100.0, d) + 0.125 * np.arange(d) ** 1.5)


# ---- 1. one GPU equals many, bit for bit ------------------------------------------------------------------------------
@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
def test_planted_scene_on_the_bench_grid(f32):
    """The planted scene on the 400-row bench grid: the default window, the delay-only window of the CFAR tests (guard 32,
    the largest row reach), a loose threshold that yields 64 detections, and detect's min_ratio."""
    needle, hay = planted()
    S, fd, _, _ = surface_of(needle, hay, bench_shifts(), f32)
    for det in (DET, CA, OS):
        for w, k in ((windows(det, 2, 2, 4, 16), 16), (windows(det, 32, 2, 0, 64), 8)):
            check_all_worlds(det, S, fd, k, w)
    check_all_worlds(CA, S, fd, 64, windows(CA, 1, 1, 2, 8, scale=1.5))
    check_all_worlds(OS, S, fd, 64, windows(OS, 1, 1, 2, 8, scale=1.5))
    check_all_worlds(DET, S, fd, 64, windows(DET, 2, 2, min_ratio=0.01))
    assert check_all_worlds(DET, S, fd, 1024, windows(DET, 1, 1))[1] == 1024


@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
@pytest.mark.parametrize("k_max", [1, 16, 1024])
def test_tie_heavy_integer_surfaces(f32, k_max):
    """Few distinct values: plateaus everywhere, equal values in every shard, and far more local maxima per shard than
    k_max.  Windows up to gr + tr = 32 (training rows reach past every shard of 8 ranks)."""
    rng = np.random.default_rng(3 + k_max)
    S = tensor(rng.integers(0, 4, (61, 300)).astype(np.float32 if f32 else np.float64))
    fd = grid(61)
    for det in (DET, CA, OS):
        for (gr, gd, tr, tc) in ((1, 1, 2, 3), (0, 0, 1, 1), (3, 2, 29, 5), (32, 4, 0, 8)):
            check_all_worlds(det, S, fd, k_max, windows(det, gr, gd, tr, tc, scale=0.9 if det != DET else None))


@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
def test_shards_narrower_than_the_halo(f32):
    """d = 20 rows over 8 ranks (2 or 3 rows each) with halos of 1 ... 12 rows: a block holds several neighbours' rows."""
    rng = np.random.default_rng(5)
    S = tensor(rng.exponential(1.0, (20, 512)).astype(np.float32 if f32 else np.float64))
    fd = grid(20)
    for det in (DET, CA, OS):
        for (gr, gd, tr, tc) in ((1, 1, 2, 4), (4, 2, 8, 6), (2, 0, 0, 3)):
            check_all_worlds(det, S, fd, 32, windows(det, gr, gd, tr, tc, scale=1.2 if det != DET else None), (8, 3))


@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
def test_long_rows(f32):
    """n = 65 536 cells per row, a few dozen rows."""
    rng = np.random.default_rng(9)
    S = tensor(rng.exponential(1.0, (36, 65536)).astype(np.float32 if f32 else np.float64))
    fd = grid(36)
    for det in (DET, CA, OS):
        check_all_worlds(det, S, fd, 64, windows(det, 2, 2, 4, 16, scale=3.0 if det != DET else None), (2, 3, 8))


# ---- 2. blocks computed from sub-grids ------------------------------------------------------------------------------
@pytest.mark.parametrize("f32", [False, True], ids=["f64", "f32"])
@pytest.mark.parametrize("l", [4096, 32768], ids=["bench", "long"])
def test_blocks_from_sub_grids_equal_carved_blocks(f32, l):
    """A rank's block computed over its halo'd sub-grid equals the same rows of the whole surface bit for bit, and the
    path dist.detect_sharded runs per rank (_block_detect) merges into the whole-surface answer."""
    import torch
    rng = np.random.default_rng(11)
    needle = np.hanning(l) * (rng.standard_normal(l) + 1j * rng.standard_normal(l))
    hay = np.concatenate([np.zeros(77), needle])[:l] * np.exp(2j * np.pi * 31.0 * np.arange(l) / FS)
    hay = hay + 0.05 * (rng.standard_normal(l) + 1j * rng.standard_normal(l))
    freqs = bench_shifts()[150:210] if l == 4096 else np.linspace(-40.0, 40.0, 24)
    S, fd, nd, hd = surface_of(needle, hay, freqs, f32)
    d = freqs.size
    for det, w in ((DET, windows(DET, 2, 2)), (CA, windows(CA, 2, 2, 4, 16)), (OS, windows(OS, 2, 2, 4, 16))):
        H = halo(det, w)
        for world in (3, 8):
            lists = torch.empty((world, 16, width(det)), dtype=torch.float64, device=dev())
            counts = torch.empty(world, dtype=torch.int64, device=dev())
            for r in range(world):
                lo, hi = shard_bounds(d, world, r)
                b_lo, b_hi = max(lo - H, 0), min(hi + H, d)
                blk, _, _, _ = surface_of(needle, hay, freqs[b_lo:b_hi], f32)
                assert torch.equal(blk, S[b_lo:b_hi])
                out, cnt = _block_detect(det, nd, hd, fd, FS, 16, world, r, guard_doppler=w["gr"], guard_delay=w["gd"],
                                         train_doppler=w["tr"], train_delay=w["tc"], os_rank=w.get("rank"),
                                         scale=w.get("scale"), min_ratio=0.0, handle=None)
                lists[r] = out
                counts[r] = cnt[0]
            torch.cuda.synchronize()
            assert merge(det, lists, counts, 16, w) == whole(det, S, fd, 16, w)


# ---- 3. boundaries ----------------------------------------------------------------------------------------------------
def records(raw, det):
    a = np.frombuffer(raw, dtype=np.float64).reshape(-1, width(det))
    return [(float(x[0]), int(x[2:4].view(np.uint64)[0]), int(x[2:4].view(np.uint64)[1])) for x in a]


def test_plateau_across_a_shard_boundary_is_one_detection():
    """A plateau on the last owned row of rank 0 and the first of rank 1 is one detection: its lowest flat index."""
    S = np.zeros((16, 256))
    S[7, 100:103] = 5.0
    S[8, 100:103] = 5.0
    S, fd = tensor(S), grid(16)
    for det in (DET, CA, OS):
        w = windows(det, 1, 1, 2, 3, scale=1.0)
        raw, cnt = check_all_worlds(det, S, fd, 8, w, (2,))
        assert cnt == 1 and records(raw, det)[0] == (5.0, 7, 100)


def test_equal_values_in_different_shards_come_out_in_flat_order():
    S = np.zeros((24, 128))
    for r, k in ((20, 5), (2, 50), (10, 20), (10, 90), (15, 3)):
        S[r, k] = 7.0
    S[12, 60] = 9.0
    S, fd = tensor(S), grid(24)
    for det in (DET, CA, OS):
        raw, cnt = check_all_worlds(det, S, fd, 8, windows(det, 1, 1, 1, 2, scale=1.0))
        got = [(r, k) for _, r, k in records(raw, det)[:cnt]]
        assert got == [(12, 60), (2, 50), (10, 20), (10, 90), (15, 3), (20, 5)]


def test_min_ratio_is_cut_against_the_global_first():
    """Rank 1 holds the global first (100); rank 0's 60 survives, its 40 passes rank 0's own cut (30) but not the
    global one (50)."""
    S = np.zeros((16, 128))
    S[2, 10], S[4, 40], S[6, 70] = 60.0, 40.0, 10.0
    S[12, 20] = 100.0
    S, fd = tensor(S), grid(16)
    w = windows(DET, 1, 1, min_ratio=0.5)
    (raw, cnt), lists, counts = sharded(DET, S, fd, 8, w, 2, ret_ranks=True)
    assert (raw, cnt) == whole(DET, S, fd, 8, w)
    assert [v for v, _, _ in records(raw, DET)[:cnt]] == [100.0, 60.0]
    assert counts.cpu().tolist() == [2, 1]


def test_ranks_without_rows_contribute_nothing():
    """d = 3 over 8 ranks: five ranks own no rows and report count 0 and unused slots; an empty block needs no halo."""
    import torch
    rng = np.random.default_rng(2)
    S, fd = tensor(rng.exponential(1.0, (3, 256))), grid(3)
    for det in (DET, CA, OS):
        w = windows(det, 1, 1, 1, 2, scale=1.0)
        (raw, cnt), lists, counts = sharded(det, S, fd, 8, w, 8, ret_ranks=True)
        assert (raw, cnt) == whole(det, S, fd, 8, w)
        empty = [r for r in range(8) if shard_bounds(3, 8, r)[0] == shard_bounds(3, 8, r)[1]]
        assert len(empty) == 5 and all(int(counts[r]) == 0 for r in empty)
        unused = lists[empty[0]].cpu().numpy()
        assert np.all(unused[:, 2:4].view(np.uint64)[:, 0] == api.UINT64_MAX)
    out = torch.zeros((4, 6), dtype=torch.float64, device=dev())
    cnt = torch.full((1,), -1, dtype=torch.int64, device=dev())
    torch.cuda.synchronize()
    api.detect_rows_dev(0, 0, 256, 0, 0, 0, 5, 10, 4, out.data_ptr(), cnt.data_ptr())
    torch.cuda.synchronize()
    assert int(cnt.cpu()[0]) == 0


def test_failed_rank_mark_is_skipped_by_the_merge():
    """A count above k_max (what the library's exchange sends for a rank that failed) drops that rank's list."""
    rng = np.random.default_rng(4)
    S, fd = tensor(rng.exponential(1.0, (40, 256))), grid(40)
    w = windows(DET, 1, 1)
    (_, _), lists, counts = sharded(DET, S, fd, 16, w, 4, ret_ranks=True)
    keep = [0, 1, 3]
    want = merge(DET, lists[keep].contiguous(), counts[keep].contiguous(), 16, w)
    counts[2] = -2                                          # UINT64_MAX - 1
    assert merge(DET, lists, counts, 16, w) == want


# ---- 4. errors --------------------------------------------------------------------------------------------------------
def test_errors_write_nothing():
    """Every rejected call returns its status and leaves both the records and the count as they were."""
    import torch
    lib = _lib.load()
    h = api.default_handle()
    rng = np.random.default_rng(8)
    S = torch.from_numpy(rng.exponential(1.0, (20, 64))).to(dev())
    f = torch.zeros(20, dtype=torch.float64, device=dev())
    lists = torch.from_numpy(rng.exponential(1.0, (2, 4, 8))).to(dev())      # merge inputs
    counts = torch.tensor([1, 2], dtype=torch.int64, device=dev())
    o = torch.from_numpy(rng.standard_normal((4, 8))).to(dev())              # every output starts as noise
    c = torch.tensor([12345], dtype=torch.int64, device=dev())
    P = lambda t: C.c_void_p(t.data_ptr())

    def rejected(status, call):
        torch.cuda.synchronize()
        o0, c0 = o.clone(), c.clone()
        torch.cuda.synchronize()
        assert call() == status
        h.sync()
        torch.cuda.synchronize()
        assert torch.equal(o.view(torch.int64), o0.view(torch.int64)) and torch.equal(c, c0)

    def det(*rows, k=4, gr=2, gd=1, mr=0.0, out=True):
        return lib.caf_b200_detect_rows_f64_dev(h.raw, P(S), *rows, k, gr, gd, mr, P(o) if out else None, P(c))

    def ca(*rows, k=4, gr=1, tr=2, scale=2.0):
        return lib.caf_b200_detect_cfar_rows_f64_dev(h.raw, P(S), *rows, k, gr, 1, tr, 2, scale, P(o), P(c))

    def os_(*rows, k=4, gr=1, tr=2, rank=3, scale=2.0):
        return lib.caf_b200_detect_cfar_os_rows_f64_dev(h.raw, P(S), *rows, k, gr, 1, tr, 2, rank, scale, P(o), P(c))

    # (d_buf, n, freqs, row_lo, row_hi, row_offset, d_global)
    good = (20, 64, P(f), 5, 15, 10, 100)
    bad = [
        (20, 64, P(f), 1, 15, 10, 100),        # one row above, H = 2 (detect) / 3 (CFAR), not the surface's top
        (20, 64, P(f), 5, 19, 10, 100),        # one row below, not the surface's end
        (20, 64, P(f), 9, 8, 10, 100),         # row_lo > row_hi
        (20, 64, P(f), 5, 21, 10, 100),        # row_hi > d_buf
        (20, 64, P(f), 5, 15, 90, 100),        # row_offset + d_buf > d_global
    ]
    for rows in bad:
        for fn in (det, ca, os_):
            rejected(-1, lambda: fn(*rows))
    for call in (lambda: det(*good, k=0), lambda: det(*good, gr=33), lambda: det(*good, mr=1.5),
                 lambda: det(20, 64, None, 5, 15, 10, 100), lambda: ca(*good, k=1025), lambda: ca(*good, tr=32),
                 lambda: ca(*good, scale=0.0), lambda: os_(*good, rank=0), lambda: os_(*good, rank=10 ** 6),
                 lambda: os_(*good, tr=32),
                 lambda: lib.caf_b200_detect_merge_dev(h.raw, P(lists), P(counts), 0, 4, 0.0, P(o), P(c)),
                 lambda: lib.caf_b200_detect_merge_dev(h.raw, P(lists), P(counts), 2, 0, 0.0, P(o), P(c)),
                 lambda: lib.caf_b200_detect_merge_dev(h.raw, P(lists), P(counts), 2, 4, -0.5, P(o), P(c)),
                 lambda: lib.caf_b200_detect_merge_dev(h.raw, P(lists), P(counts), 2, 4, 0.0, P(o), None),
                 lambda: lib.caf_b200_cfar_merge_dev(h.raw, None, P(counts), 2, 4, P(o), P(c)),
                 lambda: lib.caf_b200_cfar_merge_dev(h.raw, P(lists), P(counts), 2, 1025, P(o), P(c)),
                 lambda: lib.caf_b200_cfar_merge_dev(h.raw, P(lists), None, 2, 4, P(o), P(c))):
        rejected(-1, call)
    rejected(-1, lambda: lib.caf_b200_detect_rows_f64_dev(h.raw, P(S), *good, 4, 2, 1, 0.0, None, P(c)))
    rejected(-3, lambda: det(20, 64, P(f), 5, 15, 10, 2 ** 31 + 1))
    # the legal calls (H <= 3 rows): a block that starts or ends the surface needs no halo on that side, whatever rows it
    # owns
    torch.cuda.synchronize()
    for rows in (good, (20, 64, P(f), 0, 17, 0, 100), (20, 64, P(f), 3, 20, 80, 100), (20, 64, P(f), 1, 17, 0, 100),
                 (20, 64, P(f), 3, 19, 80, 100)):
        assert det(*rows) == 0 and ca(*rows) == 0 and os_(*rows) == 0, rows
    h.sync()


# ---- 5. the library's communicator on one GPU -----------------------------------------------------------------------
def test_world1_communicator_detect_sharded(tmp_path):
    """Comm.detect_sharded (block, exchange over caf_b200_*_allgather_dev, merge) and dist.detect_sharded without an
    initialised process group equal the whole-surface call, for all three detectors."""
    from caf_cookoff_b200.dist import Comm, detect_sharded
    needle, hay = planted()
    S, fd, nd, hd = surface_of(needle, hay, bench_shifts(), False)
    comm = Comm(api.default_handle(), 1, 0, str(tmp_path / "id"))
    try:
        for det in (DET, CA, OS):
            w = windows(det, 2, 2, 4, 16)
            kw = dict(guard_doppler=2, guard_delay=2, train_doppler=4, train_delay=16)
            want = whole(det, S, fd, 16, w)
            for fn in (comm.detect_sharded, detect_sharded):
                res, cnt = fn(det, nd, hd, fd, FS, 16, **kw)
                import torch
                torch.cuda.synchronize()
                assert (res.cpu().numpy().tobytes(), int(cnt.cpu()[0])) == want, (det, fn)
    finally:
        comm.close()


def test_detect_sharded_waits_for_torch_work():
    """dist.detect_sharded on inputs torch's stream is still producing, called without a synchronise: the library's stream
    is not ordered after torch's, so the call must wait for them (and for the buffers it takes from torch's allocator)."""
    import torch
    from caf_cookoff_b200.dist import detect_sharded
    needle, hay = planted()
    S, fd, nd, hd = surface_of(needle, hay, bench_shifts(), False)
    kw = dict(guard_doppler=2, guard_delay=2, train_doppler=4, train_delay=16)
    for det in (DET, CA):
        want = whole(det, S, fd, 16, windows(det, 2, 2, 4, 16))
        busy = torch.randn((8192, 8192), device=dev())
        for _ in range(3):
            busy = busy @ busy                       # tens of ms of torch work queued ahead of the inputs
        nd2, hd2, fd2 = nd * 1.0, hd * 1.0, fd * 1.0  # the same values, written behind that work
        res, cnt = detect_sharded(det, nd2, hd2, fd2, FS, 16, **kw)
        torch.cuda.synchronize()
        assert (res.cpu().numpy().tobytes(), int(cnt.cpu()[0])) == want, det
