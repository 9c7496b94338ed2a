"""Multi-GPU plumbing for the CAF path: one process per GPU, torch.distributed (NCCL on GPUs, gloo in CPU tests).

The path shards without any data-path collective (SURVEY.md section 8e): doppler rows are independent
(mod.rs:185,283 — the reference's own par_iter) and so are signal pairs.  The only cross-rank step is find_peak's
maximum (mod.rs:36-40): each rank packs its local peak into 4 uint64 words (caf_b200_peak_pack), ONE all_gather of
32 bytes per rank moves them, and every rank resolves the same winner with the reference's tie-break
(caf_b200_peak_resolve: larger value, then lower global doppler row).
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

from . import _lib, api
from .api import _check, peak_pack, peak_resolve


def shard_bounds(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous block of the n rows (or pairs) owned by `rank`: [lo, hi)."""
    return n * rank // world, n * (rank + 1) // world


def exchange_peak(local: _lib.Peak, global_row_offset: int, device=None, group=None) -> _lib.Peak:
    """All ranks call this with their shard's peak; all ranks get the global find_peak result."""
    import torch
    import torch.distributed as dist
    words = peak_pack(local, global_row_offset)                       # uint64[4]
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return peak_resolve(words.reshape(1, 4))
    world = dist.get_world_size(group)
    t = torch.from_numpy(words.view(np.int64).copy())
    if device is not None:
        t = t.to(device)
    out = torch.empty(world * 4, dtype=torch.int64, device=t.device)
    dist.all_gather_into_tensor(out, t, group=group)
    return peak_resolve(out.cpu().numpy().view(np.uint64).reshape(world, 4))


def gather_pair_peaks(local_peaks, n_pairs: int, device=None, group=None) -> np.ndarray:
    """Pairs sharded across ranks (BASELINE config 4): rank r holds the peaks of pairs shard_bounds(n_pairs, world, r),
    as an array of caf_b200_peak records viewed as uint64 [p_local, 4] (value bits, freq bits, doppler_idx,
    delay_idx).  ONE all_gather of the padded blocks (32 bytes per pair) gives every rank all n_pairs records in pair
    order.  Pairs are independent, so unlike exchange_peak nothing is resolved: this is a pure gather."""
    import torch
    import torch.distributed as dist
    loc = np.ascontiguousarray(local_peaks).view(np.uint64).reshape(-1, 4)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        if loc.shape[0] != n_pairs:
            raise ValueError(f"one rank must hold all {n_pairs} pairs, got {loc.shape[0]}")
        return loc.copy()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    lo, hi = shard_bounds(n_pairs, world, rank)
    if loc.shape[0] != hi - lo:
        raise ValueError(f"rank {rank} owns pairs [{lo}, {hi}) but passed {loc.shape[0]} peaks")
    width = max(b - a for a, b in (shard_bounds(n_pairs, world, r) for r in range(world)))
    block = np.zeros((width, 4), dtype=np.uint64)
    block[: hi - lo] = loc
    t = torch.from_numpy(block.view(np.int64))
    if device is not None:
        t = t.to(device)
    out = torch.empty((world * width, 4), dtype=torch.int64, device=t.device)      # blocks concatenated along dim 0
    dist.all_gather_into_tensor(out, t, group=group)
    allw = out.cpu().numpy().view(np.uint64).reshape(world, width, 4)
    parts = []
    for r in range(world):
        a, b = shard_bounds(n_pairs, world, r)
        parts.append(allw[r, : b - a])
    return np.concatenate(parts, axis=0) if parts else np.zeros((0, 4), dtype=np.uint64)


def gather_pair_peaks_dev(local_peaks_dev, n_pairs: int, group=None):
    """gather_pair_peaks for peaks that are still on the GPU: a CUDA int64 tensor [p_local, 4] in, a CUDA tensor
    [n_pairs, 4] out, ONE all_gather_into_tensor over NCCL and no host round trip (uneven shards are padded to the widest
    block and trimmed afterwards).  Stream-ordered on the current torch stream."""
    import torch
    import torch.distributed as dist
    t = local_peaks_dev.reshape(-1, 4)
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        if t.shape[0] != n_pairs:
            raise ValueError(f"one rank must hold all {n_pairs} pairs, got {t.shape[0]}")
        return t
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    lo, hi = shard_bounds(n_pairs, world, rank)
    if t.shape[0] != hi - lo:
        raise ValueError(f"rank {rank} owns pairs [{lo}, {hi}) but passed {t.shape[0]} peaks")
    bounds = [shard_bounds(n_pairs, world, r) for r in range(world)]
    width = max(b - a for a, b in bounds)
    if hi - lo == width:
        block = t.contiguous()
    else:
        block = torch.zeros((width, 4), dtype=t.dtype, device=t.device)
        block[: hi - lo] = t
    out = torch.empty((world * width, 4), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, block, group=group)
    if all(b - a == width for a, b in bounds):
        return out
    return torch.cat([out[r * width: r * width + (b - a)] for r, (a, b) in enumerate(bounds)], dim=0)


def gather_surface(local_rows, n_rows: int, group=None):
    """The full surface, only when asked for (the path itself never needs it): rank r holds rows
    shard_bounds(n_rows, world, r) of the doppler grid as [hi - lo, 2L] (a numpy array, or a torch tensor — a CUDA
    tensor under NCCL, so the rows travel GPU to GPU over NVLink); ONE all_gather of the padded blocks gives every rank
    the [n_rows, 2L] surface in freqs_hz order, exactly the Vec<CafSurfaceRow> order of the ordered strategies
    (mod.rs:135-162).  Uneven shards are padded to the widest block and trimmed after the exchange."""
    import torch
    import torch.distributed as dist
    is_np = isinstance(local_rows, np.ndarray)
    t = torch.from_numpy(np.ascontiguousarray(local_rows)) if is_np else local_rows.contiguous()
    if t.dim() != 2:
        raise ValueError("local_rows must be [rows, 2L]")
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        if t.shape[0] != n_rows:
            raise ValueError(f"one rank must hold all {n_rows} rows, got {t.shape[0]}")
        return local_rows
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    lo, hi = shard_bounds(n_rows, world, rank)
    if t.shape[0] != hi - lo:
        raise ValueError(f"rank {rank} owns rows [{lo}, {hi}) but passed {t.shape[0]}")
    bounds = [shard_bounds(n_rows, world, r) for r in range(world)]
    width = max(b - a for a, b in bounds)
    cols = t.shape[1]
    if hi - lo == width:
        block = t
    else:
        block = torch.zeros((width, cols), dtype=t.dtype, device=t.device)
        block[: hi - lo] = t
    out = torch.empty((world * width, cols), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, block, group=group)
    if all(b - a == width for a, b in bounds):
        full = out
    else:
        full = torch.cat([out[r * width: r * width + (b - a)] for r, (a, b) in enumerate(bounds)], dim=0)
    return full.numpy() if is_np else full


def peaks_as_tuples(words: np.ndarray):
    """[(freq_hz, delay_idx)] per pair from gather_pair_peaks' uint64 records: what find_peak returns (mod.rs:31-42)."""
    w = np.ascontiguousarray(words, dtype=np.uint64).reshape(-1, 4)
    return [(float(w[i, 1:2].view(np.float64)[0]), int(w[i, 3])) for i in range(w.shape[0])]


_FAILED = -2        # UINT64_MAX - 1 as int64: the failure mark of a rank's count (above any k_max), as in the library


def _block_detect(detector: str, needle, haystack, freqs, fs: int, k_max: int, world: int, rank: int, *,
                  guard_doppler: int, guard_delay: int, train_doppler: int, train_delay: int, os_rank, scale,
                  min_ratio: float, handle):
    """One rank's half of sharded detection: the halo'd block of its rows shard_bounds(d, world, rank) computed with
    caf_b200_batch_*_dev from the same inputs every rank holds, then the block detector over the owned rows.  Returns
    (records [k_max, 6 or 8] float64 tensor, count int64 tensor [1]) on the handle's device, complete.  The handle's
    stream and torch's are not ordered with each other, so torch's is synchronised before the first launch (the inputs
    as torch last wrote them, and buffers from torch's allocator that torch's pending work may still use) and the
    handle's before the return (the block is freed on return)."""
    import torch
    if detector not in ("detect", "cfar", "cfar_os"):
        raise ValueError("detector must be 'detect', 'cfar' or 'cfar_os'")
    h = handle or api.default_handle()
    f32 = needle.dtype == torch.complex64
    l, d = int(needle.numel()), int(freqs.numel())
    n = 2 * l
    lo, hi = shard_bounds(d, world, rank)
    H = api.halo_rows(detector, guard_doppler, 0 if detector == "detect" else train_doppler)
    b_lo, b_hi = max(lo - H, 0), min(hi + H, d)
    dev = needle.device
    surf = torch.empty((b_hi - b_lo, n), dtype=torch.float32 if f32 else torch.float64, device=dev)
    peak = torch.empty(4, dtype=torch.float64, device=dev)
    out = torch.empty((k_max, 6 if detector == "detect" else 8), dtype=torch.float64, device=dev)
    cnt = torch.empty(1, dtype=torch.int64, device=dev)
    torch.cuda.current_stream(dev).synchronize()
    try:
        f_ptr = freqs.data_ptr() + 8 * b_lo
        if b_hi > b_lo:
            fn = getattr(_lib.load(), "caf_b200_batch_f32_dev" if f32 else "caf_b200_batch_f64_dev")
            _check(fn(h.raw, needle.data_ptr(), haystack.data_ptr(), 1, l, f_ptr, b_hi - b_lo, int(fs), surf.data_ptr(),
                      None, None, peak.data_ptr()))
        args = (surf.data_ptr(), b_hi - b_lo, n, f_ptr, lo - b_lo, hi - b_lo, b_lo, d, k_max, out.data_ptr(),
                cnt.data_ptr())
        win = dict(guard_doppler=guard_doppler, guard_delay=guard_delay, f32=f32, handle=h)
        if detector == "detect":
            api.detect_rows_dev(*args, min_ratio=min_ratio, **win)
        else:
            N = api.cfar_train_cells(guard_doppler, guard_delay, train_doppler, train_delay)
            win.update(train_doppler=train_doppler, train_delay=train_delay)
            if detector == "cfar":
                api.detect_cfar_rows_dev(*args, scale=api.cfar_scale(1e-6, N) if scale is None else scale, **win)
            else:
                os_rank = (3 * N + 3) // 4 if os_rank is None else os_rank
                api.detect_cfar_os_rows_dev(*args, rank=os_rank,
                                            scale=api.cfar_os_scale(1e-6, N, os_rank) if scale is None else scale, **win)
    finally:
        h.sync()                      # also when a call raised after the batch launch: surf dies here
    return out, cnt


def detect_sharded(detector: str, needle, haystack, freqs, fs: int, k_max: int, *, guard_doppler: int = 1,
                   guard_delay: int = 1, train_doppler: int = 2, train_delay: int = 16, rank=None, scale=None,
                   min_ratio: float = 0.0, handle=None, group=None):
    """Detection on a row-sharded surface over torch.distributed (DESIGN.md section 12).  detector is "detect", "cfar" or
    "cfar_os"; every rank passes the same CUDA tensors needle, haystack [l] (complex128, or complex64 for f32 surfaces)
    and freqs [d] (float64, the whole grid).  Rank r computes rows shard_bounds(d, world, r) plus a halo of
    api.halo_rows(...) rows, detects over its own rows, and ONE all_gather_into_tensor of the records and count feeds
    the merge.  Every rank returns (records [k_max, 6] (detect) or [k_max, 8] float64 tensor, count int64 tensor [1])
    equal bit for bit to the same detector on the whole surface.  rank and scale of the CFAR detectors default as in
    DeviceSurface.detect_cfar / detect_cfar_os; min_ratio is detect's.  k_max and the window must be the same on every
    rank.  A rank whose block detection raises still takes part in the gather, with a count above k_max as its failure
    mark, and then re-raises; its peers skip its list and raise CafError with CAF_B200_EREMOTE (-7), as the library's
    exchange does."""
    import torch
    import torch.distributed as dist
    on = dist.is_available() and dist.is_initialized()
    world, me = (dist.get_world_size(group), dist.get_rank(group)) if on else (1, 0)
    h = handle or api.default_handle()
    width = 6 if detector == "detect" else 8
    failed = None
    try:
        out, cnt = _block_detect(detector, needle, haystack, freqs, fs, k_max, world, me, guard_doppler=guard_doppler,
                                 guard_delay=guard_delay, train_doppler=train_doppler, train_delay=train_delay,
                                 os_rank=rank, scale=scale, min_ratio=min_ratio, handle=h)
        mine = torch.cat([out.view(torch.int64).reshape(-1), cnt])
    except Exception as e:
        if world == 1:
            raise
        failed = e                    # never leave the peers alone in the collective
        mine = torch.zeros(k_max * width + 1, dtype=torch.int64, device=needle.device)
        mine[-1] = _FAILED
    if world > 1:
        allw = torch.empty((world, mine.numel()), dtype=torch.int64, device=mine.device)
        dist.all_gather_into_tensor(allw, mine, group=group)
    else:
        allw = mine.reshape(1, -1)
    if failed is not None:
        raise failed
    lists = allw[:, :-1].contiguous()
    counts = allw[:, -1].contiguous()
    res = torch.empty((k_max, width), dtype=torch.float64, device=mine.device)
    count = torch.empty(1, dtype=torch.int64, device=mine.device)
    torch.cuda.current_stream(mine.device).synchronize()  # the gathered lists, before the library's stream reads them
    if detector == "detect":
        api.detect_merge_dev(lists.data_ptr(), counts.data_ptr(), world, k_max, res.data_ptr(), count.data_ptr(),
                             min_ratio=min_ratio, handle=h)
    else:
        api.cfar_merge_dev(lists.data_ptr(), counts.data_ptr(), world, k_max, res.data_ptr(), count.data_ptr(), handle=h)
    h.sync()
    c = counts.cpu()
    if bool(((c < 0) | (c > k_max)).any()):
        raise api.CafError(-7, "a peer rank failed before the detection exchange")
    return res, count


class Comm:
    """The library's own NCCL communicator (caf_b200_comm_*): what a caller without torch.distributed (the Rust
    shim) uses.  The 128-byte NCCL id travels out of band; here through a small file any rank can read.

    The file carries a per-run nonce in front of the id (`run_id`: TORCHELASTIC_RUN_ID / CAF_RUN_ID by default, which
    every rank of one launch shares and two launches do not), so a file left behind by an earlier run is never taken
    for this run's id; rank 0 removes the file again once every rank has joined the communicator."""

    _MAGIC = b"CAFNCCL1"

    def __init__(self, handle, world: int, rank: int, id_path: str, timeout_s: float = 120.0, run_id: str | None = None):
        import ctypes as C
        import hashlib
        import os
        import time
        self._lib = _lib.load()
        self.world, self.rank, self.handle = world, rank, handle
        if run_id is None:
            run_id = os.environ.get("CAF_RUN_ID") or os.environ.get("TORCHELASTIC_RUN_ID") or ""
        nonce = hashlib.sha256(("%s|%s|%d" % (run_id, id_path, world)).encode()).digest()[:16]
        buf = (C.c_ubyte * 128)()
        if rank == 0:
            _check(self._lib.caf_b200_comm_unique_id(C.cast(buf, C.c_void_p)))
            tmp = id_path + ".tmp%d" % os.getpid()
            with open(tmp, "wb") as f:
                f.write(self._MAGIC + nonce + bytes(buf))
            os.replace(tmp, id_path)                      # atomic publish (replaces a stale file of an earlier run)
        else:
            t_end = time.time() + timeout_s
            want = self._MAGIC + nonce
            while True:
                try:
                    blob = open(id_path, "rb").read()
                except OSError:
                    blob = b""
                # the nonce tells this run's file from one an earlier run left behind (launchers without a run id:
                # pass run_id=, or use a path that is unique per launch)
                if len(blob) == len(want) + 128 and blob.startswith(want):
                    C.memmove(buf, blob[len(want):], 128)
                    break
                if time.time() > t_end:
                    raise TimeoutError(f"rank {rank}: no NCCL id of this run at {id_path}")
                time.sleep(0.01)
        self._c = C.c_void_p()
        _check(self._lib.caf_b200_comm_create(handle.raw, world, rank, C.cast(buf, C.c_void_p), C.byref(self._c)))
        if rank == 0:                                     # ncclCommInitRank returned: every rank has read the id
            try:
                os.unlink(id_path)
            except OSError:
                pass

    @property
    def raw(self):
        return self._c

    def shard(self, n: int) -> Tuple[int, int]:
        import ctypes as C
        lo, hi = C.c_size_t(), C.c_size_t()
        _check(self._lib.caf_b200_comm_shard(self._c, n, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value

    def peak_allgather_dev(self, local_peak_dev_ptr: int, global_row_offset: int) -> _lib.Peak:
        import ctypes as C
        out = _lib.Peak()
        _check(self._lib.caf_b200_peak_allgather_dev(self.handle.raw, self._c, C.c_void_p(local_peak_dev_ptr),
                                                     int(global_row_offset), C.byref(out)))
        return out

    def peak_allgather_async(self, local_peak_dev_ptr: int, global_row_offset: int, out_dev_ptr: int) -> None:
        """No host synchronisation: the global peak is in out_dev (32 bytes, device or pinned memory) once the
        handle's stream gets there."""
        import ctypes as C
        _check(self._lib.caf_b200_peak_allgather_async(self.handle.raw, self._c, C.c_void_p(local_peak_dev_ptr or None),
                                                       int(global_row_offset), C.c_void_p(out_dev_ptr)))

    def sharded_dev(self, needle_dev: int, hay_dev: int, l: int, freqs_local_dev: int, d_local: int, row_offset: int,
                    fs: int, peak_out_dev: int, surface_local_dev: int = 0, row_val_dev: int = 0, row_idx_dev: int = 0,
                    f32: bool = False) -> None:
        """caf_b200_sharded_{f64,f32}_dev: this rank's block of doppler rows + the cross-rank find_peak, all on the
        handle's stream with no host synchronisation (device pointers as integers)."""
        import ctypes as C
        fn = self._lib.caf_b200_sharded_f32_dev if f32 else self._lib.caf_b200_sharded_f64_dev
        vp = lambda x: C.c_void_p(x or None)
        _check(fn(self.handle.raw, self._c, vp(needle_dev), vp(hay_dev), int(l), vp(freqs_local_dev), int(d_local),
                  int(row_offset), int(fs), vp(surface_local_dev), vp(row_val_dev), vp(row_idx_dev), vp(peak_out_dev)))

    def detect_sharded(self, detector: str, needle, haystack, freqs, fs: int, k_max: int, *, guard_doppler: int = 1,
                       guard_delay: int = 1, train_doppler: int = 2, train_delay: int = 16, rank=None, scale=None,
                       min_ratio: float = 0.0):
        """dist.detect_sharded over this communicator: the halo'd block and the block detector on this rank, then
        caf_b200_detect_allgather_dev / caf_b200_cfar_allgather_dev.  If this rank's block cannot be computed it still
        enters the exchange with the failure mark (its peers raise CafError EREMOTE) and raises the local error."""
        import ctypes as C
        import torch
        try:
            out, cnt = _block_detect(detector, needle, haystack, freqs, fs, k_max, self.world, self.rank,
                                     guard_doppler=guard_doppler, guard_delay=guard_delay, train_doppler=train_doppler,
                                     train_delay=train_delay, os_rank=rank, scale=scale, min_ratio=min_ratio,
                                     handle=self.handle)
        except Exception:
            if detector == "detect":
                self._lib.caf_b200_detect_allgather_dev(self.handle.raw, self._c, None, None, int(k_max),
                                                        float(min_ratio), None, None)
            else:
                self._lib.caf_b200_cfar_allgather_dev(self.handle.raw, self._c, None, None, int(k_max), None, None)
            raise
        res = torch.empty_like(out)
        count = torch.empty(1, dtype=torch.int64, device=out.device)
        torch.cuda.current_stream(out.device).synchronize()   # res / count from torch's allocator, as in _block_detect
        vp = lambda t: C.c_void_p(t.data_ptr())
        if detector == "detect":
            _check(self._lib.caf_b200_detect_allgather_dev(self.handle.raw, self._c, vp(out), vp(cnt), int(k_max),
                                                           float(min_ratio), vp(res), vp(count)))
        else:
            _check(self._lib.caf_b200_cfar_allgather_dev(self.handle.raw, self._c, vp(out), vp(cnt), int(k_max), vp(res),
                                                         vp(count)))
        return res, count

    def uses_p2p(self) -> bool:
        """True when the exchange is the one-kernel peer-memory mailbox (NVLink), False when it is ncclAllGather."""
        import ctypes as C
        flag = C.c_int()
        _check(self._lib.caf_b200_comm_uses_p2p(self._c, C.byref(flag)))
        return bool(flag.value)

    def remote_error(self) -> bool:
        """After a synchronise: did a peer report a failure in the last exchange?"""
        import ctypes as C
        flag = C.c_int()
        _check(self._lib.caf_b200_comm_remote_error(self._c, C.byref(flag)))
        return bool(flag.value)

    def surface_sharded(self, needle, haystack, freqs_hz, fs: int, want_surface: bool = True):
        """caf_b200_surface_sharded_f64: (local rows [hi-lo, 2L] or None, global Peak)."""
        import ctypes as C
        n_ = np.ascontiguousarray(needle, dtype=np.complex128).ravel()
        h_ = np.ascontiguousarray(haystack, dtype=np.complex128).ravel()
        f_ = np.ascontiguousarray(freqs_hz, dtype=np.float64).ravel()
        lo, hi = self.shard(f_.size)
        surf = np.empty((hi - lo, 2 * n_.size), dtype=np.float64) if want_surface else None
        pk = _lib.Peak()
        _check(self._lib.caf_b200_surface_sharded_f64(
            self.handle.raw, self._c, n_.ctypes.data_as(C.c_void_p), h_.ctypes.data_as(C.c_void_p), n_.size,
            f_.ctypes.data_as(C.c_void_p), f_.size, int(fs), None if surf is None else surf.ctypes.data_as(C.c_void_p),
            C.byref(pk)))
        return surf, pk

    def close(self):
        if self._c:
            self._lib.caf_b200_comm_destroy(self._c)
            import ctypes as C
            self._c = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
