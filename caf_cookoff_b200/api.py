"""Host-side mirror of caf_rust's public API over the C ABI (include/caf_b200.h).

The reference interface (paths relative to /root/reference/caf_rust):
    pub trait CafSurface { fn caf_surface(needle, haystack, freqs_hz, fs) -> Vec<CafSurfaceRow>;
                           fn find_peak(arr) -> (f64, usize);
                           fn apply_freq_shift(samples, freq_shift, fs) -> Vec<Complex64>; }   src/caf/mod.rs:23-66
    pub struct CafSurfaceRow { freq, xcor_mag, xcor_peak_idx, xcor_peak_val }                  src/caf/mod.rs:17-22
    struct Xcor { fn new(n); fn run(&mut self, a, b) -> Vec<Complex64> }                       src/caf/xcor_rustfft.rs:14-78
Same names, argument order and meaning; the reference's panics become exceptions (CafPanic).
All arithmetic happens in libcaf_b200.so on the GPU — this module never computes a surface itself.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib

UINT64_MAX = (1 << 64) - 1


class CafError(RuntimeError):
    """A non-zero status from the C ABI."""

    def __init__(self, status: int, msg: str):
        super().__init__(f"caf_b200 status {status}: {msg}")
        self.status = status


class CafPanic(AssertionError):
    """Where the reference panics (xcor_rustfft.rs:54-55 assert!, Iter variants indexing an empty row)."""


def _check(rc: int):
    if rc != 0:
        msg = _lib.load().caf_b200_last_error().decode("utf-8", "replace")
        if rc == -2:
            raise CafPanic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55): " + msg)
        raise CafError(rc, msg)


class Handle:
    """One device + stream + twiddle tables + workspace (caf_b200_create / _destroy)."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        if stream is not None:
            _check(self._lib.caf_b200_create_on_stream(int(device), C.c_void_p(int(stream)), C.byref(self._h)))
        else:
            _check(self._lib.caf_b200_create(int(device), C.byref(self._h)))
        self.device = device

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.caf_b200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        _check(self._lib.caf_b200_sync(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._lib.caf_b200_launch_count(self._h))

    @property
    def raw(self):
        return self._h


_default_handles = {}


def default_handle(device: int = 0) -> Handle:
    h = _default_handles.get(device)
    if h is None:
        h = _default_handles[device] = Handle(device)
    return h


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class CafSurfaceRow:
    """mod.rs:17-22.  xcor_mag is a view into the contiguous D x 2L surface."""
    __slots__ = ("freq", "xcor_mag", "xcor_peak_idx", "xcor_peak_val")

    def __init__(self, freq: float, xcor_mag: np.ndarray, xcor_peak_idx: int, xcor_peak_val: float):
        self.freq = freq
        self.xcor_mag = xcor_mag
        self.xcor_peak_idx = xcor_peak_idx
        self.xcor_peak_val = xcor_peak_val


class Surface(list):
    """Vec<CafSurfaceRow> plus what the GPU already knows: the dense surface and the fused peak."""
    array: Optional[np.ndarray] = None          # [D, 2L] |xcor|^2
    row_peak_idx: Optional[np.ndarray] = None   # [D] uint64
    row_peak_val: Optional[np.ndarray] = None   # [D]
    peak: Optional[_lib.Peak] = None            # caf_b200_peak from the fused find_peak kernel


class _Variant:
    cdt = np.complex128
    rdt = np.float64
    sfx = "f64"


class _Variant32:
    cdt = np.complex64
    rdt = np.float32
    sfx = "f32"


def surface_arrays(needle, haystack, freqs_hz, fs: int, *, variant=_Variant, want_surface=True,
                   handle: Optional[Handle] = None):
    """caf_b200_surface_{f64,f32}: returns (surface or None, row_peak_idx, row_peak_val, Peak)."""
    n_ = np.ascontiguousarray(needle, dtype=variant.cdt).ravel()
    h_ = np.ascontiguousarray(haystack, dtype=variant.cdt).ravel()
    f_ = np.ascontiguousarray(freqs_hz, dtype=np.float64).ravel()
    if n_.size != h_.size:
        # the reference pads each to 2*len and Xcor::run asserts equal length (xcor_rustfft.rs:54-55)
        raise CafPanic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55)")
    h = handle or default_handle()
    lib = _lib.load()
    l, d = n_.size, f_.size
    surf = np.empty((d, 2 * l), dtype=variant.rdt) if want_surface else None
    pidx = np.zeros(d, dtype=np.uint64)
    pval = np.zeros(d, dtype=variant.rdt)
    pk = _lib.Peak()
    fn = getattr(lib, "caf_b200_surface_" + variant.sfx)
    _check(fn(h.raw, _ptr(n_), _ptr(h_), l, _ptr(f_), d, int(fs), _ptr(surf), _ptr(pval), _ptr(pidx),
              C.cast(C.byref(pk), C.c_void_p)))
    return surf, pidx, pval, pk


def batch_arrays(needles, haystacks, freqs_hz, fs: int, *, variant=_Variant, want_surface=False,
                 handle: Optional[Handle] = None):
    """caf_b200_batch_*: needles/haystacks [P, L].  Returns (surface[P,D,2L] or None, pidx[P,D], pval[P,D], peaks)."""
    n_ = np.ascontiguousarray(needles, dtype=variant.cdt)
    h_ = np.ascontiguousarray(haystacks, dtype=variant.cdt)
    f_ = np.ascontiguousarray(freqs_hz, dtype=np.float64).ravel()
    if n_.shape != h_.shape or n_.ndim != 2:
        raise CafPanic("needles and haystacks must both be [P, L] (xcor_rustfft.rs:54-55)")
    h = handle or default_handle()
    lib = _lib.load()
    p, l = n_.shape
    d = f_.size
    surf = np.empty((p, d, 2 * l), dtype=variant.rdt) if want_surface else None
    pidx = np.zeros((p, d), dtype=np.uint64)
    pval = np.zeros((p, d), dtype=variant.rdt)
    peaks = (_lib.Peak * max(p, 1))()
    fn = getattr(lib, "caf_b200_batch_" + variant.sfx)
    _check(fn(h.raw, _ptr(n_), _ptr(h_), p, l, _ptr(f_), d, int(fs), _ptr(surf), _ptr(pval), _ptr(pidx),
              C.cast(peaks, C.c_void_p)))
    return surf, pidx, pval, list(peaks)[:p]


class CafSurface:
    """The trait (mod.rs:23-66).  Associated functions, no self — exactly as in Rust."""
    _variant = _Variant

    @classmethod
    def caf_surface(cls, needle, haystack, freqs_hz, fs: int) -> Surface:
        surf, pidx, pval, pk = surface_arrays(needle, haystack, freqs_hz, fs, variant=cls._variant)
        f_ = np.ascontiguousarray(freqs_hz, dtype=np.float64).ravel()
        rows = Surface(CafSurfaceRow(float(f_[r]), surf[r], int(pidx[r]), float(pval[r])) for r in range(f_.size))
        rows.array, rows.row_peak_idx, rows.row_peak_val, rows.peak = surf, pidx, pval, pk
        return rows

    @staticmethod
    def find_peak(arr: Sequence[CafSurfaceRow]) -> Tuple[float, int]:
        """mod.rs:31-42: strict > from a dummy row (freq 0.0, peak 0.0) -> first row holding the max."""
        best_val, best = 0.0, (0.0, 0)
        for row in arr:
            if row.xcor_peak_val > best_val:
                best_val, best = row.xcor_peak_val, (row.freq, row.xcor_peak_idx)
        return best

    @classmethod
    def apply_freq_shift(cls, samples, freq_shift: float, fs: int) -> np.ndarray:
        """mod.rs:46-65."""
        v = cls._variant
        x = np.ascontiguousarray(samples, dtype=v.cdt).ravel()
        out = np.empty_like(x)
        fn = getattr(_lib.load(), "caf_b200_apply_freq_shift_" + v.sfx)
        _check(fn(default_handle().raw, _ptr(x), x.size, float(freq_shift), int(fs), _ptr(out)))
        return out

    apply_shift = apply_freq_shift   # README.md:124 name

    @classmethod
    def caf_peak(cls, needle, haystack, freqs_hz, fs: int) -> Tuple[float, int]:
        """caf_surface + find_peak fused on the GPU; the surface never leaves the chip."""
        _, _, _, pk = surface_arrays(needle, haystack, freqs_hz, fs, variant=cls._variant, want_surface=False)
        return pk.freq_hz, int(pk.delay_idx)


class CafB200(CafSurface):
    """fp64 / complex128 (the reference's I/O types, README.md:22)."""


class CafB200F32(CafSurface):
    """complex64 / float32 throughput variant (phasor phase still fp64)."""
    _variant = _Variant32


# The seven strategy structs of the reference (mod.rs:67,118,169,219,266,313,388; caf_bench.rs:12-19) all
# name the same computation; here every one of them is the B200 path.  Rows come back in freqs_hz order
# (the reference's Threads/Threadpool variants return arrival order, mod.rs:377,453).
class CafFFTW(CafB200): pass
class CafRustFFT(CafB200): pass
class CafRustFFTRayon(CafB200): pass
class CafRustFFTIter(CafB200):
    @classmethod
    def caf_surface(cls, needle, haystack, freqs_hz, fs):
        if np.size(needle) == 0 and np.size(freqs_hz):
            raise CafPanic("index out of bounds: xcor_mag[0] on an empty row (mod.rs:248)")
        return super().caf_surface(needle, haystack, freqs_hz, fs)
class CafRustFFTIterRayon(CafRustFFTIter): pass
class CafRustFFTThreads(CafB200): pass
class CafRustFFTThreadpool(CafB200): pass


class Xcor:
    """xcor_rustfft.rs:14-93 (crate-private in the reference, exposed here for parity checks)."""
    _variant = _Variant

    def __init__(self, n: int):
        self.n = int(n)

    @classmethod
    def new(cls, n: int) -> "Xcor":
        return cls(n)

    def clone(self) -> "Xcor":
        return type(self)(self.n)

    def run(self, a, b) -> np.ndarray:
        v = self._variant
        a_ = np.ascontiguousarray(a, dtype=v.cdt).ravel()
        b_ = np.ascontiguousarray(b, dtype=v.cdt).ravel()
        if a_.size != self.n or b_.size != self.n:
            raise CafPanic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55)")
        out = np.empty(self.n, dtype=v.cdt)
        fn = getattr(_lib.load(), "caf_b200_xcor_" + v.sfx)
        _check(fn(default_handle().raw, _ptr(a_), _ptr(b_), self.n, _ptr(out)))
        return out


class XcorF32(Xcor):
    _variant = _Variant32


class DeviceSurface:
    """A surface kept in device memory (caf_b200_surface_create_*): find_peak and row peaks come back at once, rows
    cross PCIe only when fetched, and detect() searches the surface where it lies."""

    def __init__(self, needle, haystack, freqs_hz, fs: int, *, variant=_Variant, handle: Optional[Handle] = None):
        n_ = np.ascontiguousarray(needle, dtype=variant.cdt).ravel()
        h_ = np.ascontiguousarray(haystack, dtype=variant.cdt).ravel()
        f_ = np.ascontiguousarray(freqs_hz, dtype=np.float64).ravel()
        if n_.size != h_.size:
            raise CafPanic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55)")
        self.handle = handle or default_handle()
        self.variant = variant
        self._lib = _lib.load()
        self._s = C.c_void_p()
        fn = getattr(self._lib, "caf_b200_surface_create_" + variant.sfx)
        _check(fn(self.handle.raw, _ptr(n_), _ptr(h_), n_.size, _ptr(f_), f_.size, int(fs), C.byref(self._s)))
        self.freqs_hz = f_
        rows, cells = C.c_size_t(), C.c_size_t()
        _check(self._lib.caf_b200_surface_shape(self._s, C.byref(rows), C.byref(cells)))
        self.shape = (rows.value, cells.value)

    @property
    def raw(self):
        return self._s

    def find_peak(self) -> _lib.Peak:
        pk = _lib.Peak()
        _check(self._lib.caf_b200_surface_find_peak(self._s, C.byref(pk)))
        return pk

    def fetch_rows(self, row0: int = 0, count: Optional[int] = None) -> np.ndarray:
        count = self.shape[0] - row0 if count is None else count
        out = np.empty((count, self.shape[1]), dtype=self.variant.rdt)
        _check(self._lib.caf_b200_surface_fetch_rows(self._s, int(row0), int(count), _ptr(out)))
        return out

    def detect(self, k_max: int, guard_doppler: int = 1, guard_delay: int = 1,
               min_ratio: float = 0.0) -> List[_lib.Detection]:
        """caf_b200_surface_detect: the strongest local maxima, best first (only the `count` valid records).  It runs on
        self.handle, so like every call on a handle it must not run at the same time as another call on that handle."""
        out = (_lib.Detection * max(int(k_max), 1))()
        count = C.c_size_t()
        _check(self._lib.caf_b200_surface_detect(self._s, int(k_max), int(guard_doppler), int(guard_delay),
                                                 float(min_ratio), out, C.byref(count)))
        return list(out)[:count.value]

    def detect_cfar(self, k_max: int, guard_doppler: int = 1, guard_delay: int = 1, train_doppler: int = 2,
                    train_delay: int = 16, scale: Optional[float] = None) -> List[_lib.CfarDetection]:
        """caf_b200_surface_detect_cfar: the local maxima that exceed scale x their local noise estimate, best first (only
        the `count` valid records; possibly none).  scale defaults to cfar_scale(1e-6, cfar_train_cells(...)).  Same
        handle rule as detect()."""
        if scale is None:
            scale = cfar_scale(1e-6, cfar_train_cells(guard_doppler, guard_delay, train_doppler, train_delay))
        out = (_lib.CfarDetection * max(int(k_max), 1))()
        count = C.c_size_t()
        _check(self._lib.caf_b200_surface_detect_cfar(self._s, int(k_max), int(guard_doppler), int(guard_delay),
                                                      int(train_doppler), int(train_delay), float(scale), out,
                                                      C.byref(count)))
        return list(out)[:count.value]

    def close(self):
        if getattr(self, "_s", None) is not None and self._s:
            self._lib.caf_b200_surface_destroy(self._s)
            self._s = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def detect_dev(surface_ptr: int, p: int, d: int, n: int, freqs_ptr: int, k_max: int, out_ptr: int, counts_ptr: int, *,
               guard_doppler: int = 1, guard_delay: int = 1, min_ratio: float = 0.0, f32: bool = False,
               handle: Optional[Handle] = None):
    """caf_b200_detect_{f64,f32}_dev on device pointers (e.g. torch tensors' data_ptr()): surface [p][d][n], freqs [d],
    out [p][k_max] caf_b200_detection records (48 bytes each), counts [p] uint64.  Asynchronous on the handle's stream."""
    h = handle or default_handle()
    fn = getattr(_lib.load(), "caf_b200_detect_f32_dev" if f32 else "caf_b200_detect_f64_dev")
    _check(fn(h.raw, C.c_void_p(surface_ptr), int(p), int(d), int(n), C.c_void_p(freqs_ptr), int(k_max),
              int(guard_doppler), int(guard_delay), float(min_ratio), C.c_void_p(out_ptr), C.c_void_p(counts_ptr)))


def cfar_train_cells(guard_doppler: int, guard_delay: int, train_doppler: int, train_delay: int) -> int:
    """N = (2R+1)(2C+1) - (2gr+1)(2gd+1), R = gr + tr, C = gd + tc: the training cells of a cell at least R rows from
    either edge of the surface (rows nearer an edge have fewer) and without NaN neighbours."""
    R, Cd = guard_doppler + train_doppler, guard_delay + train_delay
    return (2 * R + 1) * (2 * Cd + 1) - (2 * guard_doppler + 1) * (2 * guard_delay + 1)


def cfar_scale(pfa: float, train_cells: int) -> float:
    """The CA-CFAR threshold factor alpha = N (Pfa^(-1/N) - 1) for N training cells.

    For N i.i.d. exponential training cells (|.|^2 of complex Gaussian noise) and a test cell of the same law,
    P(v > alpha * mean) = (1 + alpha / N)^-N = Pfa.  That is the false-alarm probability of the threshold test alone,
    before the local-maximum rule, at a cell with all N training cells; edge rows have fewer, and the correlation a CAF
    puts between neighbouring cells is not modelled.  Pure host arithmetic."""
    pfa, n = float(pfa), int(train_cells)
    if not 0.0 < pfa < 1.0:
        raise ValueError("pfa must be in (0, 1)")
    if n < 1:
        raise ValueError("train_cells must be >= 1")
    return n * (pfa ** (-1.0 / n) - 1.0)


def detect_cfar_dev(surface_ptr: int, p: int, d: int, n: int, freqs_ptr: int, k_max: int, out_ptr: int, counts_ptr: int,
                    *, scale: float, guard_doppler: int = 1, guard_delay: int = 1, train_doppler: int = 2,
                    train_delay: int = 16, f32: bool = False, handle: Optional[Handle] = None):
    """caf_b200_detect_cfar_{f64,f32}_dev on device pointers: surface [p][d][n], freqs [d], out [p][k_max]
    caf_b200_cfar_detection records (64 bytes each), counts [p] uint64.  Asynchronous on the handle's stream."""
    h = handle or default_handle()
    fn = getattr(_lib.load(), "caf_b200_detect_cfar_f32_dev" if f32 else "caf_b200_detect_cfar_f64_dev")
    _check(fn(h.raw, C.c_void_p(surface_ptr), int(p), int(d), int(n), C.c_void_p(freqs_ptr), int(k_max),
              int(guard_doppler), int(guard_delay), int(train_doppler), int(train_delay), float(scale),
              C.c_void_p(out_ptr), C.c_void_p(counts_ptr)))


def cfar_noise_dev(surface_ptr: int, p: int, d: int, n: int, noise_ptr: int, *, guard_doppler: int = 1,
                   guard_delay: int = 1, train_doppler: int = 2, train_delay: int = 16, f32: bool = False,
                   handle: Optional[Handle] = None):
    """caf_b200_cfar_noise_{f64,f32}_dev: noise [p][d][n] doubles (NaN where a cell has no training cell), the same bits
    as the `noise` of detect_cfar's records.  Asynchronous on the handle's stream."""
    h = handle or default_handle()
    fn = getattr(_lib.load(), "caf_b200_cfar_noise_f32_dev" if f32 else "caf_b200_cfar_noise_f64_dev")
    _check(fn(h.raw, C.c_void_p(surface_ptr), int(p), int(d), int(n), int(guard_doppler), int(guard_delay),
              int(train_doppler), int(train_delay), C.c_void_p(noise_ptr)))


def peak_pack(pk: _lib.Peak, global_row_offset: int) -> np.ndarray:
    """caf_b200_peak_pack -> 4 uint64 words for the NCCL exchange."""
    words = (C.c_uint64 * 4)()
    _lib.load().caf_b200_peak_pack(C.byref(pk), int(global_row_offset), words)
    return np.array(list(words), dtype=np.uint64)


def peak_resolve(words: np.ndarray) -> _lib.Peak:
    """caf_b200_peak_resolve over [world, 4] words."""
    w = np.ascontiguousarray(words, dtype=np.uint64).reshape(-1, 4)
    out = _lib.Peak()
    _lib.load().caf_b200_peak_resolve(w.ctypes.data_as(C.POINTER(C.c_uint64)), w.shape[0], C.byref(out))
    return out
