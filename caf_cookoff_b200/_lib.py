"""Build and load libcaf_b200.so (the C ABI in include/caf_b200.h) with ctypes.

The library is compiled IN-TREE by nvcc for sm_100a only; there is no other backend and no CPU
fallback: `load()` raises if the shared object is missing, and handle creation fails loudly when no
sm_100 GPU is visible.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
CSRC = os.path.join(_PKG, "csrc")
SO_PATH = os.environ.get("CAF_B200_SO") or os.path.join(_PKG, "libcaf_b200.so")   # override: development builds
HEADER = os.path.join(_ROOT, "include", "caf_b200.h")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "-ldl",
]


def _sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".hpp"))] + [HEADER]


def needs_build() -> bool:
    if not os.path.exists(SO_PATH):
        return True
    so_m = os.path.getmtime(SO_PATH)
    return any(os.path.getmtime(s) > so_m for s in _sources())


def build(force: bool = False, verbose: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> caf_cookoff_b200/libcaf_b200.so"""
    if not force and not needs_build():
        return SO_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libcaf_b200.so (no prebuilt fallback exists)")
    tmp = SO_PATH + ".tmp%d.so" % os.getpid()   # link next to the target, then rename: nobody sees a half-written library
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [
        "-o", tmp, os.path.join(CSRC, "caf_b200.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    os.replace(tmp, SO_PATH)
    if verbose:
        print(res.stderr)
    return SO_PATH


class Peak(C.Structure):
    """caf_b200_peak"""
    _fields_ = [("value", C.c_double), ("freq_hz", C.c_double),
                ("doppler_idx", C.c_uint64), ("delay_idx", C.c_uint64)]


class Detection(C.Structure):
    """caf_b200_detection: the first four fields are caf_b200_peak's"""
    _fields_ = [("value", C.c_double), ("freq_hz", C.c_double),
                ("doppler_idx", C.c_uint64), ("delay_idx", C.c_uint64),
                ("lag_samples", C.c_double), ("freq_hz_interp", C.c_double)]


class CfarDetection(C.Structure):
    """caf_b200_cfar_detection: caf_b200_detection's six fields, then the cell's noise estimate and its training cells"""
    _fields_ = Detection._fields_ + [("noise", C.c_double), ("train_cells", C.c_uint64)]


# every symbol include/caf_b200.h declares: name -> (restype, argtypes)
_vp, _sz, _u32, _dbl, _int = C.c_void_p, C.c_size_t, C.c_uint32, C.c_double, C.c_int
_PK = C.POINTER(Peak)
_batch = [_vp, _vp, _vp, _sz, _sz, _vp, _sz, _u32, _vp, _vp, _vp, _vp]
_surf = [_vp, _vp, _vp, _sz, _vp, _sz, _u32, _vp, _vp, _vp, _vp]
_peak = [_vp, _vp, _vp, _sz, _vp, _sz, _u32, _vp]
_shift = [_vp, _vp, _sz, _dbl, _u32, _vp]
_xcor = [_vp, _vp, _vp, _sz, _vp]
_detect_dev = [_vp, _vp, _sz, _sz, _sz, _vp, _sz, _u32, _u32, _dbl, _vp, _vp]
_cfar_dev = [_vp, _vp, _sz, _sz, _sz, _vp, _sz, _u32, _u32, _u32, _u32, _dbl, _vp, _vp]
_cfar_noise = [_vp, _vp, _sz, _sz, _sz, _u32, _u32, _u32, _u32, _vp]
_cfar_os_dev = [_vp, _vp, _sz, _sz, _sz, _vp, _sz, _u32, _u32, _u32, _u32, _u32, _dbl, _vp, _vp]
_cfar_os_noise = [_vp, _vp, _sz, _sz, _sz, _u32, _u32, _u32, _u32, _u32, _vp]
_rows = [_vp, _vp, _sz, _sz, _vp, _sz, _sz, C.c_uint64, _sz, _sz]    # handle ... k_max: what every block detector starts with
_detect_rows = _rows + [_u32, _u32, _dbl, _vp, _vp]
_cfar_rows = _rows + [_u32, _u32, _u32, _u32, _dbl, _vp, _vp]
_cfar_os_rows = _rows + [_u32, _u32, _u32, _u32, _u32, _dbl, _vp, _vp]
SYMBOLS = {
    "caf_b200_create": (_int, [_int, C.POINTER(_vp)]),
    "caf_b200_create_on_stream": (_int, [_int, _vp, C.POINTER(_vp)]),
    "caf_b200_destroy": (_int, [_vp]),
    "caf_b200_sync": (_int, [_vp]),
    "caf_b200_last_error": (C.c_char_p, []),
    "caf_b200_version": (C.c_char_p, []),
    "caf_b200_launch_count": (C.c_uint64, [_vp]),
    "caf_b200_set_overlap": (_int, [_vp, _int]),
    "caf_b200_set_profiling": (_int, [_vp, _int]),
    "caf_b200_last_kernel_ms": (_int, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "caf_b200_probe_fma_tflops": (_int, [_vp, _int, C.POINTER(C.c_double)]),
    "caf_b200_debug_trace": (_int, [_vp, _vp, _sz]),
    "caf_b200_host_alloc": (_int, [C.POINTER(_vp), _sz]),
    "caf_b200_host_free": (_int, [_vp]),
    "caf_b200_load_c64_dev_f64": (_int, [_vp, C.c_char_p, _sz, _sz, C.POINTER(_vp), C.POINTER(_sz)]),
    "caf_b200_load_c64_dev_f32": (_int, [_vp, C.c_char_p, _sz, _sz, C.POINTER(_vp), C.POINTER(_sz)]),
    "caf_b200_dev_free": (_int, [_vp]),
    "caf_b200_dev_alloc": (_int, [_vp, _sz, C.POINTER(_vp)]),
    "caf_b200_dev_upload": (_int, [_vp, _vp, _vp, _sz]),
    "caf_b200_dev_download": (_int, [_vp, _vp, _vp, _sz]),
    "caf_b200_apply_freq_shift_f64": (_int, _shift),
    "caf_b200_apply_freq_shift_f32": (_int, _shift),
    "caf_b200_apply_shift_f64": (_int, _shift),
    "caf_b200_apply_shift_f32": (_int, _shift),
    "caf_b200_xcor_f64": (_int, _xcor),
    "caf_b200_xcor_f32": (_int, _xcor),
    "caf_b200_surface_f64": (_int, _surf),
    "caf_b200_surface_f32": (_int, _surf),
    "caf_b200_peak_f64": (_int, _peak),
    "caf_b200_peak_f32": (_int, _peak),
    "caf_b200_batch_f64": (_int, _batch),
    "caf_b200_batch_f32": (_int, _batch),
    "caf_b200_batch_f64_dev": (_int, _batch),
    "caf_b200_batch_f32_dev": (_int, _batch),
    "caf_b200_surface_layout_f64": (_int, [_vp, _vp, _vp, _sz, _vp, _sz, _u32, _int, _vp, _vp]),
    "caf_b200_surface_layout_f32": (_int, [_vp, _vp, _vp, _sz, _vp, _sz, _u32, _int, _vp, _vp]),
    "caf_b200_comm_unique_id": (_int, [_vp]),
    "caf_b200_comm_create": (_int, [_vp, _int, _int, _vp, C.POINTER(_vp)]),
    "caf_b200_comm_adopt": (_int, [_vp, _vp, _int, _int, C.POINTER(_vp)]),
    "caf_b200_comm_destroy": (_int, [_vp]),
    "caf_b200_comm_shard": (_int, [_vp, _sz, C.POINTER(_sz), C.POINTER(_sz)]),
    "caf_b200_peak_allgather_dev": (_int, [_vp, _vp, _vp, C.c_uint64, _PK]),
    "caf_b200_surface_sharded_f64": (_int, [_vp, _vp, _vp, _vp, _sz, _vp, _sz, _u32, _vp, _PK]),
    "caf_b200_surface_sharded_f32": (_int, [_vp, _vp, _vp, _vp, _sz, _vp, _sz, _u32, _vp, _PK]),
    "caf_b200_peak_pack": (None, [_PK, C.c_uint64, C.POINTER(C.c_uint64)]),
    "caf_b200_peak_resolve": (None, [C.POINTER(C.c_uint64), _sz, _PK]),
    "caf_b200_surface_create_f64": (_int, [_vp, _vp, _vp, _sz, _vp, _sz, _u32, C.POINTER(_vp)]),
    "caf_b200_surface_create_f32": (_int, [_vp, _vp, _vp, _sz, _vp, _sz, _u32, C.POINTER(_vp)]),
    "caf_b200_surface_shape": (_int, [_vp, C.POINTER(_sz), C.POINTER(_sz)]),
    "caf_b200_surface_row_peaks": (_int, [_vp, _vp, _vp, _vp]),
    "caf_b200_surface_find_peak": (_int, [_vp, _PK]),
    "caf_b200_surface_fetch_rows": (_int, [_vp, _sz, _sz, _vp]),
    "caf_b200_surface_destroy": (_int, [_vp]),
    "caf_b200_surface_detect": (_int, [_vp, _sz, _u32, _u32, _dbl, C.POINTER(Detection), C.POINTER(_sz)]),
    "caf_b200_detect_f64_dev": (_int, _detect_dev),
    "caf_b200_detect_f32_dev": (_int, _detect_dev),
    "caf_b200_surface_detect_cfar": (_int, [_vp, _sz, _u32, _u32, _u32, _u32, _dbl, C.POINTER(CfarDetection),
                                            C.POINTER(_sz)]),
    "caf_b200_detect_cfar_f64_dev": (_int, _cfar_dev),
    "caf_b200_detect_cfar_f32_dev": (_int, _cfar_dev),
    "caf_b200_cfar_noise_f64_dev": (_int, _cfar_noise),
    "caf_b200_cfar_noise_f32_dev": (_int, _cfar_noise),
    "caf_b200_surface_detect_cfar_os": (_int, [_vp, _sz, _u32, _u32, _u32, _u32, _u32, _dbl, C.POINTER(CfarDetection),
                                               C.POINTER(_sz)]),
    "caf_b200_detect_cfar_os_f64_dev": (_int, _cfar_os_dev),
    "caf_b200_detect_cfar_os_f32_dev": (_int, _cfar_os_dev),
    "caf_b200_cfar_os_noise_f64_dev": (_int, _cfar_os_noise),
    "caf_b200_cfar_os_noise_f32_dev": (_int, _cfar_os_noise),
    "caf_b200_peak_resolve_status": (_int, [C.POINTER(C.c_uint64), _sz, _PK]),
    "caf_b200_peak_allgather_async": (_int, [_vp, _vp, _vp, C.c_uint64, _vp]),
    "caf_b200_comm_remote_error": (_int, [_vp, C.POINTER(_int)]),
    "caf_b200_comm_uses_p2p": (_int, [_vp, C.POINTER(_int)]),
    "caf_b200_sharded_f64_dev": (_int, [_vp, _vp, _vp, _vp, _sz, _vp, _sz, C.c_uint64, _u32, _vp, _vp, _vp, _vp]),
    "caf_b200_sharded_f32_dev": (_int, [_vp, _vp, _vp, _vp, _sz, _vp, _sz, C.c_uint64, _u32, _vp, _vp, _vp, _vp]),
    "caf_b200_detect_rows_f64_dev": (_int, _detect_rows),
    "caf_b200_detect_rows_f32_dev": (_int, _detect_rows),
    "caf_b200_detect_cfar_rows_f64_dev": (_int, _cfar_rows),
    "caf_b200_detect_cfar_rows_f32_dev": (_int, _cfar_rows),
    "caf_b200_detect_cfar_os_rows_f64_dev": (_int, _cfar_os_rows),
    "caf_b200_detect_cfar_os_rows_f32_dev": (_int, _cfar_os_rows),
    "caf_b200_detect_merge_dev": (_int, [_vp, _vp, _vp, _sz, _sz, _dbl, _vp, _vp]),
    "caf_b200_cfar_merge_dev": (_int, [_vp, _vp, _vp, _sz, _sz, _vp, _vp]),
    "caf_b200_detect_allgather_dev": (_int, [_vp, _vp, _vp, _vp, _sz, _dbl, _vp, _vp]),
    "caf_b200_cfar_allgather_dev": (_int, [_vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    "caf_b200_integrate_f64_dev": (_int, _batch),
    "caf_b200_integrate_f32_dev": (_int, _batch),
    "caf_b200_surface_create_integrated_f64": (_int, [_vp, _vp, _vp, _sz, _sz, _vp, _sz, _u32, C.POINTER(_vp)]),
    "caf_b200_surface_create_integrated_f32": (_int, [_vp, _vp, _vp, _sz, _sz, _vp, _sz, _u32, C.POINTER(_vp)]),
}

_lib = None


def _prefer_bundled_nccl():
    """The library dlopen()s libnccl.so.2 lazily (caf_b200_comm_*).  In a Python process that may later import torch,
    the copy loaded first wins for everybody (same soname), and torch needs ITS bundled NCCL: point the library at
    that copy unless the caller chose one (CAF_B200_NCCL_LIB).  A process without the wheel uses the system NCCL."""
    if os.environ.get("CAF_B200_NCCL_LIB"):
        return
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for base in (list(spec.submodule_search_locations or []) if spec else []):
            cand = os.path.join(base, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ["CAF_B200_NCCL_LIB"] = cand
                return
    except Exception:
        pass


def load():
    """dlopen the in-tree library and type every entry point.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        _prefer_bundled_nccl()
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        lib = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)   # AttributeError if the header and the library ever disagree
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
