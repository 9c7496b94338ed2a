"""caf_cookoff_b200 — B200-native filterbank cross-ambiguity function behind caf_rust's API.

Only the hot path of Teque5/caf_cookoff lives here (SURVEY.md section 8): csrc/ holds the sm_100a
kernels and the C ABI (include/caf_b200.h); api.py mirrors `caf_rust::caf::*`; io.py mirrors
`caf_rust::utils`; siblings.py reproduces the Go / Python programs' layouts from the same kernels; generate.py is the seeded port of utils/generate.py.
"""
from .api import (CafB200, CafB200F32, CafError, CafFFTW, CafPanic, CafRustFFT, CafRustFFTIter,
                  CafRustFFTIterRayon, CafRustFFTRayon, CafRustFFTThreadpool, CafRustFFTThreads,
                  CafSurface, CafSurfaceRow, DeviceSurface, Handle, Surface, Xcor, XcorF32, batch_arrays, default_handle, detect_dev,
                  peak_pack, peak_resolve, surface_arrays)
from .io import DeviceSamples, bench_shifts, gen_float_shifts, read_file_c64, read_file_c64_dev, write_file_binary
from .siblings import GoSibling, PythonSibling, surface_layout

__all__ = [n for n in dir() if not n.startswith("_")]
