/*
 * caf_b200.h — C ABI of the B200-native filterbank cross-ambiguity function (libcaf_b200.so).
 *
 * The reference (Teque5/caf_cookoff, caf_rust) has no FFI: its boundary is the Rust crate API
 *     pub trait CafSurface { caf_surface, find_peak, apply_freq_shift }   caf_rust/src/caf/mod.rs:23-66
 *     pub struct CafSurfaceRow                                            caf_rust/src/caf/mod.rs:17-22
 *     struct Xcor { new, run }  (crate-private)                           caf_rust/src/caf/xcor_rustfft.rs:14-78
 * Each entry point below names the reference function it replaces; INTEGRATION.md shows the Rust
 * `extern "C"` block + trait impl a maintainer adds to bind them (rust/ holds that shim as source).
 *
 * Conventions
 *  - every function returns 0 on success, a negative caf_b200_status otherwise; the message of the
 *    last failure on the calling thread is caf_b200_last_error().  Nothing aborts or throws.
 *    (The reference panics instead — xcor_rustfft.rs:54-55 assert!, unwrap()s; the Rust shim turns a
 *    non-zero status into panic! to preserve that.)
 *  - caf_c128 / caf_c64 are interleaved (re, im) and layout-identical to num_complex::Complex<f64> /
 *    Complex<f32> (#[repr(C)]) and to numpy complex128 / complex64.
 *  - pointers are caller-owned HOST memory unless the function name ends in _dev (device memory on the
 *    handle's device; those calls are asynchronous on the handle's stream — caf_b200_sync() to wait).
 *  - a handle owns one device, one stream, the twiddle tables and a grow-only workspace.  A handle is
 *    not thread-safe; distinct handles are independent.
 *  - there is NO CPU fallback: if no sm_100 device is usable, create() fails.
 *
 * Environment (development / measurement switches, read ONCE when a handle is created; none is needed for normal use):
 *    CAF_B200_CHUNK_MB=<n>   scratch budget for rows longer than 8192 cells (default 6144)
 *    CAF_B200_INTEGRATE_MB=<n>  caf_b200_integrate_*: scratch budget for one chunk of segment surfaces (default 256)
 *    CAF_B200_PIPELINE=0     host surface calls: one launch + one D2H copy instead of head/rest overlap
 *    CAF_B200_PEAK_ZEROCOPY=0  single-pair host calls: copy the peak back instead of storing it into pinned host memory
 *    CAF_B200_PULL=0         single-pair host calls: one H2D copy in front of the kernel instead of the kernel's own CTAs
 *                            reading the pinned input block across PCIe
 *    CAF_B200_OVERLAP=0      caf_b200_set_overlap is accepted and ignored: every launch keeps full stream order
 *    CAF_B200_P2P=0          cross-rank find_peak by ncclAllGather instead of the peer-memory mailbox kernel (read at comm creation)
 *    CAF_B200_NCCL_LIB=<so>  which libnccl to dlopen for caf_b200_comm_* (default: the loaded one, then libnccl.so.2)
 *
 * Sizes.  l = samples per input signal (needle and haystack must be equal length, as the reference's
 * Xcor asserts).  A surface row has n = 2*l delay cells (both inputs zero-padded at the end to 2*l,
 * mod.rs:130-131); cell k < l is lag +k, cell k > l is lag k - 2l.  Rows stay in on-chip memory for l <= 4096
 * (the reference's only shape is l = 4096); 4096 < l <= 2^19 runs a four- or six-step FFT through L2 (BASELINE
 * configs 3 and 5); larger l returns CAF_B200_EUNSUPPORTED.
 */
#ifndef CAF_B200_H
#define CAF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct caf_b200_handle_s* caf_b200_handle;

typedef struct { double re, im; } caf_c128;   /* == num_complex::Complex64  (utils.rs:8-9) */
typedef struct { float re, im; } caf_c64;     /* == num_complex::Complex32 */

typedef enum {
    CAF_B200_OK = 0,
    CAF_B200_EINVAL = -1,        /* null pointer / bad argument */
    CAF_B200_ELENGTH = -2,       /* needle.len() != haystack.len()  (xcor_rustfft.rs:54-55 assert) */
    CAF_B200_EUNSUPPORTED = -3,  /* size outside what this build implements */
    CAF_B200_ECUDA = -4,         /* CUDA runtime error (message in last_error) */
    CAF_B200_ENODEVICE = -5,     /* no usable sm_100 GPU — there is no CPU fallback */
    CAF_B200_ENCCL = -6,         /* NCCL missing or an NCCL call failed (message in last_error) */
    CAF_B200_EREMOTE = -7,       /* sharded call: a PEER rank failed before the peak exchange (every rank still left the collective) */
    CAF_B200_EIO = -8            /* a sample file could not be opened or read (utils.rs:10's io::Result Err) */
} caf_b200_status;

/* Result of CafSurface::find_peak (mod.rs:31-42).  When no row beats the dummy 0.0 row (empty or
 * all-zero surface) the reference returns (0.0, 0): value = 0, freq_hz = 0, delay_idx = 0 and
 * doppler_idx = UINT64_MAX. */
typedef struct {
    double value;          /* |xcor|^2 at the peak */
    double freq_hz;        /* freqs_hz[doppler_idx] */
    uint64_t doppler_idx;  /* first row holding the maximum (rows in freqs_hz order) */
    uint64_t delay_idx;    /* xcor_peak_idx of that row */
} caf_b200_peak;

/* ---- lifecycle ------------------------------------------------------------------------------- */
int caf_b200_create(int device, caf_b200_handle* out);
/* Same, but all work is issued on an existing CUDA stream (a cudaStream_t passed as void*; NULL is the
 * legacy default stream, exactly as in the CUDA runtime). */
int caf_b200_create_on_stream(int device, void* cuda_stream, caf_b200_handle* out);
int caf_b200_destroy(caf_b200_handle h);
int caf_b200_sync(caf_b200_handle h);
const char* caf_b200_last_error(void);
const char* caf_b200_version(void);
/* number of kernels this handle has launched since creation (bench.py's gpu_launches) */
uint64_t caf_b200_launch_count(caf_b200_handle h);

/* Per-kernel device times of the LAST surface/batch call on this handle, in milliseconds, measured with
 * CUDA events on the handle's stream.  Off by default (the events cost a little); when on, every
 * surface/batch call records spectrum (FFT(s1)), rows (the fused row kernel) and peak (find_peak). */
/* Overlap of consecutive single-pair device launches (caf_b200_batch_*_dev with p = 1): mode 0 = off (the default).
 * Such a launch is issued with programmatic stream serialisation.  With mode >= 1, when it directly follows another one
 * on the handle, has at least one row per SM, and the library finds every buffer of this launch disjoint from those of the
 * previous SEVEN launches wherever one side writes, it does not wait for the grid before it: its CTAs start their rows on
 * whatever SMs are free.  mode 1 keeps one CTA per SM (400 rows on 148 SMs leave 44 SMs a row early: 37.9 -> 33.4 us per
 * surface).  mode n = 2..4 gives an overlapped launch only ceil(SMs / n) CTAs, so that about n launches share the GPU and
 * every CTA spreads its set-up over n times as many rows: 29.1 / 27.9 / 27.2 us per surface for n = 2 / 3 / 4 -- at the
 * price of latency, a single surface then takes ~n x 30 us from launch to completion.  Results are bit-identical in every
 * mode.  Switching it on is the caller's promise that (a) nothing it enqueues on the handle's stream between two library
 * calls produces data the later call reads, and (b) it does not rely on a launch being complete before the next one has
 * begun (results are complete, in order, when the stream reaches whatever follows the last launch: an event, a copy, a
 * synchronise).  Launches that alias their predecessors' buffers, problems with fewer rows than SMs, host-pointer calls
 * and everything else keep full stream order -- so a caller who wants the overlap sustained rotates its output buffers
 * (surface, row peaks, peak) over at least eight sets; inputs may be shared freely, they are only read. */
int caf_b200_set_overlap(caf_b200_handle h, int mode);
int caf_b200_set_profiling(caf_b200_handle h, int on);
int caf_b200_last_kernel_ms(caf_b200_handle h, float* spectrum_ms, float* rows_ms, float* peak_ms);
/* FMA-pipe peak probe used as the roofline denominator: runs a dependent-FMA kernel on every SM and
 * returns achieved TFLOP/s (2 flops per FMA).  is_f64 != 0 -> double, else float. */
int caf_b200_probe_fma_tflops(caf_b200_handle h, int is_f64, double* tflops);

/* development hook: phase time stamps of the row kernel; only in -DCAF_TRACE builds (else EUNSUPPORTED) */
int caf_b200_debug_trace(caf_b200_handle h, long long* out, size_t n_cta);

/* pinned host buffers: surfaces DMA straight into them (any host pointer is accepted, pinned is faster) */
int caf_b200_host_alloc(void** out, size_t bytes);
int caf_b200_host_free(void* p);

/* ---- read_file_c64 (utils.rs:10-35) straight onto the device ------------------------------------------------------
 * The file's packed little-endian f32 I/Q pairs are read into pinned memory, cross PCIe as they are (8 bytes per sample
 * instead of the 16 of the widened Vec<Complex64>) and are widened on the GPU (f32 -> f64 is exact: the device samples
 * equal read_file_c64's bit for bit).  first_sample / max_samples select a window of the file (max_samples = 0: to its
 * end).  *dev_out is device memory on the handle's device -- complex128 for _f64, complex64 for _f32 -- for the *_dev
 * entry points; release it with caf_b200_dev_free.  A file that cannot be opened is CAF_B200_EIO (the reference returns
 * io::Result Err, utils.rs:10); a trailing partial sample is CAF_B200_EINVAL (the reference's slice index panics). */
int caf_b200_load_c64_dev_f64(caf_b200_handle h, const char* path, size_t first_sample, size_t max_samples,
                              caf_c128** dev_out, size_t* n_out);
int caf_b200_load_c64_dev_f32(caf_b200_handle h, const char* path, size_t first_sample, size_t max_samples,
                              caf_c64** dev_out, size_t* n_out);
int caf_b200_dev_free(void* dev_ptr);
/* device memory for callers that do not link the CUDA runtime themselves (the Rust shim, the C++ mirror): what the *_dev
 * entry points take and fill.  upload / download are synchronous on the handle's stream. */
int caf_b200_dev_alloc(caf_b200_handle h, size_t bytes, void** dev_out);
int caf_b200_dev_upload(caf_b200_handle h, void* dev_dst, const void* host_src, size_t bytes);
int caf_b200_dev_download(caf_b200_handle h, void* host_dst, const void* dev_src, size_t bytes);

/* ---- CafSurface::apply_freq_shift (mod.rs:46-65); README.md:124 calls it apply_shift ------------ */
/* out[i] = in[i] * e^{+j 2 pi freq_hz i / fs}.  in == out allowed. */
int caf_b200_apply_freq_shift_f64(caf_b200_handle h, const caf_c128* in, size_t n, double freq_hz,
                                  uint32_t fs, caf_c128* out);
int caf_b200_apply_freq_shift_f32(caf_b200_handle h, const caf_c64* in, size_t n, double freq_hz,
                                  uint32_t fs, caf_c64* out);
int caf_b200_apply_shift_f64(caf_b200_handle h, const caf_c128* in, size_t n, double freq_hz,
                             uint32_t fs, caf_c128* out);   /* alias */
int caf_b200_apply_shift_f32(caf_b200_handle h, const caf_c64* in, size_t n, double freq_hz,
                             uint32_t fs, caf_c64* out);    /* alias */

/* ---- Xcor::run (xcor_rustfft.rs:51-78 / xcor_fftw.rs:51-78) ----------------------------------------
 * out = IFFT( FFT(a) * conj(FFT(b)) / n ), unnormalised transforms: the length-n CIRCULAR correlation
 * out[k] = sum_m a[(m+k) mod n] conj(b[m]).  Any n <= 2^19 (n <= 4096 and n == 8192 stay
 * on chip; other lengths run one row of the long-row kernels and fold the linear correlation). */
int caf_b200_xcor_f64(caf_b200_handle h, const caf_c128* a, const caf_c128* b, size_t n, caf_c128* out);
int caf_b200_xcor_f32(caf_b200_handle h, const caf_c64* a, const caf_c64* b, size_t n, caf_c64* out);

/* ---- CafSurface::caf_surface + find_peak (mod.rs:121-166, 31-42) -----------------------------------
 * needle, haystack: l samples each.  freqs_hz: d doppler shifts.  fs: sample rate (u32 as in the trait).
 * surface: d x 2l row-major |xcor|^2 (norm_sqr, mod.rs:147) or NULL to skip materialising it.
 * row_peak_val / row_peak_idx: CafSurfaceRow::xcor_peak_val / xcor_peak_idx per row, or NULL.
 * peak: find_peak over the rows in freqs_hz order, or NULL. */
int caf_b200_surface_f64(caf_b200_handle h, const caf_c128* needle, const caf_c128* haystack, size_t l,
                         const double* freqs_hz, size_t d, uint32_t fs,
                         double* surface, double* row_peak_val, uint64_t* row_peak_idx, caf_b200_peak* peak);
int caf_b200_surface_f32(caf_b200_handle h, const caf_c64* needle, const caf_c64* haystack, size_t l,
                         const double* freqs_hz, size_t d, uint32_t fs,
                         float* surface, float* row_peak_val, uint64_t* row_peak_idx, caf_b200_peak* peak);

/* peak only: caf_surface followed by find_peak with the surface never leaving the chip */
int caf_b200_peak_f64(caf_b200_handle h, const caf_c128* needle, const caf_c128* haystack, size_t l,
                      const double* freqs_hz, size_t d, uint32_t fs, caf_b200_peak* peak);
int caf_b200_peak_f32(caf_b200_handle h, const caf_c64* needle, const caf_c64* haystack, size_t l,
                      const double* freqs_hz, size_t d, uint32_t fs, caf_b200_peak* peak);

/* p independent pairs, each l samples, one shared doppler grid: needles / haystacks are [p][l],
 * surface [p][d][2l] or NULL, row_peak_* [p][d] or NULL, peaks [p] or NULL. */
int caf_b200_batch_f64(caf_b200_handle h, const caf_c128* needles, const caf_c128* haystacks, size_t p,
                       size_t l, const double* freqs_hz, size_t d, uint32_t fs,
                       double* surface, double* row_peak_val, uint64_t* row_peak_idx, caf_b200_peak* peaks);
int caf_b200_batch_f32(caf_b200_handle h, const caf_c64* needles, const caf_c64* haystacks, size_t p,
                       size_t l, const double* freqs_hz, size_t d, uint32_t fs,
                       float* surface, float* row_peak_val, uint64_t* row_peak_idx, caf_b200_peak* peaks);

/* device-resident variants: every pointer is device memory (peaks too); asynchronous on the handle's
 * stream.  Same argument meaning as the batch calls. */
int caf_b200_batch_f64_dev(caf_b200_handle h, const caf_c128* needles, const caf_c128* haystacks, size_t p,
                           size_t l, const double* freqs_hz, size_t d, uint32_t fs,
                           double* surface, double* row_peak_val, uint64_t* row_peak_idx, caf_b200_peak* peaks);
int caf_b200_batch_f32_dev(caf_b200_handle h, const caf_c64* needles, const caf_c64* haystacks, size_t p,
                           size_t l, const double* freqs_hz, size_t d, uint32_t fs,
                           float* surface, float* row_peak_val, uint64_t* row_peak_idx, caf_b200_peak* peaks);

/* ---- device-resident surface objects ---------------------------------------------------------------------
 * CafSurfaceRow's fields are PRIVATE in the reference (mod.rs:17-22): a caller of caf_surface can hand the rows to
 * find_peak and nothing else, so copying 26 MB of |xcor|^2 to the host on every call (0.5 ms against a ~45 us kernel)
 * buys nothing.  caf_b200_surface_create_* runs caf_surface and keeps the surface on the GPU; what comes back at once is
 * per row (freq, xcor_peak_val, xcor_peak_idx) -- 24 bytes -- and find_peak's answer.  The Rust shim's CafSurfaceRow holds
 * a reference-counted surface object + its row number and fetches xcor_mag only if asked (rust/src/caf/mod.rs).
 * A surface object belongs to the handle that made it (its buffer returns to that handle's pool on destroy; destroying
 * the handle first is allowed).  fetch_rows is thread-safe; create / destroy follow the handle's threading rule. */
typedef struct caf_b200_surface_s* caf_b200_surface;
int caf_b200_surface_create_f64(caf_b200_handle h, const caf_c128* needle, const caf_c128* haystack, size_t l,
                                const double* freqs_hz, size_t d, uint32_t fs, caf_b200_surface* out);
int caf_b200_surface_create_f32(caf_b200_handle h, const caf_c64* needle, const caf_c64* haystack, size_t l,
                                const double* freqs_hz, size_t d, uint32_t fs, caf_b200_surface* out);
int caf_b200_surface_shape(caf_b200_surface s, size_t* rows, size_t* cells_per_row);
/* CafSurfaceRow::{freq, xcor_peak_val, xcor_peak_idx} of every row (any pointer may be NULL) */
int caf_b200_surface_row_peaks(caf_b200_surface s, double* freq_hz, double* peak_val, uint64_t* peak_idx);
/* CafSurface::find_peak (mod.rs:31-42) over the rows in freqs_hz order, computed by the kernel that made them */
int caf_b200_surface_find_peak(caf_b200_surface s, caf_b200_peak* out);
/* CafSurfaceRow::xcor_mag of rows [row0, row0 + count): count * cells_per_row doubles (floats for an f32 surface) */
int caf_b200_surface_fetch_rows(caf_b200_surface s, size_t row0, size_t count, void* out);
int caf_b200_surface_destroy(caf_b200_surface s);

/* ---- detection: the k_max strongest local maxima of a stored surface, refined below the grid -----------------------
 * Surfaces are the Rust layout above: p pairs x d rows x n cells of |xcor|^2, rows in freqs_hz order, cell k holding lag k
 * when 2k < n and k - n otherwise.  The window of cell (r, k) is rows r +- guard_doppler (clipped to the surface) times
 * cells (k + j) mod n for |j| <= guard_delay (the delay axis is circular), without the cell itself.  A cell of value v is a
 * local maximum when v > 0, no window cell exceeds v, and no window cell equal to v has a smaller flat index r * n + k
 * (one cell per plateau; NaN cells never qualify and never block).  Local maxima are ordered by value descending, then
 * flat index ascending; the first k_max are kept, then every one below min_ratio x the first is dropped.  Detection 0 is
 * therefore find_peak's cell whenever the surface has a positive cell.
 * Refinement, in double from the stored values: a 3-point parabola through (k - 1, k, k + 1) of the row (cells wrap; no fit
 * when n < 3) and through rows (r - 1, r, r + 1) at cell k (no fit on the first and last row); each offset is clamped to
 * +-0.5 and is 0 where the three points do not curve down.  lag_samples = signed lag + delay offset; freq_hz_interp moves
 * from freqs_hz[r] by the Doppler offset times the grid step on that side (non-uniform grids work).
 * Slots [count, k_max) hold value 0, freq 0, doppler_idx UINT64_MAX, delay 0, lag 0, freq_interp 0.
 * Limits: 1 <= k_max <= 1024, guard_doppler <= 32, guard_delay <= 256 with 2 * guard_delay + 1 <= n (n > 0),
 * 0 <= min_ratio <= 1; anything else, or a null pointer, is CAF_B200_EINVAL and writes nothing.  An empty surface gives a
 * count of 0.  Scratch comes from the handle's grow-only workspace: per tile of tr <= 16 rows x 256 cells, 16 bytes x
 * min(k_max, ceil(tr / (guard_doppler + 1)) x ceil(256 / (guard_delay + 1))) -- no tile holds more local maxima than that
 * (at most 4 bytes per cell with guards of 1 x 1, 16 with none). */
typedef struct {
    double value;           /* |xcor|^2 at the cell (the first four fields are caf_b200_peak's) */
    double freq_hz;         /* freqs_hz[doppler_idx] */
    uint64_t doppler_idx;   /* row */
    uint64_t delay_idx;     /* cell */
    double lag_samples;     /* signed lag of delay_idx + parabolic offset */
    double freq_hz_interp;  /* freqs_hz interpolated at doppler_idx + parabolic offset */
} caf_b200_detection;
/* a surface object (f64 or f32); synchronous, host output (k_max records); needs the surface's handle alive (else EINVAL).
 * It runs on the surface's handle (its stream, workspace and launch count), so unlike fetch_rows it follows the handle's
 * threading rule: call it where that handle may be used, never at the same time as another call on it. */
int caf_b200_surface_detect(caf_b200_surface s, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                            double min_ratio, caf_b200_detection* out, size_t* count);
/* device surfaces [p][d][n] (e.g. from caf_b200_batch_*_dev); out [p][k_max] and counts [p] in device memory; two plain
 * stream-ordered launches on the handle's stream (they see every earlier launch complete and count in launch_count) */
int caf_b200_detect_f64_dev(caf_b200_handle h, const double* surface, size_t p, size_t d, size_t n,
                            const double* freqs_hz, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                            double min_ratio, caf_b200_detection* out, uint64_t* counts);
int caf_b200_detect_f32_dev(caf_b200_handle h, const float* surface, size_t p, size_t d, size_t n,
                            const double* freqs_hz, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                            double min_ratio, caf_b200_detection* out, uint64_t* counts);

/* ---- CFAR detection: local maxima that stand above a local noise estimate (cell-averaging CFAR) ---------------------
 * detect() ranks candidates; this decides whether anything is there.  Surfaces and the window rule are detect's; gr, gd
 * are guard_doppler, guard_delay (the local-maximum window and the CFAR guard region), tr, tc are train_doppler,
 * train_delay, and R = gr + tr, C = gd + tc.
 * Training cells of (r, k): rows r' in [r - R, r + R] clipped to [0, d), each taking cells (k + j) mod n for |j| <= C,
 * without those with |r' - r| <= gr and |j| <= gd; NaN cells are skipped.  m = how many remain.
 * noise, in ONE summation order (so the GPU, the dense map and any restatement agree bit for bit): each row r' sums +0.0
 * plus its training cells in ascending j, in double (f32 values widened first); the cell sums +0.0 plus those row sums in
 * ascending r'; noise = sum / m, correctly rounded, NaN when m = 0.  Only non-negative additions: no cancellation next to
 * a strong peak (which a running sum, adding the entering cell and subtracting the leaving one, would suffer).
 * Cell (r, k) of value v is a detection when it is a local maximum under detect's rule with (gr, gd), m > 0 and
 * v > scale * noise (correctly rounded product).  Detections are ordered by value descending, then flat index ascending,
 * and cut to k_max (no min_ratio); each is refined exactly as in detect.  Detection 0 need not be find_peak's cell, and
 * the list may be empty: a surface that holds nothing above its noise gives count 0.
 * Limits: 1 <= k_max <= 1024, gr + tr <= 32, gd + tc <= 256, tr + tc >= 1, 2C + 1 <= n (n > 0), scale finite and > 0, no
 * null pointer; anything else is CAF_B200_EINVAL and writes nothing.  An empty surface gives a count of 0.
 * Threshold: for N i.i.d. exponential training cells (|.|^2 of complex Gaussian noise) and a test cell of the same law,
 * P(v > a * mean) = (1 + a / N)^-N, so scale = N (Pfa^(-1/N) - 1) with N = (2R+1)(2C+1) - (2gr+1)(2gd+1) gives false-alarm
 * probability Pfa for the threshold test alone (before the local-maximum rule; edge rows have fewer training cells; the
 * correlation between CAF cells is not modelled).  The Python package's cfar_scale / cfar_train_cells compute it.
 * Scratch: as detect, 32 bytes per candidate slot. */
typedef struct {
    double value;           /* the first six fields are caf_b200_detection's, in its order */
    double freq_hz;
    uint64_t doppler_idx;   /* UINT64_MAX in unused slots */
    uint64_t delay_idx;
    double lag_samples;
    double freq_hz_interp;
    double noise;           /* the cell's noise estimate (0 in unused slots) */
    uint64_t train_cells;   /* m, the training cells averaged (0 in unused slots) */
} caf_b200_cfar_detection;
/* a surface object; synchronous, host records; same handle rule as caf_b200_surface_detect */
int caf_b200_surface_detect_cfar(caf_b200_surface s, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                 uint32_t train_doppler, uint32_t train_delay, double scale, caf_b200_cfar_detection* out,
                                 size_t* count);
/* device surfaces [p][d][n]; out [p][k_max] and counts [p] in device memory; two plain stream-ordered launches */
int caf_b200_detect_cfar_f64_dev(caf_b200_handle h, const double* surface, size_t p, size_t d, size_t n,
                                 const double* freqs_hz, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                 uint32_t train_doppler, uint32_t train_delay, double scale, caf_b200_cfar_detection* out,
                                 uint64_t* counts);
int caf_b200_detect_cfar_f32_dev(caf_b200_handle h, const float* surface, size_t p, size_t d, size_t n,
                                 const double* freqs_hz, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                 uint32_t train_doppler, uint32_t train_delay, double scale, caf_b200_cfar_detection* out,
                                 uint64_t* counts);
/* the dense noise map: noise_out [p][d][n] doubles (device), NaN where m = 0, bit for bit the noise of every record above;
 * one stream-ordered launch (none for an empty surface).  Limits as above without k_max and scale. */
int caf_b200_cfar_noise_f64_dev(caf_b200_handle h, const double* surface, size_t p, size_t d, size_t n,
                                uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler, uint32_t train_delay,
                                double* noise_out);
int caf_b200_cfar_noise_f32_dev(caf_b200_handle h, const float* surface, size_t p, size_t d, size_t n,
                                uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler, uint32_t train_delay,
                                double* noise_out);

/* ---- OS-CFAR detection: the same, against an order statistic of the training cells (ordered-statistic CFAR) ---------
 * CA-CFAR's mean moves with every strong cell in the training region: an emitter's own Doppler main lobe raises its
 * threshold, and a weak emitter inside a strong one's region is masked.  Here the noise estimate is the rank-th smallest of
 * N training cells instead, which a few strong cells do not move.  Surfaces, windows, training cells, m, N, the detection
 * rule, records and refinement are CA-CFAR's above; only noise differs:
 * each training value is widened to double and +0.0 is added (-0.0 counts as +0.0); with k_m = ceil(rank * m / N) in
 * 64-bit integers, noise is the k_m-th smallest of those m values, NaN when m = 0.  It is one of the values, not a rounded
 * sum, so every path (records, the dense map, any restatement) agrees bit for bit.  A record's train_cells is m.
 * Limits: CA-CFAR's, plus 1 <= rank <= N; anything else is CAF_B200_EINVAL and writes nothing.
 * Threshold: for N i.i.d. exponential cells and a test cell of the same law, P(v > a * X_(k)) = prod_{i<k} (N-i)/(N-i+a);
 * the Python package's cfar_os_scale solves it for a.  The caveats of cfar_scale apply (the threshold test alone, edge rows
 * with fewer cells, correlated CAF cells), and order statistics of correlated cells stray further from the model: expect
 * more crossings on noise than the nominal Pfa.
 * Scratch: as CA-CFAR. */
/* a surface object; synchronous, host records; same handle rule as caf_b200_surface_detect */
int caf_b200_surface_detect_cfar_os(caf_b200_surface s, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                    uint32_t train_doppler, uint32_t train_delay, uint32_t rank, double scale,
                                    caf_b200_cfar_detection* out, size_t* count);
/* device surfaces [p][d][n]; out [p][k_max] and counts [p] in device memory; two plain stream-ordered launches */
int caf_b200_detect_cfar_os_f64_dev(caf_b200_handle h, const double* surface, size_t p, size_t d, size_t n,
                                    const double* freqs_hz, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                    uint32_t train_doppler, uint32_t train_delay, uint32_t rank, double scale,
                                    caf_b200_cfar_detection* out, uint64_t* counts);
int caf_b200_detect_cfar_os_f32_dev(caf_b200_handle h, const float* surface, size_t p, size_t d, size_t n,
                                    const double* freqs_hz, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                    uint32_t train_doppler, uint32_t train_delay, uint32_t rank, double scale,
                                    caf_b200_cfar_detection* out, uint64_t* counts);
/* the dense map: noise_out [p][d][n] doubles (device), NaN where m = 0, bit for bit the noise of every record above; one
 * stream-ordered launch (none for an empty surface).  Limits as above without k_max and scale. */
int caf_b200_cfar_os_noise_f64_dev(caf_b200_handle h, const double* surface, size_t p, size_t d, size_t n,
                                   uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler,
                                   uint32_t train_delay, uint32_t rank, double* noise_out);
int caf_b200_cfar_os_noise_f32_dev(caf_b200_handle h, const float* surface, size_t p, size_t d, size_t n,
                                   uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler,
                                   uint32_t train_delay, uint32_t rank, double* noise_out);

/* ---- detection on row-sharded surfaces: each rank searches its rows with a halo, one merge gives the one-GPU answer --
 * A rank owns global rows [lo, hi) of a surface of d_global rows (e.g. from caf_b200_comm_shard).  It computes a BLOCK of
 * d_buf rows whose row 0 is global row row_offset and that covers its owned rows plus H rows on each side, clipped to the
 * surface (the surface calls give bit-identical rows for any sub-grid, so nothing is exchanged for the halo).  In the
 * block the owned rows are [row_lo, row_hi) = [lo - row_offset, hi - row_offset).  H is the depth of a detector's
 * neighbourhood: max(guard_doppler, 1) for detect (window, equal-value rule, Doppler parabola) and
 * max(guard_doppler + train_doppler, 1) for both CFAR detectors (their training rows).
 * The *_rows_* calls run a detector over the owned rows only, reading the rest of the block as neighbourhood: every owned
 * cell sees exactly what it sees on the whole surface, so its decision, refinement, noise and m are the whole-surface
 * ones.  Records carry the GLOBAL row in doppler_idx; freq_hz and freq_hz_interp come from freqs_hz, the block's own grid
 * (d_buf values).  The list is the rank's best k_max (detect: also cut at min_ratio x the rank's first, which never drops
 * a record the global cut keeps).  p = 1; out [k_max] and count in device memory; two stream-ordered launches.
 * Limits: each detector's own (with d = d_buf), and row_lo <= row_hi <= d_buf, row_offset + d_buf <= d_global <= 2^31,
 * and at least H block rows above row_lo unless the block starts the surface (row_offset == 0), and below row_hi unless
 * it ends the surface (row_offset + d_buf == d_global); anything else is CAF_B200_EINVAL and writes nothing.  An empty owned range
 * (row_lo == row_hi: a rank may own no rows) needs no halo and gives count 0. */
int caf_b200_detect_rows_f64_dev(caf_b200_handle h, const double* surface, size_t d_buf, size_t n, const double* freqs_hz,
                                 size_t row_lo, size_t row_hi, uint64_t row_offset, size_t d_global, size_t k_max,
                                 uint32_t guard_doppler, uint32_t guard_delay, double min_ratio, caf_b200_detection* out,
                                 uint64_t* count);
int caf_b200_detect_rows_f32_dev(caf_b200_handle h, const float* surface, size_t d_buf, size_t n, const double* freqs_hz,
                                 size_t row_lo, size_t row_hi, uint64_t row_offset, size_t d_global, size_t k_max,
                                 uint32_t guard_doppler, uint32_t guard_delay, double min_ratio, caf_b200_detection* out,
                                 uint64_t* count);
int caf_b200_detect_cfar_rows_f64_dev(caf_b200_handle h, const double* surface, size_t d_buf, size_t n,
                                      const double* freqs_hz, size_t row_lo, size_t row_hi, uint64_t row_offset,
                                      size_t d_global, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                      uint32_t train_doppler, uint32_t train_delay, double scale,
                                      caf_b200_cfar_detection* out, uint64_t* count);
int caf_b200_detect_cfar_rows_f32_dev(caf_b200_handle h, const float* surface, size_t d_buf, size_t n,
                                      const double* freqs_hz, size_t row_lo, size_t row_hi, uint64_t row_offset,
                                      size_t d_global, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                      uint32_t train_doppler, uint32_t train_delay, double scale,
                                      caf_b200_cfar_detection* out, uint64_t* count);
int caf_b200_detect_cfar_os_rows_f64_dev(caf_b200_handle h, const double* surface, size_t d_buf, size_t n,
                                         const double* freqs_hz, size_t row_lo, size_t row_hi, uint64_t row_offset,
                                         size_t d_global, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                         uint32_t train_doppler, uint32_t train_delay, uint32_t rank, double scale,
                                         caf_b200_cfar_detection* out, uint64_t* count);
int caf_b200_detect_cfar_os_rows_f32_dev(caf_b200_handle h, const float* surface, size_t d_buf, size_t n,
                                         const double* freqs_hz, size_t row_lo, size_t row_hi, uint64_t row_offset,
                                         size_t d_global, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                         uint32_t train_doppler, uint32_t train_delay, uint32_t rank, double scale,
                                         caf_b200_cfar_detection* out, uint64_t* count);
/* The merge: lists [world][k_max] and counts [world] (device memory) hold each rank's block records and count, from
 * DISJOINT owned rows.  The global best k_max are among them.  One stream-ordered launch (one CTA) selects them by value
 * descending, then global flat index doppler_idx * n + delay_idx ascending, copies the whole records (no refit), applies
 * min_ratio against the global first (detect only) and writes out [k_max] (device; unused slots as above) and *count
 * (device): the records and count of the same detector run on the whole surface, bit for bit.  A count above k_max marks
 * a rank that failed: its list is skipped.  For callers with their own collective layer (torch.distributed).
 * Limits: 1 <= k_max <= 1024, 1 <= world <= 65536, 0 <= min_ratio <= 1, no null pointer; else CAF_B200_EINVAL. */
int caf_b200_detect_merge_dev(caf_b200_handle h, const caf_b200_detection* lists, const uint64_t* counts, size_t world,
                              size_t k_max, double min_ratio, caf_b200_detection* out, uint64_t* count);
int caf_b200_cfar_merge_dev(caf_b200_handle h, const caf_b200_cfar_detection* lists, const uint64_t* counts, size_t world,
                            size_t k_max, caf_b200_cfar_detection* out, uint64_t* count);

/* ---- non-coherent integration: the CAF surfaces of K signal segments summed cell by cell ----------------------------
 * A longer coherent window stops paying past a point (Doppler drift and oscillator instability decorrelate it, and the
 * Doppler bins narrow as 1/T); the standard remedy is to cut the capture into K segments, compute each segment's CAF on
 * the same Doppler grid and add the K |xcor|^2 surfaces.  The relative spread of the noise floor shrinks as 1/sqrt(K).
 * needles, haystacks: [k][l] (the batch calls' layout: a capture split into consecutive segments is a [k, l] view);
 * freqs_hz: d shifts shared by every segment; fs as in the surface calls.  s_i is the surface caf_b200_batch_*_dev gives
 * for pair i.  The integrated surface, double [d][2l] for BOTH input precisions, is
 *     S[r][c] = (((+0.0 + s_0[r][c]) + s_1[r][c]) + ...) + s_{k-1}[r][c]
 * with f32 cells widened to double first (exact) and the adds in double in ascending i, nothing reassociated: the result
 * does not depend on how the work is chunked, and a numpy loop `acc += s_i.astype(np.float64)` gives it bit for bit
 * (np.sum, which adds pairwise, does not).  Row peaks and peak follow the surface calls' rules in double: a row's peak is
 * its first cell holding the row's maximum (mod.rs:141-153), 0.0 at cell 0 for an all-zero row; peak is find_peak over
 * the rows (mod.rs:31-42), the lowest row winning a tie.  l == 0 or d == 0 behave as in the batch calls.
 * The detectors above run on S unchanged.  Their CFAR scales assume exponential cells, which one segment's |.|^2 of noise
 * is; a sum of k is Gamma(k): the Python package's cfar_scale(pfa, N, looks=k) gives the CA-CFAR scale for it (no closed
 * form exists for OS-CFAR).
 * Limits: check_common's with p = k (k * d <= 2e9 and k, d <= 2^30); k == 0, a null required pointer or fs == 0 is
 * CAF_B200_EINVAL, l > 2^19 is CAF_B200_EUNSUPPORTED; a call that fails writes nothing.
 * Scratch, independent of k: the handle's grow-only workspace holds one chunk of c segment surfaces, c = max(1, min(k,
 * CAF_B200_INTEGRATE_MB MB / (sizeof(cell) * d * 2l))), plus 20 + 12 * ceil(2l / 1024) bytes per row, plus what the batch
 * calls use for c pairs. */
/* every pointer is device memory; surface is required (unless d * l == 0), row_peak_val / row_peak_idx [d] and peak may be NULL.  Asynchronous
 * on the handle's stream: per chunk the batch path's launches and one plain stream-ordered accumulation launch (they count
 * in launch_count and end any overlap, caf_b200_set_overlap), then find_peak when peak is wanted. */
int caf_b200_integrate_f64_dev(caf_b200_handle h, const caf_c128* needles, const caf_c128* haystacks, size_t k, size_t l,
                               const double* freqs_hz, size_t d, uint32_t fs, double* surface, double* row_peak_val,
                               uint64_t* row_peak_idx, caf_b200_peak* peak);
int caf_b200_integrate_f32_dev(caf_b200_handle h, const caf_c64* needles, const caf_c64* haystacks, size_t k, size_t l,
                               const double* freqs_hz, size_t d, uint32_t fs, double* surface, double* row_peak_val,
                               uint64_t* row_peak_idx, caf_b200_peak* peak);
/* host inputs; the result is an f64 surface object (whatever the input precision) on which caf_b200_surface_{shape,
 * row_peaks, find_peak, fetch_rows (doubles), detect, detect_cfar, detect_cfar_os, destroy} work unchanged; synchronous */
int caf_b200_surface_create_integrated_f64(caf_b200_handle h, const caf_c128* needles, const caf_c128* haystacks, size_t k,
                                           size_t l, const double* freqs_hz, size_t d, uint32_t fs, caf_b200_surface* out);
int caf_b200_surface_create_integrated_f32(caf_b200_handle h, const caf_c64* needles, const caf_c64* haystacks, size_t k,
                                           size_t l, const double* freqs_hz, size_t d, uint32_t fs, caf_b200_surface* out);

/* ---- the sibling programs' layouts of the same surface (SURVEY.md section 8(f)4) -------------------
 * The reference's Go and Python programs compute this correlation with the operands swapped and keep the
 * magnitude |xcor| (cmplx.Abs, np.abs) where the Rust crate keeps |xcor|^2 (norm_sqr):
 *   CAF_B200_LAYOUT_PYTHON  caf_python/caf.py:12-13,101-122  amb_surf: out is d x l, row =
 *                           |scipy.signal.correlate(shifted, haystack, 'same')|, column j holds Rust lag l/2 - j;
 *                           caf.py:145 reports tau = l//2 - argmax column.
 *   CAF_B200_LAYOUT_GO      caf_go/caf.go:93-116,162-173  amb_surf: out is d x 2l (banana zero-padded in FRONT),
 *                           column k holds Rust lag l - k (mod 2l); main.go:35 reports len - tdx.
 * The surface is computed once on the GPU (Rust layout, |.|^2) and converted there; `out` may be NULL.
 * peak: the sibling's 2-D argmax (first strict-> maximum in row-major order, caf.go:183-195 / np.argmax):
 * value = |xcor|, freq_hz, doppler_idx = row, delay_idx = COLUMN of the converted surface. */
typedef enum { CAF_B200_LAYOUT_RUST = 0, CAF_B200_LAYOUT_PYTHON = 1, CAF_B200_LAYOUT_GO = 2 } caf_b200_layout;
int caf_b200_surface_layout_f64(caf_b200_handle h, const caf_c128* needle, const caf_c128* haystack, size_t l,
                                const double* freqs_hz, size_t d, uint32_t fs, int layout,
                                double* out, caf_b200_peak* peak);
int caf_b200_surface_layout_f32(caf_b200_handle h, const caf_c64* needle, const caf_c64* haystack, size_t l,
                                const double* freqs_hz, size_t d, uint32_t fs, int layout,
                                float* out, caf_b200_peak* peak);

/* ---- multi-GPU peak reduction (doppler rows or pairs sharded across ranks; SURVEY.md section 8e) ----
 * Each rank computes the peak of its shard, packs it with its GLOBAL first-row offset into 4 uint64
 * words, the caller all-gathers (or all-reduces a zero-initialised 4*world buffer with SUM/MAX) the
 * words over NCCL, and every rank resolves the same winner with find_peak's tie-break (lowest global
 * doppler row).  Pure host helpers; no GPU work. */
void caf_b200_peak_pack(const caf_b200_peak* local, uint64_t global_row_offset, uint64_t words[4]);
void caf_b200_peak_resolve(const uint64_t* words, size_t world, caf_b200_peak* out);
/* same, and returns 1 when some rank's words carry the failure mark (words[1] == UINT64_MAX - 1: that rank could not
 * compute its shard but still took part in the collective), else 0 */
int caf_b200_peak_resolve_status(const uint64_t* words, size_t world, caf_b200_peak* out);

/* ---- the same exchange inside the library: NCCL over NVLink, one process per GPU ---------------------
 * For callers without their own collective layer (the Rust shim).  libnccl.so.2 is dlopen()ed on first use —
 * no link-time dependency; CAF_B200_ENCCL if it cannot be found.  Rank 0 obtains an id with
 * caf_b200_comm_unique_id and hands the 128 bytes to the other ranks out of band (file, env, MPI, socket);
 * every rank then calls caf_b200_comm_create (collective, = ncclCommInitRank on the handle's device).
 * caf_b200_comm_adopt wraps an ncclComm_t the caller already owns (not destroyed with the communicator). */
#define CAF_B200_NCCL_ID_BYTES 128
typedef struct caf_b200_comm_s* caf_b200_comm;
int caf_b200_comm_unique_id(unsigned char id[CAF_B200_NCCL_ID_BYTES]);
int caf_b200_comm_create(caf_b200_handle h, int world, int rank, const unsigned char id[CAF_B200_NCCL_ID_BYTES],
                         caf_b200_comm* out);
int caf_b200_comm_adopt(caf_b200_handle h, void* nccl_comm, int world, int rank, caf_b200_comm* out);
int caf_b200_comm_destroy(caf_b200_comm c);
/* contiguous block [lo, hi) of n doppler rows (or pairs) owned by this rank */
int caf_b200_comm_shard(caf_b200_comm c, size_t n, size_t* lo, size_t* hi);
/* find_peak across ranks: local_peak_dev is the DEVICE peak a *_dev call of this rank produced for its shard
 * (rows global_row_offset ...); it is packed on the device, all-gathered (32 bytes per rank, ncclAllGather on
 * the handle's stream) and resolved with find_peak's tie-break.  Every rank gets the same `out` (host). */
int caf_b200_peak_allgather_dev(caf_b200_handle h, caf_b200_comm c, const caf_b200_peak* local_peak_dev,
                                uint64_t global_row_offset, caf_b200_peak* out);
/* The same exchange with NO host synchronisation: pack (local_peak_dev == NULL packs "this rank owns no row"),
 * ncclAllGather and the resolution all run on the handle's stream; out_dev (device memory, or pinned host memory) holds
 * the global peak once the stream reaches that point.  caf_b200_comm_remote_error() afterwards (after a sync) tells
 * whether a peer had failed. */
int caf_b200_peak_allgather_async(caf_b200_handle h, caf_b200_comm c, const caf_b200_peak* local_peak_dev,
                                  uint64_t global_row_offset, caf_b200_peak* out_dev);
int caf_b200_comm_remote_error(caf_b200_comm c, int* flag);
/* Transport of the 32-byte exchange.  When every rank of the communicator could map every peer's mailbox at creation (CUDA
 * IPC over NVLink / NVSwitch peer memory; the handles travel in one ncclAllGather), the exchange is ONE kernel per rank:
 * it stores this rank's packed words straight into every peer's mailbox, acquire-polls its own mailbox for the world's
 * records and resolves them (caf_peak_exchange_kernel) -- flag = 1.  Otherwise, or with CAF_B200_P2P=0 in the environment
 * at creation, ncclAllGather + a resolve kernel -- flag = 0.  Same results either way. */
int caf_b200_comm_uses_p2p(caf_b200_comm c, int* flag);
/* Device-resident sharded surface (mod.rs:185 par_iter over rows + mod.rs:31-42 across GPUs), fully asynchronous:
 * this rank's rows freqs_local[0..d_local) are global rows row_offset.., every pointer is device memory; the local
 * find_peak writes its result already packed for the exchange, then ONE ncclAllGather of 32 bytes per rank and a
 * device-side resolve leave the global peak in peak_out (device or pinned host memory).  No host synchronisation.
 * If the local computation cannot be issued, the rank still enters the collective with a failure mark, every peer's
 * next resolve reports CAF_B200_EREMOTE / remote_error, and this call returns the local error. */
int caf_b200_sharded_f64_dev(caf_b200_handle h, caf_b200_comm c, const caf_c128* needle, const caf_c128* haystack, size_t l,
                             const double* freqs_local, size_t d_local, uint64_t row_offset, uint32_t fs,
                             double* surface_local, double* row_peak_val, uint64_t* row_peak_idx, caf_b200_peak* peak_out);
int caf_b200_sharded_f32_dev(caf_b200_handle h, caf_b200_comm c, const caf_c64* needle, const caf_c64* haystack, size_t l,
                             const double* freqs_local, size_t d_local, uint64_t row_offset, uint32_t fs,
                             float* surface_local, float* row_peak_val, uint64_t* row_peak_idx, caf_b200_peak* peak_out);
/* CafSurface::caf_surface + find_peak with the doppler ROWS sharded across the communicator (mod.rs:185 par_iter
 * over rows, one GPU per block of rows): every rank passes the SAME host inputs and the full grid; rank r computes
 * rows [lo, hi) = caf_b200_comm_shard(d), writes them to surface_local ((hi-lo) x 2l, or NULL) and receives the
 * global peak (doppler_idx is the global row). */
int caf_b200_surface_sharded_f64(caf_b200_handle h, caf_b200_comm c, const caf_c128* needle, const caf_c128* haystack,
                                 size_t l, const double* freqs_hz, size_t d, uint32_t fs,
                                 double* surface_local, caf_b200_peak* peak);
int caf_b200_surface_sharded_f32(caf_b200_handle h, caf_b200_comm c, const caf_c64* needle, const caf_c64* haystack,
                                 size_t l, const double* freqs_hz, size_t d, uint32_t fs,
                                 float* surface_local, caf_b200_peak* peak);
/* Detection on row-sharded surfaces (caf_b200_detect_rows_* and the merge, above) across this communicator's ranks. */
/* The exchange over the library's communicator (caf_b200_comm): ONE ncclAllGather of this rank's k_max records and
 * count (local, local_count: device memory) on the handle's stream, then the merge into out / count (device memory) on
 * every rank; synchronous.  k_max (and min_ratio) must be the same on every rank; a bad one fails on every rank before
 * the collective.  A rank that passes a null pointer still enters the collective with a failure mark and returns
 * CAF_B200_EINVAL; its peers skip its list and return CAF_B200_EREMOTE. */
int caf_b200_detect_allgather_dev(caf_b200_handle h, caf_b200_comm c, const caf_b200_detection* local,
                                  const uint64_t* local_count, size_t k_max, double min_ratio, caf_b200_detection* out,
                                  uint64_t* count);
int caf_b200_cfar_allgather_dev(caf_b200_handle h, caf_b200_comm c, const caf_b200_cfar_detection* local,
                                const uint64_t* local_count, size_t k_max, caf_b200_cfar_detection* out, uint64_t* count);

#ifdef __cplusplus
}
#endif
#endif /* CAF_B200_H */
