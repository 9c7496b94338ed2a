// caf_b200.hpp — C++ host-side mirror of caf_rust's public API over the C ABI (caf_b200.h).
//
// The reference's host language is Rust and no Rust toolchain exists in this build image, so the host side above
// the C ABI is written in C++ with the reference's names, argument order and error behaviour:
//     trait CafSurface { caf_surface, find_peak, apply_freq_shift }     caf_rust/src/caf/mod.rs:23-66
//     struct CafSurfaceRow { freq, xcor_mag, xcor_peak_idx, xcor_peak_val }  caf_rust/src/caf/mod.rs:17-22
//     struct Xcor { new, run, clone }                                    caf_rust/src/caf/xcor_rustfft.rs:14-93
//     read_file_c64 / BinaryIO::write_file_binary                        caf_rust/src/utils.rs:10-63
// The reference panics on bad input (assert!/unwrap); here that is a thrown caf::Panic.
// Header only; link with libcaf_b200.so.  rust/ holds the equivalent Rust shim as (uncompiled) source.
#pragma once
#include <complex>
#include <cstdint>
#include <cstdio>
#include <fstream>
#include <memory>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "caf_b200.h"

namespace caf {

using Complex64 = std::complex<double>;   // Rust's num_complex::Complex64 = Complex<f64> (utils.rs:8-9)
using Complex32 = std::complex<float>;

struct Panic : std::runtime_error { using std::runtime_error::runtime_error; };

inline void check(int rc) {
    if (rc != CAF_B200_OK) throw Panic(std::string("caf_b200 status ") + std::to_string(rc) + ": " + caf_b200_last_error());
}

// one lazily created handle per thread: the trait functions are static and must be callable from any thread
// (caf::set_overlap(true) lets consecutive independent device launches of this thread's handle overlap, caf_b200.h)
inline caf_b200_handle thread_handle() {
    struct Holder {
        caf_b200_handle h = nullptr;
        ~Holder() { if (h) caf_b200_destroy(h); }
    };
    thread_local Holder holder;
    if (!holder.h) check(caf_b200_create(0, &holder.h));
    return holder.h;
}

using Detection = caf_b200_detection;   // the strongest local maxima of a surface, refined below the grid (caf_b200.h)
using CfarDetection = caf_b200_cfar_detection;   // the same, above a local noise estimate, with that estimate

// One surface on the GPU, shared by its rows (caf_b200_surface_*).  The reference's CafSurfaceRow owns a Vec<f64> per row
// (mod.rs:17-22) but keeps every field PRIVATE, so no caller of the crate can read it: here a row is (surface, row number)
// and the 2L doubles of xcor_mag cross PCIe only when xcor_mag() is called.
class DeviceSurface {
    caf_b200_surface s_ = nullptr;
    std::thread::id owner_ = std::this_thread::get_id();   // the thread whose handle made it (thread_handle())
    std::size_t rows_ = 0, cells_ = 0;
    mutable bool have_peaks_ = false;
    mutable std::vector<double> freq_, pval_;
    mutable std::vector<uint64_t> pidx_;
public:
    explicit DeviceSurface(caf_b200_surface s) : s_(s) { check(caf_b200_surface_shape(s_, &rows_, &cells_)); }
    DeviceSurface(const DeviceSurface&) = delete;
    DeviceSurface& operator=(const DeviceSurface&) = delete;
    ~DeviceSurface() { if (s_) caf_b200_surface_destroy(s_); }
    std::size_t rows() const { return rows_; }
    std::size_t cells_per_row() const { return cells_; }
    caf_b200_peak fused_peak() const { caf_b200_peak p; check(caf_b200_surface_find_peak(s_, &p)); return p; }
    void need_peaks() const {                      // one 16-byte-per-row copy, the first time a row's peak is looked at
        if (have_peaks_) return;
        freq_.resize(rows_); pval_.resize(rows_); pidx_.resize(rows_);
        check(caf_b200_surface_row_peaks(s_, freq_.data(), pval_.data(), pidx_.data()));
        have_peaks_ = true;
    }
    double freq(std::size_t r) const { need_peaks(); return freq_[r]; }
    double peak_val(std::size_t r) const { need_peaks(); return pval_[r]; }
    std::size_t peak_idx(std::size_t r) const { need_peaks(); return (std::size_t)pidx_[r]; }
    std::vector<double> fetch_rows(std::size_t row0, std::size_t count) const {
        std::vector<double> out(count * cells_);
        check(caf_b200_surface_fetch_rows(s_, row0, count, out.data()));
        return out;
    }
    // caf_b200_surface_detect: the count valid detections, best first
    std::vector<Detection> detect(std::size_t k_max, uint32_t guard_doppler = 1, uint32_t guard_delay = 1,
                                  double min_ratio = 0.0) const {
        // detection runs on the surface's handle, which belongs to the creating thread (caf_b200.h threading rule)
        if (std::this_thread::get_id() != owner_) throw Panic("detect: a surface is searched on the thread that created it");
        std::vector<Detection> out(k_max);
        std::size_t count = 0;
        check(caf_b200_surface_detect(s_, k_max, guard_doppler, guard_delay, min_ratio, out.data(), &count));
        out.resize(count);
        return out;
    }
    // caf_b200_surface_detect_cfar: the count valid CFAR detections, best first (possibly none)
    std::vector<CfarDetection> detect_cfar(std::size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                           uint32_t train_doppler, uint32_t train_delay, double scale) const {
        if (std::this_thread::get_id() != owner_) throw Panic("detect_cfar: a surface is searched on the thread that created it");
        std::vector<CfarDetection> out(k_max);
        std::size_t count = 0;
        check(caf_b200_surface_detect_cfar(s_, k_max, guard_doppler, guard_delay, train_doppler, train_delay, scale,
                                           out.data(), &count));
        out.resize(count);
        return out;
    }
    // caf_b200_surface_detect_cfar_os: the same against the rank-th smallest training cell (OS-CFAR)
    std::vector<CfarDetection> detect_cfar_os(std::size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                              uint32_t train_doppler, uint32_t train_delay, uint32_t rank,
                                              double scale) const {
        if (std::this_thread::get_id() != owner_) throw Panic("detect_cfar_os: a surface is searched on the thread that created it");
        std::vector<CfarDetection> out(k_max);
        std::size_t count = 0;
        check(caf_b200_surface_detect_cfar_os(s_, k_max, guard_doppler, guard_delay, train_doppler, train_delay, rank,
                                              scale, out.data(), &count));
        out.resize(count);
        return out;
    }
};

// mod.rs:17-22 (fields are private in the reference; accessors added so results can be inspected)
class CafSurfaceRow {
    std::shared_ptr<const DeviceSurface> surf_;
    std::size_t row_ = 0;
public:
    CafSurfaceRow() = default;
    CafSurfaceRow(std::shared_ptr<const DeviceSurface> s, std::size_t row) : surf_(std::move(s)), row_(row) {}
    double freq() const { return surf_ ? surf_->freq(row_) : 0.0; }
    std::size_t xcor_peak_idx() const { return surf_ ? surf_->peak_idx(row_) : 0; }
    double xcor_peak_val() const { return surf_ ? surf_->peak_val(row_) : 0.0; }
    std::vector<double> xcor_mag() const { return surf_ ? surf_->fetch_rows(row_, 1) : std::vector<double>(); }   // lazy: one row over PCIe
    const std::shared_ptr<const DeviceSurface>& surface() const { return surf_; }
    std::size_t row() const { return row_; }
};

inline void set_overlap(bool on) { check(caf_b200_set_overlap(thread_handle(), on ? 1 : 0)); }

struct CafB200 {
    // mod.rs:121-166 (every strategy struct computes this).  Costs a peak-only call: inputs up, one fused launch, the
    // 32-byte find_peak result down; the surface and its row peaks stay on the GPU behind the rows.
    static std::vector<CafSurfaceRow> caf_surface(const std::vector<Complex64>& needle, const std::vector<Complex64>& haystack,
                                                  const std::vector<double>& freqs_hz, uint32_t fs) {
        if (needle.size() != haystack.size()) throw Panic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55)");
        caf_b200_surface raw = nullptr;
        check(caf_b200_surface_create_f64(thread_handle(), reinterpret_cast<const caf_c128*>(needle.data()),
                                          reinterpret_cast<const caf_c128*>(haystack.data()), needle.size(), freqs_hz.data(),
                                          freqs_hz.size(), fs, &raw));
        auto surf = std::make_shared<const DeviceSurface>(raw);
        std::vector<CafSurfaceRow> rows;
        rows.reserve(freqs_hz.size());
        for (std::size_t r = 0; r < freqs_hz.size(); ++r) rows.emplace_back(surf, r);
        return rows;
    }
    // Non-coherent integration (caf_b200_surface_create_integrated_f64): needles and haystacks hold k consecutive segments
    // of l = needles.size() / k samples; the rows are ONE surface on the GPU, the cell-by-cell sum of the k segments'
    // |xcor|^2 surfaces in double.  find_peak, the rows' fields and the detectors work on it as on caf_surface's rows, and
    // like those it belongs to the calling thread's handle (detection refuses other threads).
    static std::vector<CafSurfaceRow> integrate(const std::vector<Complex64>& needles, const std::vector<Complex64>& haystacks,
                                                std::size_t k, const std::vector<double>& freqs_hz, uint32_t fs) {
        if (needles.size() != haystacks.size()) throw Panic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55)");
        if (k == 0 || needles.size() % k) throw Panic("integrate needs k > 0 segments of equal length");
        caf_b200_surface raw = nullptr;
        check(caf_b200_surface_create_integrated_f64(thread_handle(), reinterpret_cast<const caf_c128*>(needles.data()),
                                                     reinterpret_cast<const caf_c128*>(haystacks.data()), k, needles.size() / k,
                                                     freqs_hz.data(), freqs_hz.size(), fs, &raw));
        auto surf = std::make_shared<const DeviceSurface>(raw);
        std::vector<CafSurfaceRow> rows;
        rows.reserve(freqs_hz.size());
        for (std::size_t r = 0; r < freqs_hz.size(); ++r) rows.emplace_back(surf, r);
        return rows;
    }
    // mod.rs:31-42: strict > from a dummy row (0.0, peak 0.0) in VECTOR order; consumes the surface like the reference.
    // When `arr` is what caf_surface returned, untouched (all rows of one surface, in order), that scan is exactly what
    // the kernel's fused find_peak already did; any other vector (reordered, truncated, rows of several surfaces) is
    // scanned here from the rows' peaks.
    static std::pair<double, std::size_t> find_peak(std::vector<CafSurfaceRow> arr) {
        if (!arr.empty() && arr[0].surface() && arr.size() == arr[0].surface()->rows()) {
            bool whole = true;
            for (std::size_t i = 0; i < arr.size() && whole; ++i) whole = arr[i].surface() == arr[0].surface() && arr[i].row() == i;
            if (whole) {
                const caf_b200_peak pk = arr[0].surface()->fused_peak();
                return {pk.freq_hz, (std::size_t)pk.delay_idx};
            }
        }
        double best = 0.0, f = 0.0;
        std::size_t idx = 0;
        for (const auto& row : arr)
            if (row.xcor_peak_val() > best) { best = row.xcor_peak_val(); f = row.freq(); idx = row.xcor_peak_idx(); }
        return {f, idx};
    }
    // Detection on the surface behind `arr`, which must be what caf_surface returned, untouched (every row of one surface,
    // in order): a reordered or partial vector no longer names a surface, so it is refused (Panic).
    static std::vector<Detection> detect(const std::vector<CafSurfaceRow>& arr, std::size_t k_max, uint32_t guard_doppler = 1,
                                         uint32_t guard_delay = 1, double min_ratio = 0.0) {
        bool whole = !arr.empty() && arr[0].surface() && arr.size() == arr[0].surface()->rows();
        for (std::size_t i = 0; i < arr.size() && whole; ++i) whole = arr[i].surface() == arr[0].surface() && arr[i].row() == i;
        if (!whole) throw Panic("detect needs the untouched rows of one caf_surface call");
        return arr[0].surface()->detect(k_max, guard_doppler, guard_delay, min_ratio);
    }
    // CFAR detection on the surface behind `arr` (same rule for `arr` and the calling thread as detect)
    static std::vector<CfarDetection> detect_cfar(const std::vector<CafSurfaceRow>& arr, std::size_t k_max,
                                                  uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler,
                                                  uint32_t train_delay, double scale) {
        bool whole = !arr.empty() && arr[0].surface() && arr.size() == arr[0].surface()->rows();
        for (std::size_t i = 0; i < arr.size() && whole; ++i) whole = arr[i].surface() == arr[0].surface() && arr[i].row() == i;
        if (!whole) throw Panic("detect_cfar needs the untouched rows of one caf_surface call");
        return arr[0].surface()->detect_cfar(k_max, guard_doppler, guard_delay, train_doppler, train_delay, scale);
    }
    // OS-CFAR detection on the surface behind `arr` (same rule for `arr` and the calling thread as detect)
    static std::vector<CfarDetection> detect_cfar_os(const std::vector<CafSurfaceRow>& arr, std::size_t k_max,
                                                     uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler,
                                                     uint32_t train_delay, uint32_t rank, double scale) {
        bool whole = !arr.empty() && arr[0].surface() && arr.size() == arr[0].surface()->rows();
        for (std::size_t i = 0; i < arr.size() && whole; ++i) whole = arr[i].surface() == arr[0].surface() && arr[i].row() == i;
        if (!whole) throw Panic("detect_cfar_os needs the untouched rows of one caf_surface call");
        return arr[0].surface()->detect_cfar_os(k_max, guard_doppler, guard_delay, train_doppler, train_delay, rank, scale);
    }
    // caf_surface + find_peak fused on the GPU, the surface never leaves the chip
    static std::pair<double, std::size_t> caf_peak(const std::vector<Complex64>& needle, const std::vector<Complex64>& haystack,
                                                   const std::vector<double>& freqs_hz, uint32_t fs) {
        if (needle.size() != haystack.size()) throw Panic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55)");
        caf_b200_peak pk;
        check(caf_b200_peak_f64(thread_handle(), reinterpret_cast<const caf_c128*>(needle.data()),
                                reinterpret_cast<const caf_c128*>(haystack.data()), needle.size(), freqs_hz.data(),
                                freqs_hz.size(), fs, &pk));
        return {pk.freq_hz, (std::size_t)pk.delay_idx};
    }
    // mod.rs:46-65
    static std::vector<Complex64> apply_freq_shift(const std::vector<Complex64>& samples, double freq_shift, uint32_t fs) {
        std::vector<Complex64> out(samples.size());
        check(caf_b200_apply_freq_shift_f64(thread_handle(), reinterpret_cast<const caf_c128*>(samples.data()), samples.size(),
                                            freq_shift, fs, reinterpret_cast<caf_c128*>(out.data())));
        return out;
    }
    static std::vector<Complex64> apply_shift(const std::vector<Complex64>& s, double f, uint32_t fs) { return apply_freq_shift(s, f, fs); }
};

// the seven strategy structs of the reference (mod.rs:67,118,169,219,266,313,388): one computation, one path
using CafFFTW = CafB200;
using CafRustFFT = CafB200;
using CafRustFFTRayon = CafB200;
using CafRustFFTIter = CafB200;
using CafRustFFTIterRayon = CafB200;
using CafRustFFTThreads = CafB200;
using CafRustFFTThreadpool = CafB200;

// xcor_rustfft.rs:14-93
class Xcor {
    std::size_t n_;
public:
    explicit Xcor(std::size_t n) : n_(n) {}
    static Xcor make(std::size_t n) { return Xcor(n); }       // Xcor::new
    Xcor clone() const { return Xcor(n_); }
    std::vector<Complex64> run(const std::vector<Complex64>& a, const std::vector<Complex64>& b) const {
        if (a.size() != n_ || b.size() != n_) throw Panic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55)");
        std::vector<Complex64> out(n_);
        check(caf_b200_xcor_f64(thread_handle(), reinterpret_cast<const caf_c128*>(a.data()),
                                reinterpret_cast<const caf_c128*>(b.data()), n_, reinterpret_cast<caf_c128*>(out.data())));
        return out;
    }
};

// The Go program of the reference (caf_go/caf.go) from the same kernels: amb_surf (caf.go:162-173) returns
// [][]float64 of 2L columns, |xcor|, column k = Rust lag L - k; find_2d_peak (caf.go:183-195) is the first
// strict-> maximum in row-major order; main.go:35 reports len(apple) - tdx.
struct GoSibling {
    // caf.go:118 takes a float64 sample rate, the C ABI the Rust crate's u32 (mod.rs:46): a rate the u32 cannot hold
    // exactly would silently give a different phasor than the Go program, so it is refused
    static uint32_t whole_sample_rate(double samp_rate) {
        if (!(samp_rate >= 1.0 && samp_rate <= 4294967295.0) || samp_rate != (double)(uint64_t)samp_rate)
            throw Panic("samp_rate must be a whole number of Hz in [1, 2^32 - 1] (the library's sample rate is the Rust crate's u32, mod.rs:46)");
        return (uint32_t)samp_rate;
    }
    static std::vector<std::vector<double>> amb_surf(const std::vector<Complex64>& needle, const std::vector<Complex64>& haystack,
                                                     const std::vector<double>& freqs_hz, double samp_rate) {
        if (needle.size() != haystack.size()) throw Panic("input arrays should be same size (caf.go:97-99)");
        const std::size_t l = needle.size(), d = freqs_hz.size(), w = 2 * l;
        std::vector<double> flat(d * w);
        check(caf_b200_surface_layout_f64(thread_handle(), reinterpret_cast<const caf_c128*>(needle.data()),
                                          reinterpret_cast<const caf_c128*>(haystack.data()), l, freqs_hz.data(), d,
                                          whole_sample_rate(samp_rate), CAF_B200_LAYOUT_GO, flat.data(), nullptr));
        std::vector<std::vector<double>> surf(d);
        for (std::size_t r = 0; r < d; ++r) surf[r].assign(flat.begin() + r * w, flat.begin() + (r + 1) * w);
        return surf;
    }
    struct Peak2d { int fdx, tdx; double max; };
    static Peak2d find_2d_peak(const std::vector<std::vector<double>>& surf) {
        Peak2d p{0, 0, 0.0};
        for (std::size_t i = 0; i < surf.size(); ++i)
            for (std::size_t j = 0; j < surf[i].size(); ++j)
                if (surf[i][j] > p.max) p = Peak2d{(int)i, (int)j, surf[i][j]};
        return p;
    }
};

// Detection on the owned rows [row_lo, row_hi) of a device block of d_buf rows whose row 0 is global row row_offset of a
// d_global-row surface, and the merge of the ranks' lists (caf_b200.h: caf_b200_detect_rows_* ... caf_b200_cfar_merge_dev).
// Device pointers, asynchronous on the calling thread's handle.
inline void detect_rows_dev(const double* surface, std::size_t d_buf, std::size_t n, const double* freqs_hz,
                            std::size_t row_lo, std::size_t row_hi, uint64_t row_offset, std::size_t d_global,
                            std::size_t k_max, uint32_t guard_doppler, uint32_t guard_delay, double min_ratio,
                            Detection* out, uint64_t* count) {
    check(caf_b200_detect_rows_f64_dev(thread_handle(), surface, d_buf, n, freqs_hz, row_lo, row_hi, row_offset, d_global,
                                       k_max, guard_doppler, guard_delay, min_ratio, out, count));
}
inline void detect_rows_dev(const float* surface, std::size_t d_buf, std::size_t n, const double* freqs_hz,
                            std::size_t row_lo, std::size_t row_hi, uint64_t row_offset, std::size_t d_global,
                            std::size_t k_max, uint32_t guard_doppler, uint32_t guard_delay, double min_ratio,
                            Detection* out, uint64_t* count) {
    check(caf_b200_detect_rows_f32_dev(thread_handle(), surface, d_buf, n, freqs_hz, row_lo, row_hi, row_offset, d_global,
                                       k_max, guard_doppler, guard_delay, min_ratio, out, count));
}
inline void detect_cfar_rows_dev(const double* surface, std::size_t d_buf, std::size_t n, const double* freqs_hz,
                                 std::size_t row_lo, std::size_t row_hi, uint64_t row_offset, std::size_t d_global,
                                 std::size_t k_max, uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler,
                                 uint32_t train_delay, double scale, CfarDetection* out, uint64_t* count) {
    check(caf_b200_detect_cfar_rows_f64_dev(thread_handle(), surface, d_buf, n, freqs_hz, row_lo, row_hi, row_offset,
                                            d_global, k_max, guard_doppler, guard_delay, train_doppler, train_delay, scale,
                                            out, count));
}
inline void detect_cfar_rows_dev(const float* surface, std::size_t d_buf, std::size_t n, const double* freqs_hz,
                                 std::size_t row_lo, std::size_t row_hi, uint64_t row_offset, std::size_t d_global,
                                 std::size_t k_max, uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler,
                                 uint32_t train_delay, double scale, CfarDetection* out, uint64_t* count) {
    check(caf_b200_detect_cfar_rows_f32_dev(thread_handle(), surface, d_buf, n, freqs_hz, row_lo, row_hi, row_offset,
                                            d_global, k_max, guard_doppler, guard_delay, train_doppler, train_delay, scale,
                                            out, count));
}
inline void detect_cfar_os_rows_dev(const double* surface, std::size_t d_buf, std::size_t n, const double* freqs_hz,
                                    std::size_t row_lo, std::size_t row_hi, uint64_t row_offset, std::size_t d_global,
                                    std::size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                    uint32_t train_doppler, uint32_t train_delay, uint32_t rank, double scale,
                                    CfarDetection* out, uint64_t* count) {
    check(caf_b200_detect_cfar_os_rows_f64_dev(thread_handle(), surface, d_buf, n, freqs_hz, row_lo, row_hi, row_offset,
                                               d_global, k_max, guard_doppler, guard_delay, train_doppler, train_delay,
                                               rank, scale, out, count));
}
inline void detect_cfar_os_rows_dev(const float* surface, std::size_t d_buf, std::size_t n, const double* freqs_hz,
                                    std::size_t row_lo, std::size_t row_hi, uint64_t row_offset, std::size_t d_global,
                                    std::size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                    uint32_t train_doppler, uint32_t train_delay, uint32_t rank, double scale,
                                    CfarDetection* out, uint64_t* count) {
    check(caf_b200_detect_cfar_os_rows_f32_dev(thread_handle(), surface, d_buf, n, freqs_hz, row_lo, row_hi, row_offset,
                                               d_global, k_max, guard_doppler, guard_delay, train_doppler, train_delay,
                                               rank, scale, out, count));
}
inline void detect_merge_dev(const Detection* lists, const uint64_t* counts, std::size_t world, std::size_t k_max,
                             double min_ratio, Detection* out, uint64_t* count) {
    check(caf_b200_detect_merge_dev(thread_handle(), lists, counts, world, k_max, min_ratio, out, count));
}
inline void cfar_merge_dev(const CfarDetection* lists, const uint64_t* counts, std::size_t world, std::size_t k_max,
                           CfarDetection* out, uint64_t* count) {
    check(caf_b200_cfar_merge_dev(thread_handle(), lists, counts, world, k_max, out, count));
}

// Doppler rows sharded over one process per GPU (mod.rs:185's par_iter with GPUs for workers): the library's own NCCL
// communicator.  Rank 0 makes the 128-byte id (ShardedCaf::unique_id) and hands it to the other ranks out of band.
class ShardedCaf {
    caf_b200_comm comm_ = nullptr;
public:
    static std::vector<unsigned char> unique_id() {
        std::vector<unsigned char> id(CAF_B200_NCCL_ID_BYTES);
        check(caf_b200_comm_unique_id(id.data()));
        return id;
    }
    ShardedCaf(int world, int rank, const std::vector<unsigned char>& id) {
        if (id.size() != CAF_B200_NCCL_ID_BYTES) throw Panic("NCCL id must be 128 bytes");
        check(caf_b200_comm_create(thread_handle(), world, rank, id.data(), &comm_));
    }
    ShardedCaf(const ShardedCaf&) = delete;
    ShardedCaf& operator=(const ShardedCaf&) = delete;
    ~ShardedCaf() { if (comm_) caf_b200_comm_destroy(comm_); }
    std::pair<std::size_t, std::size_t> shard(std::size_t n) const {
        std::size_t lo = 0, hi = 0;
        check(caf_b200_comm_shard(comm_, n, &lo, &hi));
        return {lo, hi};
    }
    // this rank's rows [lo, hi) of the surface (row-major, 2l cells each) and the GLOBAL find_peak answer
    std::pair<std::vector<double>, std::pair<double, std::size_t>> caf_surface_peak(
        const std::vector<Complex64>& needle, const std::vector<Complex64>& haystack, const std::vector<double>& freqs_hz, uint32_t fs) const {
        if (needle.size() != haystack.size()) throw Panic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55)");
        const auto [lo, hi] = shard(freqs_hz.size());
        std::vector<double> rows((hi - lo) * 2 * needle.size());
        caf_b200_peak pk;
        check(caf_b200_surface_sharded_f64(thread_handle(), comm_, reinterpret_cast<const caf_c128*>(needle.data()),
                                           reinterpret_cast<const caf_c128*>(haystack.data()), needle.size(), freqs_hz.data(),
                                           freqs_hz.size(), fs, rows.data(), &pk));
        return {std::move(rows), {pk.freq_hz, (std::size_t)pk.delay_idx}};
    }
    // the exchange of the ranks' block detections (device records and counts; caf_b200_*_allgather_dev)
    void detect_allgather_dev(const Detection* local, const uint64_t* local_count, std::size_t k_max, double min_ratio,
                              Detection* out, uint64_t* count) const {
        check(caf_b200_detect_allgather_dev(thread_handle(), comm_, local, local_count, k_max, min_ratio, out, count));
    }
    void cfar_allgather_dev(const CfarDetection* local, const uint64_t* local_count, std::size_t k_max,
                            CfarDetection* out, uint64_t* count) const {
        check(caf_b200_cfar_allgather_dev(thread_handle(), comm_, local, local_count, k_max, out, count));
    }
};

// utils.rs:10-35: packed little-endian f32 I/Q -> Complex64
inline std::vector<Complex64> read_file_c64(const std::string& filename) {
    std::ifstream f(filename, std::ios::binary);
    if (!f) throw std::runtime_error("read_file_c64: cannot open " + filename);      // io::Result Err in the reference
    std::vector<char> buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    if (buf.size() % 8) throw Panic("read_file_c64: trailing partial sample");
    std::vector<Complex64> out(buf.size() / 8);
    const float* p = reinterpret_cast<const float*>(buf.data());
    for (std::size_t i = 0; i < out.size(); ++i) out[i] = Complex64((double)p[2 * i], (double)p[2 * i + 1]);
    return out;
}

// Samples resident on the GPU and the loader that puts them there: read_file_c64 (utils.rs:10-35) through pinned memory,
// 8 bytes per sample across PCIe, widened on the device (bit-identical to the host loader).  window: first sample and
// count (0 = to the end of the file; main.rs:15 truncates the haystack to the needle's length).
class DeviceSamples {
    caf_c128* p_ = nullptr;
    std::size_t n_ = 0;
public:
    DeviceSamples() = default;
    DeviceSamples(caf_c128* p, std::size_t n) : p_(p), n_(n) {}
    DeviceSamples(const DeviceSamples&) = delete;
    DeviceSamples& operator=(const DeviceSamples&) = delete;
    DeviceSamples(DeviceSamples&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    DeviceSamples& operator=(DeviceSamples&& o) noexcept { std::swap(p_, o.p_); std::swap(n_, o.n_); return *this; }
    ~DeviceSamples() { if (p_) caf_b200_dev_free(p_); }
    const caf_c128* data() const { return p_; }
    std::size_t size() const { return n_; }
    std::vector<Complex64> to_host() const {
        std::vector<Complex64> out(n_);
        check(caf_b200_dev_download(thread_handle(), out.data(), p_, n_ * sizeof(Complex64)));
        return out;
    }
};
inline DeviceSamples read_file_c64_dev(const std::string& filename, std::size_t first_sample = 0, std::size_t max_samples = 0) {
    caf_c128* p = nullptr;
    std::size_t n = 0;
    const int rc = caf_b200_load_c64_dev_f64(thread_handle(), filename.c_str(), first_sample, max_samples, &p, &n);
    if (rc == CAF_B200_EIO) throw std::runtime_error(std::string("read_file_c64: ") + caf_b200_last_error());   // io::Result Err
    check(rc);
    return DeviceSamples(p, n);
}
// caf_surface + find_peak on device-resident samples (caf_b200_batch_f64_dev): only the doppler grid goes up and the
// 32-byte peak comes down
inline std::pair<double, std::size_t> caf_peak_dev(const DeviceSamples& needle, const DeviceSamples& haystack,
                                                   const std::vector<double>& freqs_hz, uint32_t fs) {
    if (needle.size() != haystack.size()) throw Panic("assertion failed: a.len() == self.n (xcor_rustfft.rs:54-55)");
    caf_b200_handle h = thread_handle();
    void* scratch = nullptr;
    const std::size_t fb = freqs_hz.size() * sizeof(double);
    check(caf_b200_dev_alloc(h, fb + sizeof(caf_b200_peak), &scratch));
    struct Free { void* p; ~Free() { if (p) caf_b200_dev_free(p); } } guard{scratch};
    caf_b200_peak pk{0.0, 0.0, ~0ull, 0};
    if (scratch) {
        check(caf_b200_dev_upload(h, scratch, freqs_hz.data(), fb));
        caf_b200_peak* d_pk = reinterpret_cast<caf_b200_peak*>(static_cast<char*>(scratch) + fb);
        check(caf_b200_batch_f64_dev(h, needle.data(), haystack.data(), 1, needle.size(), static_cast<const double*>(scratch),
                                     freqs_hz.size(), fs, nullptr, nullptr, nullptr, d_pk));
        check(caf_b200_dev_download(h, &pk, d_pk, sizeof pk));
    }
    return {pk.freq_hz, (std::size_t)pk.delay_idx};
}

// utils.rs:39-63: raw little-endian f64 pairs (numpy complex128)
inline void write_file_binary(const std::vector<Complex64>& v, const std::string& filename) {
    std::ofstream f(filename, std::ios::binary);
    if (!f) throw Panic("write_file_binary: cannot create " + filename);
    f.write(reinterpret_cast<const char*>(v.data()), (std::streamsize)(v.size() * sizeof(Complex64)));
}

// tests/test.rs:335-352
inline std::vector<double> gen_float_shifts(double start, double end, double step) {
    const int s = (int)(start * 1000.0), e = (int)(end * 1000.0);
    const std::size_t st = (std::size_t)(step * 1000.0);
    std::vector<double> out;
    for (int m = s; m < e; m += (int)st) out.push_back((double)m / 1e3);
    return out;
}

}  // namespace caf
