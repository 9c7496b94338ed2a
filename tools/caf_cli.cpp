// caf_cli — the reference's command-line program on the B200 library.
//
// /root/reference/caf_rust/src/main.rs:10-32 hard-codes two files and a -100..100 Hz / 0.5 Hz grid and carries a TODO
// ("Use CLAP to take in two c64 files as arguments", main.rs:1-2).  This is that program with the arguments:
//
//   caf_cli NEEDLE.c64 HAYSTACK.c64 [--fmin HZ] [--fmax HZ] [--fstep HZ] [--fs HZ]
//           [--layout rust|go|python] [--dump FILE] [--device-load] [--segments K]
//           [--detect K [--guard-doppler R] [--guard-delay C] [--min-db X |
//                        --cfar-db X [--train-doppler A] [--train-delay B] [--cfar-rank K]]]
//
// With no options it prints exactly what main.rs prints for the same two files:
//     Frequency offset: 69.0Hz
//     Time offset: 202 samples (4.208ms)
// --dump writes the surface as row-major little-endian f64 (caf_go/caf.go:14-29 dump_surf); --layout picks the
// sibling program's convention for the dump and for the reported delay (caf.go / caf.py, include/caf_b200.h).
// --device-load reads both files through pinned memory straight onto the GPU (read_file_c64_dev): the samples never exist
// as a widened Vec on the host.
// --detect K prints, after those two lines, one line per detection: the K strongest local maxima of the surface
// (caf_b200_surface_detect; guards default to 1 row x 1 cell), each refined below the grid, dropping those more than X dB
// below the first (--min-db X, min_ratio = 10^(-X/10); default: keep all K).
// --cfar-db X (with --detect K, instead of --min-db) keeps only the local maxima more than X dB above their local noise
// estimate (caf_b200_surface_detect_cfar, scale = 10^(X/10); training region --train-doppler A rows x --train-delay B
// cells beyond the guards, default 2 x 16), at most K of them and possibly none; each line ends with its SNR.
// --cfar-rank K (with --cfar-db) estimates the noise as the K-th smallest training cell instead of their mean
// (ordered-statistic CFAR, caf_b200_surface_detect_cfar_os; 1 <= K <= the training cells); the lines are the same.
// --segments K (default 1) integrates non-coherently: the needle file supplies K consecutive segments of L = len / K
// samples (the tail is dropped) and the haystack file the same K windows; the report lines and --detect / --cfar-db /
// --cfar-rank then run on the sum of the K segments' surfaces (caf_b200_surface_create_integrated_f64).  --cfar-db is a
// scale in dB either way; cfar_scale(pfa, N, looks=K) of the Python package gives the one for a sum of K.  --segments 1
// is the plain program.
// Build: g++ -std=c++17 -O2 -Iinclude tools/caf_cli.cpp -Lcaf_cookoff_b200 -lcaf_b200 -Wl,-rpath,$PWD/caf_cookoff_b200
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>
#include <vector>

#include "caf_b200.hpp"

// a whole number in [lo, hi] or exit 2 (no sign, no trailing characters)
static std::size_t count_arg(const char* what, const char* v, unsigned long lo, unsigned long hi) {
    char* end = nullptr;
    const unsigned long x = std::strtoul(v, &end, 10);
    if (!(*v >= '0' && *v <= '9') || *end || x < lo || x > hi) {
        std::fprintf(stderr, "caf_cli: %s needs a whole number in [%lu, %lu], got '%s'\n", what, lo, hi, v);
        std::exit(2);
    }
    return (std::size_t)x;
}

int main(int argc, char** argv) {
    using namespace caf;
    std::vector<std::string> pos;
    double fmin = -100.0, fmax = 100.0, fstep = 0.5;
    uint32_t fs = 48000;
    std::string layout = "rust", dump;
    bool device_load = false;
    std::size_t detect_k = 0;
    uint32_t guard_doppler = 1, guard_delay = 1;
    double min_db = INFINITY, cfar_db = NAN;
    uint32_t train_doppler = 2, train_delay = 16;
    bool train_given = false;
    uint32_t cfar_rank = 0;                                     // 0: cell-averaging CFAR
    std::size_t segments = 1;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto need = [&](const char* what) -> const char* {
            if (i + 1 >= argc) { std::fprintf(stderr, "caf_cli: %s needs a value\n", what); std::exit(2); }
            return argv[++i];
        };
        if (a == "--fmin") fmin = std::atof(need("--fmin"));
        else if (a == "--fmax") fmax = std::atof(need("--fmax"));
        else if (a == "--fstep") fstep = std::atof(need("--fstep"));
        else if (a == "--fs") fs = (uint32_t)std::atol(need("--fs"));
        else if (a == "--layout") layout = need("--layout");
        else if (a == "--dump") dump = need("--dump");
        else if (a == "--device-load") device_load = true;
        else if (a == "--detect") detect_k = count_arg("--detect", need("--detect"), 1, 1024);
        else if (a == "--guard-doppler") guard_doppler = (uint32_t)count_arg("--guard-doppler", need("--guard-doppler"), 0, 32);
        else if (a == "--guard-delay") guard_delay = (uint32_t)count_arg("--guard-delay", need("--guard-delay"), 0, 256);
        else if (a == "--min-db") {
            const char* v = need("--min-db");
            char* end = nullptr;
            min_db = std::strtod(v, &end);
            if (end == v || *end || !(min_db >= 0.0)) { std::fprintf(stderr, "caf_cli: --min-db needs a number >= 0, got '%s'\n", v); std::exit(2); }
        }
        else if (a == "--cfar-db") {
            const char* v = need("--cfar-db");
            char* end = nullptr;
            cfar_db = std::strtod(v, &end);
            if (end == v || *end || !std::isfinite(cfar_db) || !std::isfinite(std::pow(10.0, cfar_db / 10.0)) ||
                !(std::pow(10.0, cfar_db / 10.0) > 0.0)) {
                std::fprintf(stderr, "caf_cli: --cfar-db needs a finite number of dB, got '%s'\n", v);
                std::exit(2);
            }
        }
        else if (a == "--train-doppler") { train_doppler = (uint32_t)count_arg("--train-doppler", need("--train-doppler"), 0, 32); train_given = true; }
        else if (a == "--train-delay") { train_delay = (uint32_t)count_arg("--train-delay", need("--train-delay"), 0, 256); train_given = true; }
        else if (a == "--segments") segments = count_arg("--segments", need("--segments"), 1, 1ul << 20);
        else if (a == "--cfar-rank") cfar_rank = (uint32_t)count_arg("--cfar-rank", need("--cfar-rank"), 1, 65 * 513);
        else if (a == "-h" || a == "--help") {
            std::printf("usage: caf_cli NEEDLE.c64 HAYSTACK.c64 [--fmin HZ] [--fmax HZ] [--fstep HZ] [--fs HZ] "
                        "[--layout rust|go|python] [--dump FILE] [--device-load] [--segments K] "
                        "[--detect K [--guard-doppler R] [--guard-delay C] "
                        "[--min-db X | --cfar-db X [--train-doppler A] [--train-delay B] [--cfar-rank K]]]\n");
            return 0;
        } else if (a.rfind("--", 0) == 0) { std::fprintf(stderr, "caf_cli: unknown option %s\n", a.c_str()); return 2; }
        else pos.push_back(a);
    }
    if (pos.size() != 2) { std::fprintf(stderr, "caf_cli: expected NEEDLE.c64 HAYSTACK.c64 (see --help)\n"); return 2; }
    if (!(fstep > 0.0) || fs == 0) { std::fprintf(stderr, "caf_cli: --fstep and --fs must be positive\n"); return 2; }
    const bool detecting = detect_k > 0, cfar = !std::isnan(cfar_db);
    if (cfar && !detecting) { std::fprintf(stderr, "caf_cli: --cfar-db needs --detect K\n"); return 2; }
    if (cfar && !std::isinf(min_db)) { std::fprintf(stderr, "caf_cli: --cfar-db and --min-db exclude each other\n"); return 2; }
    if (train_given && !cfar) { std::fprintf(stderr, "caf_cli: --train-doppler / --train-delay need --cfar-db\n"); return 2; }
    if (cfar_rank && !cfar) { std::fprintf(stderr, "caf_cli: --cfar-rank needs --cfar-db\n"); return 2; }
    if (detecting && (device_load || layout != "rust" || !dump.empty())) {
        std::fprintf(stderr, "caf_cli: --detect goes with the default report (no --layout / --dump / --device-load)\n");
        return 2;
    }
    if (segments > 1 && (device_load || layout != "rust" || !dump.empty())) {
        std::fprintf(stderr, "caf_cli: --segments goes with the default report (no --layout / --dump / --device-load)\n");
        return 2;
    }
    try {
        if (device_load) {
            if (layout != "rust" || !dump.empty()) { std::fprintf(stderr, "caf_cli: --device-load goes with the default report (no --layout / --dump)\n"); return 2; }
            const auto needle_d = read_file_c64_dev(pos[0]);
            const auto hay_d = read_file_c64_dev(pos[1], 0, needle_d.size());        // main.rs:15
            const auto [freq, idx] = caf_peak_dev(needle_d, hay_d, gen_float_shifts(fmin, fmax, fstep), fs);
            std::printf("Frequency offset: %.1fHz\nTime offset: %zu samples (%.3fms)\n", freq, idx, (double)idx / ((double)fs / 1e3));
            return 0;
        }
        auto needle = read_file_c64(pos[0]);
        auto haystack = read_file_c64(pos[1]);
        haystack.resize(needle.size());                                  // main.rs:15
        if (segments > 1) {                                              // K windows of L samples, the tail dropped
            const std::size_t seg_l = needle.size() / segments;
            if (seg_l == 0) { std::fprintf(stderr, "caf_cli: --segments %zu needs at least that many samples\n", segments); return 2; }
            needle.resize(segments * seg_l);
            haystack.resize(segments * seg_l);
        }
        const auto shifts = gen_float_shifts(fmin, fmax, fstep);         // integer milli-Hz range, main.rs:18-22 / test.rs:335-352
        const std::size_t l = needle.size(), d = shifts.size();
        if (layout == "rust") {
            if (detecting || segments > 1) {
                // the surface (or the sum of the segments' surfaces) stays on the GPU
                const auto rows = segments > 1 ? CafB200::integrate(needle, haystack, segments, shifts, fs)
                                               : CafB200::caf_surface(needle, haystack, shifts, fs);
                const auto [freq, idx] = CafB200::find_peak(rows);
                std::printf("Frequency offset: %.1fHz\nTime offset: %zu samples (%.3fms)\n", freq, idx, (double)idx / ((double)fs / 1e3));
                if (!detecting) return 0;
                if (cfar) {
                    const double scale = std::pow(10.0, cfar_db / 10.0);
                    const auto dets = cfar_rank ? CafB200::detect_cfar_os(rows, detect_k, guard_doppler, guard_delay,
                                                                          train_doppler, train_delay, cfar_rank, scale)
                                                : CafB200::detect_cfar(rows, detect_k, guard_doppler, guard_delay,
                                                                       train_doppler, train_delay, scale);
                    for (std::size_t i = 0; i < dets.size(); ++i)
                        std::printf("Detection %zu: %.4fHz (grid %.2fHz), %.3f samples (cell %llu), %.2f dB below the first, "
                                    "%.2f dB above the noise\n", i, dets[i].freq_hz_interp, dets[i].freq_hz,
                                    dets[i].lag_samples, (unsigned long long)dets[i].delay_idx,
                                    10.0 * std::log10(dets[0].value / dets[i].value),
                                    10.0 * std::log10(dets[i].value / dets[i].noise));
                    return 0;
                }
                const double min_ratio = std::isinf(min_db) ? 0.0 : std::pow(10.0, -min_db / 10.0);
                const auto dets = CafB200::detect(rows, detect_k, guard_doppler, guard_delay, min_ratio);
                for (std::size_t i = 0; i < dets.size(); ++i)
                    std::printf("Detection %zu: %.4fHz (grid %.2fHz), %.3f samples (cell %llu), %.2f dB below the first\n", i,
                                dets[i].freq_hz_interp, dets[i].freq_hz, dets[i].lag_samples,
                                (unsigned long long)dets[i].delay_idx, 10.0 * std::log10(dets[0].value / dets[i].value));
            } else if (dump.empty()) {
                const auto [freq, idx] = CafB200::caf_peak(needle, haystack, shifts, fs);     // the surface never leaves the GPU
                std::printf("Frequency offset: %.1fHz\nTime offset: %zu samples (%.3fms)\n", freq, idx, (double)idx / ((double)fs / 1e3));
            } else {
                std::vector<double> surf(d * 2 * l);
                caf_b200_peak pk;
                check(caf_b200_surface_f64(thread_handle(), reinterpret_cast<const caf_c128*>(needle.data()),
                                           reinterpret_cast<const caf_c128*>(haystack.data()), l, shifts.data(), d, fs,
                                           surf.data(), nullptr, nullptr, &pk));
                std::ofstream(dump, std::ios::binary).write(reinterpret_cast<const char*>(surf.data()), (std::streamsize)(surf.size() * 8));
                std::printf("Frequency offset: %.1fHz\nTime offset: %zu samples (%.3fms)\n", pk.freq_hz, (std::size_t)pk.delay_idx,
                            (double)pk.delay_idx / ((double)fs / 1e3));
                std::printf("wrote (%zux%zu) surf to file\n", d, 2 * l);
            }
        } else if (layout == "go" || layout == "python") {
            const bool go = layout == "go";
            const std::size_t w = go ? 2 * l : l;
            std::vector<double> surf(dump.empty() ? 0 : d * w);
            caf_b200_peak pk;
            check(caf_b200_surface_layout_f64(thread_handle(), reinterpret_cast<const caf_c128*>(needle.data()),
                                              reinterpret_cast<const caf_c128*>(haystack.data()), l, shifts.data(), d, fs,
                                              go ? CAF_B200_LAYOUT_GO : CAF_B200_LAYOUT_PYTHON, dump.empty() ? nullptr : surf.data(), &pk));
            const long tau = go ? (long)l - (long)pk.delay_idx : (long)(l / 2) - (long)pk.delay_idx;     // main.go:35 / caf.py:145
            if (go) std::printf("caf result: %ld samples %g hz @ amb = %g\n", tau, pk.freq_hz, pk.value);
            else std::printf("amb_surf (%zu, %zu) float64 -> %ld %g\n", d, w, tau, pk.freq_hz);
            if (!dump.empty()) {
                std::ofstream(dump, std::ios::binary).write(reinterpret_cast<const char*>(surf.data()), (std::streamsize)(surf.size() * 8));
                std::printf("wrote (%zux%zu) surf to file\n", d, w);
            }
        } else {
            std::fprintf(stderr, "caf_cli: --layout must be rust, go or python\n");
            return 2;
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "caf_cli: %s\n", e.what());
        return 1;
    }
    return 0;
}
