// caf_b200.cu — C ABI (include/caf_b200.h) over the sm_100a kernels in caf_kernels.cuh.
//
// Host-side responsibilities only: argument checks that mirror the reference's panics
// (/root/reference/caf_rust/src/caf/xcor_rustfft.rs:54-55), workspace management, H2D/D2H,
// kernel launches on the handle's stream.  No CPU compute path exists here: without an
// sm_100 device create() fails (CAF_B200_ENODEVICE).
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <set>
#include <string>
#include <vector>

#include <cuda_runtime.h>
#include <dlfcn.h>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "../../include/caf_b200.h"
#include "caf_kernels.cuh"
#include "caf_large.cuh"
#include "caf_detect.cuh"
#include "caf_cfar.cuh"
#include "overlap_policy.hpp"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char b_[512];                                                                          \
            snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return fail(CAF_B200_ECUDA, b_);                                                       \
        }                                                                                          \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

template <typename T> struct Tables { caf::cx<T>* tw1 = nullptr; caf::cx<T>* tw2 = nullptr; caf::cx<T>* g = nullptr; };

}  // namespace

// ---- NCCL, bound at run time --------------------------------------------------------------------------------
// The library has no link-time NCCL dependency: libnccl.so.2 is dlopen()ed on first use (inside a torch process
// that is the copy torch already loaded, otherwise the system one).  Only the handful of entry points the peak
// exchange needs are bound; the types below are NCCL's stable 2.x ABI (nccl.h: ncclUniqueId is 128 opaque bytes,
// ncclUint64 == 5, ncclSuccess == 0).
namespace {
struct NcclUniqueId { char internal[CAF_B200_NCCL_ID_BYTES]; };
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(NcclUniqueId*) = nullptr;
    int (*CommInitRank)(void**, int, NcclUniqueId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string why;
    bool ok() const { return lib && GetUniqueId && CommInitRank && CommDestroy && AllGather && GetErrorString; }
};
NcclApi& nccl_api() {
    static NcclApi api = [] {
        NcclApi a;
        // a copy the process already holds (torch's) wins; then the caller's choice; then the system library
        a.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        const char* names[] = {getenv("CAF_B200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (a.lib) break;
            if (!n || !*n) continue;
            a.lib = dlopen(n, RTLD_NOW | RTLD_LOCAL);
            if (!a.lib) a.why = dlerror();
        }
        if (!a.lib) return a;
        a.GetUniqueId = (int (*)(NcclUniqueId*))dlsym(a.lib, "ncclGetUniqueId");
        a.CommInitRank = (int (*)(void**, int, NcclUniqueId, int))dlsym(a.lib, "ncclCommInitRank");
        a.CommDestroy = (int (*)(void*))dlsym(a.lib, "ncclCommDestroy");
        a.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(a.lib, "ncclAllGather");
        a.GetErrorString = (const char* (*)(int))dlsym(a.lib, "ncclGetErrorString");
        if (!a.ok()) a.why = "libnccl is missing one of ncclGetUniqueId/CommInitRank/CommDestroy/AllGather/GetErrorString";
        return a;
    }();
    return api;
}
constexpr int kNcclUint64 = 5;
}  // namespace

struct caf_b200_comm_s {
    caf_b200_handle h = nullptr;          // identity check only (never dereferenced: the handle may die first)
    int device = 0;
    void* comm = nullptr;       // ncclComm_t
    bool own = false;
    int world = 1, rank = 0;
    unsigned long long* send = nullptr;   // device: 4 words
    unsigned long long* recv = nullptr;   // device: 4 * world words
    unsigned long long* host = nullptr;   // pinned: 4 * world words
    int* status = nullptr;                // pinned, device-addressable: 1 when a peer reported a failure in the last exchange
    // find_peak across ranks over NVLink peer memory (caf_peak_exchange_kernel): this rank's mailbox, mapped by every peer
    // through CUDA IPC, and the peers' mailboxes mapped here.  p2p is false (NCCL all-gather instead) when any rank could
    // not map any peer, or with CAF_B200_P2P=0.
    bool p2p = false;
    unsigned long long* mail = nullptr;           // device: [2][world][8] words
    unsigned long long** peer_mail = nullptr;     // device: [world] pointers (own entry = mail)
    std::vector<void*> opened;                    // IPC mappings to close
    unsigned long long p2p_epoch = 0;
};

struct caf_b200_handle_s {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    unsigned long long launches = 0;
    Tables<double> td;
    Tables<float> tf;
    int occ_d = 1, occ_f = 1;   // resident CTAs per SM of the surface kernel
    DevBuf needle, hay, hperm, freqs, surface, rowval, rowidx, peaks, scratch, layout;
    std::vector<std::pair<void*, size_t>> surf_pool;   // device buffers of released surface objects, reused by the next one
    DevBuf in_block;            // small host calls: needle | haystack | freqs in ONE device block (one H2D instead of three)
    void* h_stage = nullptr;    // pinned host mirror of in_block for callers whose three inputs are not one contiguous block
    size_t h_stage_cap = 0;
    DevBuf lwbuf, lhtmp, lhbig, lpart;      // long-row path: chunk scratch, scratch of the H transform, H, partial row maxima
    DevBuf det, det_io;                     // detection: counters | candidate lists; host calls' grid | records | count
    long long* trace = nullptr;   // CAF_TRACE builds: device buffer for phase stamps
    // Launch-private state of single-pair surface launches, a ring of kRing slots indexed by launch number (epoch % kRing):
    // several such launches can be in flight at once (overlap, below).
    static constexpr int kRing = 8;
    unsigned int* done_counter = nullptr;   // [kRing] last-CTA-done tickets of the fused find_peak, monotonic
    void* hshare = nullptr;                 // [kRing][8192 complex128] H published by the publishing CTAs
    unsigned int* hflag = nullptr;          // [kRing][2] publish counters, monotonic
    unsigned int epoch = 0;
    unsigned int done_total[kRing] = {};    // tickets drawn so far from done_counter[slot]
    // Overlap of consecutive single-pair surface launches (RowArgs::flags bit 0; include/caf_b200.h, caf_b200_set_overlap).
    // overlap = 0: off.  1: a launch independent of its predecessors skips the wait for the grid before it, full grids.
    // n >= 2: such a launch also uses only ceil(SMs / n) CTAs, so that ~n launches share the GPU and every CTA amortises
    // its set-up over n times as many rows.
    int overlap = 0;
    bool overlap_killed = false;            // CAF_B200_OVERLAP=0 in the environment at handle creation
    using Range = caf_host::Range;
    static constexpr int kHist = kRing - 1;          // launches whose buffers are compared (overlap_policy.hpp)
    caf_host::OverlapHistory<kHist> hist;
    // small single-pair host calls: the kernel pulls its inputs out of pinned host memory itself (RowArgs::pull_*)
    unsigned int* pull_counter = nullptr;       // device word the grid meets on, monotonic
    unsigned int pull_total = 0;                // its value after every launch issued so far
    const void* pull_src = nullptr;             // set by run_batch_host around ONE run_batch_dev call
    size_t pull_bytes = 0;
    bool allow_pull = true;                     // CAF_B200_PULL
    int gather_ahead = 2;                       // two-level gather: L2 tile prefetch distance in blocks per SM (CAF_B200_GATHER_AHEAD, development)
    unsigned int* seq_ptr = nullptr;            // single-pair host calls: pinned word the fused find_peak signals (see run_batch_host)
    unsigned int seq_val = 0, seq_counter = 0;
    unsigned long long* pack_words = nullptr;   // sharded rows: find_peak also writes its result packed for the exchange
    unsigned long long pack_offset = 0;         // global index of the first local doppler row
    void* h_peaks = nullptr;    // pinned staging for peaks
    size_t h_peaks_cap = 0;
    bool profiling = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // around spectrum | rows | peak
    cudaStream_t copy_stream = nullptr;     // side stream: D2H of the head rows while the rest is computed; the long rows' H transform
    cudaEvent_t ev_head = nullptr, ev_copy = nullptr;
    // switches read ONCE, at handle creation (include/caf_b200.h lists them)
    size_t chunk_mb = 6144;                 // CAF_B200_CHUNK_MB
    bool allow_pipeline = true;             // CAF_B200_PIPELINE
    bool peak_zero_copy = true;             // CAF_B200_PEAK_ZEROCOPY
    bool ev_valid = false;
};

// ---- device-resident surface objects (caf_b200_surface_*): CafSurfaceRow's fields are private in the reference
//      (mod.rs:17-22), so the drop-in caller can only observe find_peak's result; the 26 MB of a surface stay on the GPU
//      and a row crosses PCIe when somebody asks for it. ----
struct caf_b200_surface_s {
    caf_b200_handle h = nullptr;
    int device = 0;
    bool f32 = false;
    size_t d = 0, n = 0, bytes = 0;
    void* dev = nullptr;
    void* dev_rv = nullptr;             // row peaks on the device (tail of the same buffer), fetched on first request
    unsigned long long* dev_ri = nullptr;
    bool peaks_on_host = false;
    std::vector<double> pval;
    std::vector<uint64_t> pidx;
    std::vector<double> freqs;
    caf_b200_peak peak{};
};

namespace {

// Copy into the pinned staging block the GPU is about to read across PCIe.  The CPU never reads that block again, so the
// stores are non-temporal: no read-for-ownership of 134 KB of lines the previous call's PCIe reads pushed out of the caches,
// and the data is on its way to DRAM when the kernel's loads arrive.  dst is 16-byte aligned (offsets in the block are).
inline void stage_copy(void* dst, const void* src, size_t n) {
#if defined(__x86_64__)
    if (((uintptr_t)dst & 15) == 0) {
        char* d = (char*)dst; const char* s_ = (const char*)src;
        size_t i = 0;
        for (; i + 64 <= n; i += 64) {
            const __m128i a0 = _mm_loadu_si128((const __m128i*)(s_ + i)), a1 = _mm_loadu_si128((const __m128i*)(s_ + i + 16));
            const __m128i a2 = _mm_loadu_si128((const __m128i*)(s_ + i + 32)), a3 = _mm_loadu_si128((const __m128i*)(s_ + i + 48));
            _mm_stream_si128((__m128i*)(d + i), a0); _mm_stream_si128((__m128i*)(d + i + 16), a1);
            _mm_stream_si128((__m128i*)(d + i + 32), a2); _mm_stream_si128((__m128i*)(d + i + 48), a3);
        }
        if (i < n) std::memcpy(d + i, s_ + i, n - i);
        return;
    }
#endif
    std::memcpy(dst, src, n);
}
inline void stage_fence() {
#if defined(__x86_64__)
    _mm_sfence();      // the streamed data is globally visible before the launch's doorbell is rung
#endif
}

// blocks handed out by caf_b200_host_alloc: pinned and device-addressable, so a kernel may read inputs straight from them
std::mutex g_pinned_mu;
std::vector<std::pair<const char*, size_t>> g_pinned_blocks;
bool pinned_block_holds(const void* p, size_t bytes) {
    std::lock_guard<std::mutex> lk(g_pinned_mu);
    for (const auto& b : g_pinned_blocks)
        if ((const char*)p >= b.first && (const char*)p + bytes <= b.first + b.second) return true;
    return false;
}

std::mutex g_live_mu;
std::set<caf_b200_handle> g_live_handles;     // a surface object outliving its handle frees its buffer itself

template <typename T> Tables<T>& tables(caf_b200_handle h);
template <> Tables<double>& tables<double>(caf_b200_handle h) { return h->td; }
template <> Tables<float>& tables<float>(caf_b200_handle h) { return h->tf; }

template <typename T> size_t smem_bytes() { return caf::SmemLayout<T>::kTotal; }

template <typename T>
cudaError_t upload_tables(Tables<T>& t, cudaStream_t s) {
    using C = caf::cx<T>;
    const long double TWO_PI = 6.283185307179586476925286766559005768L;
    std::vector<C> tw1(16 * 256), tw2(256), g(4096);
    for (int k = 0; k < 16; ++k)
        for (int tt = 0; tt < 256; ++tt) {
            long double a = -TWO_PI * (long double)((k * tt) % 4096) / 4096.0L;
            tw1[k * 256 + tt].x = (T)cosl(a); tw1[k * 256 + tt].y = (T)sinl(a);
        }
    for (int a_ = 0; a_ < 16; ++a_)
        for (int b_ = 0; b_ < 16; ++b_) {
            long double a = -TWO_PI * (long double)((a_ * b_) % 256) / 256.0L;
            tw2[a_ * 16 + b_].x = (T)cosl(a); tw2[a_ * 16 + b_].y = (T)sinl(a);
        }
    for (int n = 0; n < 4096; ++n) {
        long double a = TWO_PI * (long double)n / 8192.0L;
        g[n].x = (T)cosl(a); g[n].y = (T)sinl(a);
    }
    cudaError_t e;
    if ((e = cudaMalloc(&t.tw1, sizeof(C) * tw1.size())) != cudaSuccess) return e;
    if ((e = cudaMalloc(&t.tw2, sizeof(C) * tw2.size())) != cudaSuccess) return e;
    if ((e = cudaMalloc(&t.g, sizeof(C) * g.size())) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(t.tw1, tw1.data(), sizeof(C) * tw1.size(), cudaMemcpyHostToDevice, s)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(t.tw2, tw2.data(), sizeof(C) * tw2.size(), cudaMemcpyHostToDevice, s)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(t.g, g.data(), sizeof(C) * g.size(), cudaMemcpyHostToDevice, s)) != cudaSuccess) return e;
    return cudaStreamSynchronize(s);   // the host vectors die at scope exit
}

template <typename T, int MODE, bool FULL = false, bool SHARED = false>
cudaError_t configure_kernel(int* occ_out) {
    auto k = caf::caf_rows_kernel<T, MODE, FULL, SHARED>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes<T>());
    if (e != cudaSuccess) return e;
    if (occ_out) {
        int occ = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, caf::kThreads, smem_bytes<T>());
        if (e != cudaSuccess) return e;
        // the occupancy calculator does not know about tensor memory: a CTA allocates TmemGeom<T>::kAlloc of the SM's 512
        // columns, and a single-pair launch needs its whole grid co-resident (consumer CTAs wait for the publisher's H)
        const int tmem_cap = 512 / caf::TmemGeom<T>::kAlloc;
        if (occ > tmem_cap) occ = tmem_cap;
        *occ_out = occ < 1 ? 1 : occ;
    }
    return cudaSuccess;
}

// fused two-level kernels: tile of 2 * RT * 16 * J cells in dynamic shared memory.  Function attributes are per
// device, so this runs for every handle (create_impl), not once per process.
constexpr int kFusedJ = 16;
template <typename T, int RT>
cudaError_t configure_fused() {
    const int smem = (int)(sizeof(caf::cx<T>) * 2 * RT * 16 * kFusedJ);
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(caf::caf_large_spread2<T, RT, kFusedJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(caf::caf_large_gather2<T, RT, kFusedJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess) return e;
    return cudaFuncSetAttribute(caf::caf_large_gather2<T, RT, kFusedJ, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

// detection tiles: allowed the largest dynamic shared memory run_detect_dev can ask for, once per handle (the attribute
// belongs to the device, so every handle sets the same value and no handle can lower it under another)
template <typename T>
cudaError_t configure_detect() {
    return cudaFuncSetAttribute(caf::caf_detect_tiles_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)caf::det_tile_smem_max<T>());
}

// CFAR tiles: the same rule, at the most run_cfar_dev can ask for (a one-row tile staging its training region)
template <typename T>
cudaError_t configure_cfar() {
    return cudaFuncSetAttribute(caf::caf_cfar_tiles_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)caf::kCfarSmemMax);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point query: no link-time dependency on libcuda
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}
// The scratch buffer of a chunk as a 2-D tensor for the TMA engine: [units][4096 complex] seen as [units][8192 reals];
// a box is `box_units` consecutive units x `j` positions (caf_large.cuh, Fused2).
template <typename T>
cudaError_t make_unit_map(CUtensorMap* tm, void* base, size_t units, int j, int box_units) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return cudaErrorNotSupported;
    const cuuint64_t gdim[2] = {(cuuint64_t)(2 * caf::kL0), (cuuint64_t)units};
    const cuuint64_t gstride[1] = {(cuuint64_t)(caf::kL0 * sizeof(caf::cx<T>))};
    const cuuint32_t box[2] = {(cuuint32_t)(2 * j), (cuuint32_t)box_units};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(tm, std::is_same<T, double>::value ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                           base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

template <typename T>
cudaError_t configure_all(int* occ) {
    cudaError_t e;
    if ((e = configure_fused<T, 2>()) != cudaSuccess) return e;
    if ((e = configure_fused<T, 4>()) != cudaSuccess) return e;
    if ((e = configure_fused<T, 8>()) != cudaSuccess) return e;
    if ((e = configure_kernel<T, caf::kSurface, true, true>(occ)) != cudaSuccess) return e;
    if ((e = configure_kernel<T, caf::kSurface, false, true>(nullptr)) != cudaSuccess) return e;
    if ((e = configure_kernel<T, caf::kSurface, true, false>(nullptr)) != cudaSuccess) return e;
    if ((e = configure_kernel<T, caf::kSurface, false, false>(nullptr)) != cudaSuccess) return e;
    if ((e = configure_kernel<T, caf::kSpectrumHalf>(nullptr)) != cudaSuccess) return e;
    if ((e = configure_kernel<T, caf::kSpectrumFull>(nullptr)) != cudaSuccess) return e;
    if ((e = configure_kernel<T, caf::kXcorFull>(nullptr)) != cudaSuccess) return e;
    if ((e = configure_kernel<T, caf::kXcorHalf>(nullptr)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(caf::caf_large_core<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)caf::SmemLayout<T>::kTotalNoNeedle)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(caf::caf_large_core<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)caf::SmemLayout<T>::kTotalNoNeedle)) != cudaSuccess) return e;
    return cudaSuccess;
}

template <typename T, int MODE, bool FULL = false>
cudaError_t launch_rows(caf_b200_handle h, const caf::RowArgs<T>& a, long long n_items, long long grid_cap = 0) {
    if (n_items <= 0) return cudaSuccess;
    const int occ = std::is_same<T, double>::value ? h->occ_d : h->occ_f;
    long long cap = (long long)h->sm_count * occ;
    if (grid_cap > 0 && grid_cap < cap) cap = grid_cap;
    int grid = (int)(n_items < cap ? n_items : cap);
    h->launches++;
    if (MODE == caf::kSurface) {
        // programmatic stream serialisation: this launch may begin (TMEM, tables -- nothing that touches caller memory)
        // while the kernel before it on the stream drains; see griddepcontrol.wait in caf_rows_kernel
        cudaLaunchConfig_t cfg{};
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(caf::kThreads);
        cfg.dynamicSmemBytes = smem_bytes<T>(); cfg.stream = h->stream;
        if (a.hshare != nullptr) return cudaLaunchKernelEx(&cfg, caf::caf_rows_kernel<T, MODE, FULL, true>, a);
        return cudaLaunchKernelEx(&cfg, caf::caf_rows_kernel<T, MODE, FULL, false>, a);
    }
    caf::caf_rows_kernel<T, MODE, FULL><<<grid, caf::kThreads, smem_bytes<T>(), h->stream>>>(a);
    return cudaGetLastError();
}

template <typename T>
caf::RowArgs<T> base_args(caf_b200_handle h) {
    caf::RowArgs<T> a{};
    Tables<T>& t = tables<T>(h);
    a.tw1 = t.tw1; a.tw2 = t.tw2; a.g = t.g;
    a.dt = 0.0; a.L = 0; a.D = 1; a.P = 1;
    a.trace = h->trace;
    return a;
}

// ---- rows longer than 8192 cells: four-/six-step FFT (caf_large.cuh), one pair at a time, rows in L2-sized chunks ----
template <typename T, int R>
cudaError_t launch_large_top_rt(caf_b200_handle h, const caf::LargeArgs<T>& a, bool gather) {
    dim3 grid((unsigned)(a.inner_top / 256), (unsigned)a.rows);
    if (!gather) caf::caf_large_spread_top<T, R><<<grid, 256, 0, h->stream>>>(a);
    else if (a.cplx) caf::caf_large_gather_top<T, R, true><<<grid, 256, 0, h->stream>>>(a);
    else caf::caf_large_gather_top<T, R><<<grid, 256, 0, h->stream>>>(a);
    h->launches++;
    return cudaGetLastError();
}
template <typename T>
cudaError_t launch_large_top(caf_b200_handle h, const caf::LargeArgs<T>& a, bool gather) {
    switch (a.Rtop) {
        case 2: return launch_large_top_rt<T, 2>(h, a, gather);
        case 4: return launch_large_top_rt<T, 4>(h, a, gather);
        case 8: return launch_large_top_rt<T, 8>(h, a, gather);
        case 16: return launch_large_top_rt<T, 16>(h, a, gather);
        default: return cudaErrorInvalidValue;
    }
}
// two-level rows: fused spread (top + mid) and gather (mid + top), J innermost positions per block
template <typename T, int RT, int J>
cudaError_t launch_large_fused_rt(caf_b200_handle h, const caf::LargeArgs<T>& a, bool gather) {
    dim3 grid((unsigned)(caf::kL0 / J), (unsigned)a.rows);
    const size_t smem = sizeof(caf::cx<T>) * 2 * RT * 16 * J;
    if (!gather) {
        caf::caf_large_spread2<T, RT, J><<<grid, 16 * J, smem, h->stream>>>(a);
    } else {
        // the gather's tiles are prefetched into L2 by the TMA engine, `ahead` blocks ahead of the block that loads them
        CUtensorMap tm;
        const int box_units = 2 * RT * 16;
        cudaError_t e = make_unit_map<T>(&tm, a.wbuf, (size_t)a.rows * box_units, J, box_units);
        if (e != cudaSuccess) return e;
        const int ahead = h->gather_ahead * h->sm_count;
        if (a.cplx) caf::caf_large_gather2<T, RT, J, true><<<grid, 16 * J, smem, h->stream>>>(a, tm, ahead);
        else caf::caf_large_gather2<T, RT, J><<<grid, 16 * J, smem, h->stream>>>(a, tm, ahead);
    }
    h->launches++;
    return cudaGetLastError();
}
template <typename T>
cudaError_t launch_large_fused(caf_b200_handle h, const caf::LargeArgs<T>& a, bool gather) {
    // 16 positions per block (256-byte runs, 64 KB tile, three blocks per SM) measured best: 32 positions (one block per
    // SM) 44.2 ms against 40.9 ms on 2048 config-5 rows, 8 positions the same as 16
    switch (a.Rtop) {
        case 2: return launch_large_fused_rt<T, 2, kFusedJ>(h, a, gather);
        case 4: return launch_large_fused_rt<T, 4, kFusedJ>(h, a, gather);
        case 8: return launch_large_fused_rt<T, 8, kFusedJ>(h, a, gather);
        default: return cudaErrorInvalidValue;
    }
}
template <typename T, bool HMODE>
cudaError_t launch_large_core(caf_b200_handle h, const caf::LargeArgs<T>& a) {
    // two warp groups per SM; the kernel cuts the (position, row) units into one contiguous share per group
    const long long upr = a.N / caf::kL0;
    const long long units = (long long)a.rows * upr;
    const long long groups = units < 2LL * h->sm_count ? units : 2LL * h->sm_count;
    const long long ctas = (groups + 1) / 2;
    caf::caf_large_core<T, HMODE><<<(unsigned)ctas, caf::kThreads, caf::SmemLayout<T>::kTotalNoNeedle, h->stream>>>(a);
    h->launches++;
    return cudaGetLastError();
}
// The three stages of a chunk of long rows: spread (one level: spread_top; two levels: the fused spread2), core, and
// -- unless H is being built -- gather (gather_top / gather2: inverse top step, radix-2, |.|^2, row argmax).
template <typename T>
int large_spread(caf_b200_handle h, const caf::LargeArgs<T>& a) {
    if (a.inner_top != caf::kL0) CK(launch_large_fused<T>(h, a, false));
    else CK(launch_large_top<T>(h, a, false));
    return CAF_B200_OK;
}
template <typename T>
int large_gather(caf_b200_handle h, const caf::LargeArgs<T>& a) {
    if (a.inner_top != caf::kL0) CK(launch_large_fused<T>(h, a, true));
    else CK(launch_large_top<T>(h, a, true));
    return CAF_B200_OK;
}

template <typename T>
int run_large_dev(caf_b200_handle h, const caf::cx<T>* needles, const caf::cx<T>* hays, size_t p, size_t l,
                  const double* freqs, size_t d, uint32_t fs, T* surface, T* rowval,
                  unsigned long long* rowidx, caf::PeakOut* peaks, caf::cx<T>* cplx = nullptr) {
    using namespace caf;
    long long n = 16384;
    while ((size_t)n < 2 * l) n *= 2;
    const bool two = n > 131072;
    const int inner = two ? 65536 : kL0;
    const int rtop = (int)(n / 2 / inner);
    const size_t row_bytes = sizeof(cx<T>) * (size_t)n;
    // Rows are processed in chunks whose scratch is bounded by a budget.  Round 1 first sized the chunks to stay inside
    // the 126 MB L2; measured with the final kernels the opposite holds -- the streaming spread / gather kernels run as
    // fast out of HBM, and every extra chunk costs launches, a TMEM/H prologue per core launch and a partly filled last
    // pass (config 3: 72 MB chunks 5.54 ms, 432 MB 4.70 ms, one chunk 4.23 ms; config 5 rows: 48 MB 34.3 us, 4 GB
    // 27.3 us per row).  Default budget 6 GB; CAF_B200_CHUNK_MB (read at handle creation) overrides.
    size_t chunk = (h->chunk_mb << 20) / row_bytes;
    if (chunk < 1) chunk = 1;
    if (chunk < d) {
        // equal chunks, each a whole number of "sets" of rows (groups / positions): the core keeps every warp group on one
        // position of the row, so such a chunk leaves no group idle in its last pass
        const size_t upr = (size_t)(n / kL0), groups = 2 * (size_t)h->sm_count;
        const size_t sets = groups >= upr ? groups / upr : 1;
        const size_t nch = (d + chunk - 1) / chunk;
        chunk = (d + nch - 1) / nch;
        chunk = (chunk + sets - 1) / sets * sets;
    }
    if (chunk < 1) chunk = 1;
    if (chunk > d) chunk = d;
    if (chunk > 65535) chunk = 65535;                       // rows of a chunk are grid.y of the one-level spread / gather launches
    const int nparts = two ? kL0 / kFusedJ : inner / 256;   // gather blocks per row (each leaves one partial maximum)
    CK(h->lwbuf.ensure(row_bytes * chunk));
    CK(h->lhtmp.ensure(row_bytes));
    CK(h->lhbig.ensure(row_bytes));
    CK(h->lpart.ensure((sizeof(double) + sizeof(int)) * (size_t)nparts * chunk + sizeof(unsigned int) * chunk));
    T* rv = rowval; unsigned long long* ri = rowidx;
    if (!rv || !ri) {
        CK(h->scratch.ensure((sizeof(T) + sizeof(unsigned long long)) * p * d + 16));
        ri = reinterpret_cast<unsigned long long*>(h->scratch.p);
        rv = reinterpret_cast<T*>(ri + p * d);
    }
    if (!h->copy_stream) CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    if (!h->ev_head) CK(cudaEventCreateWithFlags(&h->ev_head, cudaEventDisableTiming));
    if (!h->ev_copy) CK(cudaEventCreateWithFlags(&h->ev_copy, cudaEventDisableTiming));
    Tables<T>& t = tables<T>(h);
    LargeArgs<T> a{};
    a.wbuf = (cx<T>*)h->lwbuf.p; a.hbig = (cx<T>*)h->lhbig.p;
    a.part_val = (double*)h->lpart.p; a.part_idx = (int*)((double*)h->lpart.p + (size_t)nparts * chunk);
    a.row_ticket = (unsigned int*)(a.part_idx + (size_t)nparts * chunk);
    CK(cudaMemsetAsync(a.row_ticket, 0, sizeof(unsigned int) * chunk, h->stream));   // tickets start at zero (the layout moves with the shape)
    a.tw1 = t.tw1; a.tw2 = t.tw2; a.g = t.g;
    a.dt = 1.0 / (double)fs; a.L = (int)l; a.N = (int)n; a.Rtop = rtop; a.inner_top = inner;
    a.trace = h->trace;
    cudaStream_t const main_s = h->stream, side_s = h->copy_stream;
    for (size_t pi = 0; pi < p; ++pi) {
        // H = FFT(haystack)/N once per pair (the reference recomputes it per row, xcor_rustfft.rs:58-59).  It is a chain of
        // under-filled launches (one row), so it runs on the side stream, with its own one-row scratch, WHILE the main
        // stream already spreads the first chunk of needle rows; the core of that chunk waits for it.
        CK(cudaEventRecord(h->ev_head, main_s));             // the previous pair's cores are done with hbig
        CK(cudaStreamWaitEvent(side_s, h->ev_head, 0));
        {
            LargeArgs<T> ah = a;
            ah.wbuf = (cx<T>*)h->lhtmp.p; ah.in = hays + pi * l; ah.freqs = nullptr; ah.rows = 1; ah.surface = nullptr;
            h->stream = side_s;
            int rc = large_spread<T>(h, ah);
            if (!rc) { cudaError_t e = launch_large_core<T, true>(h, ah); if (e != cudaSuccess) rc = fail(CAF_B200_ECUDA, cudaGetErrorString(e)); }
            h->stream = main_s;
            if (rc) return rc;
            CK(cudaEventRecord(h->ev_copy, side_s));
        }
        bool h_pending = true;
        for (size_t off = 0; off < d; off += chunk) {
            const size_t c = (d - off < chunk) ? d - off : chunk;
            a.in = needles + pi * l; a.freqs = freqs + off; a.rows = (int)c;
            a.surface = surface ? surface + (pi * d + off) * 2 * l : nullptr;
            a.cplx = cplx ? cplx + (pi * d + off) * (size_t)n : nullptr;
            a.row_peak_val = rv + pi * d + off; a.row_peak_idx = ri + pi * d + off;
            int rc = large_spread<T>(h, a);
            if (rc) return rc;
            if (h_pending) { CK(cudaStreamWaitEvent(main_s, h->ev_copy, 0)); h_pending = false; }
            CK((launch_large_core<T, false>(h, a)));
            rc = large_gather<T>(h, a);
            if (rc) return rc;
        }
        if (h_pending) CK(cudaStreamWaitEvent(main_s, h->ev_copy, 0));     // d == 0 cannot happen here, but never leave the side stream unjoined
    }
    if (peaks || h->pack_words) {
        caf_peak_kernel<T><<<(unsigned)p, 256, 0, h->stream>>>(rv, ri, freqs, (int)d, peaks, h->pack_words, h->pack_offset);
        h->launches++;
        CK(cudaGetLastError());
    }
    return CAF_B200_OK;
}

// The whole device-side pipeline for p pairs; every pointer is device memory.
template <typename T>
int run_batch_dev(caf_b200_handle h, const caf::cx<T>* needles, const caf::cx<T>* hays, size_t p, size_t l,
                  const double* freqs, size_t d, uint32_t fs, T* surface, T* rowval,
                  unsigned long long* rowidx, caf::PeakOut* peaks) {
    using namespace caf;
    if (p == 0) return CAF_B200_OK;
    if (l == 0 || d == 0) {
        // empty rows: xcor_peak_idx = 0, xcor_peak_val = 0.0 (mod.rs:143-144); find_peak -> dummy row
        if (d && rowval) CK(cudaMemsetAsync(rowval, 0, sizeof(T) * p * d, h->stream));
        if (d && rowidx) CK(cudaMemsetAsync(rowidx, 0, sizeof(unsigned long long) * p * d, h->stream));
        if (peaks) {
            std::vector<PeakOut> z(p);
            for (auto& q : z) { q.value = 0.0; q.freq_hz = 0.0; q.doppler_idx = ~0ull; q.delay_idx = 0; }
            CK(cudaMemcpyAsync(peaks, z.data(), sizeof(PeakOut) * p, cudaMemcpyDefault, h->stream));   // peaks may be pinned host memory
            CK(cudaStreamSynchronize(h->stream));
        }
        if (h->pack_words) {      // a rank that owns no rows still contributes "no row" to the exchange
            caf_peak_pack_kernel<<<1, 32, 0, h->stream>>>(nullptr, 0ull, h->pack_words);
            h->launches++;
            CK(cudaGetLastError());
        }
        return CAF_B200_OK;
    }
    if (l > (size_t)kL0) return run_large_dev<T>(h, needles, hays, p, l, freqs, d, fs, surface, rowval, rowidx, peaks);
    // row peaks are needed internally for find_peak even when the caller does not want them
    T* rv = rowval; unsigned long long* ri = rowidx;
    if (peaks && (!rv || !ri)) {
        CK(h->scratch.ensure((sizeof(T) + sizeof(unsigned long long)) * p * d + 16));
        ri = reinterpret_cast<unsigned long long*>(h->scratch.p);
        rv = reinterpret_cast<T*>(ri + p * d);
    }
    RowArgs<T> a = base_args<T>(h);
    a.L = (int)l; a.P = (int)p; a.D = (int)d;
    a.in = needles; a.in2 = hays; a.freqs = freqs; a.dt = 1.0 / (double)fs;   // dt: mod.rs:53
    a.out = surface; a.row_peak_val = rv; a.row_peak_idx = ri;
    const bool fused_peak = peaks && p == 1 && d > 1;      // single pair over many CTAs: find_peak rides in the same launch
    if (fused_peak) {
        a.peak = peaks; a.done_counter = h->done_counter; a.peak_words = h->pack_words; a.row_offset = h->pack_offset;
        a.peak_seq = h->seq_ptr; a.seq_val = h->seq_val;
    }
    const bool prof = h->profiling;
    // ---- may this launch overlap its predecessors?  Only a single-pair device launch directly behind another overlappable
    //      one (no other library launch in between), with every buffer disjoint from those of the launches in the history
    //      (the previous kHist = 7) wherever one side writes.  Why 7 is enough: a CTA of launch k is placed only after every
    //      CTA of k-1 has started (launch_dependents is issued at entry), hence after every CTA of k-2 ... k-7 has started;
    //      those are 7 x grid >= 7 x 37 = 259 CTAs on 148 SMs, so at least 112 of them must have run to completion while a
    //      CTA of k-8 was still running -- it would have to take twice as long as its peers, which all carry the same
    //      rows +- 1.  (A formal version, a second griddepcontrol.wait at the END of an overlapped launch, was measured and
    //      cancels the whole gain: caf_kernels.cuh.) ----
    caf_b200_handle_s::Range cur_in[3] = {}, cur_out[6] = {};
    bool overlappable = false;
    long long grid_cap = 0;                       // 0 = one CTA per SM
    if (p == 1 && d > 1 && h->overlap > 0 && !h->pull_src && !h->seq_ptr && !prof) {
        const int occ_ = std::is_same<T, double>::value ? h->occ_d : h->occ_f;
        const long long full = (long long)h->sm_count * occ_;
        const long long want = caf_host::overlapped_grid(full, h->overlap);      // CTAs of an overlapped launch
        if ((long long)d >= full) {               // (smaller problems keep full stream order)
            overlappable = true;
            cur_in[0] = {(const char*)needles, sizeof(cx<T>) * l}; cur_in[1] = {(const char*)hays, sizeof(cx<T>) * l};
            cur_in[2] = {(const char*)freqs, sizeof(double) * d};
            cur_out[0] = {(const char*)surface, surface ? sizeof(T) * d * 2 * l : 0};
            cur_out[1] = {(const char*)rv, rv ? sizeof(T) * d : 0}; cur_out[2] = {(const char*)ri, ri ? sizeof(unsigned long long) * d : 0};
            cur_out[3] = {(const char*)peaks, peaks ? sizeof(PeakOut) : 0};
            cur_out[4] = {(const char*)h->pack_words, h->pack_words ? (size_t)32 : (size_t)0};
            const bool indep = h->hist.independent(cur_in, cur_out, h->launches);
            if (indep) { a.flags |= 1u; grid_cap = want; }
        }
    }
    if (p == 1 && d > 1) {                        // one pair over many CTAs: CTA 0 publishes H, the rest consume it
        a.epoch = ++h->epoch;
        const unsigned int slot = a.epoch % (unsigned int)caf_b200_handle_s::kRing;
        a.hshare = reinterpret_cast<cx<T>*>(reinterpret_cast<double2*>(h->hshare) + (size_t)slot * caf::kM); a.hflag = h->hflag + 2 * slot;
        // H_1's publisher: the lowest-index CTA other than 0 that owns the fewest rows (same split as the kernel)
        const long long n_items = (long long)d;
        const int occ = std::is_same<T, double>::value ? h->occ_d : h->occ_f;
        long long cap = (long long)h->sm_count * occ;
        if (grid_cap > 0 && grid_cap < cap) cap = grid_cap;
        const long long grid = n_items < cap ? n_items : cap;
        if (fused_peak) { a.done_counter = h->done_counter + slot; a.done_last = h->done_total[slot] + (unsigned int)grid - 1u; }
        a.hprod1 = 0;
        long long best = -1;
        for (long long b = 1; b < grid; ++b) {
            const long long cnt = n_items * (b + 1) / grid - n_items * b / grid;
            if (best < 0 || cnt < best) { best = cnt; a.hprod1 = (int)b; }
        }
        if (h->pull_src) {      // the grid fetches needle | haystack | freqs from pinned host memory itself
            a.pull_src = reinterpret_cast<const uint4*>(h->pull_src);
            a.pull_dst = reinterpret_cast<uint4*>(const_cast<cx<T>*>(needles));
            a.pull_n16 = (unsigned int)(h->pull_bytes / 16);
            a.pull_counter = h->pull_counter;
            a.pull_target = h->pull_total + 2u * (unsigned int)grid;      // two pulling warps per CTA
        }
    }
    if (prof) {
        for (auto& e : h->ev) if (!e) CK(cudaEventCreate(&e));
        h->ev_valid = false;
        CK(cudaEventRecord(h->ev[0], h->stream));
        CK(cudaEventRecord(h->ev[1], h->stream));
    }
    // one fused launch: per pair FFT(s1) -> TMEM, then per row shift -> FFT -> xH -> IFFT -> |.|^2 -> argmax
    if (l == (size_t)kL0) CK((launch_rows<T, kSurface, true>(h, a, (long long)p * (long long)d, grid_cap)));
    else CK((launch_rows<T, kSurface, false>(h, a, (long long)p * (long long)d, grid_cap)));
    if (overlappable) h->hist.push(cur_in, cur_out, h->launches, !(a.flags & 1u));
    else h->hist.reset();
    if (a.pull_src) h->pull_total = a.pull_target;      // only a launch that was accepted moves the meeting point
    if (a.done_counter) h->done_total[a.epoch % (unsigned int)caf_b200_handle_s::kRing] = a.done_last + 1u;
    if (prof) CK(cudaEventRecord(h->ev[2], h->stream));
    if (peaks && !fused_peak) {
        caf_peak_kernel<T><<<(unsigned)p, 256, 0, h->stream>>>(rv, ri, freqs, (int)d, peaks, h->pack_words, h->pack_offset);
        h->launches++;
        CK(cudaGetLastError());
    }
    if (prof) { CK(cudaEventRecord(h->ev[3], h->stream)); h->ev_valid = true; }
    return CAF_B200_OK;
}

void to_public(const caf::PeakOut& s, caf_b200_peak* o) {
    o->value = s.value; o->freq_hz = s.freq_hz; o->doppler_idx = s.doppler_idx; o->delay_idx = s.delay_idx;
}

template <typename T>
int check_common(caf_b200_handle h, const void* needle, const void* hay, size_t p, size_t l, const double* freqs,
                 size_t d, uint32_t fs) {
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    if (p && l && (!needle || !hay)) return fail(CAF_B200_EINVAL, "null needle/haystack");
    if (d && !freqs) return fail(CAF_B200_EINVAL, "null freqs_hz");
    if (fs == 0) return fail(CAF_B200_EINVAL, "fs must be non-zero");
    if (l > (1u << 19))
        return fail(CAF_B200_EUNSUPPORTED, "l > 2^19: rows longer than 2^20 delay cells are not built");
    if (p > (1u << 30) || d > (1u << 30) || (double)p * (double)d > 2.0e9)
        return fail(CAF_B200_EUNSUPPORTED, "p*d too large");
    return CAF_B200_OK;
}

// Host-pointer batch: stage in, run, stage out.
// keep: compute the surface and the row peaks into these DEVICE buffers and leave them there (surface objects).
template <typename T> struct DevKeep { T* surface; T* rv; unsigned long long* ri; };
template <typename T>
int run_batch_host(caf_b200_handle h, const caf::cx<T>* needles, const caf::cx<T>* hays, size_t p, size_t l,
                   const double* freqs, size_t d, uint32_t fs, T* surface, T* rowval, uint64_t* rowidx,
                   caf_b200_peak* peaks, const DevKeep<T>* keep = nullptr) {
    using namespace caf;
    int rc = check_common<T>(h, needles, hays, p, l, freqs, d, fs);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if (p == 0) return CAF_B200_OK;
    const size_t n = 2 * l, rows = p * d;
    cudaStream_t s = h->stream;
    struct PullReset { caf_b200_handle h; ~PullReset() { h->pull_src = nullptr; } } pull_reset{h};   // never outlives this call
    // ---- inputs.  Three small H2D copies cost ~6 us EACH on B200 (DMA set-up, not bytes: 19 us of a 69 us peak-only
    //      call), so a small call moves needle | haystack | freqs as ONE block: straight from the caller's memory when the
    //      three already sit back to back (a caller that stages them in one caf_b200_host_alloc block), else through a
    //      pinned staging block (one 131 KB memcpy on the CPU is cheaper than two more DMAs). ----
    const cx<T>* d_needle = nullptr; const cx<T>* d_hay = nullptr; const double* d_freqs = nullptr;
    const size_t sig_bytes = sizeof(cx<T>) * p * l, fr_bytes = sizeof(double) * d;
    const size_t sig_pad = (sig_bytes + 15) & ~(size_t)15;
    if (l && d && 2 * sig_pad + fr_bytes <= ((size_t)1 << 20)) {
        const size_t tot = 2 * sig_pad + fr_bytes;
        const size_t tot16 = (tot + 15) & ~(size_t)15;
        CK(h->in_block.ensure(tot16));
        bool moved = false;
        // One pair over many CTAs, nothing pipelined behind it: no copy at all -- the kernel's own CTAs read the block out
        // of pinned host memory while they set up (caf_kernels.cuh, RowArgs::pull_*).  The caller's memory is used as it
        // is when the three inputs are one run inside a caf_b200_host_alloc block, else the staging block.
        const bool pipelined = h->allow_pipeline && surface && p == 1 && l <= (size_t)kL0 && d >= 2 * (size_t)h->sm_count;
        if (h->allow_pull && h->pull_counter && p == 1 && d > 1 && l <= (size_t)kL0 && !pipelined) {
            const bool one_run = sig_pad == sig_bytes && (const char*)hays == (const char*)needles + sig_bytes &&
                                 (const char*)freqs == (const char*)hays + sig_bytes;
            if (one_run && ((uintptr_t)needles & 15) == 0 && pinned_block_holds(needles, tot16)) {
                h->pull_src = needles;
            } else {
                if (h->h_stage_cap < tot16) {
                    if (h->h_stage) cudaFreeHost(h->h_stage);
                    h->h_stage = nullptr; h->h_stage_cap = 0;
                    CK(cudaMallocHost(&h->h_stage, tot16 + tot16 / 4));
                    h->h_stage_cap = tot16 + tot16 / 4;
                }
                char* st = (char*)h->h_stage;
                stage_copy(st, needles, sig_bytes); stage_copy(st + sig_pad, hays, sig_bytes); stage_copy(st + 2 * sig_pad, freqs, fr_bytes);
                stage_fence();
                h->pull_src = st;
            }
            h->pull_bytes = tot16;
            moved = true;
        }
        if (!moved && sig_pad == sig_bytes && (const char*)hays == (const char*)needles + sig_bytes &&
            (const char*)freqs == (const char*)hays + sig_bytes) {
            // already one block in the caller's memory.  Adjacent addresses need not be ONE pinned allocation (a copy may
            // not span two): such a copy is refused at once and the staging block below takes over.
            if (cudaMemcpyAsync(h->in_block.p, needles, tot, cudaMemcpyHostToDevice, s) == cudaSuccess) moved = true;
            else (void)cudaGetLastError();
        }
        if (!moved) {
            if (h->h_stage_cap < tot) {
                if (h->h_stage) cudaFreeHost(h->h_stage);
                h->h_stage = nullptr; h->h_stage_cap = 0;
                CK(cudaMallocHost(&h->h_stage, tot + tot / 4));
                h->h_stage_cap = tot + tot / 4;
            }
            // the previous call on this handle ended with a stream synchronise (or saw its result), so the block is free
            char* st = (char*)h->h_stage;
            std::memcpy(st, needles, sig_bytes); std::memcpy(st + sig_pad, hays, sig_bytes); std::memcpy(st + 2 * sig_pad, freqs, fr_bytes);
            CK(cudaMemcpyAsync(h->in_block.p, st, tot, cudaMemcpyHostToDevice, s));
        }
        d_needle = (const cx<T>*)h->in_block.p; d_hay = (const cx<T>*)((char*)h->in_block.p + sig_pad);
        d_freqs = (const double*)((char*)h->in_block.p + 2 * sig_pad);
    } else {
        if (l) {
            CK(h->needle.ensure(sig_bytes));
            CK(h->hay.ensure(sig_bytes));
            CK(cudaMemcpyAsync(h->needle.p, needles, sig_bytes, cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(h->hay.p, hays, sig_bytes, cudaMemcpyHostToDevice, s));
        }
        if (d) {
            CK(h->freqs.ensure(fr_bytes));
            CK(cudaMemcpyAsync(h->freqs.p, freqs, fr_bytes, cudaMemcpyHostToDevice, s));
        }
        d_needle = (const cx<T>*)h->needle.p; d_hay = (const cx<T>*)h->hay.p; d_freqs = (const double*)h->freqs.p;
    }
    T* d_surface = nullptr;
    if (keep) d_surface = keep->surface;
    else if (surface && rows && n) { CK(h->surface.ensure(sizeof(T) * rows * n)); d_surface = (T*)h->surface.p; }
    T* d_rv = nullptr; unsigned long long* d_ri = nullptr;
    if (keep) { d_rv = keep->rv; d_ri = keep->ri; }
    else if (rows && (rowval || rowidx || peaks)) {
        CK(h->rowval.ensure(sizeof(T) * rows)); CK(h->rowidx.ensure(sizeof(unsigned long long) * rows));
        d_rv = (T*)h->rowval.p; d_ri = (unsigned long long*)h->rowidx.p;
    }
    PeakOut* d_pk = nullptr;
    if (peaks) {
        CK(h->peaks.ensure(sizeof(PeakOut) * p)); d_pk = (PeakOut*)h->peaks.p;
        if (h->h_peaks_cap < sizeof(PeakOut) * p) {
            if (h->h_peaks) cudaFreeHost(h->h_peaks);
            h->h_peaks = nullptr; h->h_peaks_cap = 0;
            CK(cudaMallocHost(&h->h_peaks, sizeof(PeakOut) * p + 64));      // + the completion word of the spin wait
            h->h_peaks_cap = sizeof(PeakOut) * p;
            *reinterpret_cast<volatile unsigned int*>((char*)h->h_peaks + h->h_peaks_cap) = 0u;
        }
    }
    // A single pair's peak is stored by the kernel straight into the pinned staging buffer (cudaMallocHost memory is
    // device-addressable under unified addressing): no 32-byte D2H copy and no DMA set-up on the call's tail.  Measured
    // on B200, two A/B pairs on one box: peak-only call 82.3 / 82.8 us -> 74.5 / 77.9 us, surface call 550 / 549 us ->
    // 541 / 542 us.  CAF_B200_PEAK_ZEROCOPY=0 keeps the copy; batches (p > 1) always use it.
    const bool peak_zero_copy = h->peak_zero_copy && peaks && p == 1;
    if (peak_zero_copy) d_pk = (PeakOut*)h->h_peaks;
    // One pair with the surface wanted on the host: the D2H copy (26 MB at PCIe speed, ~0.5 ms) dwarfs the kernels
    // (~50 us), so the rows are issued as a short head (one wave of CTAs) and the rest; the head's cells start
    // crossing PCIe on a second stream while the rest is still being computed.  find_peak then runs as its own
    // small kernel over all row peaks.  CAF_B200_PIPELINE=0 in the environment keeps the single-launch path.
    const size_t d0 = (size_t)h->sm_count;
    bool spin = false;
    if (h->allow_pipeline && surface && d_surface && p == 1 && l <= (size_t)kL0 && d >= 2 * d0 && d_rv && d_ri) {
        if (!h->copy_stream) CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        if (!h->ev_head) CK(cudaEventCreateWithFlags(&h->ev_head, cudaEventDisableTiming));
        if (!h->ev_copy) CK(cudaEventCreateWithFlags(&h->ev_copy, cudaEventDisableTiming));
        const double* fq = d_freqs;
        // an error return below must not leave the head's DMA into the caller's buffer in flight
        struct Drain {
            cudaStream_t a, b; bool armed = true;
            ~Drain() { if (armed) { cudaStreamSynchronize(a); cudaStreamSynchronize(b); } }
        } drain{h->copy_stream, s};
        rc = run_batch_dev<T>(h, d_needle, d_hay, 1, l, fq, d0, fs, d_surface, d_rv, d_ri, nullptr);
        if (rc) return rc;
        CK(cudaEventRecord(h->ev_head, s));
        CK(cudaStreamWaitEvent(h->copy_stream, h->ev_head, 0));
        CK(cudaMemcpyAsync(surface, d_surface, sizeof(T) * d0 * n, cudaMemcpyDeviceToHost, h->copy_stream));
        CK(cudaEventRecord(h->ev_copy, h->copy_stream));
        rc = run_batch_dev<T>(h, d_needle, d_hay, 1, l, fq + d0, d - d0, fs,
                              d_surface + d0 * n, d_rv + d0, d_ri + d0, nullptr);
        if (rc) return rc;
        if (d_pk) {
            caf_peak_kernel<T><<<1, 256, 0, s>>>(d_rv, d_ri, fq, (int)d, d_pk);
            h->launches++;
            CK(cudaGetLastError());
        }
        CK(cudaMemcpyAsync(surface + d0 * n, d_surface + d0 * n, sizeof(T) * (d - d0) * n, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamWaitEvent(s, h->ev_copy, 0));
        drain.armed = false;      // from here on the final synchronise of s covers both streams
    } else {
        // Peak-only call on the fused path: the kernel stores the peak into pinned host memory and then a sequence word
        // next to it; the host spins on that word (with a stream query now and then, so a failed launch cannot hang it)
        // instead of cudaStreamSynchronize, whose wake-up alone costs several microseconds of a ~55 us call.
        spin = peak_zero_copy && !surface && !rowval && !rowidx && l && d > 1 && l <= (size_t)kL0;
        if (spin) { h->seq_ptr = reinterpret_cast<unsigned int*>((char*)h->h_peaks + h->h_peaks_cap); h->seq_val = ++h->seq_counter; }
        rc = run_batch_dev<T>(h, d_needle, d_hay, p, l, d_freqs, d, fs, d_surface, d_rv, d_ri, d_pk);
        h->seq_ptr = nullptr; h->pull_src = nullptr;
        if (rc) return rc;
        if (surface && d_surface) CK(cudaMemcpyAsync(surface, d_surface, sizeof(T) * rows * n, cudaMemcpyDeviceToHost, s));
    }
    if (rowval && rows) CK(cudaMemcpyAsync(rowval, d_rv, sizeof(T) * rows, cudaMemcpyDeviceToHost, s));
    if (rowidx && rows) CK(cudaMemcpyAsync(rowidx, d_ri, sizeof(uint64_t) * rows, cudaMemcpyDeviceToHost, s));
    if (peaks && !peak_zero_copy) CK(cudaMemcpyAsync(h->h_peaks, d_pk, sizeof(PeakOut) * p, cudaMemcpyDeviceToHost, s));
    if (spin) {
        volatile unsigned int* seq = reinterpret_cast<volatile unsigned int*>((char*)h->h_peaks + h->h_peaks_cap);
        const unsigned int want = h->seq_counter;
        unsigned int polls = 0;
        while (*seq != want) {
            if ((++polls & 0xfffu) == 0u && cudaStreamQuery(s) != cudaErrorNotReady) break;   // finished (or failed) without the word
        }
        if (*seq != want) CK(cudaStreamSynchronize(s));      // surfaces a launch / execution error
    } else {
        CK(cudaStreamSynchronize(s));
    }
    if (peaks)
        for (size_t i = 0; i < p; ++i) to_public(reinterpret_cast<PeakOut*>(h->h_peaks)[i], &peaks[i]);
    return CAF_B200_OK;
}

// Sibling layouts (caf_layout_kernel): the surface is computed in the Rust layout on the device, converted there,
// and only the converted array crosses PCIe.
template <typename T>
int run_layout_host(caf_b200_handle h, const caf::cx<T>* needle, const caf::cx<T>* hay, size_t l, const double* freqs,
                    size_t d, uint32_t fs, int layout, T* out, caf_b200_peak* peak) {
    using namespace caf;
    int rc = check_common<T>(h, needle, hay, 1, l, freqs, d, fs);
    if (rc) return rc;
    if (layout != CAF_B200_LAYOUT_PYTHON && layout != CAF_B200_LAYOUT_GO)
        return fail(CAF_B200_EINVAL, "layout must be CAF_B200_LAYOUT_PYTHON or CAF_B200_LAYOUT_GO");
    if (l > (1u << 26)) return fail(CAF_B200_EUNSUPPORTED, "l too large");
    CK(cudaSetDevice(h->device));
    const size_t W = (layout == CAF_B200_LAYOUT_PYTHON) ? l : 2 * l;
    const int lag0 = (layout == CAF_B200_LAYOUT_PYTHON) ? (int)(l / 2) : (int)l;
    if (peak) { peak->value = 0.0; peak->freq_hz = 0.0; peak->doppler_idx = ~0ull; peak->delay_idx = 0; }
    if (l == 0 || d == 0) return CAF_B200_OK;
    cudaStream_t s = h->stream;
    CK(h->needle.ensure(sizeof(cx<T>) * l));
    CK(h->hay.ensure(sizeof(cx<T>) * l));
    CK(h->freqs.ensure(sizeof(double) * d));
    CK(cudaMemcpyAsync(h->needle.p, needle, sizeof(cx<T>) * l, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(h->hay.p, hay, sizeof(cx<T>) * l, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(h->freqs.p, freqs, sizeof(double) * d, cudaMemcpyHostToDevice, s));
    CK(h->surface.ensure(sizeof(T) * d * 2 * l));
    CK(h->layout.ensure(sizeof(T) * d * W));
    CK(h->rowval.ensure(sizeof(T) * d));
    CK(h->rowidx.ensure(sizeof(unsigned long long) * d));
    CK(h->peaks.ensure(sizeof(PeakOut)));
    rc = run_batch_dev<T>(h, (const cx<T>*)h->needle.p, (const cx<T>*)h->hay.p, 1, l, (const double*)h->freqs.p, d, fs,
                          (T*)h->surface.p, nullptr, nullptr, nullptr);
    if (rc) return rc;
    caf_layout_kernel<T><<<(unsigned)d, 256, 0, s>>>((const T*)h->surface.p, (T*)h->layout.p, (int)l, (int)W, lag0,
                                                     (T*)h->rowval.p, (unsigned long long*)h->rowidx.p);
    h->launches++;
    CK(cudaGetLastError());
    caf_peak_kernel<T><<<1, 256, 0, s>>>((const T*)h->rowval.p, (const unsigned long long*)h->rowidx.p,
                                         (const double*)h->freqs.p, (int)d, (PeakOut*)h->peaks.p);
    h->launches++;
    CK(cudaGetLastError());
    if (out) CK(cudaMemcpyAsync(out, h->layout.p, sizeof(T) * d * W, cudaMemcpyDeviceToHost, s));
    PeakOut pk;
    CK(cudaMemcpyAsync(&pk, h->peaks.p, sizeof(PeakOut), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (peak) to_public(pk, peak);
    return CAF_B200_OK;
}

template <typename T>
int run_shift(caf_b200_handle h, const caf::cx<T>* in, size_t n, double f, uint32_t fs, caf::cx<T>* out) {
    using namespace caf;
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    if (n && (!in || !out)) return fail(CAF_B200_EINVAL, "null samples");
    if (fs == 0) return fail(CAF_B200_EINVAL, "fs must be non-zero");
    if (n == 0) return CAF_B200_OK;
    CK(cudaSetDevice(h->device));
    CK(h->needle.ensure(sizeof(cx<T>) * n));
    CK(h->scratch.ensure(sizeof(cx<T>) * n));
    cudaStream_t s = h->stream;
    CK(cudaMemcpyAsync(h->needle.p, in, sizeof(cx<T>) * n, cudaMemcpyHostToDevice, s));
    const double dt = 1.0 / (double)fs;   // mod.rs:53
    long long blocks = (long long)((n + 255) / 256);
    if (blocks > 4 * h->sm_count) blocks = 4 * h->sm_count;
    caf_apply_shift_kernel<T><<<(unsigned)blocks, 256, 0, s>>>((const cx<T>*)h->needle.p, (cx<T>*)h->scratch.p,
                                                              (long long)n, f * dt);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, h->scratch.p, sizeof(cx<T>) * n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return CAF_B200_OK;
}

template <typename T>
int run_xcor(caf_b200_handle h, const caf::cx<T>* a_, const caf::cx<T>* b_, size_t n, caf::cx<T>* out) {
    using namespace caf;
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    if (n && (!a_ || !b_ || !out)) return fail(CAF_B200_EINVAL, "null operand");
    if (n == 0) return CAF_B200_OK;
    if (n > (1u << 19))
        return fail(CAF_B200_EUNSUPPORTED, "xcor: n > 2^19 (rows longer than 2^20 cells are not built)");
    CK(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    CK(h->needle.ensure(sizeof(cx<T>) * n)); CK(h->hay.ensure(sizeof(cx<T>) * n));
    if (n > (size_t)kL0 && n != (size_t)kM) {
        // any other length: the linear correlation of the two n-sample signals through the long-row kernels (one row,
        // no doppler shift, complex cells kept), folded to the circular one: c[k] = R(k) + R(k - n)
        size_t big_n = 16384;
        while (big_n < 2 * n) big_n *= 2;
        CK(h->layout.ensure(sizeof(cx<T>) * (big_n + n)));
        CK(h->freqs.ensure(sizeof(double)));
        CK(cudaMemsetAsync(h->freqs.p, 0, sizeof(double), s));           // one row at 0.0 Hz: the phasor is exactly 1
        CK(cudaMemcpyAsync(h->hay.p, a_, sizeof(cx<T>) * n, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(h->needle.p, b_, sizeof(cx<T>) * n, cudaMemcpyHostToDevice, s));
        cx<T>* y = (cx<T>*)h->layout.p;
        int rc = run_large_dev<T>(h, (const cx<T>*)h->needle.p, (const cx<T>*)h->hay.p, 1, n, (const double*)h->freqs.p, 1, 1u,
                                  nullptr, nullptr, nullptr, nullptr, y);
        if (rc) return rc;
        caf_fold_circular_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(y, y + big_n, (int)n, (int)big_n);
        h->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(out, y + big_n, sizeof(cx<T>) * n, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return CAF_B200_OK;
    }
    CK(h->hperm.ensure(sizeof(cx<T>) * kM)); CK(h->scratch.ensure(sizeof(cx<T>) * (kM + n)));
    CK(cudaMemcpyAsync(h->hay.p, a_, sizeof(cx<T>) * n, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(h->needle.p, b_, sizeof(cx<T>) * n, cudaMemcpyHostToDevice, s));
    RowArgs<T> a = base_args<T>(h);
    a.hperm = (cx<T>*)h->hperm.p; a.P = 1; a.D = 1; a.L = (int)n;
    cx<T>* y = (cx<T>*)h->scratch.p;
    cx<T>* res = y;
    if (n == (size_t)kM) {
        a.in = (const cx<T>*)h->hay.p;
        CK((launch_rows<T, kSpectrumFull>(h, a, 1)));
        a.in = (const cx<T>*)h->needle.p; a.out = y;
        CK((launch_rows<T, kXcorFull>(h, a, 1)));
    } else {
        a.in = (const cx<T>*)h->hay.p;
        CK((launch_rows<T, kSpectrumHalf>(h, a, 1)));
        a.in = (const cx<T>*)h->needle.p; a.out = y;
        CK((launch_rows<T, kXcorHalf>(h, a, 1)));
        res = y + kM;
        caf_fold_circular_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(y, res, (int)n, kM);
        h->launches++;
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(out, res, sizeof(cx<T>) * n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return CAF_B200_OK;
}

// read_file_c64 (utils.rs:10-35) onto the device: see include/caf_b200.h
template <typename T>
int load_c64_dev(caf_b200_handle h, const char* path, size_t first, size_t max_samples, void** dev_out, size_t* n_out) {
    if (!h || !path || !dev_out || !n_out) return fail(CAF_B200_EINVAL, "null argument");
    *dev_out = nullptr; *n_out = 0;
    FILE* f = std::fopen(path, "rb");
    if (!f) return fail(CAF_B200_EIO, std::string("read_file_c64: cannot open ") + path);
    struct Close { FILE* f; ~Close() { std::fclose(f); } } closer{f};
    if (std::fseek(f, 0, SEEK_END) != 0) return fail(CAF_B200_EIO, "read_file_c64: seek failed");
    const long long bytes = (long long)std::ftell(f);
    if (bytes < 0) return fail(CAF_B200_EIO, "read_file_c64: tell failed");
    if (bytes % 8) return fail(CAF_B200_EINVAL, "read_file_c64: trailing partial sample (utils.rs:19-32 indexes past the end)");
    const size_t total = (size_t)bytes / 8;
    if (first > total) first = total;
    size_t n = total - first;
    if (max_samples && n > max_samples) n = max_samples;
    if (n == 0) return CAF_B200_OK;
    CK(cudaSetDevice(h->device));
    // file -> pinned staging (the read lands where the DMA starts) -> device, 8 bytes per sample
    const size_t raw = n * 8;
    if (h->h_stage_cap < raw) {
        if (h->h_stage) cudaFreeHost(h->h_stage);
        h->h_stage = nullptr; h->h_stage_cap = 0;
        CK(cudaMallocHost(&h->h_stage, raw));
        h->h_stage_cap = raw;
    }
    if (std::fseek(f, (long)(first * 8), SEEK_SET) != 0 || std::fread(h->h_stage, 1, raw, f) != raw)
        return fail(CAF_B200_EIO, std::string("read_file_c64: short read from ") + path);
    void* out = nullptr;
    CK(cudaMalloc(&out, n * sizeof(caf::cx<T>)));
    cudaError_t e;
    if (std::is_same<T, float>::value) {
        e = cudaMemcpyAsync(out, h->h_stage, raw, cudaMemcpyHostToDevice, h->stream);
    } else {
        e = h->scratch.ensure(raw);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h->scratch.p, h->h_stage, raw, cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) {
            long long blocks = (long long)((n + 255) / 256);
            if (blocks > 8LL * h->sm_count) blocks = 8LL * h->sm_count;
            caf::caf_widen_c64_kernel<<<(unsigned)blocks, 256, 0, h->stream>>>((const float2*)h->scratch.p, (double2*)out, (long long)n);
            h->launches++;
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);      // the staging block is the handle's: free it for the next call
    if (e != cudaSuccess) { cudaFree(out); return fail(CAF_B200_ECUDA, cudaGetErrorString(e)); }
    *dev_out = out; *n_out = n;
    return CAF_B200_OK;
}
}  // namespace

// ================================================ C ABI ================================================
extern "C" {

const char* caf_b200_last_error(void) { return g_err.c_str(); }
const char* caf_b200_version(void) { return "caf_b200 0.1 (sm_100a)"; }

static int create_impl(int device, bool own_stream, void* cuda_stream, caf_b200_handle* out) {
    if (!out) return fail(CAF_B200_EINVAL, "null out");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(CAF_B200_ENODEVICE, std::string("no CUDA device (there is no CPU fallback): ") +
                                            (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0"));
    if (device < 0 || device >= ndev) return fail(CAF_B200_EINVAL, "device index out of range");
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10 || prop.minor != 0)   // sm_100a SASS is arch-specific: it does not load on sm_103 or sm_120 either
        return fail(CAF_B200_ENODEVICE, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                                            ", this library carries sm_100a code only (no fallback)");
    CK(cudaSetDevice(device));
    caf_b200_handle h = new (std::nothrow) caf_b200_handle_s();
    if (!h) return fail(CAF_B200_EINVAL, "out of host memory");
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    if (const char* e_ = getenv("CAF_B200_CHUNK_MB")) { const long v_ = atol(e_); if (v_ > 0) h->chunk_mb = (size_t)v_; }
    if (const char* e_ = getenv("CAF_B200_PIPELINE")) h->allow_pipeline = e_[0] != '0';
    if (const char* e_ = getenv("CAF_B200_PEAK_ZEROCOPY")) h->peak_zero_copy = e_[0] != '0';
    if (const char* e_ = getenv("CAF_B200_PULL")) h->allow_pull = e_[0] != '0';
    if (const char* e_ = getenv("CAF_B200_OVERLAP")) h->overlap_killed = e_[0] == '0';
    if (const char* e_ = getenv("CAF_B200_GATHER_AHEAD")) h->gather_ahead = atoi(e_);

    if (!own_stream) { h->stream = (cudaStream_t)cuda_stream; h->own_stream = false; }   // 0 = legacy default stream
    else {
        e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { delete h; return fail(CAF_B200_ECUDA, cudaGetErrorString(e)); }
        h->own_stream = true;
    }
    constexpr size_t kRing_ = (size_t)caf_b200_handle_s::kRing;
    if ((e = cudaMalloc(&h->hshare, kRing_ * sizeof(double2) * caf::kM)) != cudaSuccess ||
        (e = cudaMalloc(&h->hflag, 2 * kRing_ * sizeof(unsigned int))) != cudaSuccess ||
        (e = cudaMemsetAsync(h->hflag, 0, 2 * kRing_ * sizeof(unsigned int), h->stream)) != cudaSuccess ||
        (e = cudaMalloc(&h->pull_counter, sizeof(unsigned int))) != cudaSuccess ||
        (e = cudaMemsetAsync(h->pull_counter, 0, sizeof(unsigned int), h->stream)) != cudaSuccess ||
        (e = cudaMalloc(&h->done_counter, kRing_ * sizeof(unsigned int))) != cudaSuccess ||
        (e = cudaMemsetAsync(h->done_counter, 0, kRing_ * sizeof(unsigned int), h->stream)) != cudaSuccess ||
        (e = upload_tables<double>(h->td, h->stream)) != cudaSuccess ||
        (e = upload_tables<float>(h->tf, h->stream)) != cudaSuccess ||
        (e = configure_all<double>(&h->occ_d)) != cudaSuccess ||
        (e = configure_all<float>(&h->occ_f)) != cudaSuccess ||
        (e = configure_detect<double>()) != cudaSuccess ||
        (e = configure_detect<float>()) != cudaSuccess ||
        (e = configure_cfar<double>()) != cudaSuccess ||
        (e = configure_cfar<float>()) != cudaSuccess) {
        std::string m = std::string("handle setup failed: ") + cudaGetErrorString(e);
        caf_b200_destroy(h);
        return fail(CAF_B200_ECUDA, m);
    }
    { std::lock_guard<std::mutex> lk(g_live_mu); g_live_handles.insert(h); }
    *out = h;
    return CAF_B200_OK;
}

int caf_b200_create(int device, caf_b200_handle* out) { return create_impl(device, true, nullptr, out); }
int caf_b200_create_on_stream(int device, void* cuda_stream, caf_b200_handle* out) {
    return create_impl(device, false, cuda_stream, out);
}

int caf_b200_destroy(caf_b200_handle h) {
    if (!h) return CAF_B200_OK;
    { std::lock_guard<std::mutex> lk(g_live_mu); g_live_handles.erase(h); }
    cudaSetDevice(h->device);
    for (auto& b : h->surf_pool) if (b.first) cudaFree(b.first);
    h->surf_pool.clear();
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (DevBuf* b : {&h->in_block, &h->needle, &h->hay, &h->hperm, &h->freqs, &h->surface, &h->rowval, &h->rowidx, &h->peaks, &h->scratch, &h->layout, &h->lwbuf, &h->lhtmp, &h->lhbig, &h->lpart, &h->det, &h->det_io})
        b->release();
    for (void* q : {(void*)h->td.tw1, (void*)h->td.tw2, (void*)h->td.g, (void*)h->tf.tw1, (void*)h->tf.tw2, (void*)h->tf.g})
        if (q) cudaFree(q);
    if (h->h_peaks) cudaFreeHost(h->h_peaks);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    if (h->done_counter) cudaFree(h->done_counter);
    if (h->pull_counter) cudaFree(h->pull_counter);
    if (h->hshare) cudaFree(h->hshare);
    if (h->hflag) cudaFree(h->hflag);
    for (auto& e : h->ev) if (e) cudaEventDestroy(e);
    if (h->ev_head) cudaEventDestroy(h->ev_head);
    if (h->ev_copy) cudaEventDestroy(h->ev_copy);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CAF_B200_OK;
}

int caf_b200_sync(caf_b200_handle h) {
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    CK(cudaStreamSynchronize(h->stream));
    return CAF_B200_OK;
}

uint64_t caf_b200_launch_count(caf_b200_handle h) { return h ? h->launches : 0; }

int caf_b200_set_overlap(caf_b200_handle h, int mode) {
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    if (mode < 0 || mode > 4) return fail(CAF_B200_EINVAL, "overlap mode must be 0 (off), 1 (full grids) or 2..4 (that many launches share the GPU)");
    h->overlap = h->overlap_killed ? 0 : mode;      // CAF_B200_OVERLAP=0: the switch is accepted and ignored
    h->hist.reset();
    return CAF_B200_OK;
}
int caf_b200_set_profiling(caf_b200_handle h, int on) {
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    h->profiling = on != 0;
    return CAF_B200_OK;
}

int caf_b200_last_kernel_ms(caf_b200_handle h, float* spectrum_ms, float* rows_ms, float* peak_ms) {
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    if (!h->ev_valid) return fail(CAF_B200_EINVAL, "no profiled call recorded (caf_b200_set_profiling first)");
    CK(cudaEventSynchronize(h->ev[3]));
    float a = 0, b = 0, c = 0;
    CK(cudaEventElapsedTime(&a, h->ev[0], h->ev[1]));
    CK(cudaEventElapsedTime(&b, h->ev[1], h->ev[2]));
    CK(cudaEventElapsedTime(&c, h->ev[2], h->ev[3]));
    if (spectrum_ms) *spectrum_ms = a;
    if (rows_ms) *rows_ms = b;
    if (peak_ms) *peak_ms = c;
    return CAF_B200_OK;
}

int caf_b200_probe_fma_tflops(caf_b200_handle h, int is_f64, double* tflops) {
    if (!h || !tflops) return fail(CAF_B200_EINVAL, "null argument");
    CK(cudaSetDevice(h->device));
    CK(h->scratch.ensure(64));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    const int iters = is_f64 ? 4096 : 16384, blocks = h->sm_count * 4, threads = 512;
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        CK(cudaEventRecord(e0, h->stream));
        if (is_f64) caf::caf_fma_probe_kernel<double><<<blocks, threads, 0, h->stream>>>((double*)h->scratch.p, iters, 1.0);
        else caf::caf_fma_probe_kernel<float><<<blocks, threads, 0, h->stream>>>((float*)h->scratch.p, iters, 1.0f);
        h->launches++;
        CK(cudaGetLastError());
        CK(cudaEventRecord(e1, h->stream));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        double fl = 2.0 * 64.0 * (double)iters * (double)blocks * (double)threads;
        double tf = fl / ((double)ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *tflops = best;
    return CAF_B200_OK;
}

/* development hook (CAF_TRACE builds): copy the per-warp phase stamps of the last surface launch to `out`
 * (n_cta * 16 * 8 * 32 int64).  Allocates the trace buffer on first use; returns EUNSUPPORTED otherwise. */
int caf_b200_debug_trace(caf_b200_handle h, long long* out, size_t n_cta) {
#ifdef CAF_TRACE
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    const size_t bytes = sizeof(long long) * 512 * 16 * 8 * 32;
    if (!h->trace) { CK(cudaMalloc(&h->trace, bytes)); CK(cudaMemset(h->trace, 0, bytes)); return CAF_B200_OK; }
    CK(cudaStreamSynchronize(h->stream));
    if (out) CK(cudaMemcpy(out, h->trace, sizeof(long long) * n_cta * 16 * 8 * 32, cudaMemcpyDeviceToHost));
    return CAF_B200_OK;
#else
    (void)h; (void)out; (void)n_cta;
    return fail(CAF_B200_EUNSUPPORTED, "library built without CAF_TRACE");
#endif
}

int caf_b200_host_alloc(void** out, size_t bytes) {
    if (!out) return fail(CAF_B200_EINVAL, "null out");
    *out = nullptr;
    if (bytes == 0) return CAF_B200_OK;
    // (a few bytes of slack: the kernel-side input pull reads whole 16-byte chunks)
    CK(cudaMallocHost(out, bytes + 16));
    std::lock_guard<std::mutex> lk(g_pinned_mu);
    g_pinned_blocks.emplace_back((const char*)*out, bytes + 16);
    return CAF_B200_OK;
}
int caf_b200_host_free(void* p) {
    if (p) {
        {
            std::lock_guard<std::mutex> lk(g_pinned_mu);
            for (size_t i = 0; i < g_pinned_blocks.size(); ++i)
                if (g_pinned_blocks[i].first == (const char*)p) { g_pinned_blocks.erase(g_pinned_blocks.begin() + (long)i); break; }
        }
        CK(cudaFreeHost(p));
    }
    return CAF_B200_OK;
}

int caf_b200_load_c64_dev_f64(caf_b200_handle h, const char* path, size_t first_sample, size_t max_samples, caf_c128** dev_out, size_t* n_out) {
    return load_c64_dev<double>(h, path, first_sample, max_samples, reinterpret_cast<void**>(dev_out), n_out);
}
int caf_b200_load_c64_dev_f32(caf_b200_handle h, const char* path, size_t first_sample, size_t max_samples, caf_c64** dev_out, size_t* n_out) {
    return load_c64_dev<float>(h, path, first_sample, max_samples, reinterpret_cast<void**>(dev_out), n_out);
}
int caf_b200_dev_free(void* dev_ptr) {
    if (dev_ptr) CK(cudaFree(dev_ptr));
    return CAF_B200_OK;
}
int caf_b200_dev_alloc(caf_b200_handle h, size_t bytes, void** dev_out) {
    if (!h || !dev_out) return fail(CAF_B200_EINVAL, "null argument");
    *dev_out = nullptr;
    if (bytes == 0) return CAF_B200_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaMalloc(dev_out, bytes));
    return CAF_B200_OK;
}
int caf_b200_dev_upload(caf_b200_handle h, void* dev_dst, const void* host_src, size_t bytes) {
    if (!h || (bytes && (!dev_dst || !host_src))) return fail(CAF_B200_EINVAL, "null argument");
    if (bytes == 0) return CAF_B200_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(dev_dst, host_src, bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return CAF_B200_OK;
}
int caf_b200_dev_download(caf_b200_handle h, void* host_dst, const void* dev_src, size_t bytes) {
    if (!h || (bytes && (!host_dst || !dev_src))) return fail(CAF_B200_EINVAL, "null argument");
    if (bytes == 0) return CAF_B200_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return CAF_B200_OK;
}

int caf_b200_apply_freq_shift_f64(caf_b200_handle h, const caf_c128* in, size_t n, double f, uint32_t fs, caf_c128* out) {
    return run_shift<double>(h, (const double2*)in, n, f, fs, (double2*)out);
}
int caf_b200_apply_freq_shift_f32(caf_b200_handle h, const caf_c64* in, size_t n, double f, uint32_t fs, caf_c64* out) {
    return run_shift<float>(h, (const float2*)in, n, f, fs, (float2*)out);
}
int caf_b200_apply_shift_f64(caf_b200_handle h, const caf_c128* in, size_t n, double f, uint32_t fs, caf_c128* out) {
    return caf_b200_apply_freq_shift_f64(h, in, n, f, fs, out);
}
int caf_b200_apply_shift_f32(caf_b200_handle h, const caf_c64* in, size_t n, double f, uint32_t fs, caf_c64* out) {
    return caf_b200_apply_freq_shift_f32(h, in, n, f, fs, out);
}

int caf_b200_xcor_f64(caf_b200_handle h, const caf_c128* a, const caf_c128* b, size_t n, caf_c128* out) {
    return run_xcor<double>(h, (const double2*)a, (const double2*)b, n, (double2*)out);
}
int caf_b200_xcor_f32(caf_b200_handle h, const caf_c64* a, const caf_c64* b, size_t n, caf_c64* out) {
    return run_xcor<float>(h, (const float2*)a, (const float2*)b, n, (float2*)out);
}

int caf_b200_batch_f64(caf_b200_handle h, const caf_c128* needles, const caf_c128* hays, size_t p, size_t l,
                       const double* freqs, size_t d, uint32_t fs, double* surface, double* rv, uint64_t* ri,
                       caf_b200_peak* peaks) {
    return run_batch_host<double>(h, (const double2*)needles, (const double2*)hays, p, l, freqs, d, fs, surface, rv, ri, peaks);
}
int caf_b200_batch_f32(caf_b200_handle h, const caf_c64* needles, const caf_c64* hays, size_t p, size_t l,
                       const double* freqs, size_t d, uint32_t fs, float* surface, float* rv, uint64_t* ri,
                       caf_b200_peak* peaks) {
    return run_batch_host<float>(h, (const float2*)needles, (const float2*)hays, p, l, freqs, d, fs, surface, rv, ri, peaks);
}

int caf_b200_surface_f64(caf_b200_handle h, const caf_c128* needle, const caf_c128* hay, size_t l, const double* freqs,
                         size_t d, uint32_t fs, double* surface, double* rv, uint64_t* ri, caf_b200_peak* peak) {
    return caf_b200_batch_f64(h, needle, hay, 1, l, freqs, d, fs, surface, rv, ri, peak);
}
int caf_b200_surface_f32(caf_b200_handle h, const caf_c64* needle, const caf_c64* hay, size_t l, const double* freqs,
                         size_t d, uint32_t fs, float* surface, float* rv, uint64_t* ri, caf_b200_peak* peak) {
    return caf_b200_batch_f32(h, needle, hay, 1, l, freqs, d, fs, surface, rv, ri, peak);
}
int caf_b200_peak_f64(caf_b200_handle h, const caf_c128* needle, const caf_c128* hay, size_t l, const double* freqs,
                      size_t d, uint32_t fs, caf_b200_peak* peak) {
    if (!peak) return fail(CAF_B200_EINVAL, "null peak");
    return caf_b200_batch_f64(h, needle, hay, 1, l, freqs, d, fs, nullptr, nullptr, nullptr, peak);
}
int caf_b200_peak_f32(caf_b200_handle h, const caf_c64* needle, const caf_c64* hay, size_t l, const double* freqs,
                      size_t d, uint32_t fs, caf_b200_peak* peak) {
    if (!peak) return fail(CAF_B200_EINVAL, "null peak");
    return caf_b200_batch_f32(h, needle, hay, 1, l, freqs, d, fs, nullptr, nullptr, nullptr, peak);
}

int caf_b200_surface_layout_f64(caf_b200_handle h, const caf_c128* needle, const caf_c128* hay, size_t l,
                                const double* freqs, size_t d, uint32_t fs, int layout, double* out, caf_b200_peak* peak) {
    return run_layout_host<double>(h, (const double2*)needle, (const double2*)hay, l, freqs, d, fs, layout, out, peak);
}
int caf_b200_surface_layout_f32(caf_b200_handle h, const caf_c64* needle, const caf_c64* hay, size_t l,
                                const double* freqs, size_t d, uint32_t fs, int layout, float* out, caf_b200_peak* peak) {
    return run_layout_host<float>(h, (const float2*)needle, (const float2*)hay, l, freqs, d, fs, layout, out, peak);
}

static_assert(sizeof(caf_b200_peak) == sizeof(caf::PeakOut), "peak layouts must match");

int caf_b200_batch_f64_dev(caf_b200_handle h, const caf_c128* needles, const caf_c128* hays, size_t p, size_t l,
                           const double* freqs, size_t d, uint32_t fs, double* surface, double* rv, uint64_t* ri,
                           caf_b200_peak* peaks) {
    int rc = check_common<double>(h, needles, hays, p, l, freqs, d, fs);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    return run_batch_dev<double>(h, (const double2*)needles, (const double2*)hays, p, l, freqs, d, fs, surface, rv,
                                 (unsigned long long*)ri, (caf::PeakOut*)peaks);
}
int caf_b200_batch_f32_dev(caf_b200_handle h, const caf_c64* needles, const caf_c64* hays, size_t p, size_t l,
                           const double* freqs, size_t d, uint32_t fs, float* surface, float* rv, uint64_t* ri,
                           caf_b200_peak* peaks) {
    int rc = check_common<float>(h, needles, hays, p, l, freqs, d, fs);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    return run_batch_dev<float>(h, (const float2*)needles, (const float2*)hays, p, l, freqs, d, fs, surface, rv,
                                (unsigned long long*)ri, (caf::PeakOut*)peaks);
}


// ---- device-resident surface objects ------------------------------------------------------------------------
extern "C++" {
namespace {
template <typename T>
int surface_create_impl(caf_b200_handle h, const caf::cx<T>* needle, const caf::cx<T>* hay, size_t l, const double* freqs,
                        size_t d, uint32_t fs, caf_b200_surface* out) {
    if (!out) return fail(CAF_B200_EINVAL, "null out");
    *out = nullptr;
    int rc = check_common<T>(h, needle, hay, 1, l, freqs, d, fs);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    caf_b200_surface s = new (std::nothrow) caf_b200_surface_s();
    if (!s) return fail(CAF_B200_EINVAL, "out of host memory");
    s->h = h; s->device = h->device; s->f32 = std::is_same<T, float>::value; s->d = d; s->n = 2 * l;
    const size_t surf_bytes = (sizeof(T) * d * 2 * l + 255) & ~(size_t)255;
    s->bytes = surf_bytes + 16 * d;                       // surface | row_peak_idx (u64) | row_peak_val
    s->freqs.assign(freqs, freqs + d);
    s->peak.value = 0.0; s->peak.freq_hz = 0.0; s->peak.doppler_idx = UINT64_MAX; s->peak.delay_idx = 0;
    if (d && l) {
        // a buffer a released surface left behind, else a fresh one (cudaMalloc costs more than the whole computation)
        size_t best = (size_t)-1;
        for (size_t i = 0; i < h->surf_pool.size(); ++i)
            if (h->surf_pool[i].second >= s->bytes && (best == (size_t)-1 || h->surf_pool[i].second < h->surf_pool[best].second)) best = i;
        if (best != (size_t)-1) {
            s->dev = h->surf_pool[best].first; s->bytes = h->surf_pool[best].second;
            h->surf_pool.erase(h->surf_pool.begin() + (long)best);
        } else {
            cudaError_t e = cudaMalloc(&s->dev, s->bytes);
            if (e != cudaSuccess) { delete s; return fail(CAF_B200_ECUDA, std::string("surface buffer: ") + cudaGetErrorString(e)); }
        }
        s->dev_ri = (unsigned long long*)((char*)s->dev + surf_bytes);
        s->dev_rv = (void*)(s->dev_ri + d);
        // nothing but the fused find_peak result comes back now: the call is a peak-only call that leaves the surface
        // and its row peaks on the device
        const DevKeep<T> keep{(T*)s->dev, (T*)s->dev_rv, s->dev_ri};
        rc = run_batch_host<T>(h, needle, hay, 1, l, freqs, d, fs, nullptr, nullptr, nullptr, &s->peak, &keep);
        if (rc) { const std::string why = g_err; caf_b200_surface_destroy(s); return fail(rc, why); }
    } else {
        s->peaks_on_host = true; s->pval.assign(d, 0.0); s->pidx.assign(d, 0);      // empty rows: peak 0.0 at index 0 (mod.rs:143-144)
    }
    *out = s;
    return CAF_B200_OK;
}
}  // namespace
}  // extern "C++"

int caf_b200_surface_create_f64(caf_b200_handle h, const caf_c128* needle, const caf_c128* hay, size_t l, const double* freqs,
                                size_t d, uint32_t fs, caf_b200_surface* out) {
    return surface_create_impl<double>(h, (const double2*)needle, (const double2*)hay, l, freqs, d, fs, out);
}
int caf_b200_surface_create_f32(caf_b200_handle h, const caf_c64* needle, const caf_c64* hay, size_t l, const double* freqs,
                                size_t d, uint32_t fs, caf_b200_surface* out) {
    return surface_create_impl<float>(h, (const float2*)needle, (const float2*)hay, l, freqs, d, fs, out);
}
int caf_b200_surface_shape(caf_b200_surface s, size_t* rows, size_t* cells_per_row) {
    if (!s) return fail(CAF_B200_EINVAL, "null surface");
    if (rows) *rows = s->d;
    if (cells_per_row) *cells_per_row = s->n;
    return CAF_B200_OK;
}
int caf_b200_surface_row_peaks(caf_b200_surface s, double* freq_hz, double* peak_val, uint64_t* peak_idx) {
    if (!s) return fail(CAF_B200_EINVAL, "null surface");
    if (!s->peaks_on_host && (peak_val || peak_idx)) {       // first request: one copy of 16 bytes per row
        CK(cudaSetDevice(s->device));
        std::vector<unsigned char> raw(16 * s->d);
        CK(cudaMemcpy(raw.data(), s->dev_ri, 16 * s->d, cudaMemcpyDeviceToHost));
        s->pidx.resize(s->d); s->pval.resize(s->d);
        std::memcpy(s->pidx.data(), raw.data(), 8 * s->d);
        if (s->f32) { const float* v = (const float*)(raw.data() + 8 * s->d); for (size_t i = 0; i < s->d; ++i) s->pval[i] = (double)v[i]; }
        else std::memcpy(s->pval.data(), raw.data() + 8 * s->d, 8 * s->d);
        s->peaks_on_host = true;
    }
    for (size_t i = 0; i < s->d; ++i) {
        if (freq_hz) freq_hz[i] = s->freqs[i];
        if (peak_val) peak_val[i] = s->pval[i];
        if (peak_idx) peak_idx[i] = s->pidx[i];
    }
    return CAF_B200_OK;
}
int caf_b200_surface_find_peak(caf_b200_surface s, caf_b200_peak* out) {
    if (!s || !out) return fail(CAF_B200_EINVAL, "null argument");
    *out = s->peak;
    return CAF_B200_OK;
}
// rows [row0, row0 + count) of the surface, count * cells_per_row values of the surface's precision.  Thread-safe: the
// surface was complete when create returned, and the copy does not touch the handle or its stream.
int caf_b200_surface_fetch_rows(caf_b200_surface s, size_t row0, size_t count, void* out) {
    if (!s || (count && !out)) return fail(CAF_B200_EINVAL, "null argument");
    if (row0 > s->d || count > s->d - row0) return fail(CAF_B200_EINVAL, "row range outside the surface");
    if (!count || !s->n) return CAF_B200_OK;
    CK(cudaSetDevice(s->device));
    const size_t esz = s->f32 ? sizeof(float) : sizeof(double);
    CK(cudaMemcpy(out, (const char*)s->dev + row0 * s->n * esz, count * s->n * esz, cudaMemcpyDeviceToHost));
    return CAF_B200_OK;
}
int caf_b200_surface_destroy(caf_b200_surface s) {
    if (!s) return CAF_B200_OK;
    if (s->dev) {
        bool pooled = false;
        {
            std::lock_guard<std::mutex> lk(g_live_mu);
            if (g_live_handles.count(s->h) && s->h->surf_pool.size() < 4) { s->h->surf_pool.emplace_back(s->dev, s->bytes); pooled = true; }
        }
        if (!pooled) { cudaSetDevice(s->device); cudaFree(s->dev); }
    }
    delete s;
    return CAF_B200_OK;
}

// ---- detection: the K strongest local maxima of stored surfaces (caf_detect.cuh) ------------------------------------
static_assert(sizeof(caf_b200_detection) == sizeof(caf::DetectOut), "detection layouts must match");
extern "C++" {
namespace {
int check_detect(size_t d, size_t n, size_t k_max, uint32_t gr, uint32_t gd, double min_ratio) {
    if (k_max < 1 || k_max > (size_t)caf::kDetMaxK) return fail(CAF_B200_EINVAL, "k_max must be 1 ... 1024");
    if (gr > (uint32_t)caf::kDetMaxGuardDoppler) return fail(CAF_B200_EINVAL, "guard_doppler must be 0 ... 32 rows");
    if (gd > (uint32_t)caf::kDetMaxGuardDelay) return fail(CAF_B200_EINVAL, "guard_delay must be 0 ... 256 cells");
    if (d && n && 2 * (size_t)gd + 1 > n) return fail(CAF_B200_EINVAL, "2 * guard_delay + 1 exceeds the cells per row");
    if (!(min_ratio >= 0.0 && min_ratio <= 1.0)) return fail(CAF_B200_EINVAL, "min_ratio must be in [0, 1]");
    if (d > (1ull << 31) || n > (1ull << 31)) return fail(CAF_B200_EUNSUPPORTED, "more than 2^31 rows or cells per row");
    return CAF_B200_OK;
}

// Both passes on the handle's stream; every pointer is device memory.  Arguments are already checked.
template <typename T>
int run_detect_dev(caf_b200_handle h, const T* surface, size_t p, size_t d, size_t n, const double* freqs, size_t k_max,
                   uint32_t gr, uint32_t gd, double min_ratio, caf::DetectOut* out, unsigned long long* counts) {
    using namespace caf;
    if (p == 0) return CAF_B200_OK;
    const bool cells = d && n;
    // tile height: the tallest of 16 / 8 / 4 / 2 / 1 rows whose shared memory leaves room for two CTAs per SM; rows
    // beyond the surface's own are not worth their halo
    int tr = 16;
    while (tr > 1 && (det_tile_smem<T>(tr, (int)gr, (int)gd) > kDetSmemBudget || (size_t)(tr / 2) >= d)) tr /= 2;
    const size_t smem = det_tile_smem<T>(tr, (int)gr, (int)gd);      // <= det_tile_smem_max<T>(), set at handle creation
    const long long tiles_c = (long long)((n + kDetCols - 1) / kDetCols), tiles_r = (long long)((d + tr - 1) / tr);
    const long long tiles = cells ? tiles_c * tiles_r : 0;
    const long long slots = (long long)std::min(k_max, det_tile_max_maxima(tr, (int)gr, (int)gd));   // entries one tile can append
    const long long cap = tiles * slots;
    if ((double)p * (double)tiles > 2147483647.0) return fail(CAF_B200_EUNSUPPORTED, "too many tiles for one launch");
    const size_t ctr_bytes = (16 * p + 255) & ~(size_t)255;
    CK(h->det.ensure(ctr_bytes + sizeof(DetEntry) * (size_t)cap * p));
    unsigned long long* ctr = reinterpret_cast<unsigned long long*>(h->det.p);
    DetEntry* entries = reinterpret_cast<DetEntry*>((char*)h->det.p + ctr_bytes);
    CK(cudaMemsetAsync(ctr, 0, 16 * p, h->stream));
    if (tiles) {
        caf_detect_tiles_kernel<T><<<(unsigned)(p * tiles), kDetCols, smem, h->stream>>>(
            surface, (long long)d, (long long)n, (int)gr, (int)gd, tr, tiles_c, tiles, (unsigned)k_max, cap, entries, ctr);
        h->launches++;
        CK(cudaGetLastError());
    }
    caf_detect_merge_kernel<T><<<(unsigned)p, kDetMergeThreads, 0, h->stream>>>(
        surface, (long long)d, (long long)n, freqs, entries, cap, ctr, (unsigned)k_max, min_ratio, out, counts);
    h->launches++;
    CK(cudaGetLastError());
    return CAF_B200_OK;
}

template <typename T>
int detect_dev_impl(caf_b200_handle h, const T* surface, size_t p, size_t d, size_t n, const double* freqs, size_t k_max,
                    uint32_t gr, uint32_t gd, double min_ratio, caf_b200_detection* out, uint64_t* counts) {
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    int rc = check_detect(d, n, k_max, gr, gd, min_ratio);
    if (rc) return rc;
    if (p && (!out || !counts)) return fail(CAF_B200_EINVAL, "null out / counts");
    if (p && d && n && !surface) return fail(CAF_B200_EINVAL, "null surface");
    if (p && d && !freqs) return fail(CAF_B200_EINVAL, "null freqs_hz");
    if ((double)p * (double)d * (double)n > 9.0e18) return fail(CAF_B200_EUNSUPPORTED, "surface too large");
    CK(cudaSetDevice(h->device));
    return run_detect_dev<T>(h, surface, p, d, n, freqs, k_max, gr, gd, min_ratio, (caf::DetectOut*)out,
                             (unsigned long long*)counts);
}
}  // namespace
}  // extern "C++"

int caf_b200_surface_detect(caf_b200_surface s, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                            double min_ratio, caf_b200_detection* out, size_t* count) {
    if (!s || !out || !count) return fail(CAF_B200_EINVAL, "null argument");
    int rc = check_detect(s->d, s->n, k_max, guard_doppler, guard_delay, min_ratio);
    if (rc) return rc;
    {
        std::lock_guard<std::mutex> lk(g_live_mu);
        if (!g_live_handles.count(s->h)) return fail(CAF_B200_EINVAL, "the surface's handle was destroyed");
    }
    caf_b200_handle h = s->h;
    CK(cudaSetDevice(h->device));
    // device block: grid | records | count
    const size_t fr_bytes = (sizeof(double) * s->d + 255) & ~(size_t)255, rec_bytes = sizeof(caf_b200_detection) * k_max;
    CK(h->det_io.ensure(fr_bytes + rec_bytes + 8));
    double* d_freqs = (double*)h->det_io.p;
    caf::DetectOut* d_out = (caf::DetectOut*)((char*)h->det_io.p + fr_bytes);
    unsigned long long* d_count = (unsigned long long*)((char*)d_out + rec_bytes);
    if (s->d) CK(cudaMemcpyAsync(d_freqs, s->freqs.data(), sizeof(double) * s->d, cudaMemcpyHostToDevice, h->stream));
    if (s->f32) rc = run_detect_dev<float>(h, (const float*)s->dev, 1, s->d, s->n, d_freqs, k_max, guard_doppler, guard_delay, min_ratio, d_out, d_count);
    else rc = run_detect_dev<double>(h, (const double*)s->dev, 1, s->d, s->n, d_freqs, k_max, guard_doppler, guard_delay, min_ratio, d_out, d_count);
    if (rc) return rc;
    std::vector<caf_b200_detection> rec(k_max);
    unsigned long long cnt = 0;
    CK(cudaMemcpyAsync(rec.data(), d_out, rec_bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&cnt, d_count, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    std::memcpy(out, rec.data(), rec_bytes);
    *count = (size_t)cnt;
    return CAF_B200_OK;
}
int caf_b200_detect_f64_dev(caf_b200_handle h, const double* surface, size_t p, size_t d, size_t n, const double* freqs_hz,
                            size_t k_max, uint32_t guard_doppler, uint32_t guard_delay, double min_ratio,
                            caf_b200_detection* out, uint64_t* counts) {
    return detect_dev_impl<double>(h, surface, p, d, n, freqs_hz, k_max, guard_doppler, guard_delay, min_ratio, out, counts);
}
int caf_b200_detect_f32_dev(caf_b200_handle h, const float* surface, size_t p, size_t d, size_t n, const double* freqs_hz,
                            size_t k_max, uint32_t guard_doppler, uint32_t guard_delay, double min_ratio,
                            caf_b200_detection* out, uint64_t* counts) {
    return detect_dev_impl<float>(h, surface, p, d, n, freqs_hz, k_max, guard_doppler, guard_delay, min_ratio, out, counts);
}

// ---- CFAR detection and the noise map (caf_cfar.cuh) ----------------------------------------------------------------
static_assert(sizeof(caf_b200_cfar_detection) == sizeof(caf::CfarOut) && sizeof(caf::CfarOut) == 64,
              "CFAR record layouts must match");
extern "C++" {
namespace {
int check_cfar_window(size_t d, size_t n, uint32_t gr, uint32_t gd, uint32_t tr, uint32_t tc) {
    if ((uint64_t)gr + tr > (uint64_t)caf::kCfarMaxTrainDoppler) return fail(CAF_B200_EINVAL, "guard_doppler + train_doppler must be <= 32 rows");
    if ((uint64_t)gd + tc > (uint64_t)caf::kCfarMaxTrainDelay) return fail(CAF_B200_EINVAL, "guard_delay + train_delay must be <= 256 cells");
    if ((uint64_t)tr + tc < 1) return fail(CAF_B200_EINVAL, "train_doppler + train_delay must be >= 1");
    if (d && n && 2 * ((size_t)gd + tc) + 1 > n) return fail(CAF_B200_EINVAL, "2 * (guard_delay + train_delay) + 1 exceeds the cells per row");
    if (d > (1ull << 31) || n > (1ull << 31)) return fail(CAF_B200_EUNSUPPORTED, "more than 2^31 rows or cells per row");
    return CAF_B200_OK;
}
int check_cfar(size_t d, size_t n, size_t k_max, uint32_t gr, uint32_t gd, uint32_t tr, uint32_t tc, double scale) {
    if (k_max < 1 || k_max > (size_t)caf::kDetMaxK) return fail(CAF_B200_EINVAL, "k_max must be 1 ... 1024");
    if (!(scale > 0.0 && scale <= 1.7976931348623157e308)) return fail(CAF_B200_EINVAL, "scale must be finite and > 0");
    return check_cfar_window(d, n, gr, gd, tr, tc);
}

// Both passes on the handle's stream; every pointer is device memory.  Arguments are already checked.
template <typename T>
int run_cfar_dev(caf_b200_handle h, const T* surface, size_t p, size_t d, size_t n, const double* freqs, size_t k_max,
                 uint32_t gr, uint32_t gd, uint32_t trd, uint32_t tcd, double scale, caf::CfarOut* out,
                 unsigned long long* counts) {
    using namespace caf;
    if (p == 0) return CAF_B200_OK;
    const bool cells = d && n;
    const int R = (int)(gr + trd), C = (int)(gd + tcd);
    // tile height: the tallest of 16 / 8 / 4 / 2 / 1 rows that stages its training region and leaves room for two CTAs
    // per SM; else one row staging up to kCfarSmemMax; else (the largest windows) the tallest tile that reads its
    // training cells from the surface
    auto smem = [&](int tr, bool staged) {
        return cfar_tile_layout<T>(tr, (int)gr, (int)gd, R, C, staged, (int)det_tile_max_maxima(tr, (int)gr, (int)gd)).total;
    };
    int tr = 16;
    bool staged = true;
    while (tr > 1 && (smem(tr, true) > kDetSmemBudget || (size_t)(tr / 2) >= d)) tr /= 2;
    if (smem(tr, true) > kCfarSmemMax) {
        staged = false;
        tr = 16;
        while (tr > 1 && (smem(tr, false) > kDetSmemBudget || (size_t)(tr / 2) >= d)) tr /= 2;
    }
    const size_t bytes = smem(tr, staged);                       // <= kCfarSmemMax, set at handle creation
    const int mx = (int)det_tile_max_maxima(tr, (int)gr, (int)gd);
    const long long tiles_c = (long long)((n + kDetCols - 1) / kDetCols), tiles_r = (long long)((d + tr - 1) / tr);
    const long long tiles = cells ? tiles_c * tiles_r : 0;
    const long long slots = (long long)std::min(k_max, (size_t)mx);   // entries one tile can append
    const long long cap = tiles * slots;
    if ((double)p * (double)tiles > 2147483647.0) return fail(CAF_B200_EUNSUPPORTED, "too many tiles for one launch");
    const size_t ctr_bytes = (16 * p + 255) & ~(size_t)255;
    CK(h->det.ensure(ctr_bytes + sizeof(CfarEntry) * (size_t)cap * p));
    unsigned long long* ctr = reinterpret_cast<unsigned long long*>(h->det.p);
    CfarEntry* entries = reinterpret_cast<CfarEntry*>((char*)h->det.p + ctr_bytes);
    CK(cudaMemsetAsync(ctr, 0, 16 * p, h->stream));
    if (tiles) {
        caf_cfar_tiles_kernel<T><<<(unsigned)(p * tiles), kDetCols, bytes, h->stream>>>(
            surface, (long long)d, (long long)n, (int)gr, (int)gd, R, C, tr, staged, mx, scale, tiles_c, tiles,
            (unsigned)k_max, cap, entries, ctr);
        h->launches++;
        CK(cudaGetLastError());
    }
    caf_cfar_merge_kernel<T><<<(unsigned)p, kDetMergeThreads, 0, h->stream>>>(
        surface, (long long)d, (long long)n, freqs, entries, cap, ctr, (unsigned)k_max, out, counts);
    h->launches++;
    CK(cudaGetLastError());
    return CAF_B200_OK;
}

template <typename T>
int detect_cfar_dev_impl(caf_b200_handle h, const T* surface, size_t p, size_t d, size_t n, const double* freqs,
                         size_t k_max, uint32_t gr, uint32_t gd, uint32_t tr, uint32_t tc, double scale,
                         caf_b200_cfar_detection* out, uint64_t* counts) {
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    int rc = check_cfar(d, n, k_max, gr, gd, tr, tc, scale);
    if (rc) return rc;
    if (!out || !counts) return fail(CAF_B200_EINVAL, "null out / counts");
    if (!surface) return fail(CAF_B200_EINVAL, "null surface");
    if (!freqs) return fail(CAF_B200_EINVAL, "null freqs_hz");
    if ((double)p * (double)d * (double)n > 9.0e18) return fail(CAF_B200_EUNSUPPORTED, "surface too large");
    CK(cudaSetDevice(h->device));
    return run_cfar_dev<T>(h, surface, p, d, n, freqs, k_max, gr, gd, tr, tc, scale, (caf::CfarOut*)out,
                           (unsigned long long*)counts);
}

template <typename T>
int cfar_noise_dev_impl(caf_b200_handle h, const T* surface, size_t p, size_t d, size_t n, uint32_t gr, uint32_t gd,
                        uint32_t tr, uint32_t tc, double* noise_out) {
    if (!h) return fail(CAF_B200_EINVAL, "null handle");
    int rc = check_cfar_window(d, n, gr, gd, tr, tc);
    if (rc) return rc;
    if (!surface || !noise_out) return fail(CAF_B200_EINVAL, "null surface / noise_out");
    if ((double)p * (double)d * (double)n > 9.0e18) return fail(CAF_B200_EUNSUPPORTED, "surface too large");
    const long long cells = (long long)(p * d * n);
    if (cells == 0) return CAF_B200_OK;
    CK(cudaSetDevice(h->device));
    const long long blocks = std::min<long long>((cells + 255) / 256, (long long)h->sm_count * 64);
    caf::caf_cfar_noise_kernel<T><<<(unsigned)blocks, 256, 0, h->stream>>>(
        surface, (long long)p, (long long)d, (long long)n, (int)gr, (int)gd, (int)(gr + tr), (int)(gd + tc), noise_out);
    h->launches++;
    CK(cudaGetLastError());
    return CAF_B200_OK;
}
}  // namespace
}  // extern "C++"

int caf_b200_surface_detect_cfar(caf_b200_surface s, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                 uint32_t train_doppler, uint32_t train_delay, double scale, caf_b200_cfar_detection* out,
                                 size_t* count) {
    if (!s || !out || !count) return fail(CAF_B200_EINVAL, "null argument");
    int rc = check_cfar(s->d, s->n, k_max, guard_doppler, guard_delay, train_doppler, train_delay, scale);
    if (rc) return rc;
    {
        std::lock_guard<std::mutex> lk(g_live_mu);
        if (!g_live_handles.count(s->h)) return fail(CAF_B200_EINVAL, "the surface's handle was destroyed");
    }
    caf_b200_handle h = s->h;
    CK(cudaSetDevice(h->device));
    // device block: grid | records | count
    const size_t fr_bytes = (sizeof(double) * s->d + 255) & ~(size_t)255, rec_bytes = sizeof(caf_b200_cfar_detection) * k_max;
    CK(h->det_io.ensure(fr_bytes + rec_bytes + 8));
    double* d_freqs = (double*)h->det_io.p;
    caf::CfarOut* d_out = (caf::CfarOut*)((char*)h->det_io.p + fr_bytes);
    unsigned long long* d_count = (unsigned long long*)((char*)d_out + rec_bytes);
    if (s->d) CK(cudaMemcpyAsync(d_freqs, s->freqs.data(), sizeof(double) * s->d, cudaMemcpyHostToDevice, h->stream));
    if (s->f32) rc = run_cfar_dev<float>(h, (const float*)s->dev, 1, s->d, s->n, d_freqs, k_max, guard_doppler, guard_delay, train_doppler, train_delay, scale, d_out, d_count);
    else rc = run_cfar_dev<double>(h, (const double*)s->dev, 1, s->d, s->n, d_freqs, k_max, guard_doppler, guard_delay, train_doppler, train_delay, scale, d_out, d_count);
    if (rc) return rc;
    std::vector<caf_b200_cfar_detection> rec(k_max);
    unsigned long long cnt = 0;
    CK(cudaMemcpyAsync(rec.data(), d_out, rec_bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&cnt, d_count, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    std::memcpy(out, rec.data(), rec_bytes);
    *count = (size_t)cnt;
    return CAF_B200_OK;
}
int caf_b200_detect_cfar_f64_dev(caf_b200_handle h, const double* surface, size_t p, size_t d, size_t n,
                                 const double* freqs_hz, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                 uint32_t train_doppler, uint32_t train_delay, double scale, caf_b200_cfar_detection* out,
                                 uint64_t* counts) {
    return detect_cfar_dev_impl<double>(h, surface, p, d, n, freqs_hz, k_max, guard_doppler, guard_delay, train_doppler,
                                        train_delay, scale, out, counts);
}
int caf_b200_detect_cfar_f32_dev(caf_b200_handle h, const float* surface, size_t p, size_t d, size_t n,
                                 const double* freqs_hz, size_t k_max, uint32_t guard_doppler, uint32_t guard_delay,
                                 uint32_t train_doppler, uint32_t train_delay, double scale, caf_b200_cfar_detection* out,
                                 uint64_t* counts) {
    return detect_cfar_dev_impl<float>(h, surface, p, d, n, freqs_hz, k_max, guard_doppler, guard_delay, train_doppler,
                                       train_delay, scale, out, counts);
}
int caf_b200_cfar_noise_f64_dev(caf_b200_handle h, const double* surface, size_t p, size_t d, size_t n,
                                uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler, uint32_t train_delay,
                                double* noise_out) {
    return cfar_noise_dev_impl<double>(h, surface, p, d, n, guard_doppler, guard_delay, train_doppler, train_delay, noise_out);
}
int caf_b200_cfar_noise_f32_dev(caf_b200_handle h, const float* surface, size_t p, size_t d, size_t n,
                                uint32_t guard_doppler, uint32_t guard_delay, uint32_t train_doppler, uint32_t train_delay,
                                double* noise_out) {
    return cfar_noise_dev_impl<float>(h, surface, p, d, n, guard_doppler, guard_delay, train_doppler, train_delay, noise_out);
}

// ---- multi-GPU peak words: [0] = bits(value), [1] = global doppler row (UINT64_MAX if none),
//      [2] = delay index, [3] = bits(freq_hz) ----
#define CKN(call)                                                                                   \
    do {                                                                                            \
        int e_ = (call);                                                                            \
        if (e_ != 0) return fail(CAF_B200_ENCCL, std::string(#call " failed: ") + nccl_api().GetErrorString(e_)); \
    } while (0)

int caf_b200_comm_unique_id(unsigned char id[CAF_B200_NCCL_ID_BYTES]) {
    if (!id) return fail(CAF_B200_EINVAL, "null id");
    NcclApi& n = nccl_api();
    if (!n.ok()) return fail(CAF_B200_ENCCL, "NCCL is not available: " + n.why);
    NcclUniqueId u;
    CKN(n.GetUniqueId(&u));
    std::memcpy(id, u.internal, CAF_B200_NCCL_ID_BYTES);
    return CAF_B200_OK;
}

// Map every peer's mailbox (one NCCL all-gather of the IPC handles, one of the outcomes: either every rank has every peer
// mapped or all fall back to the NCCL exchange).  Collective: every rank of the communicator runs it, in comm_finish.
static void setup_p2p(caf_b200_comm c) {
    c->p2p = false;
    if (c->world < 2) return;
    bool want = true;
    if (const char* e_ = getenv("CAF_B200_P2P")) want = e_[0] != '0';
    cudaStream_t s = c->h->stream;
    const size_t W = (size_t)c->world;
    struct Rec { cudaIpcMemHandle_t hd; unsigned long long ok; };
    static_assert(sizeof(Rec) % 8 == 0, "record is sent as u64 words");
    Rec mine{}; mine.ok = 0;
    if (want && cudaMalloc(&c->mail, 2 * W * 8 * 8) == cudaSuccess && cudaMemset(c->mail, 0, 2 * W * 8 * 8) == cudaSuccess &&
        cudaIpcGetMemHandle(&mine.hd, c->mail) == cudaSuccess) mine.ok = 1;
    (void)cudaGetLastError();
    // the exchange of handles is itself collective: every rank takes part whatever its local outcome
    void* d_send = nullptr; void* d_recv = nullptr;
    std::vector<Rec> all(W);
    bool moved = cudaMalloc(&d_send, sizeof(Rec)) == cudaSuccess && cudaMalloc(&d_recv, sizeof(Rec) * W) == cudaSuccess &&
                 cudaMemcpyAsync(d_send, &mine, sizeof(Rec), cudaMemcpyHostToDevice, s) == cudaSuccess &&
                 nccl_api().AllGather(d_send, d_recv, sizeof(Rec) / 8, kNcclUint64, c->comm, s) == 0 &&
                 cudaMemcpyAsync(all.data(), d_recv, sizeof(Rec) * W, cudaMemcpyDeviceToHost, s) == cudaSuccess &&
                 cudaStreamSynchronize(s) == cudaSuccess;
    unsigned long long good = moved ? 1ull : 0ull;
    for (size_t r = 0; good && r < W; ++r) good = all[r].ok;
    std::vector<unsigned long long*> peers(W, nullptr);
    for (size_t r = 0; good && r < W; ++r) {
        if ((int)r == c->rank) { peers[r] = c->mail; continue; }
        void* p = nullptr;
        if (cudaIpcOpenMemHandle(&p, all[r].hd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { good = 0; (void)cudaGetLastError(); break; }
        c->opened.push_back(p);
        peers[r] = (unsigned long long*)p;
    }
    if (good && (cudaMalloc(&c->peer_mail, sizeof(void*) * W) != cudaSuccess ||
                 cudaMemcpy(c->peer_mail, peers.data(), sizeof(void*) * W, cudaMemcpyHostToDevice) != cudaSuccess)) good = 0;
    // second round: everybody mapped everybody?
    unsigned long long verdict = 0;
    if (moved) {
        std::vector<unsigned long long> oks(W, 0ull);
        if (cudaMemcpyAsync(d_send, &good, 8, cudaMemcpyHostToDevice, s) == cudaSuccess &&
            nccl_api().AllGather(d_send, d_recv, 1, kNcclUint64, c->comm, s) == 0 &&
            cudaMemcpyAsync(oks.data(), d_recv, 8 * W, cudaMemcpyDeviceToHost, s) == cudaSuccess &&
            cudaStreamSynchronize(s) == cudaSuccess) {
            verdict = 1;
            for (size_t r = 0; r < W; ++r) verdict &= oks[r];
        }
    }
    if (d_send) cudaFree(d_send);
    if (d_recv) cudaFree(d_recv);
    (void)cudaGetLastError();
    c->p2p = verdict != 0;
}

static int comm_finish(caf_b200_comm c, caf_b200_comm* out) {
    cudaError_t e;
    if ((e = cudaMalloc(&c->send, 8 * 4)) != cudaSuccess || (e = cudaMalloc(&c->recv, 8 * 4 * (size_t)c->world)) != cudaSuccess ||
        (e = cudaMallocHost(&c->host, 8 * 4 * (size_t)c->world)) != cudaSuccess ||
        (e = cudaMallocHost(&c->status, sizeof(int))) != cudaSuccess) {
        caf_b200_comm_destroy(c);
        return fail(CAF_B200_ECUDA, std::string("communicator buffers: ") + cudaGetErrorString(e));
    }
    *c->status = 0;
    setup_p2p(c);
    *out = c;
    return CAF_B200_OK;
}

int caf_b200_comm_create(caf_b200_handle h, int world, int rank, const unsigned char id[CAF_B200_NCCL_ID_BYTES],
                         caf_b200_comm* out) {
    if (!h || !out || !id) return fail(CAF_B200_EINVAL, "null argument");
    if (world < 1 || rank < 0 || rank >= world) return fail(CAF_B200_EINVAL, "bad world / rank");
    NcclApi& n = nccl_api();
    if (!n.ok()) return fail(CAF_B200_ENCCL, "NCCL is not available: " + n.why);
    CK(cudaSetDevice(h->device));
    caf_b200_comm c = new (std::nothrow) caf_b200_comm_s();
    if (!c) return fail(CAF_B200_EINVAL, "out of memory");
    c->h = h; c->device = h->device; c->world = world; c->rank = rank; c->own = true;
    NcclUniqueId u;
    std::memcpy(u.internal, id, CAF_B200_NCCL_ID_BYTES);
    int e = n.CommInitRank(&c->comm, world, u, rank);
    if (e != 0) { delete c; return fail(CAF_B200_ENCCL, std::string("ncclCommInitRank failed: ") + n.GetErrorString(e)); }
    return comm_finish(c, out);
}

int caf_b200_comm_adopt(caf_b200_handle h, void* nccl_comm, int world, int rank, caf_b200_comm* out) {
    if (!h || !out || !nccl_comm) return fail(CAF_B200_EINVAL, "null argument");
    if (world < 1 || rank < 0 || rank >= world) return fail(CAF_B200_EINVAL, "bad world / rank");
    NcclApi& n = nccl_api();
    if (!n.ok()) return fail(CAF_B200_ENCCL, "NCCL is not available: " + n.why);
    CK(cudaSetDevice(h->device));
    caf_b200_comm c = new (std::nothrow) caf_b200_comm_s();
    if (!c) return fail(CAF_B200_EINVAL, "out of memory");
    c->h = h; c->device = h->device; c->world = world; c->rank = rank; c->own = false; c->comm = nccl_comm;
    return comm_finish(c, out);
}

int caf_b200_comm_destroy(caf_b200_comm c) {
    if (!c) return CAF_B200_OK;
    cudaSetDevice(c->device);             // the handle may already be gone: the communicator remembers its own device
    for (void* p : c->opened) cudaIpcCloseMemHandle(p);
    if (c->peer_mail) cudaFree(c->peer_mail);
    if (c->mail) cudaFree(c->mail);
    if (c->send) cudaFree(c->send);
    if (c->recv) cudaFree(c->recv);
    if (c->host) cudaFreeHost(c->host);
    if (c->status) cudaFreeHost(c->status);
    if (c->own && c->comm && nccl_api().ok()) nccl_api().CommDestroy(c->comm);
    delete c;
    return CAF_B200_OK;
}

int caf_b200_comm_shard(caf_b200_comm c, size_t n, size_t* lo, size_t* hi) {
    if (!c || !lo || !hi) return fail(CAF_B200_EINVAL, "null argument");
    *lo = n * (size_t)c->rank / (size_t)c->world;
    *hi = n * ((size_t)c->rank + 1) / (size_t)c->world;
    return CAF_B200_OK;
}

int caf_b200_comm_uses_p2p(caf_b200_comm c, int* flag) {
    if (!c || !flag) return fail(CAF_B200_EINVAL, "null argument");
    *flag = c->p2p ? 1 : 0;
    return CAF_B200_OK;
}

int caf_b200_comm_remote_error(caf_b200_comm c, int* flag) {
    if (!c || !flag) return fail(CAF_B200_EINVAL, "null argument");
    *flag = *c->status;
    return CAF_B200_OK;
}

extern "C++" {
namespace {
int check_comm(caf_b200_handle h, caf_b200_comm c) {
    if (!h || !c) return fail(CAF_B200_EINVAL, "null handle / communicator");
    if (c->h != h) return fail(CAF_B200_EINVAL, "communicator belongs to another handle");
    return CAF_B200_OK;
}
// c->send holds this rank's packed words (device): all-gather them and resolve on the DEVICE into out_dev (device or
// pinned host memory).  Everything is stream-ordered; nothing waits on the host.
int exchange_async(caf_b200_handle h, caf_b200_comm c, caf_b200_peak* out_dev) {
    if (c->p2p) {
        // one kernel: post to every peer's mailbox over NVLink, collect the world's records, resolve
        caf::caf_peak_exchange_kernel<<<1, 32, 0, h->stream>>>(c->send, c->peer_mail, c->mail, c->world, c->rank, ++c->p2p_epoch,
                                                               (caf::PeakOut*)out_dev, c->status);
        h->launches++;
        CK(cudaGetLastError());
        return CAF_B200_OK;
    }
    CKN(nccl_api().AllGather(c->send, c->recv, 4, kNcclUint64, c->comm, h->stream));
    caf::caf_peak_resolve_kernel<<<1, 32, 0, h->stream>>>(c->recv, c->world, (caf::PeakOut*)out_dev, c->status);
    h->launches++;
    CK(cudaGetLastError());
    return CAF_B200_OK;
}
// Words that tell every peer "this rank failed": the collective is still entered, so nobody hangs in it.
int post_failure_and_exchange(caf_b200_handle h, caf_b200_comm c) {
    const unsigned long long w[4] = {0ull, caf::kPeakRemoteError, 0ull, 0ull};
    if (cudaMemcpyAsync(c->send, w, sizeof w, cudaMemcpyHostToDevice, h->stream) != cudaSuccess) return CAF_B200_ECUDA;
    const int rc = exchange_async(h, c, reinterpret_cast<caf_b200_peak*>(c->host));     // the same transport the healthy ranks use
    cudaStreamSynchronize(h->stream);
    return rc;
}
// c->send -> the world's resolved peak on the HOST (through the pinned block c->host), whichever transport is in use
int exchange_sync(caf_b200_handle h, caf_b200_comm c, caf_b200_peak* out) {
    int rc = exchange_async(h, c, reinterpret_cast<caf_b200_peak*>(c->host));
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));
    to_public(*reinterpret_cast<const caf::PeakOut*>(c->host), out);
    if (*c->status) return fail(CAF_B200_EREMOTE, "a peer rank failed before the peak exchange");
    return CAF_B200_OK;
}
}  // namespace
}  // extern "C++"

int caf_b200_peak_allgather_async(caf_b200_handle h, caf_b200_comm c, const caf_b200_peak* local_peak_dev,
                                  uint64_t global_row_offset, caf_b200_peak* out_dev) {
    int rc = check_comm(h, c);
    if (rc) return rc;
    if (!out_dev) return fail(CAF_B200_EINVAL, "null out");
    CK(cudaSetDevice(h->device));
    caf::caf_peak_pack_kernel<<<1, 32, 0, h->stream>>>((const caf::PeakOut*)local_peak_dev, (unsigned long long)global_row_offset, c->send);
    h->launches++;
    CK(cudaGetLastError());
    return exchange_async(h, c, out_dev);
}

int caf_b200_peak_allgather_dev(caf_b200_handle h, caf_b200_comm c, const caf_b200_peak* local_dev,
                                uint64_t global_row_offset, caf_b200_peak* out) {
    if (!local_dev || !out) return fail(CAF_B200_EINVAL, "null argument");
    int rc = check_comm(h, c);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    caf::caf_peak_pack_kernel<<<1, 32, 0, h->stream>>>((const caf::PeakOut*)local_dev, (unsigned long long)global_row_offset, c->send);
    h->launches++;
    CK(cudaGetLastError());
    return exchange_sync(h, c, out);
}

extern "C++" {
namespace {
// Device-resident rows [row_offset, row_offset + d_local) of the doppler grid on this rank, find_peak across ranks:
// the local find_peak writes its result already packed into c->send, then ncclAllGather + device resolve.  No host
// synchronisation anywhere; out_dev is valid once the stream has reached this point.
template <typename T>
int run_sharded_dev(caf_b200_handle h, caf_b200_comm c, const caf::cx<T>* needle, const caf::cx<T>* hay, size_t l,
                    const double* freqs_local, size_t d_local, uint64_t row_offset, uint32_t fs, T* surface_local,
                    T* rv, unsigned long long* ri, caf_b200_peak* out_dev) {
    int rc = check_comm(h, c);
    if (rc) return rc;
    if (!out_dev) return fail(CAF_B200_EINVAL, "null out");
    rc = check_common<T>(h, needle, hay, 1, l, freqs_local, d_local, fs);
    cudaError_t ce = cudaSuccess;
    if (!rc && (ce = cudaSetDevice(h->device)) != cudaSuccess) rc = fail(CAF_B200_ECUDA, cudaGetErrorString(ce));
    if (!rc && (ce = h->peaks.ensure(sizeof(caf::PeakOut))) != cudaSuccess) rc = fail(CAF_B200_ECUDA, cudaGetErrorString(ce));
    if (!rc) {
        h->pack_words = c->send; h->pack_offset = (unsigned long long)row_offset;
        rc = run_batch_dev<T>(h, needle, hay, 1, l, freqs_local, d_local, fs, surface_local, rv, ri, (caf::PeakOut*)h->peaks.p);
        h->pack_words = nullptr; h->pack_offset = 0;
    }
    if (rc) {                       // never leave the peers alone in the collective (they would wait for ever)
        const std::string why = g_err;
        post_failure_and_exchange(h, c);
        return fail(rc, why);
    }
    return exchange_async(h, c, out_dev);
}

// rows [lo, hi) of the doppler grid on this rank, then find_peak across ranks (host inputs, host outputs)
template <typename T>
int run_sharded(caf_b200_handle h, caf_b200_comm c, const caf::cx<T>* needle, const caf::cx<T>* hay, size_t l,
                const double* freqs, size_t d, uint32_t fs, T* surface_local, caf_b200_peak* peak) {
    int rc = check_comm(h, c);
    if (rc) return rc;
    if (!peak) return fail(CAF_B200_EINVAL, "null peak");
    size_t lo = 0, hi = 0;
    caf_b200_comm_shard(c, d, &lo, &hi);
    caf_b200_peak local;
    rc = run_batch_host<T>(h, needle, hay, 1, l, freqs ? freqs + lo : freqs, hi - lo, fs, surface_local, nullptr, nullptr, &local);
    if (rc) {                       // every rank enters the collective, whatever happened locally
        const std::string why = g_err;
        post_failure_and_exchange(h, c);
        return fail(rc, why);
    }
    // the local peak is on the host here (run_batch_host staged it); it is tiny, so the exchange re-uploads the words
    uint64_t words[4];
    caf_b200_peak_pack(&local, lo, words);
    CK(cudaMemcpyAsync(c->send, words, sizeof words, cudaMemcpyHostToDevice, h->stream));
    return exchange_sync(h, c, peak);
}
}  // namespace
}  // extern "C++"

int caf_b200_surface_sharded_f64(caf_b200_handle h, caf_b200_comm c, const caf_c128* needle, const caf_c128* hay, size_t l,
                                 const double* freqs, size_t d, uint32_t fs, double* surface_local, caf_b200_peak* peak) {
    return run_sharded<double>(h, c, (const double2*)needle, (const double2*)hay, l, freqs, d, fs, surface_local, peak);
}
int caf_b200_surface_sharded_f32(caf_b200_handle h, caf_b200_comm c, const caf_c64* needle, const caf_c64* hay, size_t l,
                                 const double* freqs, size_t d, uint32_t fs, float* surface_local, caf_b200_peak* peak) {
    return run_sharded<float>(h, c, (const float2*)needle, (const float2*)hay, l, freqs, d, fs, surface_local, peak);
}
int caf_b200_sharded_f64_dev(caf_b200_handle h, caf_b200_comm c, const caf_c128* needle, const caf_c128* hay, size_t l,
                             const double* freqs_local, size_t d_local, uint64_t row_offset, uint32_t fs,
                             double* surface_local, double* rv, uint64_t* ri, caf_b200_peak* peak_out) {
    return run_sharded_dev<double>(h, c, (const double2*)needle, (const double2*)hay, l, freqs_local, d_local, row_offset, fs,
                                   surface_local, rv, (unsigned long long*)ri, peak_out);
}
int caf_b200_sharded_f32_dev(caf_b200_handle h, caf_b200_comm c, const caf_c64* needle, const caf_c64* hay, size_t l,
                             const double* freqs_local, size_t d_local, uint64_t row_offset, uint32_t fs,
                             float* surface_local, float* rv, uint64_t* ri, caf_b200_peak* peak_out) {
    return run_sharded_dev<float>(h, c, (const float2*)needle, (const float2*)hay, l, freqs_local, d_local, row_offset, fs,
                                  surface_local, rv, (unsigned long long*)ri, peak_out);
}

void caf_b200_peak_pack(const caf_b200_peak* local, uint64_t global_row_offset, uint64_t words[4]) {
    double v = local->value, f = local->freq_hz;
    std::memcpy(&words[0], &v, 8);
    words[1] = (local->doppler_idx == UINT64_MAX) ? UINT64_MAX : local->doppler_idx + global_row_offset;
    words[2] = local->delay_idx;
    std::memcpy(&words[3], &f, 8);
}

void caf_b200_peak_resolve(const uint64_t* words, size_t world, caf_b200_peak* out) {
    (void)caf_b200_peak_resolve_status(words, world, out);
}

int caf_b200_peak_resolve_status(const uint64_t* words, size_t world, caf_b200_peak* out) {
    caf_b200_peak best; best.value = 0.0; best.freq_hz = 0.0; best.doppler_idx = UINT64_MAX; best.delay_idx = 0;
    int failed = 0;
    for (size_t r = 0; r < world; ++r) {
        const uint64_t* w = words + 4 * r;
        double v, f;
        std::memcpy(&v, &w[0], 8); std::memcpy(&f, &w[3], 8);
        if (w[1] == UINT64_MAX - 1) { failed = 1; continue; }     // that rank failed before the exchange
        if (w[1] == UINT64_MAX) continue;
        // find_peak (mod.rs:36-40): strict > in row order  ==  larger value, ties to the lower global row
        if (v > best.value || (v == best.value && v > 0.0 && w[1] < best.doppler_idx)) {
            best.value = v; best.freq_hz = f; best.doppler_idx = w[1]; best.delay_idx = w[2];
        }
    }
    *out = best;
    return failed;
}

}  // extern "C"
