// caf_detect.cuh -- the K strongest local maxima of stored CAF surfaces, refined to sub-cell delay and Doppler
// (caf_b200_surface_detect / caf_b200_detect_*_dev, include/caf_b200.h).  The detector reads a surface after the row
// kernels have written it; it shares no code with them.
//
// The contract (DESIGN.md section 9; oracle/detect.py restates it in numpy):
//   window of cell (r, k): rows r' in [r - gr, r + gr] clipped to [0, d), cells (k + j) mod n for |j| <= gd, minus the
//   cell itself.  (r, k) with value v is a local maximum when v > 0, no window cell exceeds v and no window cell equal to
//   v has a smaller flat index r' * n + k'.  NaN cells never qualify and never block.  Local maxima are ordered by value
//   descending, then flat index ascending; the first k_max are kept, then those below min_ratio x the first are dropped.
//
// Pass 1 (caf_detect_tiles_kernel): one CTA per tile of `tr` rows x 256 cells of one pair.  Each warp stages whole rows
//   of the tile plus the halo (wrapped in delay) in shared memory and writes the row's sliding maximum over +-gd cells;
//   the column maximum of those over +-gr rows is the window maximum.  Only a cell equal to its window maximum runs the
//   equal-value rule, from shared memory except where a staged row maximum shows an equal cell in an earlier row (then
//   that row is read from the surface) and for halo or wrapped cells of its own row.  The tile's local maxima are cut to its top k_max by the 128-bit key
//   (value bits, ~flat index) -- values are >= 0, so the bit pattern of the double orders them -- and appended to the
//   pair's candidate list.  A tile with k_max or more local maxima also raises the pair's floor to its k_max-th value:
//   that many entries reach it, so nothing below it can be in the answer, and later tiles drop such entries at once.
// Pass 2 (caf_detect_merge_kernel): one CTA per pair selects the k_max best keys of the candidate list, sorts them,
//   refines each from its neighbours and writes the records.  Keys are unique (the flat index is), so the answer does not
//   depend on the order in which tiles appended their lists: it is the same for any grid and on every call.
#pragma once
#include <cstdint>

namespace caf {

struct DetectOut {                    // == caf_b200_detection
    double value;
    double freq_hz;
    unsigned long long doppler_idx;   // ~0ull in unused slots
    unsigned long long delay_idx;
    double lag_samples;
    double freq_hz_interp;
};

struct DetEntry { unsigned long long vbits, flat; };   // a candidate: bits of the value widened to double, flat index

constexpr int kDetCols = 256;                 // cells per tile row = threads of pass 1
constexpr int kDetWarps = kDetCols / 32;
constexpr int kDetMergeThreads = 512;
constexpr int kDetMaxK = 1024;
constexpr int kDetMaxGuardDoppler = 32;
constexpr int kDetMaxGuardDelay = 256;

// dynamic shared memory of pass 1: window maxima of tr + 2 gr rows, values of the tr output rows, one staged row per warp,
// the candidate list (tile-local indices) and the radix-select histogram
template <typename T>
__host__ __device__ constexpr size_t det_tile_smem(int tr, int gr, int gd) {
    return sizeof(T) * ((size_t)(tr + 2 * gr) * kDetCols + (size_t)tr * kDetCols + (size_t)kDetWarps * (kDetCols + 2 * gd)) +
           sizeof(unsigned) * ((size_t)tr * kDetCols + 256);
}

constexpr size_t kDetSmemBudget = 100 * 1024;     // tiles taller than one row stay under this: two CTAs per SM

// the most pass 1 ever asks for: the budget, or one row at the largest guards (186 KB in f64)
template <typename T>
__host__ __device__ constexpr size_t det_tile_smem_max() {
    return det_tile_smem<T>(1, kDetMaxGuardDoppler, kDetMaxGuardDelay) > kDetSmemBudget
               ? det_tile_smem<T>(1, kDetMaxGuardDoppler, kDetMaxGuardDelay) : kDetSmemBudget;
}

// Most local maxima a tile of tr rows x kDetCols cells can hold.  Two local maxima never lie in each other's window
// (the larger, or the earlier of two equal ones, blocks the other), so they differ by more than gr rows or more than gd
// cells; blocks of (gr + 1) x (gd + 1) cells hold at most one each.
inline size_t det_tile_max_maxima(int tr, int gr, int gd) {
    return (size_t)((tr + gr) / (gr + 1)) * (size_t)((kDetCols + gd) / (gd + 1));
}

template <typename T> __device__ __forceinline__ T det_max(T a, T b);      // NaN-ignoring maximum
template <> __device__ __forceinline__ double det_max<double>(double a, double b) { return fmax(a, b); }
template <> __device__ __forceinline__ float det_max<float>(float a, float b) { return fmaxf(a, b); }

__device__ __forceinline__ long long det_wrap(long long c, long long n) {   // c in (-n, 2n) -> [0, n)
    return c < 0 ? c + n : (c >= n ? c - n : c);
}

// Block-wide radix select: writes to (st->oh, st->ol) the kk-th largest (1-based, kk <= N) of N unique 128-bit keys
// get(i) = (hi, lo), compared as unsigned (hi, lo) pairs.  MSB first, 8 bits per step; stops as soon as the step's bucket
// holds that key alone.  Every thread of the block calls it; blockDim.x >= 256; hist has 256 words.
struct DetSelState { unsigned long long ph, pl, mh, ml, oh, ol; unsigned rem, done; };

template <typename Get>
__device__ void det_select_kth(Get get, long long N, unsigned kk, unsigned* hist, DetSelState* st) {
    const int tid = threadIdx.x;
    if (tid == 0) { st->ph = st->pl = st->mh = st->ml = 0ull; st->rem = kk; st->done = 0; }
    __syncthreads();
    for (int step = 0; step < 16; ++step) {
        const bool on_hi = step < 8;
        const int sh = 56 - 8 * (step & 7);
        for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0u;
        __syncthreads();
        const unsigned long long ph = st->ph, pl = st->pl, mh = st->mh, ml = st->ml;
        for (long long i = tid; i < N; i += blockDim.x) {
            unsigned long long h, l;
            get(i, h, l);
            if ((h & mh) == ph && (l & ml) == pl) atomicAdd(&hist[(unsigned)(((on_hi ? h : l) >> sh) & 0xffull)], 1u);
        }
        __syncthreads();
        if (tid < 32) {       // warp 0: lane q owns bins 255 - 8q ... 248 - 8q, scanned from the top
            unsigned b[8], s = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { b[j] = hist[255 - 8 * tid - j]; s += b[j]; }
            unsigned inc = s;
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
                if (tid >= o) inc += t;
            }
            const unsigned rem = st->rem;
            const unsigned hit = __ballot_sync(0xffffffffu, inc >= rem);
            const int q = __ffs(hit) - 1;           // rem <= the bucket total, so some lane reaches it
            if (tid == q) {
                unsigned before = inc - s;
                bool found = false;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (!found && before + b[j] >= rem) {
                        found = true;
                        const unsigned long long dig = (unsigned long long)(255 - 8 * q - j) << sh;
                        if (on_hi) { st->ph |= dig; st->mh |= 0xffull << sh; }
                        else { st->pl |= dig; st->ml |= 0xffull << sh; }
                        st->rem = rem - before;
                        st->done = b[j] == 1u;
                    }
                    if (!found) before += b[j];
                }
            }
        }
        __syncthreads();
        if (st->done) break;
    }
    if (st->done) {           // the prefix names one key: fetch the rest of it
        const unsigned long long ph = st->ph, pl = st->pl, mh = st->mh, ml = st->ml;
        for (long long i = tid; i < N; i += blockDim.x) {
            unsigned long long h, l;
            get(i, h, l);
            if ((h & mh) == ph && (l & ml) == pl) { st->oh = h; st->ol = l; }
        }
    } else if (tid == 0) {
        st->oh = st->ph; st->ol = st->pl;
    }
    __syncthreads();
}

__device__ __forceinline__ bool det_key_ge(unsigned long long h, unsigned long long l, unsigned long long th,
                                           unsigned long long tl) {
    return h > th || (h == th && l >= tl);
}

// ---- pass 1 --------------------------------------------------------------------------------------------------------
// surf [p][d][n]; grid = p * tiles_per_pair CTAs of kDetCols threads.  ctr [p][2] = (entries appended, floor value bits),
// zeroed before the launch; entries [p][cap].
template <typename T>
__global__ void __launch_bounds__(kDetCols) caf_detect_tiles_kernel(
        const T* __restrict__ surf, long long d, long long n, int gr, int gd, int tr, long long tiles_c,
        long long tiles_per_pair, unsigned kmax, long long cap, DetEntry* __restrict__ entries,
        unsigned long long* __restrict__ ctr) {
    extern __shared__ __align__(16) unsigned char det_smem[];
    T* hbuf = reinterpret_cast<T*>(det_smem);                             // [tr + 2 gr][kDetCols]
    T* vbuf = hbuf + (size_t)(tr + 2 * gr) * kDetCols;                   // [tr][kDetCols]
    const int W = kDetCols + 2 * gd;
    T* stage = vbuf + (size_t)tr * kDetCols;                              // [kDetWarps][W]
    unsigned* cand = reinterpret_cast<unsigned*>(stage + (size_t)kDetWarps * W);   // [tr * kDetCols]
    unsigned* hist = cand + (size_t)tr * kDetCols;                        // [256]
    __shared__ unsigned ncand, nkeep, wpos;
    __shared__ unsigned long long base;
    __shared__ DetSelState sel;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long pair = (long long)blockIdx.x / tiles_per_pair;
    const long long t = (long long)blockIdx.x - pair * tiles_per_pair;
    const long long r0 = (t / tiles_c) * tr, c0 = (t % tiles_c) * kDetCols;
    const T* S = surf + pair * d * n;
    unsigned long long* my_ctr = ctr + 2 * pair;
    if (tid == 0) { ncand = 0u; nkeep = 0u; wpos = 0u; }

    // rows r0 - gr ... r0 + tr + gr - 1 (clipped): stage the row with its delay halo, write its sliding maximum
    const long long rlo = r0 - gr > 0 ? r0 - gr : 0;
    const long long rhi = r0 + tr + gr < d ? r0 + tr + gr : d;
    const bool no_wrap = c0 >= gd && c0 - gd + W <= n;
    T* st = stage + (size_t)warp * W;
    for (long long rr = rlo + warp; rr < rhi; rr += kDetWarps) {
        const T* row = S + rr * n;
        if (no_wrap) {
            for (int i = lane; i < W; i += 32) st[i] = __ldg(row + (c0 - gd + i));
        } else {
            for (int i = lane; i < W; i += 32) {
                long long c = (c0 - gd + i) % n;
                if (c < 0) c += n;
                st[i] = __ldg(row + c);
            }
        }
        __syncwarp();
        T* hrow = hbuf + (size_t)(rr - r0 + gr) * kDetCols;
        const bool out_row = rr >= r0 && rr < r0 + tr;
        for (int cl = lane; cl < kDetCols; cl += 32) {
            T m = st[cl];
            for (int j = 1; j <= 2 * gd; ++j) m = det_max<T>(m, st[cl + j]);
            hrow[cl] = m;
            if (out_row) vbuf[(size_t)(rr - r0) * kDetCols + cl] = st[cl + gd];
        }
        __syncwarp();
    }
    __syncthreads();

    // local maxima of this thread's column
    const unsigned long long floor0 = *reinterpret_cast<volatile unsigned long long*>(my_ctr + 1);
    const long long c = c0 + tid;
    if (c < n) {
        for (int q = 0; q < tr && r0 + q < d; ++q) {
            const long long r = r0 + q;
            const T v = vbuf[(size_t)q * kDetCols + tid];
            if (!(v > (T)0)) continue;
            if ((unsigned long long)__double_as_longlong((double)v) < floor0) continue;
            T m = v;
            const long long qa = r - gr > 0 ? r - gr : 0, qb = r + gr < d - 1 ? r + gr : d - 1;
            for (long long qq = qa; qq <= qb; ++qq) m = det_max<T>(m, hbuf[(size_t)(qq - r0 + gr) * kDetCols + tid]);
            if (m > v) continue;
            // v is the window maximum: no window cell equal to v may come first in flat order.  An earlier row can hold
            // one only where its maximum over the window's cells (hbuf) equals v -- rare outside plateaus -- and only then
            // is that row read from the surface.
            bool blocked = false;
            for (long long qq = qa; qq < r && !blocked; ++qq) {
                if (!(hbuf[(size_t)(qq - r0 + gr) * kDetCols + tid] == v)) continue;
                for (int j = -gd; j <= gd; ++j)
                    if (__ldg(S + qq * n + det_wrap(c + j, n)) == v) { blocked = true; break; }
            }
            // this row: the cells left of c (from the tile's values where they lie in the tile) and the cells that wrap
            // past the end of the row to its start
            for (int j = 1; j <= gd && !blocked; ++j) {
                const long long kl = c - j, kr = c + j;
                if (kl >= 0 && (kl >= c0 ? vbuf[(size_t)q * kDetCols + tid - j] : __ldg(S + r * n + kl)) == v) blocked = true;
                if (kr >= n && __ldg(S + r * n + (kr - n)) == v) blocked = true;
            }
            if (!blocked) cand[atomicAdd(&ncand, 1u)] = (unsigned)(q * kDetCols + tid);
        }
    }
    __syncthreads();

    // this tile's best kmax, then the pair's floor
    const unsigned cnt = ncand;
    auto key = [&](long long i, unsigned long long& h, unsigned long long& l) {
        const unsigned li = cand[i];
        h = (unsigned long long)__double_as_longlong((double)vbuf[li]);
        l = ~(unsigned long long)((r0 + li / kDetCols) * n + c0 + li % kDetCols);
    };
    unsigned long long th = 0ull, tl = 0ull;
    if (cnt > kmax) {
        det_select_kth(key, (long long)cnt, kmax, hist, &sel);
        th = sel.oh; tl = sel.ol;
        if (tid == 0) atomicMax(my_ctr + 1, th);
    }
    const unsigned long long fl = *reinterpret_cast<volatile unsigned long long*>(my_ctr + 1);
    unsigned mine = 0;
    for (unsigned i = tid; i < cnt; i += kDetCols) {
        unsigned long long h, l;
        key(i, h, l);
        if (det_key_ge(h, l, th, tl) && h >= fl) ++mine;
    }
    if (mine) atomicAdd(&nkeep, mine);
    __syncthreads();
    if (tid == 0 && nkeep) base = atomicAdd(my_ctr, (unsigned long long)nkeep);
    __syncthreads();
    if (nkeep == 0u) return;
    DetEntry* E = entries + pair * cap + base;
    for (unsigned i = tid; i < cnt; i += kDetCols) {
        unsigned long long h, l;
        key(i, h, l);
        if (det_key_ge(h, l, th, tl) && h >= fl) E[atomicAdd(&wpos, 1u)] = DetEntry{h, ~l};
    }
}

// ---- pass 2 --------------------------------------------------------------------------------------------------------
// one CTA per pair: out [p][kmax], counts [p]
__device__ __forceinline__ double det_fit(double a, double v, double b) {   // parabola vertex offset, in cells
    const double den = __dadd_rn(__dsub_rn(a, __dmul_rn(2.0, v)), b);
    if (!(den < 0.0)) return 0.0;
    const double dl = __ddiv_rn(__dmul_rn(0.5, __dsub_rn(a, b)), den);
    return dl < -0.5 ? -0.5 : (dl > 0.5 ? 0.5 : dl);
}

template <typename T>
__global__ void __launch_bounds__(kDetMergeThreads) caf_detect_merge_kernel(
        const T* __restrict__ surf, long long d, long long n, const double* __restrict__ freqs,
        const DetEntry* __restrict__ entries, long long cap, const unsigned long long* __restrict__ ctr, unsigned kmax,
        double min_ratio, DetectOut* __restrict__ out, unsigned long long* __restrict__ counts) {
    __shared__ DetEntry win[kDetMaxK];
    __shared__ unsigned hist[256];
    __shared__ DetSelState sel;
    __shared__ unsigned nwin, nkept;
    const int tid = threadIdx.x;
    const long long pair = blockIdx.x;
    const T* S = surf + pair * d * n;
    const DetEntry* E = entries + pair * cap;
    const long long N = (long long)ctr[2 * pair];
    if (tid == 0) { nwin = 0u; nkept = 0u; }
    auto key = [&](long long i, unsigned long long& h, unsigned long long& l) { h = E[i].vbits; l = ~E[i].flat; };
    unsigned long long th = 0ull, tl = 0ull;
    if (N > (long long)kmax) { det_select_kth(key, N, kmax, hist, &sel); th = sel.oh; tl = sel.ol; }
    __syncthreads();
    for (long long i = tid; i < N; i += blockDim.x) {
        unsigned long long h, l;
        key(i, h, l);
        if (det_key_ge(h, l, th, tl)) win[atomicAdd(&nwin, 1u)] = E[i];
    }
    __syncthreads();
    const unsigned m = nwin;
    unsigned P = 1;
    while (P < m) P <<= 1;
    for (unsigned i = m + tid; i < P; i += blockDim.x) win[i] = DetEntry{0ull, ~0ull};   // sorts after every candidate
    __syncthreads();
    // bitonic sort, best key first
    for (unsigned kk = 2; kk <= P; kk <<= 1)
        for (unsigned j = kk >> 1; j > 0; j >>= 1) {
            for (unsigned i = tid; i < P; i += blockDim.x) {
                const unsigned x = i ^ j;
                if (x > i) {
                    const DetEntry a = win[i], b = win[x];
                    const bool a_first = a.vbits > b.vbits || (a.vbits == b.vbits && a.flat < b.flat);
                    if (((i & kk) == 0) != a_first) { win[i] = b; win[x] = a; }
                }
            }
            __syncthreads();
        }
    const double v0 = m ? __longlong_as_double((long long)win[0].vbits) : 0.0;
    const double bar = min_ratio * v0;
    unsigned mine = 0;
    for (unsigned i = tid; i < m; i += blockDim.x)
        if (!(__longlong_as_double((long long)win[i].vbits) < bar)) ++mine;
    if (mine) atomicAdd(&nkept, mine);
    __syncthreads();
    const unsigned kept = nkept;        // values descend, so the kept entries are a prefix
    DetectOut* O = out + pair * (long long)kmax;
    for (unsigned i = tid; i < kmax; i += blockDim.x) {
        DetectOut o;
        if (i < kept) {
            const unsigned long long flat = win[i].flat;
            const long long r = (long long)(flat / (unsigned long long)n), k = (long long)(flat % (unsigned long long)n);
            const T* row = S + r * n;
            const double v = (double)row[k];
            double dk = 0.0, df = 0.0;
            if (n >= 3) dk = det_fit((double)row[k == 0 ? n - 1 : k - 1], v, (double)row[k + 1 == n ? 0 : k + 1]);
            if (r > 0 && r + 1 < d) df = det_fit((double)row[k - n], v, (double)row[k + n]);
            const double fr = freqs[r];
            double fi = fr;
            if (df > 0.0) fi = __dadd_rn(fr, __dmul_rn(df, __dsub_rn(freqs[r + 1], fr)));
            else if (df < 0.0) fi = __dadd_rn(fr, __dmul_rn(df, __dsub_rn(fr, freqs[r - 1])));
            o.value = v; o.freq_hz = fr; o.doppler_idx = (unsigned long long)r; o.delay_idx = (unsigned long long)k;
            o.lag_samples = __dadd_rn((double)(2 * k < n ? k : k - n), dk);
            o.freq_hz_interp = fi;
        } else {
            o.value = 0.0; o.freq_hz = 0.0; o.doppler_idx = ~0ull; o.delay_idx = 0ull; o.lag_samples = 0.0; o.freq_hz_interp = 0.0;
        }
        O[i] = o;
    }
    if (tid == 0) counts[pair] = kept;
}

}  // namespace caf
