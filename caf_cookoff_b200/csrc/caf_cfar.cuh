// caf_cfar.cuh -- cell-averaging CFAR detection on stored CAF surfaces (caf_b200_surface_detect_cfar /
// caf_b200_detect_cfar_*_dev) and the dense noise map it is built on (caf_b200_cfar_noise_*_dev), include/caf_b200.h.
//
// The contract (DESIGN.md section 10; oracle/cfar.py restates it in numpy):
//   R = gr + tr, C = gd + tc.  The training cells of (r, k) are rows r' in [r - R, r + R] clipped to [0, d), cells
//   (k + j) mod n for |j| <= C, minus the guard block |r' - r| <= gr, |j| <= gd; NaN cells are skipped.  noise = sum / m,
//   the sum in ONE fixed order: per row, +0.0 plus its cells in ascending j, in double; the cell's sum, +0.0 plus the row
//   sums in ascending r'.  Only additions and one division, so every path (pass 1, the dense map, the numpy reference)
//   gives the same bits.  (r, k) is a detection when it is a local maximum under detect's rule with (gr, gd), m > 0 and
//   v > scale * noise (the correctly rounded product).
//
// Pass 1 (caf_cfar_tiles_kernel): the tiles, staging and local-maximum rule of caf_detect_tiles_kernel (restated here,
//   not factored out of it, so that detect's kernel and its code generation stay exactly as they are).  Only the local
//   maxima that pass the pair's floor then sum their training cells: one warp takes 32 / (2R + 1) candidates, a lane one
//   training row of one candidate, and the lanes' row sums are added in ascending row by shuffles.  The cells come from a
//   copy of the tile's training region in shared memory (its row pitch is odd, so the lanes of a warp, on different rows
//   of one column, hit different banks) or, when the region does not fit even in a one-row tile, from the surface.  The
//   tile's qualifying cells are cut to its best k_max and raise the pair's floor as in detect; every entry carries its
//   noise and m, so pass 2 never sums again.
// Pass 2 (caf_cfar_merge_kernel): detect's merge without min_ratio, writing the 64-byte records.
// Map (caf_cfar_noise_kernel): one thread per cell, the same row-sum code, reading the surface.
#pragma once
#include <cstdint>
#include "caf_detect.cuh"

namespace caf {

struct CfarOut {                      // == caf_b200_cfar_detection
    DetectOut det;
    double noise;
    unsigned long long train_cells;
};

struct CfarEntry { unsigned long long vbits, flat, noise_bits, m; };   // a qualifying candidate and its noise estimate

constexpr int kCfarMaxTrainDoppler = 32;      // limits of gr + tr and gd + tc: detect's staging bounds
constexpr int kCfarMaxTrainDelay = 256;
constexpr size_t kCfarSmemMax = 200 * 1024;   // one-row tiles may stage a region this large (B200: 227 KB per CTA)

// Dynamic shared memory of pass 1, in bytes from the start: detect's buffers (window maxima, output-row values, one staged
// row per warp), the training region [tr + 2R][pitch] when staged, then per candidate slot (mx of them) its noise, its
// m, its tile-local index and its place in the qualifying list, and the radix-select histogram.
struct CfarTileLayout { size_t region, noise, mcnt, cand, qual, hist, total; int pitch; };

template <typename T>
__host__ __device__ inline CfarTileLayout cfar_tile_layout(int tr, int gr, int gd, int R, int C, bool staged, int mx) {
    CfarTileLayout L;
    L.pitch = (kDetCols + 2 * C) | 1;
    size_t o = sizeof(T) * ((size_t)(tr + 2 * gr) * kDetCols + (size_t)tr * kDetCols + (size_t)kDetWarps * (kDetCols + 2 * gd));
    L.region = o;
    if (staged) o += sizeof(T) * (size_t)(tr + 2 * R) * (size_t)L.pitch;
    o = (o + 7) & ~(size_t)7;
    L.noise = o; o += sizeof(double) * (size_t)mx;
    L.mcnt = o; o += sizeof(unsigned) * (size_t)mx;
    L.cand = o; o += sizeof(unsigned) * (size_t)mx;
    L.qual = o; o += sizeof(unsigned) * (size_t)mx;
    L.hist = o; o += sizeof(unsigned) * 256;
    L.total = o;
    return L;
}

// One training row of a cell: +0.0 plus the non-NaN cells get(j) in ascending j over -C ... C, skipping |j| <= gd in a guard
// row; adds the number of cells taken to cnt.  Pass 1 and the dense map both sum through this.
template <typename Get>
__device__ __forceinline__ double cfar_row_sum(Get get, int C, int gd, bool guard_row, unsigned& cnt) {
    double s = 0.0;
    const int stop = guard_row ? -gd - 1 : C;
    for (int j = -C; j <= stop; ++j) {
        const double x = (double)get(j);
        if (x == x) { s = __dadd_rn(s, x); ++cnt; }
    }
    if (guard_row)
        for (int j = gd + 1; j <= C; ++j) {
            const double x = (double)get(j);
            if (x == x) { s = __dadd_rn(s, x); ++cnt; }
        }
    return s;
}

__device__ __forceinline__ double cfar_noise_of(double sum, unsigned m) {
    return m ? __ddiv_rn(sum, (double)m) : __longlong_as_double(0x7ff8000000000000ll);
}

// ---- pass 1 --------------------------------------------------------------------------------------------------------
// surf [p][d][n]; grid = p * tiles_per_pair CTAs of kDetCols threads.  ctr [p][2] = (entries appended, floor value bits),
// zeroed before the launch; entries [p][cap].  mx = det_tile_max_maxima(tr, gr, gd), the candidate slots of a tile.
template <typename T>
__global__ void __launch_bounds__(kDetCols) caf_cfar_tiles_kernel(
        const T* __restrict__ surf, long long d, long long n, int gr, int gd, int R, int C, int tr, bool staged, int mx,
        double scale, long long tiles_c, long long tiles_per_pair, unsigned kmax, long long cap,
        CfarEntry* __restrict__ entries, unsigned long long* __restrict__ ctr) {
    extern __shared__ __align__(16) unsigned char cfar_smem[];
    const CfarTileLayout L = cfar_tile_layout<T>(tr, gr, gd, R, C, staged, mx);
    T* hbuf = reinterpret_cast<T*>(cfar_smem);                            // [tr + 2 gr][kDetCols]
    T* vbuf = hbuf + (size_t)(tr + 2 * gr) * kDetCols;                   // [tr][kDetCols]
    const int W = kDetCols + 2 * gd;
    T* stage = vbuf + (size_t)tr * kDetCols;                              // [kDetWarps][W]
    T* region = reinterpret_cast<T*>(cfar_smem + L.region);              // [tr + 2R][pitch], cells c0 - C ...
    double* noise = reinterpret_cast<double*>(cfar_smem + L.noise);      // [mx]
    unsigned* mcnt = reinterpret_cast<unsigned*>(cfar_smem + L.mcnt);    // [mx]
    unsigned* cand = reinterpret_cast<unsigned*>(cfar_smem + L.cand);    // [mx]
    unsigned* qual = reinterpret_cast<unsigned*>(cfar_smem + L.qual);    // [mx] positions in cand
    unsigned* hist = reinterpret_cast<unsigned*>(cfar_smem + L.hist);    // [256]
    __shared__ unsigned ncand, nqual, nkeep, wpos;
    __shared__ unsigned long long base;
    __shared__ DetSelState sel;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long pair = (long long)blockIdx.x / tiles_per_pair;
    const long long t = (long long)blockIdx.x - pair * tiles_per_pair;
    const long long r0 = (t / tiles_c) * tr, c0 = (t % tiles_c) * kDetCols;
    const T* S = surf + pair * d * n;
    unsigned long long* my_ctr = ctr + 2 * pair;
    if (tid == 0) { ncand = 0u; nqual = 0u; nkeep = 0u; wpos = 0u; }

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
    // the training region: rows r0 - R ... r0 + tr + R - 1 (clipped), cells c0 - C ... c0 + kDetCols + C - 1 (wrapped)
    const long long tlo = r0 - R > 0 ? r0 - R : 0;
    const long long thi = r0 + tr + R < d ? r0 + tr + R : d;
    if (staged) {
        const int WR = kDetCols + 2 * C;
        const bool flat_rows = c0 >= C && c0 - C + WR <= n;
        for (long long rr = tlo + warp; rr < thi; rr += kDetWarps) {
            const T* row = S + rr * n;
            T* dst = region + (size_t)(rr - (r0 - R)) * L.pitch;
            if (flat_rows) {
                for (int i = lane; i < WR; i += 32) dst[i] = __ldg(row + (c0 - C + i));
            } else {
                for (int i = lane; i < WR; i += 32) {
                    long long c = (c0 - C + i) % n;
                    if (c < 0) c += n;
                    dst[i] = __ldg(row + c);
                }
            }
        }
    }
    __syncthreads();

    // local maxima of this thread's column that can still reach the answer
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
            bool blocked = false;
            for (long long qq = qa; qq < r && !blocked; ++qq) {
                if (!(hbuf[(size_t)(qq - r0 + gr) * kDetCols + tid] == v)) continue;
                for (int j = -gd; j <= gd; ++j)
                    if (__ldg(S + qq * n + det_wrap(c + j, n)) == v) { blocked = true; break; }
            }
            for (int j = 1; j <= gd && !blocked; ++j) {
                const long long kl = c - j, kr = c + j;
                if (kl >= 0 && (kl >= c0 ? vbuf[(size_t)q * kDetCols + tid - j] : __ldg(S + r * n + kl)) == v) blocked = true;
                if (kr >= n && __ldg(S + r * n + (kr - n)) == v) blocked = true;
            }
            if (!blocked) cand[atomicAdd(&ncand, 1u)] = (unsigned)(q * kDetCols + tid);
        }
    }
    __syncthreads();

    // noise of every candidate: G candidates per warp, lane sub * rows + i sums training row r - R + i of candidate sub
    // (rows > 32: one candidate, lane i sums rows i, i + 32, i + 64); the row sums are then added in ascending row
    const unsigned cnt = ncand;
    const int rows = 2 * R + 1;
    const int G = rows <= 32 ? 32 / rows : 1;
    const int sub = G > 1 ? lane / rows : 0;
    const int ri0 = G > 1 ? lane - sub * rows : lane;
    for (unsigned b0 = (unsigned)(warp * G); b0 < cnt; b0 += (unsigned)(kDetWarps * G)) {
        const unsigned ci = b0 + (unsigned)sub;
        const bool have = sub < G && ci < cnt;
        const unsigned li = have ? cand[ci] : 0u;
        const int q = (int)(li / kDetCols), cl = (int)(li % kDetCols);
        const long long r = r0 + q;
        double rs0 = 0.0, rs1 = 0.0, rs2 = 0.0;
        unsigned rc0 = 0u, rc1 = 0u, rc2 = 0u;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int ri = ri0 + 32 * s;
            if (!have || ri >= rows || (G > 1 && s > 0)) continue;
            const long long rr = r - R + ri;
            if (rr < 0 || rr >= d) continue;
            const bool guard_row = ri - R >= -gr && ri - R <= gr;
            unsigned cc = 0u;
            double x;
            if (staged) {
                const T* src = region + (size_t)(rr - (r0 - R)) * L.pitch + cl + C;
                x = cfar_row_sum([&](int j) { return src[j]; }, C, gd, guard_row, cc);
            } else {
                const T* row = S + rr * n;
                const long long cg = c0 + cl;
                x = cfar_row_sum([&](int j) { return __ldg(row + det_wrap(cg + j, n)); }, C, gd, guard_row, cc);
            }
            if (s == 0) { rs0 = x; rc0 = cc; } else if (s == 1) { rs1 = x; rc1 = cc; } else { rs2 = x; rc2 = cc; }
        }
        double sum = 0.0;
        unsigned m = 0u;
        for (int i = 0; i < rows; ++i) {
            const int s = i >> 5;
            const int src = G > 1 ? sub * rows + i : (i & 31);
            const double x = __shfl_sync(0xffffffffu, s == 0 ? rs0 : (s == 1 ? rs1 : rs2), src);
            const unsigned y = __shfl_sync(0xffffffffu, s == 0 ? rc0 : (s == 1 ? rc1 : rc2), src);
            sum = __dadd_rn(sum, x);
            m += y;
        }
        if (have && ri0 == 0) { noise[ci] = cfar_noise_of(sum, m); mcnt[ci] = m; }
    }
    __syncthreads();

    // the qualifying candidates: v > scale * noise over m > 0 training cells
    for (unsigned i = tid; i < cnt; i += kDetCols) {
        const double v = (double)vbuf[cand[i]];
        if (mcnt[i] > 0u && v > __dmul_rn(scale, noise[i])) qual[atomicAdd(&nqual, 1u)] = i;
    }
    __syncthreads();

    // this tile's best kmax, then the pair's floor
    const unsigned nq = nqual;
    auto key = [&](long long i, unsigned long long& h, unsigned long long& l) {
        const unsigned li = cand[qual[i]];
        h = (unsigned long long)__double_as_longlong((double)vbuf[li]);
        l = ~(unsigned long long)((r0 + li / kDetCols) * n + c0 + li % kDetCols);
    };
    unsigned long long th = 0ull, tl = 0ull;
    if (nq > kmax) {
        det_select_kth(key, (long long)nq, kmax, hist, &sel);
        th = sel.oh; tl = sel.ol;
        if (tid == 0) atomicMax(my_ctr + 1, th);
    }
    const unsigned long long fl = *reinterpret_cast<volatile unsigned long long*>(my_ctr + 1);
    unsigned mine = 0;
    for (unsigned i = tid; i < nq; i += kDetCols) {
        unsigned long long h, l;
        key(i, h, l);
        if (det_key_ge(h, l, th, tl) && h >= fl) ++mine;
    }
    if (mine) atomicAdd(&nkeep, mine);
    __syncthreads();
    if (tid == 0 && nkeep) base = atomicAdd(my_ctr, (unsigned long long)nkeep);
    __syncthreads();
    if (nkeep == 0u) return;
    CfarEntry* E = entries + pair * cap + base;
    for (unsigned i = tid; i < nq; i += kDetCols) {
        unsigned long long h, l;
        key(i, h, l);
        if (det_key_ge(h, l, th, tl) && h >= fl) {
            const unsigned ci = qual[i];
            E[atomicAdd(&wpos, 1u)] = CfarEntry{h, ~l, (unsigned long long)__double_as_longlong(noise[ci]),
                                                (unsigned long long)mcnt[ci]};
        }
    }
}

// ---- pass 2 --------------------------------------------------------------------------------------------------------
// one CTA per pair: out [p][kmax], counts [p]
template <typename T>
__global__ void __launch_bounds__(kDetMergeThreads) caf_cfar_merge_kernel(
        const T* __restrict__ surf, long long d, long long n, const double* __restrict__ freqs,
        const CfarEntry* __restrict__ entries, long long cap, const unsigned long long* __restrict__ ctr, unsigned kmax,
        CfarOut* __restrict__ out, unsigned long long* __restrict__ counts) {
    __shared__ CfarEntry win[kDetMaxK];
    __shared__ unsigned hist[256];
    __shared__ DetSelState sel;
    __shared__ unsigned nwin;
    const int tid = threadIdx.x;
    const long long pair = blockIdx.x;
    const T* S = surf + pair * d * n;
    const CfarEntry* E = entries + pair * cap;
    const long long N = (long long)ctr[2 * pair];
    if (tid == 0) nwin = 0u;
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
    for (unsigned i = m + tid; i < P; i += blockDim.x) win[i] = CfarEntry{0ull, ~0ull, 0ull, 0ull};   // sorts last
    __syncthreads();
    // bitonic sort, best key first
    for (unsigned kk = 2; kk <= P; kk <<= 1)
        for (unsigned j = kk >> 1; j > 0; j >>= 1) {
            for (unsigned i = tid; i < P; i += blockDim.x) {
                const unsigned x = i ^ j;
                if (x > i) {
                    const CfarEntry a = win[i], b = win[x];
                    const bool a_first = a.vbits > b.vbits || (a.vbits == b.vbits && a.flat < b.flat);
                    if (((i & kk) == 0) != a_first) { win[i] = b; win[x] = a; }
                }
            }
            __syncthreads();
        }
    CfarOut* O = out + pair * (long long)kmax;
    for (unsigned i = tid; i < kmax; i += blockDim.x) {
        CfarOut o;
        DetectOut& e = o.det;
        if (i < m) {
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
            e.value = v; e.freq_hz = fr; e.doppler_idx = (unsigned long long)r; e.delay_idx = (unsigned long long)k;
            e.lag_samples = __dadd_rn((double)(2 * k < n ? k : k - n), dk);
            e.freq_hz_interp = fi;
            o.noise = __longlong_as_double((long long)win[i].noise_bits);
            o.train_cells = win[i].m;
        } else {
            e.value = 0.0; e.freq_hz = 0.0; e.doppler_idx = ~0ull; e.delay_idx = 0ull; e.lag_samples = 0.0; e.freq_hz_interp = 0.0;
            o.noise = 0.0; o.train_cells = 0ull;
        }
        O[i] = o;
    }
    if (tid == 0) counts[pair] = m;
}

// ---- the dense noise map ---------------------------------------------------------------------------------------------
// noise [p][d][n] doubles (NaN where m = 0); one thread per cell, grid-stride
template <typename T>
__global__ void __launch_bounds__(256) caf_cfar_noise_kernel(
        const T* __restrict__ surf, long long p, long long d, long long n, int gr, int gd, int R, int C,
        double* __restrict__ noise) {
    const long long cells = p * d * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (long long)gridDim.x * blockDim.x) {
        const long long pr = i / n, c = i - pr * n, pair = pr / d, r = pr - pair * d;
        const T* S = surf + pair * d * n;
        const long long ra = r - R > 0 ? r - R : 0, rb = r + R < d - 1 ? r + R : d - 1;
        double sum = 0.0;
        unsigned m = 0u;
        for (long long rr = ra; rr <= rb; ++rr) {
            const T* row = S + rr * n;
            const bool guard_row = rr - r >= -gr && rr - r <= gr;
            sum = __dadd_rn(sum, cfar_row_sum([&](int j) { return __ldg(row + det_wrap(c + j, n)); }, C, gd, guard_row, m));
        }
        noise[i] = cfar_noise_of(sum, m);
    }
}

}  // namespace caf
