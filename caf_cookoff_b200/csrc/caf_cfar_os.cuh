// caf_cfar_os.cuh -- ordered-statistic CFAR detection on stored CAF surfaces (caf_b200_surface_detect_cfar_os /
// caf_b200_detect_cfar_os_*_dev) and its dense noise map (caf_b200_cfar_os_noise_*_dev), include/caf_b200.h.
//
// The contract (DESIGN.md section 11; oracle/cfar_os.py restates it in numpy): CA-CFAR's (caf_cfar.cuh) but for the noise
// estimate.  The training cells, m and N = (2R+1)(2C+1) - (2gr+1)(2gd+1) are CA's.  Each training value is widened to
// double and +0.0 is added (so -0.0 counts as +0.0); with k_m = ceil(rank * m / N) in 64-bit integers, noise is the k_m-th
// smallest of those m values -- an exact value, so every path gives the same bits -- and NaN when m = 0.  (r, k) is a
// detection when it is a local maximum under detect's rule with (gr, gd), m > 0 and v > scale * noise (correctly rounded).
//
// Pass 1 (caf_cfar_os_tiles_kernel): the tiles, staging, local-maximum rule, per-tile select and append of
//   caf_cfar_tiles_kernel, restated (calling shared steps changes the other tile kernels' code generation, DESIGN.md
//   section 10).  One warp takes one candidate and first COUNTS: it qualifies iff at least k_m of its training values x
//   have scale * x < v, which is exact because x -> RN(scale * x) is non-decreasing for scale > 0.  Only a qualifying
//   candidate then SELECTS its k_m-th smallest value, by an 8-bit radix select over order-preserving 64-bit keys with a
//   warp-private 256-bin histogram.  Both read the copy of the tile's training region that caf_cfar_tiles_kernel stages,
//   or the surface at the largest windows.  Entries are CfarEntry, so pass 2 is caf_cfar_merge_kernel.
// Map (caf_cfar_os_noise_kernel): one warp per cell, the same counting and selection, reading the surface.
#pragma once
#include <cstdint>
#include "caf_cfar.cuh"

namespace caf {

// pass 1's dynamic shared memory: caf_cfar_tiles_kernel's layout, then one 256-bin histogram per warp
template <typename T>
__host__ __device__ inline CfarTileLayout cfar_os_tile_layout(int tr, int gr, int gd, int R, int C, bool staged, int mx) {
    CfarTileLayout L = cfar_tile_layout<T>(tr, gr, gd, R, C, staged, mx);
    L.total += sizeof(unsigned) * 256 * kDetWarps;
    return L;
}

// Calls f(x) for the training values of one cell that fall to this lane, each widened to double with +0.0 added, NaN
// skipped.  The cell's training rows dr in [dlo, dhi] (offsets from its row, already clipped to the surface) times
// j in [-C, C] are taken in row-major order, lane-strided; get(dr, j) reads one of them.
template <typename Get, typename F>
__device__ __forceinline__ void os_cells(Get get, int dlo, int dhi, int C, int gr, int gd, int lane, F f) {
    const int w = 2 * C + 1;
    const int total = (dhi - dlo + 1) * w;
    int dr = dlo + lane / w, jj = lane % w;
    for (int t = lane; t < total; t += 32) {
        const int j = jj - C;
        if (!(dr >= -gr && dr <= gr && j >= -gd && j <= gd)) {
            const double x = __dadd_rn((double)get(dr, j), 0.0);
            if (x == x) f(x);
        }
        jj += 32;
        while (jj >= w) { jj -= w; ++dr; }
    }
}

// order-preserving keys of non-NaN doubles other than -0.0: unsigned order of the keys is numeric order of the values
__device__ __forceinline__ unsigned long long os_key(double x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double os_unkey(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// The km-th smallest (1-based, 1 <= km <= m) training value of one cell; every lane of the warp calls it with the same
// cells and gets the answer.  MSB first, 8 bits per step, in the warp's 256-word histogram hist; stops as soon as the
// step's bucket holds that value alone and fetches it.
template <typename Cells>
__device__ __forceinline__ double os_select(Cells cells, unsigned km, unsigned* hist, int lane) {
    unsigned long long prefix = 0ull, mask = 0ull;
    unsigned rem = km;
    bool done = false;
    for (int step = 0; step < 8 && !done; ++step) {
        const int sh = 56 - 8 * step;
#pragma unroll
        for (int b = 0; b < 8; ++b) hist[lane * 8 + b] = 0u;
        __syncwarp();
        cells([&](double x) {
            const unsigned long long key = os_key(x);
            if ((key & mask) == prefix) atomicAdd(&hist[(unsigned)(key >> sh) & 0xffu], 1u);
        });
        __syncwarp();
        unsigned b[8], s = 0u;               // lane q owns bins 8q ... 8q + 7, scanned from the bottom
#pragma unroll
        for (int j = 0; j < 8; ++j) { b[j] = hist[lane * 8 + j]; s += b[j]; }
        unsigned inc = s;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        const int q = __ffs(__ballot_sync(0xffffffffu, inc >= rem)) - 1;    // rem <= the bucket total
        unsigned dig = 0u, before = inc - s, cnt = 0u;
        bool found = false;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (!found && before + b[j] >= rem) { found = true; dig = (unsigned)(8 * lane + j); cnt = b[j]; }
            if (!found) before += b[j];
        }
        dig = __shfl_sync(0xffffffffu, dig, q);
        before = __shfl_sync(0xffffffffu, before, q);
        cnt = __shfl_sync(0xffffffffu, cnt, q);
        prefix |= (unsigned long long)dig << sh;
        mask |= 0xffull << sh;
        rem -= before;
        done = cnt == 1u;                    // the bucket holds the answer alone
        __syncwarp();
    }
    if (done && mask != ~0ull) {             // the prefix names one value: fetch the rest of it
        unsigned long long got = 0ull;
        cells([&](double x) {
            const unsigned long long key = os_key(x);
            if ((key & mask) == prefix) got = key;
        });
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long t = __shfl_xor_sync(0xffffffffu, got, o);
            got = t > got ? t : got;
        }
        prefix = got;
    }
    return os_unkey(prefix);
}

// k_m = ceil(rank * m / N)
__device__ __forceinline__ unsigned os_rank_of(unsigned rank, unsigned m, unsigned long long ntrain) {
    return (unsigned)(((unsigned long long)rank * m + ntrain - 1ull) / ntrain);
}

// ---- pass 1 --------------------------------------------------------------------------------------------------------
// surf [p][d][n]; grid = p * tiles_per_pair CTAs of kDetCols threads.  ctr [p][2] = (entries appended, floor value bits),
// zeroed before the launch; entries [p][cap].  mx = det_tile_max_maxima(tr, gr, gd), the candidate slots of a tile.
// BLOCK, row_lo, row_hi: as in det_tiles.
template <typename T, bool BLOCK>
__device__ __forceinline__ void cfar_os_tiles(
        const T* __restrict__ surf, long long d, long long n, int gr, int gd, int R, int C, int tr, bool staged, int mx,
        unsigned rank, unsigned long long ntrain, double scale, long long tiles_c, long long tiles_per_pair, unsigned kmax,
        long long cap, CfarEntry* __restrict__ entries, unsigned long long* __restrict__ ctr, long long row_lo,
        long long row_hi) {
    extern __shared__ __align__(16) unsigned char cfar_os_smem[];
    const CfarTileLayout L = cfar_os_tile_layout<T>(tr, gr, gd, R, C, staged, mx);
    T* hbuf = reinterpret_cast<T*>(cfar_os_smem);                         // [tr + 2 gr][kDetCols]
    T* vbuf = hbuf + (size_t)(tr + 2 * gr) * kDetCols;                   // [tr][kDetCols]
    const int W = kDetCols + 2 * gd;
    T* stage = vbuf + (size_t)tr * kDetCols;                              // [kDetWarps][W]
    T* region = reinterpret_cast<T*>(cfar_os_smem + L.region);           // [tr + 2R][pitch], cells c0 - C ...
    double* noise = reinterpret_cast<double*>(cfar_os_smem + L.noise);   // [mx]
    unsigned* mcnt = reinterpret_cast<unsigned*>(cfar_os_smem + L.mcnt); // [mx]
    unsigned* cand = reinterpret_cast<unsigned*>(cfar_os_smem + L.cand); // [mx]
    unsigned* qual = reinterpret_cast<unsigned*>(cfar_os_smem + L.qual); // [mx] positions in cand
    unsigned* hist = reinterpret_cast<unsigned*>(cfar_os_smem + L.hist); // [256]
    unsigned* whist = hist + 256;                                         // [kDetWarps][256]
    __shared__ unsigned ncand, nqual, nkeep, wpos;
    __shared__ unsigned long long base;
    __shared__ DetSelState sel;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long pair = (long long)blockIdx.x / tiles_per_pair;
    const long long t = (long long)blockIdx.x - pair * tiles_per_pair;
    const long long r0 = (BLOCK ? row_lo : 0ll) + (t / tiles_c) * tr, c0 = (t % tiles_c) * kDetCols;
    const long long rend = BLOCK ? row_hi : d;           // candidates stop here
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
        for (int q = 0; q < tr && r0 + q < rend; ++q) {
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

    // one warp per candidate: count, and select only for the qualifying ones
    const unsigned cnt = ncand;
    unsigned* wh = whist + (size_t)warp * 256;
    for (unsigned ci = (unsigned)warp; ci < cnt; ci += (unsigned)kDetWarps) {
        const unsigned li = cand[ci];
        const int q = (int)(li / kDetCols), cl = (int)(li % kDetCols);
        const long long r = r0 + q;
        const double v = (double)vbuf[li];
        const int dlo = (int)(r - R > 0 ? -R : -r), dhi = (int)(r + R < d ? R : d - 1 - r);
        auto cells = [&](auto f) {
            if (staged) {
                const T* src = region + (size_t)(r - (r0 - R)) * L.pitch + cl + C;
                os_cells([&](int dr, int j) { return src[(long long)dr * L.pitch + j]; }, dlo, dhi, C, gr, gd, lane, f);
            } else {
                const long long cg = c0 + cl;
                os_cells([&](int dr, int j) { return __ldg(S + (r + dr) * n + det_wrap(cg + j, n)); }, dlo, dhi, C, gr,
                         gd, lane, f);
            }
        };
        unsigned mc = 0u, below = 0u;
        cells([&](double x) { ++mc; if (__dmul_rn(scale, x) < v) ++below; });
        mc = __reduce_add_sync(0xffffffffu, mc);
        below = __reduce_add_sync(0xffffffffu, below);
        if (mc == 0u) continue;
        const unsigned km = os_rank_of(rank, mc, ntrain);
        if (below < km) continue;
        const double nz = os_select(cells, km, wh, lane);
        if (lane == 0) { noise[ci] = nz; mcnt[ci] = mc; qual[atomicAdd(&nqual, 1u)] = ci; }
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

template <typename T>
__global__ void __launch_bounds__(kDetCols) caf_cfar_os_tiles_kernel(
        const T* __restrict__ surf, long long d, long long n, int gr, int gd, int R, int C, int tr, bool staged, int mx,
        unsigned rank, unsigned long long ntrain, double scale, long long tiles_c, long long tiles_per_pair, unsigned kmax,
        long long cap, CfarEntry* __restrict__ entries, unsigned long long* __restrict__ ctr) {
    cfar_os_tiles<T, false>(surf, d, n, gr, gd, R, C, tr, staged, mx, rank, ntrain, scale, tiles_c, tiles_per_pair, kmax,
                            cap, entries, ctr, 0, 0);
}

// rows [row_lo, row_hi) of a block of d rows
template <typename T>
__global__ void __launch_bounds__(kDetCols) caf_cfar_os_tiles_rows_kernel(
        const T* __restrict__ surf, long long d, long long n, int gr, int gd, int R, int C, int tr, bool staged, int mx,
        unsigned rank, unsigned long long ntrain, double scale, long long tiles_c, long long tiles_per_pair, unsigned kmax,
        long long cap, CfarEntry* __restrict__ entries, unsigned long long* __restrict__ ctr, long long row_lo,
        long long row_hi) {
    cfar_os_tiles<T, true>(surf, d, n, gr, gd, R, C, tr, staged, mx, rank, ntrain, scale, tiles_c, tiles_per_pair, kmax,
                           cap, entries, ctr, row_lo, row_hi);
}

// ---- the dense noise map ---------------------------------------------------------------------------------------------
// noise [p][d][n] doubles (NaN where m = 0); one warp per cell, grid-stride; blocks of kCfarOsMapThreads
constexpr int kCfarOsMapThreads = 256;

template <typename T>
__global__ void __launch_bounds__(kCfarOsMapThreads) caf_cfar_os_noise_kernel(
        const T* __restrict__ surf, long long p, long long d, long long n, int gr, int gd, int R, int C, unsigned rank,
        unsigned long long ntrain, double* __restrict__ noise) {
    __shared__ unsigned whist[kCfarOsMapThreads / 32][256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long cells = p * d * n;
    const long long warps = (long long)gridDim.x * (kCfarOsMapThreads / 32);
    for (long long i = (long long)blockIdx.x * (kCfarOsMapThreads / 32) + warp; i < cells; i += warps) {
        const long long pr = i / n, c = i - pr * n, pair = pr / d, r = pr - pair * d;
        const T* S = surf + pair * d * n;
        const int dlo = (int)(r - R > 0 ? -R : -r), dhi = (int)(r + R < d ? R : d - 1 - r);
        auto cellf = [&](auto f) {
            os_cells([&](int dr, int j) { return __ldg(S + (r + dr) * n + det_wrap(c + j, n)); }, dlo, dhi, C, gr, gd,
                     lane, f);
        };
        unsigned mc = 0u;
        cellf([&](double) { ++mc; });
        mc = __reduce_add_sync(0xffffffffu, mc);
        const double nz = mc ? os_select(cellf, os_rank_of(rank, mc, ntrain), whist[warp], lane)
                             : __longlong_as_double(0x7ff8000000000000ll);
        if (lane == 0) noise[i] = nz;
    }
}

}  // namespace caf
