// caf_integrate.cuh -- non-coherent integration of CAF surfaces over K signal segments (caf_b200_integrate_*_dev,
// caf_b200_surface_create_integrated_*), include/caf_b200.h.
//
// The contract (DESIGN.md section 13): S[r][c] = (((+0.0 + s_0[r][c]) + s_1[r][c]) + ...) + s_{K-1}[r][c] in double, f32
// cells widened first (exact), the adds in ascending k and nothing reassociated -- so the sum does not depend on how the
// segments are chunked, and a numpy loop `acc += s_k.astype(np.float64)` gives the same bits.  Row peaks and find_peak
// follow the surface calls' rules (mod.rs:141-153, 31-42) in double.
//
// The host loop (caf_b200.cu, run_integrate_dev) computes the segments' surfaces chunk by chunk with the unchanged batch
// path into a scratch buffer [c][d][n] and runs caf_integrate_kernel after each chunk: it adds the chunk's c surfaces into
// the caller's double surface in ascending k, starting from +0.0 on the first chunk (the caller's buffer is not read
// then), and on the last chunk leaves every row's first maximum: one partial per block and a per-row ticket, as
// caf_large_gather_top does, so that rows of up to 2^20 cells spread over many blocks.
#pragma once
#include "caf_kernels.cuh"

namespace caf {

constexpr int kIntThreads = 256;
constexpr int kIntPerThread = 4;
constexpr int kIntCells = kIntThreads * kIntPerThread;   // cells of one row per block

// Arguments of one chunk.  Block b covers cells [part * kIntCells, (part + 1) * kIntCells) of row b / parts; thread t
// takes cells part * kIntCells + t + kIntThreads * j, j = 0..3 (every warp load is 32 consecutive cells).
template <typename T>
struct IntegrateArgs {
    const T* seg;                        // [c][d][n] the chunk's segment surfaces
    double* acc;                         // [d][n] the integrated surface (caller's)
    long long d, n;
    int c;                               // segments in this chunk
    int parts;                           // blocks per row = ceil(n / kIntCells)
    int first;                           // start from +0.0 instead of reading acc
    int last;                            // leave the row maxima (row_peak_* non-null)
    double* part_val;                    // [d][parts] partial row maxima (parts > 1)
    int* part_idx;
    unsigned int* row_ticket;            // [d] zero before the launch, zero again after it
    double* row_peak_val;                // [d]
    unsigned long long* row_peak_idx;    // [d]
};

template <typename T>
__global__ void __launch_bounds__(kIntThreads) caf_integrate_kernel(const IntegrateArgs<T> a) {
    const long long row = (long long)blockIdx.x / a.parts;
    const int part = (int)((long long)blockIdx.x - row * a.parts);
    const long long stride = a.d * a.n;
    const long long base = row * a.n;
    const int c0 = part * kIntCells + (int)threadIdx.x;
    double s[kIntPerThread];
#pragma unroll
    for (int j = 0; j < kIntPerThread; ++j) {
        const int cell = c0 + kIntThreads * j;
        s[j] = (a.first || cell >= a.n) ? 0.0 : a.acc[base + cell];
    }
    const T* src = a.seg + base;
    for (int k = 0; k < a.c; ++k) {
        T v[kIntPerThread];
#pragma unroll
        for (int j = 0; j < kIntPerThread; ++j) {
            const int cell = c0 + kIntThreads * j;
            v[j] = cell < a.n ? __ldcs(src + cell) : (T)0;         // read once: streaming
        }
#pragma unroll
        for (int j = 0; j < kIntPerThread; ++j) s[j] = __dadd_rn(s[j], (double)v[j]);   // ascending k, no reassociation
        src += stride;
    }
    double best = 0.0;
    int bidx = 0;
#pragma unroll
    for (int j = 0; j < kIntPerThread; ++j) {
        const int cell = c0 + kIntThreads * j;
        if (cell < a.n) {
            a.acc[base + cell] = s[j];
            if (s[j] > best) { best = s[j]; bidx = cell; }          // ascending cells, strict >: the first maximum (mod.rs:148)
        }
    }
    if (!a.last) return;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, off);
        const int oi = __shfl_xor_sync(0xffffffffu, bidx, off);
        amax_take<double>(best, bidx, ov, oi);
    }
    __shared__ double sv[kIntThreads / 32];
    __shared__ int si[kIntThreads / 32];
    __shared__ unsigned int s_last;
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = bidx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int q = 1; q < kIntThreads / 32; ++q) amax_take<double>(best, bidx, sv[q], si[q]);
        if (a.parts == 1) {
            if (!(best > 0.0)) bidx = 0;
            a.row_peak_val[row] = best;
            a.row_peak_idx[row] = (unsigned long long)bidx;
            return;
        }
        a.part_val[row * a.parts + part] = best;
        a.part_idx[row * a.parts + part] = bidx;
        __threadfence();
        const unsigned int ticket = atomicAdd(a.row_ticket + row, 1u);
        s_last = (ticket == (unsigned int)a.parts - 1u) ? 1u : 0u;
    }
    if (a.parts == 1) return;
    __syncthreads();
    if (s_last && threadIdx.x < 32) {
        // the last block of this row folds the partials: first strict-> maximum (mod.rs:141-153)
        __threadfence();
        double b2 = 0.0;
        int i2 = 0;
        for (int q = threadIdx.x; q < a.parts; q += 32)
            amax_take<double>(b2, i2, __ldcg(a.part_val + row * a.parts + q), __ldcg(a.part_idx + row * a.parts + q));
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, b2, off);
            const int oi = __shfl_xor_sync(0xffffffffu, i2, off);
            amax_take<double>(b2, i2, ov, oi);
        }
        if (threadIdx.x == 0) {
            if (!(b2 > 0.0)) i2 = 0;
            a.row_peak_val[row] = b2;
            a.row_peak_idx[row] = (unsigned long long)i2;
            a.row_ticket[row] = 0u;          // self-resetting for the next call
        }
    }
}

}  // namespace caf
