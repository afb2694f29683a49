// gc_kernel.cuh -- the sm_100a kernels of gen.gc (DESIGN.md 2b).
//
// gc_layer_kernel: one launch per layer.  A CTA takes a chunk of columns (kGcThreads threads x kGcVec
// double2) for a group of the layer's rows; per row it adds the input rows in CSR order in binary64,
// halves the sum (exact), adds the seed 1 in the row's own column and writes the row to its frontier slot
// and/or (streaming store: never read again on the device) its output-block row.  The order of the
// additions is part of the result's contract: ((0 + in_1) + in_2) + ..., then 1/2 * sum + seed.
//
// gc_gather_kernel: a 32 x 32 tile of the output block, with duplicates of either list expanded, to a
// staging buffer in the layout of the caller's matrix (row- or column-major, float64 or float32),
// transposed through shared memory where the output block's rows are the matrix's columns.
#pragma once
#include <cstdint>

namespace genlib {

#if defined(GENLIB_SOFTCHECK)       // record the source line of the FIRST violated bound in the error word, go on
#define GC_CHECK(cond) do { if (!(cond)) atomicCAS(a.err, 0, 100000 + __LINE__); } while (0)
#else
#define GC_CHECK(cond) do { } while (0)
#endif

constexpr int kGcThreads = 256;
constexpr int kGcVec = 2;                         // double2 per thread and row
constexpr int kGcChunk = kGcThreads * kGcVec;     // double2 per CTA and row

struct GcLayerArgs {
    double2 *F;                 // frontier: capacity rows of w2 double2
    double2 *O;                 // output block: n_targets rows of w2 double2
    int64_t w2;                 // double2 per row (the device's columns, padded to even)
    int32_t width;              // the device's columns
    int32_t col_lo;             // unique index of the device's first column
    int32_t n_rows;
    int64_t capacity, n_targets;
    const int32_t *row_slot, *row_seed, *row_out;
    const int64_t *in_ptr;      // the layer's n_rows + 1 entries (global offsets)
    const int32_t *in_slot;
    int32_t *err;               // GENLIB_SOFTCHECK: first violated bound
};

__global__ void __launch_bounds__(kGcThreads) gc_layer_kernel(GcLayerArgs a) {
    const int64_t c0 = (int64_t)blockIdx.x * kGcChunk + threadIdx.x;
    for (int32_t r = blockIdx.y; r < a.n_rows; r += gridDim.y) {
        const int64_t p0 = a.in_ptr[r], p1 = a.in_ptr[r + 1];
        double2 acc[kGcVec];
#pragma unroll
        for (int u = 0; u < kGcVec; u++) acc[u] = make_double2(0.0, 0.0);
        int64_t p = p0;
        for (; p + 1 < p1; p += 2) {               // two input rows in flight, added in CSR order
            const int32_t s0 = a.in_slot[p], s1 = a.in_slot[p + 1];
            GC_CHECK(s0 >= 0 && s0 < a.capacity && s1 >= 0 && s1 < a.capacity);
            const double2 *x0 = a.F + (int64_t)s0 * a.w2, *x1 = a.F + (int64_t)s1 * a.w2;
            double2 v0[kGcVec], v1[kGcVec];
#pragma unroll
            for (int u = 0; u < kGcVec; u++) {
                const int64_t c = c0 + u * kGcThreads;
                v0[u] = v1[u] = make_double2(0.0, 0.0);
                if (c < a.w2) { v0[u] = __ldg(x0 + c); v1[u] = __ldg(x1 + c); }
            }
#pragma unroll
            for (int u = 0; u < kGcVec; u++) {
                acc[u].x += v0[u].x; acc[u].y += v0[u].y;
                acc[u].x += v1[u].x; acc[u].y += v1[u].y;
            }
        }
        if (p < p1) {
            const int32_t s0 = a.in_slot[p];
            GC_CHECK(s0 >= 0 && s0 < a.capacity);
            const double2 *x0 = a.F + (int64_t)s0 * a.w2;
#pragma unroll
            for (int u = 0; u < kGcVec; u++) {
                const int64_t c = c0 + u * kGcThreads;
                if (c < a.w2) { const double2 v = __ldg(x0 + c); acc[u].x += v.x; acc[u].y += v.y; }
            }
        }
        const int32_t rs = a.row_seed[r];
        const int32_t seed = rs >= 0 ? rs - a.col_lo : -1;  // the row's own column on this device, if any
        const int32_t slot = a.row_slot[r], orow = a.row_out[r];
        GC_CHECK(slot < a.capacity && orow < a.n_targets);
#pragma unroll
        for (int u = 0; u < kGcVec; u++) {
            const int64_t c = c0 + u * kGcThreads;
            if (c >= a.w2) continue;
            double2 v = make_double2(0.5 * acc[u].x, 0.5 * acc[u].y);
            if (seed >= 0 && seed < a.width && (seed >> 1) == c) {
                if (seed & 1) v.y += 1.0; else v.x += 1.0;
            }
            if (slot >= 0) a.F[(int64_t)slot * a.w2 + c] = v;
            if (orow >= 0) __stcs(a.O + (int64_t)orow * a.w2 + c, v);
        }
    }
}

struct GcGatherArgs {
    const double *O;            // output block, rows of ws doubles
    int64_t ws;
    const int32_t *tgt_row;     // target list position -> output-block row
    const int32_t *col;         // column list position (the device's range) -> local column
    int32_t n_t, n_c;           // the block's target positions [t0, t0 + n_t), column positions [c0, c0 + n_c)
    int32_t t0, c0;
};

// stage (major x minor, minor contiguous): C_MAJOR = false: major = target, minor = column position;
// C_MAJOR = true: major = column position, minor = target.  Tiles of 32 x 32, 32 x 8 threads.
template <bool C_MAJOR, typename Out>
__global__ void __launch_bounds__(256) gc_gather_kernel(GcGatherArgs a, Out *stage) {
    __shared__ double tile[32][33];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int32_t cb = blockIdx.x * 32;                              // tile origin (relative to c0 / t0)
    const int32_t c = cb + tx;
    const int32_t lc = c < a.n_c ? a.col[a.c0 + c] : 0;
    for (int32_t tb = blockIdx.y * 32; tb < a.n_t; tb += gridDim.y * 32) {
        // read: lanes along the columns (the output block's rows are contiguous in columns)
        for (int k = ty; k < 32; k += 8) {
            const int32_t t = tb + k;
            if (t < a.n_t && c < a.n_c) tile[k][tx] = a.O[(int64_t)a.tgt_row[a.t0 + t] * a.ws + lc];
        }
        if (!C_MAJOR) {
            for (int k = ty; k < 32; k += 8) {
                const int32_t t = tb + k;
                if (t < a.n_t && c < a.n_c) stage[(int64_t)t * a.n_c + c] = (Out)tile[k][tx];
            }
            continue;
        }
        __syncthreads();
        // write: lanes along the targets
        for (int k = ty; k < 32; k += 8) {
            const int32_t cc = cb + k, t = tb + tx;
            if (t < a.n_t && cc < a.n_c) stage[(int64_t)cc * a.n_t + t] = (Out)tile[tx][k];
        }
        __syncthreads();
    }
}

}  // namespace genlib
