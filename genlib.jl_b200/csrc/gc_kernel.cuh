// gc_kernel.cuh -- the sm_100a kernels of gen.gc, gen.occ, gen.rec and gen.findMRCA (DESIGN.md 2b, 2c, 2d).
//
// gc_layer_kernel<Op>: one launch per layer.  A CTA takes a chunk of columns (threads per row x kGcVec
// 16-byte vectors) for a group of the layer's rows -- several rows per CTA when rows are narrow; per row it
// combines the input rows in CSR order, finishes the row with the seed in the row's own column and writes
// it to its frontier slot and/or (streaming store: never read again by a layer) its output-block row.  For
// gen.gc the order of the additions is part of the result's contract: ((0 + in_1) + in_2) + ..., then
// 1/2 * sum + seed.  gen.occ adds counts with saturation, gen.rec ORs bit rows, the meioses of gen.findMRCA
// take the minimum of saturating uint16 sums: all three are order-free.
//
// gc_row_reduce_kernel / gc_col_reduce_kernel: the row sums of gen.occ(typeOcc = "TOTAL") and the counts of
// gen.rec, one pass over the output block, so the matrix never leaves the device.
//
// gc_group_reduce_kernel: gen.gcGroups with the target side grouped -- every group's output-block rows summed
// into one row, so only a groups x columns block is gathered.
//
// gc_gather_kernel: a 32 x 32 tile of the output block, with duplicates of either list expanded, to a
// staging buffer in the layout of the caller's matrix (row- or column-major; float64, float32 or int64; uint16
// distances widen to int64),
// transposed through shared memory where the output block's rows are the matrix's columns.
#pragma once
#include <cstdint>
#include <type_traits>

namespace genlib {

#if defined(GENLIB_SOFTCHECK)       // record the source line of the FIRST violated bound in the error word, go on
#define GC_CHECK(cond) do { if (!(cond)) atomicCAS(a.err, 0, 100000 + __LINE__); } while (0)
#else
#define GC_CHECK(cond) do { } while (0)
#endif

constexpr int kGcThreads = 256;
constexpr int kGcThreadsLog2 = 8;
static_assert(1 << kGcThreadsLog2 == kGcThreads, "kGcThreadsLog2");
constexpr int kGcVec = 2;                         // 16-byte vectors per thread and row
constexpr unsigned long long kOccSat = 1ull << 63;   // gen.occ: a path count that does not fit an Int64

// saturating non-negative addition, capped at kOccSat (both operands <= kOccSat): associative and
// commutative, so a saturated count is the same whatever the order of the sums
__device__ __forceinline__ unsigned long long sat_add(unsigned long long a, unsigned long long b) {
    const unsigned long long s = a + b;
    return (s < a || s > kOccSat) ? kOccSat : s;
}
__device__ __forceinline__ unsigned long long sat_mul(unsigned long long a, uint32_t w) {
    if (w == 1 || a == 0) return a;
    return a > kOccSat / w ? kOccSat : a * w;
}

// The three row operations of the layer kernel: row = finish(in_1 + in_2 + ..., seed), inputs in CSR order.
struct GcOpHalfSum {            // gen.gc: binary64, seed + 1/2 * (((0 + in_1) + in_2) + ...)
    using V = double2;
    static constexpr int kColsPerVec = 2;
    __device__ static V zero() { return make_double2(0.0, 0.0); }
    __device__ static void add(V &a, V x) { a.x += x.x; a.y += x.y; }
    __device__ static V finish(V a, int64_t c, int32_t seed) {
        V v = make_double2(0.5 * a.x, 0.5 * a.y);
        if (seed >= 0 && (seed >> 1) == c) { if (seed & 1) v.y += 1.0; else v.x += 1.0; }
        return v;
    }
};
struct GcOpCount {              // gen.occ: path counts, saturating uint64 sum + seed 1
    using V = ulonglong2;
    static constexpr int kColsPerVec = 2;
    __device__ static V zero() { return make_ulonglong2(0, 0); }
    __device__ static void add(V &a, V x) { a.x = sat_add(a.x, x.x); a.y = sat_add(a.y, x.y); }
    __device__ static V finish(V a, int64_t c, int32_t seed) {
        if (seed >= 0 && (seed >> 1) == c) { if (seed & 1) a.y = sat_add(a.y, 1); else a.x = sat_add(a.x, 1); }
        return a;
    }
};
struct GcOpReach {              // gen.rec: reachability, 64 columns per uint64 word, OR + seed bit
    using V = ulonglong2;
    static constexpr int kColsPerVec = 128;
    __device__ static V zero() { return make_ulonglong2(0, 0); }
    __device__ static void add(V &a, V x) { a.x |= x.x; a.y |= x.y; }
    __device__ static V finish(V a, int64_t c, int32_t seed) {
        if (seed >= 0 && (seed >> 7) == c) {
            const unsigned long long bit = 1ull << (seed & 63);
            if (seed & 64) a.y |= bit; else a.x |= bit;
        }
        return a;
    }
};

// gen.findMRCA / gen.findDistance: the shortest descent path in the (min, +1) semiring, eight uint16 distances
// per vector, 0xFFFF = unreachable.  +1 saturates at 0xFFFF, so an unreachable input stays unreachable; the
// host refuses plans of 0xFFFF layers or more, so a reachable distance (< layers) never meets the sentinel.
// Descending the inputs are the parents and the columns ancestors, ascending the children and the columns
// probands: the same rules give d(ancestor, proband) both ways.
constexpr uint16_t kMeiosesNone = 0xFFFF;
struct GcOpMinPlus {
    using V = uint4;
    static constexpr int kColsPerVec = 8;
    __device__ static V zero() { return make_uint4(~0u, ~0u, ~0u, ~0u); }
    __device__ static void add(V &a, V x) {
        constexpr unsigned one = 0x00010001u;
        a.x = __vminu2(a.x, __vaddus2(x.x, one)); a.y = __vminu2(a.y, __vaddus2(x.y, one));
        a.z = __vminu2(a.z, __vaddus2(x.z, one)); a.w = __vminu2(a.w, __vaddus2(x.w, one));
    }
    __device__ static V finish(V a, int64_t c, int32_t seed) {
        if (seed >= 0 && (seed >> 3) == c) {
            const unsigned keep = (seed & 1) ? 0x0000FFFFu : 0xFFFF0000u;   // d(p, p) = 0
            switch ((seed >> 1) & 3) {
                case 0: a.x &= keep; break;
                case 1: a.y &= keep; break;
                case 2: a.z &= keep; break;
                default: a.w &= keep; break;
            }
        }
        return a;
    }
};

struct GcLayerArgs {
    void *F;                    // frontier: capacity rows of w2 16-byte vectors
    void *O;                    // output block: n_targets rows of w2 vectors
    int64_t w2;                 // vectors per row (the device's columns, padded to 16 bytes)
    int32_t width;              // the device's columns
    int32_t col_lo;             // unique index of the device's first column
    int32_t n_rows;
    int32_t tpr_log2;           // threads per row = 1 << tpr_log2 (<= kGcThreads): a CTA takes several narrow rows
    int64_t capacity, n_targets;
    const int32_t *row_slot, *row_seed, *row_out;
    const int64_t *in_ptr;      // the layer's n_rows + 1 entries (global offsets)
    const int32_t *in_slot;
    int32_t *err;               // GENLIB_SOFTCHECK: first violated bound
};

// Threads per row for rows of w2 vectors: the fewest that cover the row with kGcVec vectors each (at most
// kGcThreads; wider rows take several CTAs along x).
inline int gc_tpr_log2(int64_t w2) {
    int l = 0;
    while (l < kGcThreadsLog2 && (int64_t)(1 << l) * kGcVec < w2) l++;
    return l;
}

// WIDE: a row takes the whole CTA (tpr_log2 == kGcThreadsLog2), with the mapping known at compile time --
// the wide rows of gc and occ on large pedigrees run exactly the code they ran before narrow rows existed.

template <typename Op, bool WIDE>
__global__ void __launch_bounds__(kGcThreads) gc_layer_kernel(GcLayerArgs a) {
    using V = typename Op::V;
    V *F = static_cast<V *>(a.F), *O = static_cast<V *>(a.O);
    const int lg = WIDE ? kGcThreadsLog2 : a.tpr_log2;
    const int tpr = 1 << lg, rpc = kGcThreads >> lg;                      // threads per row, rows per CTA
    // WIDE: the row index is blockIdx.y, uniform over the CTA, so the row's indices load once per CTA
    const int lane = WIDE ? (int)threadIdx.x : (int)(threadIdx.x & (tpr - 1));
    const int32_t r0 = WIDE ? (int32_t)blockIdx.y : (int32_t)(blockIdx.y * rpc + (threadIdx.x >> lg));
    const int64_t c0 = (int64_t)blockIdx.x * tpr * kGcVec + lane;
    for (int32_t r = r0; r < a.n_rows; r += gridDim.y * rpc) {
        const int64_t p0 = a.in_ptr[r], p1 = a.in_ptr[r + 1];
        V acc[kGcVec];
#pragma unroll
        for (int u = 0; u < kGcVec; u++) acc[u] = Op::zero();
        int64_t p = p0;
        for (; p + 1 < p1; p += 2) {               // two input rows in flight, added in CSR order
            const int32_t s0 = a.in_slot[p], s1 = a.in_slot[p + 1];
            GC_CHECK(s0 >= 0 && s0 < a.capacity && s1 >= 0 && s1 < a.capacity);
            const V *x0 = F + (int64_t)s0 * a.w2, *x1 = F + (int64_t)s1 * a.w2;
            V v0[kGcVec], v1[kGcVec];
#pragma unroll
            for (int u = 0; u < kGcVec; u++) {
                const int64_t c = c0 + u * tpr;
                v0[u] = v1[u] = Op::zero();
                if (c < a.w2) { v0[u] = __ldg(x0 + c); v1[u] = __ldg(x1 + c); }
            }
#pragma unroll
            for (int u = 0; u < kGcVec; u++) { Op::add(acc[u], v0[u]); Op::add(acc[u], v1[u]); }
        }
        if (p < p1) {
            const int32_t s0 = a.in_slot[p];
            GC_CHECK(s0 >= 0 && s0 < a.capacity);
            const V *x0 = F + (int64_t)s0 * a.w2;
#pragma unroll
            for (int u = 0; u < kGcVec; u++) {
                const int64_t c = c0 + u * tpr;
                if (c < a.w2) Op::add(acc[u], __ldg(x0 + c));
            }
        }
        const int32_t rs = a.row_seed[r];
        int32_t seed = rs >= 0 ? rs - a.col_lo : -1;         // the row's own column on this device, if any
        if (seed >= a.width) seed = -1;
        const int32_t slot = a.row_slot[r], orow = a.row_out[r];
        GC_CHECK(slot < a.capacity && orow < a.n_targets);
#pragma unroll
        for (int u = 0; u < kGcVec; u++) {
            const int64_t c = c0 + u * tpr;
            if (c >= a.w2) continue;
            const V v = Op::finish(acc[u], c, seed);
            if (slot >= 0) F[(int64_t)slot * a.w2 + c] = v;
            if (orow >= 0) __stcs(O + (int64_t)orow * a.w2 + c, v);
        }
    }
}

// ---- reductions of the output block (gen.occ typeOcc = "TOTAL", gen.rec), one pass, after the last layer.
// Row reduction (the block's rows are the ancestors, its columns the device's probands): one warp per row,
// every column weighted by how often the device's part of the proband list names it.
//   REACH: out[t] = sum over set bits b of wt(b), with the weights as masks: popc(x & m1) counts every listed
//          column once, the bits of x & m2 (named twice or more) add wt(b) - 1 each
//   else:  out[t] = saturating sum of wt[c] * O[t][c]
struct GcRowReduceArgs {
    const ulonglong2 *O;
    int64_t w2;                 // vectors per row
    int32_t n_rows;
    const uint32_t *wt;         // weight per column (2 * w2 entries; padding 0)
    const unsigned long long *m1, *m2;   // REACH: masks per word (2 * w2 entries)
    unsigned long long *out;    // n_rows
};

template <bool REACH>
__global__ void __launch_bounds__(256) gc_row_reduce_kernel(GcRowReduceArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (t >= a.n_rows) return;
    const ulonglong2 *row = a.O + t * a.w2;
    unsigned long long s = 0;
    for (int64_t v = lane; v < a.w2; v += 32) {
        const ulonglong2 x = __ldcs(row + v);
        if (REACH) {
            unsigned long long add = (unsigned long long)(__popcll(x.x & a.m1[2 * v]) + __popcll(x.y & a.m1[2 * v + 1]));
            for (int h = 0; h < 2; h++) {
                for (unsigned long long m = (h ? x.y : x.x) & a.m2[2 * v + h]; m; m &= m - 1)
                    add += a.wt[(2 * v + h) * 64 + __ffsll((long long)m) - 1] - 1;
            }
            s += add;
        } else {
            s = sat_add(s, sat_mul(x.x, a.wt[2 * v]));
            s = sat_add(s, sat_mul(x.y, a.wt[2 * v + 1]));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long y = __shfl_xor_sync(0xffffffffu, s, o);
        s = REACH ? s + y : sat_add(s, y);
    }
    if (lane == 0) a.out[t] = s;
}

// Column reduction (the block's rows are the probands, its columns the device's ancestors): a thread per
// column and a range of rows, every row weighted by how often the proband list names it; the ranges meet in
// integer atomics (an add for REACH, a saturating compare-and-swap loop otherwise), so the sums do not depend
// on the order in which they arrive.  `out` (width entries) is zero before the launch.
struct GcColReduceArgs {
    const unsigned long long *O;
    int64_t ws;                 // uint64 per row
    int32_t n_rows, width, rows_per_cta;
    const uint32_t *wt;         // n_rows
    unsigned long long *out;
};

template <bool REACH>
__global__ void __launch_bounds__(256) gc_col_reduce_kernel(GcColReduceArgs a) {
    const int32_t c = blockIdx.x * 256 + threadIdx.x;
    if (c >= a.width) return;
    const int32_t t0 = blockIdx.y * a.rows_per_cta, t1 = min(a.n_rows, t0 + a.rows_per_cta);
    unsigned long long s = 0;
    for (int32_t t = t0; t < t1; t++) {
        const unsigned long long x = a.O[(int64_t)t * a.ws + (REACH ? c >> 6 : c)];
        if (REACH) s += ((x >> (c & 63)) & 1) ? a.wt[t] : 0;
        else       s = sat_add(s, sat_mul(x, a.wt[t]));
    }
    if (s == 0) return;
    if (REACH) { atomicAdd(a.out + c, s); return; }
    unsigned long long old = a.out[c], seen;
    do { seen = old; old = atomicCAS(a.out + c, seen, sat_add(seen, s)); } while (old != seen);
}

struct GcGatherArgs {
    const void *O;              // output block, rows of ws elements of E
    int64_t ws;
    const int32_t *tgt_row;     // target list position -> output-block row
    const int32_t *col;         // column list position (the device's range) -> local column
    int32_t n_t, n_c;           // the block's target positions [t0, t0 + n_t), column positions [c0, c0 + n_c)
    int32_t t0, c0;
    // E = unsigned long long (gen.occ): the smallest (ancestor position, proband position) whose count
    // saturated, as ancestor * n_pro + proband over the whole lists, is atomicMin-ed into *ovf
    unsigned long long *ovf;
    int32_t j0, n_pro;          // list position of the device's first column; proband list length
    int32_t tgt_is_pro;         // the targets are the probands (descend)
};

// An output-block element as the caller's type: a uint16 distance widens, the unreachable sentinel to -1.
template <typename Out, typename E>
__device__ __forceinline__ Out gc_widen(E v) {
    if constexpr (std::is_same<E, uint16_t>::value) return v == kMeiosesNone ? (Out)-1 : (Out)v;
    else return (Out)v;
}

// stage (major x minor, minor contiguous): C_MAJOR = false: major = target, minor = column position;
// C_MAJOR = true: major = column position, minor = target.  Tiles of 32 x 32, 32 x 8 threads.
template <bool C_MAJOR, typename E, typename Out>
__global__ void __launch_bounds__(256) gc_gather_kernel(GcGatherArgs a, Out *stage) {
    __shared__ E tile[32][33];
    const E *O = static_cast<const E *>(a.O);
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int32_t cb = blockIdx.x * 32;                              // tile origin (relative to c0 / t0)
    const int32_t c = cb + tx;
    const int32_t lc = c < a.n_c ? a.col[a.c0 + c] : 0;
    for (int32_t tb = blockIdx.y * 32; tb < a.n_t; tb += gridDim.y * 32) {
        // read: lanes along the columns (the output block's rows are contiguous in columns)
        for (int k = ty; k < 32; k += 8) {
            const int32_t t = tb + k;
            if (t < a.n_t && c < a.n_c) {
                const E v = O[(int64_t)a.tgt_row[a.t0 + t] * a.ws + lc];
                tile[k][tx] = v;
                if constexpr (sizeof(E) == 8 && !std::is_floating_point<E>::value) {
                    if (v >= kOccSat) {
                        const unsigned long long tp = (unsigned long long)(a.t0 + t), cp = (unsigned long long)(a.j0 + a.c0 + c);
                        atomicMin(a.ovf, a.tgt_is_pro ? cp * a.n_pro + tp : tp * a.n_pro + cp);
                    }
                }
            }
        }
        if (!C_MAJOR) {
            for (int k = ty; k < 32; k += 8) {
                const int32_t t = tb + k;
                if (t < a.n_t && c < a.n_c) stage[(int64_t)t * a.n_c + c] = gc_widen<Out>(tile[k][tx]);
            }
            continue;
        }
        __syncthreads();
        // write: lanes along the targets
        for (int k = ty; k < 32; k += 8) {
            const int32_t cc = cb + k, t = tb + tx;
            if (t < a.n_t && cc < a.n_c) stage[(int64_t)cc * a.n_t + t] = gc_widen<Out>(tile[tx][k]);
        }
        __syncthreads();
    }
}

// gen.gcGroups, target side grouped: out[g][c] = the sum of O[row][c] over group g's output-block rows, in list
// order, one binary64 running sum per (group, column).  The order is fixed and there are no atomics, and every
// column lives on one device, so the bits do not depend on the device count.  A thread per column (coalesced
// along the row), a y-stride over the groups; the row indices and values of kGcGroupBatch members are loaded
// before they are added, in order.
constexpr int kGcGroupBatch = 8;
struct GcGroupReduceArgs {
    const double *O;            // output block: rows of ws doubles
    double *out;                // n_groups rows of ws doubles
    int64_t ws;
    int32_t n_groups;
    const int64_t *grp_ptr;     // n_groups + 1 entries
    const int32_t *grp_row;
};

__global__ void __launch_bounds__(256) gc_group_reduce_kernel(GcGroupReduceArgs a) {
    const int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (c >= a.ws) return;
    for (int32_t g = blockIdx.y; g < a.n_groups; g += gridDim.y) {
        const int64_t k1 = a.grp_ptr[g + 1];
        double s = 0.0;
        int64_t k = a.grp_ptr[g];
        for (; k + kGcGroupBatch <= k1; k += kGcGroupBatch) {
            double v[kGcGroupBatch];
#pragma unroll
            for (int u = 0; u < kGcGroupBatch; u++) v[u] = __ldcs(a.O + (int64_t)a.grp_row[k + u] * a.ws + c);
#pragma unroll
            for (int u = 0; u < kGcGroupBatch; u++) s += v[u];
        }
        for (; k < k1; k++) s += __ldcs(a.O + (int64_t)a.grp_row[k] * a.ws + c);
        a.out[(int64_t)g * a.ws + c] = s;
    }
}

}  // namespace genlib
