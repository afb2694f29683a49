// kernels.cuh -- device-side vocabulary shared by the sm_100a kernels of the kinship sweep, and the
// small kernels around the layer kernel (layer_kernel.cuh): proband gather, gen.phiOver's selection, gen.phiMeanGroups'
// and phiMean's reductions, gen.phiProduct's products, the inter-GPU barrier, sparse_phi's misfiled pairs, gen.f's parents' kinships and gen.phi_pairs' reads.
//
// Arithmetic is binary64 in the reference's grouping; storage type T is float
// (GENLIB_NUMERICS_REFERENCE: one RN32 per step, like src/compute.jl:296) or double.
// STORED = true selects the arithmetic of gen.sparse_phi instead (compute.jl:321-447: every
// stored kinship is a Float32 and is halved in Float32; the plan then orders the layers and the
// members by sparse_phi's queue, see plan.hpp).  No -use_fast_math / -ftz: Float32 subnormals occur.
#pragma once
#include <cuda_runtime.h>
#include <climits>
#include <cstdint>

#include "plan.hpp"

namespace genlib {

constexpr int kMaxWorld = 16;

// Where every rank keeps its frontier rows.  Entries of other ranks are NVLink peer memory: CUDA-IPC
// mappings of their arenas (one process per GPU) or plain peer pointers (one process, several devices).
struct PeerTable {
    void *A[kMaxWorld];       // rows_cap[g] x ld frontier rows of rank g
};

struct LayerArgs {
    int32_t n_new, n_fam, rt_lo, any_carried;
    // row sharding: this rank owns couples [own_f0, own_f0 + own_nf) and members [own_m0, own_m0 + own_nm)
    int32_t own_f0, own_nf, own_m0, own_nm;
    const int32_t *mem_ind, *mem_slot, *mem_fam, *mem_lrow;     // members: rank (or queue position), column slot, couple, local row
    const int32_t *fam_pf, *fam_pm, *fam_start;                  // couples: parent slots (-1 none), first member
    const int2 *fam_q;                                           // couples: the parents' rows in a strip buffer (-1 none)
    const int8_t *fam_pf_owner, *fam_pm_owner, *live_owner;      // where the parents' / the live individuals' rows are
    const int32_t *fam_pf_lrow, *fam_pm_lrow, *live_lrow;
    const uint8_t *flags;                                        // per slot of the live range: kFlagLive | kFlagCarried
    const int4 *mt_desc;                                         // member tiles: first couple, couples, first member, members
    int32_t n_mtiles;
};

constexpr int kThreads = 256;

// ---- 4-wide row-segment stores -------------------------------------------------------
// New frontier rows are written once and read by the NEXT step's kernel at the earliest: streaming stores
// (st.global.cs, evict-first) keep them from pushing the strip buffers out of L2.
__device__ __forceinline__ void store4(float *p, const double (&d)[4]) {
    // (float)double is cvt.rn.f32.f64: round-to-nearest-even, subnormals kept (no -ftz)
    __stcs(reinterpret_cast<float4 *>(p), make_float4((float)d[0], (float)d[1], (float)d[2], (float)d[3]));
}
__device__ __forceinline__ void store4(double *p, const double (&d)[4]) {
    __stcs(reinterpret_cast<double2 *>(p), make_double2(d[0], d[1]));
    __stcs(reinterpret_cast<double2 *>(p) + 1, make_double2(d[2], d[3]));
}
__device__ __forceinline__ void store_vec4(float *p, const float (&v)[4]) {
    __stcs(reinterpret_cast<float4 *>(p), make_float4(v[0], v[1], v[2], v[3]));
}
__device__ __forceinline__ void store_vec4(double *p, const double (&v)[4]) {
    __stcs(reinterpret_cast<double2 *>(p), make_double2(v[0], v[1]));
    __stcs(reinterpret_cast<double2 *>(p) + 1, make_double2(v[2], v[3]));
}
// an L2 cache policy for data that is read once (the parents' rows): evict first
__device__ __forceinline__ unsigned long long policy_evict_first() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// 1/2 x + 1/2 y with ONE binary64 rounding (1/2 y is exact), = Julia's `0 + x/2 + y/2`
__device__ __forceinline__ double half_sum(double x, double y) { return fma(0.5, x, 0.5 * y); }
// sparse_phi's `phi[..] / 2` is a FLOAT32 division of a stored Float32 (compute.jl:350-389): it rounds
// when the stored value is a subnormal with an odd last bit; the sum is Float64 as above.
__device__ __forceinline__ double half_sum_stored(double x, double y) {
    return (double)__fmul_rn((float)x, 0.5f) + (double)__fmul_rn((float)y, 0.5f);
}
template <bool STORED>
__device__ __forceinline__ double half_sum_mode(double x, double y) {
    if constexpr (STORED) return half_sum_stored(x, y);
    else return half_sum(x, y);
}

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// mbarrier + bulk-copy (TMA, SASS UBLKCP) helpers
__device__ __forceinline__ void mbar_init(unsigned bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// returns false when the phase did not complete within ~2^26 polls (a lost bulk copy must not hang the device)
__device__ __forceinline__ bool mbar_wait(unsigned bar, unsigned parity) {
    unsigned ok;
    for (unsigned spins = 0; spins < (1u << 26); spins++) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) return true;
    }
    return false;
}
// global -> shared bulk copy (16-byte aligned, size a multiple of 16), completes on `bar`
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint(unsigned dst, const void *src, unsigned bytes, unsigned bar, unsigned long long pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
// An unknown parent contributes 0 (compute.jl:111-126): its row (`bytes`, a multiple of 16) is zeroed instead of copied.
// Bulk copies (async proxy) fill the same place at other times: the fence orders these ordinary stores against them.
__device__ __forceinline__ void zero_row_shared(unsigned smem, unsigned bytes) {
    for (unsigned c = 0; c < bytes; c += 16) asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};\n" ::"r"(smem + c), "r"(0) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void lds4(const float *p, double (&d)[4]) {
    const float4 v = *reinterpret_cast<const float4 *>(p);
    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
}
__device__ __forceinline__ void lds4(const double *p, double (&d)[4]) {
    const double2 a = reinterpret_cast<const double2 *>(p)[0], b = reinterpret_cast<const double2 *>(p)[1];
    d[0] = a.x; d[1] = a.y; d[2] = b.x; d[3] = b.y;
}
template <typename T>
__device__ __forceinline__ T lds(unsigned addr) {
    T v;
    if constexpr (sizeof(T) == 4) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    else asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

// =====================================================================================
// misfile_kernel (GENLIB_SCHEDULE_SPARSE_PHI only).  sparse_phi FILES a kinship under
// phi[earlier processed][later processed] (compute.jl:393) but every look-up reads
// phi[lower rank][higher rank] (:36-40, :350-358, :367-389): between two individuals whose queue
// order inverts their rank order the stored value is never found again and the reference goes on
// as if the pair were unrelated.  Both orders follow the depth, so this only happens between the
// members of ONE layer; the frontier keeps what a look-up finds, 0.  grid (own rows, column chunks).
// =====================================================================================
template <typename T>
__global__ void __launch_bounds__(kThreads)
misfile_kernel(T *__restrict__ A, int64_t ld, const int32_t *__restrict__ mem_rank, LayerArgs L) {
    const int i = L.own_m0 + blockIdx.x;
    const int seq_i = L.mem_ind[i], rank_i = mem_rank[i];
    T *row = A + (int64_t)L.mem_lrow[i] * ld;
    for (int j = blockIdx.y * kThreads + threadIdx.x; j < L.n_new; j += gridDim.y * kThreads)
        if (j != i && ((seq_i > L.mem_ind[j]) != (rank_i > mem_rank[j]))) row[L.mem_slot[j]] = (T)0;
}

// =====================================================================================
// couple_kinship_kernel (GENLIB_SCHEDULE_F), launched just BEFORE the layer kernel of the couples' layer: the
// inbreeding coefficient of a child is the kinship of its parents, Psi[father, mother], the entry at the mother's
// slot of the father's row.  During the layer both parents are live and nobody writes that entry; after it the
// mother's slot may be recycled, by a peer rank too.  Every rank reads the couples whose father row it holds.
// =====================================================================================
template <typename T>
__global__ void couple_kinship_kernel(const T *__restrict__ A, int64_t ld, const int8_t *__restrict__ pf_owner,
                                      const int32_t *__restrict__ pf_lrow, const int32_t *__restrict__ pm, int32_t n_fam,
                                      int rank, double *__restrict__ out) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_fam || pf_owner[f] != rank || pm[f] < 0) return;
    out[f] = (double)A[(int64_t)pf_lrow[f] * ld + pm[f]];
}

// =====================================================================================
// pair_kinship_kernel (GENLIB_SCHEDULE_PAIRS), launched just BEFORE the layer kernel of the reads' layer (or once after
// the last layer): Psi[a, b] of a pair is the entry at the other member's slot of the higher-ranked member's row.  Both
// rows are live then and nobody writes that entry; one thread per read of the layer, every rank reads the rows it holds.
// Such a plan always stores Float64.
// =====================================================================================
__global__ void pair_kinship_kernel(const double *__restrict__ A, int64_t ld, const int8_t *__restrict__ owner,
                                    const int32_t *__restrict__ lrow, const int32_t *__restrict__ col, int64_t n_reads,
                                    int rank, double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_reads || owner[i] != rank) return;
    out[i] = A[(int64_t)lrow[i] * ld + col[i]];
}

// =====================================================================================
// proband gather (compute.jl:303: the last frontier, rows/columns in probandIDs order).
// rows[] are LOCAL rows of this rank's probands, cols[] the global slots of all probands.
// =====================================================================================
template <typename T, typename O>
__global__ void gather_kernel(const T *__restrict__ A, int64_t ld, const int32_t *__restrict__ rows,
                              const int32_t *__restrict__ cols, int32_t P, int32_t row0, int32_t nrows,
                              O *__restrict__ out) {
    if (blockIdx.y >= (unsigned)nrows) return;
    const T *row = A + (int64_t)rows[row0 + blockIdx.y] * ld;
    O *dst = out + (size_t)blockIdx.y * P;
    for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < P; v += gridDim.x * blockDim.x)
        dst[v] = (O)row[cols[v]];
}

// The same for ANY proband row of a sharded frontier: row u lives on rank owner[u] at local row lrow[u]
// (a peer read over NVLink unless it is this rank's own).  One process, several devices: every device
// assembles a contiguous block of output rows and copies it to the host over its own PCIe link.
template <typename T, typename O>
__global__ void gather_peer_kernel(PeerTable PT, int64_t ld, const int8_t *__restrict__ owner, const int32_t *__restrict__ lrow,
                                   const int32_t *__restrict__ cols, int32_t P, int32_t row0, int32_t nrows,
                                   O *__restrict__ out) {
    if (blockIdx.y >= (unsigned)nrows) return;
    const int u = row0 + blockIdx.y;
    const T *row = static_cast<const T *>(PT.A[owner[u]]) + (int64_t)lrow[u] * ld;
    O *dst = out + (size_t)blockIdx.y * P;
    for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < P; v += gridDim.x * blockDim.x)
        dst[v] = (O)row[cols[v]];
}

// =====================================================================================
// gen.phiOver: the proband pairs (i, j), i < j, whose kinship reaches a threshold, selected from this rank's own
// proband rows (rows[] local rows, index[] their positions i in the proband list, ascending; columns read as
// gather_kernel reads them, so no peer reads).  M[i, j] is the entry gen.phi returns in the output type O, compared as
// a binary64 number.  Two passes over the same columns j > i, one CTA per row: the first counts them, the second writes
// (j, M[i, j]) of each row, ascending in j, from the row's offset on.
// =====================================================================================
template <typename T, typename O>
__global__ void __launch_bounds__(kThreads)
phi_over_count_kernel(const T *__restrict__ A, int64_t ld, const int32_t *__restrict__ rows, const int32_t *__restrict__ index,
                      const int32_t *__restrict__ cols, int32_t P, double threshold, int64_t *__restrict__ count) {
    __shared__ int part[kThreads / 32];
    const int r = blockIdx.x;
    const T *row = A + (int64_t)rows[r] * ld;
    int c = 0;
    for (int j = index[r] + 1 + threadIdx.x; j < P; j += kThreads) c += (double)(O)row[cols[j]] >= threshold;
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t s = 0;
        for (int w = 0; w < kThreads / 32; w++) s += part[w];
        count[r] = s;
    }
}

// The rows sel[0, gridDim.x) of one block (own rows with at least one pair), row r's pairs written from
// offset[r] - base on: per chunk of kThreads columns a warp ballot orders the hits inside a warp and a scan of the
// warps' counts in shared memory orders the warps.
template <typename T, typename O>
__global__ void __launch_bounds__(kThreads)
phi_over_select_kernel(const T *__restrict__ A, int64_t ld, const int32_t *__restrict__ rows, const int32_t *__restrict__ index,
                       const int32_t *__restrict__ cols, int32_t P, double threshold, const int32_t *__restrict__ sel,
                       const int64_t *__restrict__ offset, int64_t base, int32_t *__restrict__ col_out, O *__restrict__ val_out) {
    __shared__ int warp_hits[kThreads / 32];
    const int r = sel[blockIdx.x];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const T *row = A + (int64_t)rows[r] * ld;
    int64_t at = offset[r] - base;
    for (int j0 = index[r] + 1; j0 < P; j0 += kThreads) {       // (the same trip count for every thread of the CTA)
        const int j = j0 + threadIdx.x;
        const O v = j < P ? (O)row[cols[j]] : (O)0;
        const bool hit = j < P && (double)v >= threshold;
        const unsigned ballot = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) warp_hits[w] = __popc(ballot);
        __syncthreads();
        int before = 0, total = 0;
        for (int k = 0; k < kThreads / 32; k++) {
            const int h = warp_hits[k];
            before += k < w ? h : 0;
            total += h;
        }
        if (hit) {
            const int64_t p = at + before + __popc(ballot & ((1u << lane) - 1u));
            col_out[p] = j;
            val_out[p] = v;
        }
        at += total;
        __syncthreads();                                          // (warp_hits is written again by the next chunk)
    }
}

// =====================================================================================
// gen.phiMeanGroups: S[i][g] = sum of M[i, j] over the probands j != i of group g, for this rank's own proband rows
// row0 + blockIdx.x (rows[] local rows, index[] their list positions i; no peer reads).  The columns come in group-major
// order: column k is the proband at frontier slot gcol[k], group g holds columns [gptr[g], gptr[g + 1]), never empty,
// and list position i is column gat[i] (the diagonal, skipped).  out[r * G + g] = S[row0 + r][g].  Every entry of the
// row is read once, all sums are binary64, and their order depends only on P, the groups and kThreads:
//   - thread t adds the columns [P t / kThreads, P (t + 1) / kThreads) in ascending order, one running sum per group;
//   - a group whose columns all lie in one chunk is written by that thread;
//   - the open group at the end of each chunk enters a segmented scan over the threads (Kogge-Stone shuffles inside a
//     warp, then the warps' totals in warp order); the thread that holds a group's last column adds its own partial to
//     the scan's value before it, and writes the group.
// Work per row is P / kThreads columns and a binary search in gptr per thread, whatever G is.
// =====================================================================================
template <typename T>
__global__ void __launch_bounds__(kThreads)
phi_groups_kernel(const T *__restrict__ A, int64_t ld, const int32_t *__restrict__ rows, const int32_t *__restrict__ index,
                  const int32_t *__restrict__ gcol, const int32_t *__restrict__ gat, const int32_t *__restrict__ gptr,
                  int32_t G, int32_t P, int32_t row0, double *__restrict__ out) {
    __shared__ double warp_v[kThreads / 32];
    __shared__ int warp_f[kThreads / 32];
    const int r = row0 + blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const T *row = A + (int64_t)rows[r] * ld;
    const int diag = gat[index[r]];
    double *dst = out + (size_t)blockIdx.x * G;
    const int c0 = (int)((int64_t)P * threadIdx.x / kThreads), c1 = (int)((int64_t)P * (threadIdx.x + 1) / kThreads);
    double s = 0.0, head = 0.0;        // the open group's partial; the first group's, when it began before c0 and ends here
    int g = 0, g_head = -1;
    bool began_here = false;           // the open group began in this chunk (an empty chunk is the scan's identity)
    if (c0 < c1) {
        int lo = 0, hi = G - 1;        // the group of column c0: the last g with gptr[g] <= c0
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (gptr[mid] <= c0) lo = mid; else hi = mid - 1;
        }
        g = lo;
        began_here = gptr[g] == c0;
        int end = gptr[g + 1];
        for (int k = c0; k < c1; k++) {
            if (k == end) {            // group g ended at column k - 1
                if (began_here) dst[g] = s; else { head = s; g_head = g; }
                end = gptr[++g + 1];
                s = 0.0;
                began_here = true;
            }
            if (k != diag) s += (double)row[gcol[k]];
        }
        if (end == c1) {               // the last group ends with the chunk
            if (began_here) dst[g] = s; else { head = s; g_head = g; }
        }
    }
    // segmented inclusive scan of (began_here, s): a later element that began its group discards what came before
    double v = s;
    int f = began_here;
    for (int o = 1; o < 32; o <<= 1) {
        const double pv = __shfl_up_sync(0xffffffffu, v, o);
        const int pf = __shfl_up_sync(0xffffffffu, f, o);
        if (lane >= o) {
            if (!f) v = pv + v;
            f |= pf;
        }
    }
    if (lane == 31) { warp_v[w] = v; warp_f[w] = f; }
    double ev = __shfl_up_sync(0xffffffffu, v, 1);      // exclusive: the threads before this one
    int ef = __shfl_up_sync(0xffffffffu, f, 1);
    if (lane == 0) { ev = 0.0; ef = 0; }
    __syncthreads();
    if (g_head >= 0) {
        if (!ef) {
            double pv = 0.0;                              // the warps before this one, in warp order
            for (int k = 0; k < w; k++) pv = warp_f[k] ? warp_v[k] : pv + warp_v[k];
            ev = pv + ev;
        }
        dst[g_head] = ev + head;
    }
}

// Row sums of the proband block for phiMean (src/compute.jl:454-459), deterministic: one CTA per own
// proband row, every thread adds its columns in ascending order in binary64, then a fixed shuffle /
// shared-memory tree.  out[2 r] = sum over all proband columns of row r, out[2 r + 1] = its diagonal entry.
// The host adds the rows in proband order, so the mean does not depend on the number of ranks.
template <typename T>
__global__ void __launch_bounds__(kThreads)
rowsum_kernel(const T *__restrict__ A, int64_t ld, const int32_t *__restrict__ own_rows, const int32_t *__restrict__ own_index,
              const int32_t *__restrict__ slots, int32_t P, double *__restrict__ out) {
    __shared__ double part[kThreads / 32];
    const int r = blockIdx.x;
    const T *row = A + (int64_t)own_rows[r] * ld;
    double s = 0.0;
    for (int v = threadIdx.x; v < P; v += kThreads) s += (double)row[slots[v]];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kThreads / 32; w++) s += part[w];
        out[2 * r] = s;
        out[2 * r + 1] = (double)row[slots[own_index[r]]];
    }
}

// =====================================================================================
// gen.phiProduct: Y[i][c] = sum over all probands j of M[i, j] X[j][c], for this rank's own proband rows
// row0 + rb * R + q (rows[] local rows, index[] their list positions; columns gathered through slots[] in list order,
// as rowsum_kernel reads them, so no peer reads).  X is P x k row-major (binary64), Y is nrows x k row-major, diag[r] =
// M[i, i] (when not null, written by the first column block).  One CTA per R rows and CB columns: each M entry loaded
// from memory serves its CB columns from registers, and each X row segment its R rows.
// The order of every sum depends only on P, and is rowsum_kernel's: thread t accumulates the columns j = t, t + 256,
// ... ascending with one FMA each (acc = fma(M[i, j], X[j][c], acc), rounded once), then a shuffle tree inside each
// warp and the warps' totals in warp order.  So a column of a k-column call is the same bits as a one-column call, X
// = 1 gives rowsum_kernel's sums, and neither CB, R, the row block nor the rank changes a result.
// =====================================================================================
template <typename T, int CB, int R>
__global__ void __launch_bounds__(kThreads)
phi_product_kernel(const T *__restrict__ A, int64_t ld, const int32_t *__restrict__ rows, const int32_t *__restrict__ index,
                   const int32_t *__restrict__ slots, int32_t P, const double *__restrict__ X, int32_t k, int32_t row0,
                   int32_t nrows, double *__restrict__ Y, double *__restrict__ diag) {
    __shared__ double part[kThreads / 32][R * CB];
    const int ncb = k > 0 ? (k + CB - 1) / CB : 1;
    const int cb = blockIdx.x % ncb, r0 = (int)(blockIdx.x / ncb) * R, c0 = cb * CB;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const T *row[R];
#pragma unroll
    for (int q = 0; q < R; q++) row[q] = A + (int64_t)rows[row0 + min(r0 + q, nrows - 1)] * ld;   // (past the block: a copy, not written)
    if (k > 0) {
        double acc[R][CB];
#pragma unroll
        for (int q = 0; q < R; q++)
#pragma unroll
            for (int c = 0; c < CB; c++) acc[q][c] = 0.0;
        for (int j = threadIdx.x; j < P; j += kThreads) {
            const int s = slots[j];
            const double *xj = X + (size_t)j * k + c0;
            double x[CB];
#pragma unroll
            for (int c = 0; c < CB; c++) x[c] = c0 + c < k ? __ldg(xj + c) : 0.0;
#pragma unroll
            for (int q = 0; q < R; q++) {
                const double m = (double)row[q][s];
#pragma unroll
                for (int c = 0; c < CB; c++) acc[q][c] = __fma_rn(m, x[c], acc[q][c]);
            }
        }
#pragma unroll
        for (int q = 0; q < R; q++)
#pragma unroll
            for (int c = 0; c < CB; c++) {
                double v = acc[q][c];
                for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
                if (lane == 0) part[w][q * CB + c] = v;
            }
        __syncthreads();
        for (int e = threadIdx.x; e < R * CB; e += kThreads) {
            const int q = e / CB, c = e % CB;
            if (r0 + q >= nrows || c0 + c >= k) continue;
            double v = part[0][e];
            for (int u = 1; u < kThreads / 32; u++) v += part[u][e];
            Y[(size_t)(r0 + q) * k + c0 + c] = v;
        }
    }
    if (diag && cb == 0 && threadIdx.x < R && r0 + (int)threadIdx.x < nrows) {
        const int r = row0 + r0 + (int)threadIdx.x;
        diag[r - row0] = (double)A[(int64_t)rows[r] * ld + slots[index[r]]];
    }
}

// =====================================================================================
// barrier_kernel: all ranks of one box meet here (one process per GPU, so every rank's
// kernel is resident on its own device).  Rank r stores `epoch` into slot r of every peer's
// flag array (release, system scope, through the NVLink mapping) and waits until all slots of
// its own array have reached `epoch`.  A rank that waits longer than ~10 s (GENLIB_BARRIER_TIMEOUT_S)
// records an error in every rank's flag block instead of hanging: all ranks' genlib_engine_run fail.
// =====================================================================================
struct BarrierTable {
    unsigned *flags[kMaxWorld];   // [world] words on each rank; word kMaxWorld = error flag
};

__global__ void barrier_kernel(BarrierTable B, int rank, int world, unsigned epoch, long long timeout_cycles) {
    const int peer = threadIdx.x;
    if (peer >= world) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(B.flags[peer] + rank), "r"(epoch) : "memory");
    const unsigned *mine = B.flags[rank] + peer;
    const long long t0 = clock64();
    for (;;) {
        unsigned v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
        if ((int)(v - epoch) >= 0) break;
        if (clock64() - t0 > timeout_cycles) {               // tell EVERY rank: the peers that arrive later pass this barrier,
            for (int g = 0; g < world; g++)                   // but their genlib_engine_run must fail as well
                asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(B.flags[g] + kMaxWorld), "r"(1u) : "memory");
            break;
        }
        __nanosleep(200);
    }
    __threadfence_system();
}

}  // namespace genlib
