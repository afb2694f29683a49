// gc_engine.cu -- gen.gc, gen.occ and gen.rec on the device (DESIGN.md 2b, 2c): the C ABI entry points, the split of
// the column-side list over the devices and each device's run of the plan (gc_plan.hpp) with the kernels of
// gc_kernel.cuh.
#include <cstdio>
#include <cstring>
#include <memory>

#include "runtime.hpp"
#include "gc_kernel.cuh"
#include "gc_plan.hpp"

using namespace genlib;

struct genlib_gc_plan {
    GcPlan p;
    double ms_plan = 0;
};

namespace {

// What a run of the gc plan computes: gen.gc's matrix, gen.occ's matrix or row sums, gen.rec's counts.
enum GcFn { kFnGc = 0, kFnOcc, kFnOccTotal, kFnRec };
const char *const kGcFnName[] = {"gc", "occ", "occ", "rec"};     // gen.<name> in Python, genlib_<name> in C
bool gc_fn_reduces(int fn) { return fn == kFnOccTotal || fn == kFnRec; }

// One device's share: column positions [j0, j1) of the column-side list and the unique columns [lo, hi) they
// name (contiguous when the list has no duplicates; a duplicate may widen the range, never the result).
struct GcShare {
    int device = -1;
    int fn = kFnGc;
    int32_t j0 = 0, j1 = 0, lo = 0, hi = 0;
    // row stride in 8-byte elements (16-byte rows): a column each, or for gen.rec 64 columns per word
    int64_t ws() const {
        const int64_t w = fn == kFnRec ? ((int64_t)(hi - lo) + 63) / 64 : (int64_t)(hi - lo);
        return (w + 1) / 2 * 2;
    }
    size_t stage = 0, need = 0;
    double ms_kernels = 0, ms_fetch = 0;
    int32_t launches = 0;
    int64_t d2h = 0;
    std::vector<unsigned long long> red;   // reductions: per output-block row (ascend) or local column (descend)
    unsigned long long ovf = ~0ull;        // gen.occ matrix: the smallest saturated (ancestor, proband) key
};

// Required traffic of a share over `cols` columns: the plan's byte model over the row's 8-byte elements
// (gen.rec: its words, 16-byte padded as the kernel moves them), plus one read of the output block for a
// reduction.
double gc_fn_bytes(const GcPlan &P, int fn, int32_t cols) {
    const int64_t w = fn == kFnRec ? (((int64_t)cols + 63) / 64 + 1) / 2 * 2 : cols;
    double b = P.alg_bytes(w);
    if (gc_fn_reduces(fn)) b += (double)P.n_targets() * (double)w * 8.0;
    return b;
}

// Output layout of a share: the stage's major dimension is the column position (cmaj) or the target position.
struct GcLayout {
    bool cmaj;
    int64_t ld, nmaj, nmin, maj_off, min_off;
};

GcLayout gc_layout(const GcPlan &P, const GcShare &d, int col_major) {
    // gen.occ's ancestors x probands matrix in row-major order is gen.gc's layout in column-major order
    const bool cm = d.fn == kFnOcc ? !col_major : col_major != 0;
    GcLayout L;
    L.cmaj = (P.direction == kGcDescend) == cm;
    L.ld = cm ? P.n_pro : P.n_anc;
    const int64_t T = (int64_t)P.target_uid().size(), C = d.j1 - d.j0;
    L.nmaj = L.cmaj ? C : T; L.nmin = L.cmaj ? T : C;
    L.maj_off = L.cmaj ? d.j0 : 0; L.min_off = L.cmaj ? 0 : d.j0;
    return L;
}

// Reduction buffers: weights (ascend: per column, gen.rec also two masks per word; descend: per target row)
// and the result (ascend: per target row; descend: per local column).
size_t gc_reduce_bytes(const GcPlan &P, const GcShare &d) {
    const size_t ws = (size_t)d.ws(), T = (size_t)P.n_targets(), W = (size_t)(d.hi - d.lo);
    if (P.direction == kGcAscend)
        return DevBuf<uint32_t>::padded(d.fn == kFnRec ? ws * 64 : ws) +
               (d.fn == kFnRec ? 2 * DevBuf<unsigned long long>::padded(ws) : 0) + DevBuf<unsigned long long>::padded(T);
    return DevBuf<uint32_t>::padded(T) + DevBuf<unsigned long long>::padded(W);
}

size_t gc_device_bytes(const GcPlan &P, GcShare &d, int col_major, size_t esize) {
    const size_t ws = (size_t)d.ws(), R = (size_t)P.rows();
    d.stage = gc_fn_reduces(d.fn) ? 0 : pad256(std::max<size_t>(kFetchStageBytes, (size_t)gc_layout(P, d, col_major).nmin * esize));
    return pad256((size_t)P.capacity * ws * 8) + pad256((size_t)P.n_targets() * ws * 8) +
           3 * DevBuf<int32_t>::padded(R) + DevBuf<int64_t>::padded(R + 1) + DevBuf<int32_t>::padded((size_t)P.inputs()) +
           DevBuf<int32_t>::padded(P.target_uid().size()) + DevBuf<int32_t>::padded((size_t)(d.j1 - d.j0)) +
           DevBuf<int32_t>::padded(1) + 2 * d.stage +
           (d.fn == kFnGc ? 0 : DevBuf<unsigned long long>::padded(1)) + (gc_fn_reduces(d.fn) ? gc_reduce_bytes(P, d) : 0);
}

template <typename E, typename O>
int gc_fetch(const GcPlan &P, GcShare &d, const void *Oblk, const int32_t *tgt_row, const int32_t *col, O *out,
             int col_major, unsigned char *stage_base, unsigned long long *ovf, cudaStream_t st, cudaStream_t cst) {
    const GcLayout L = gc_layout(P, d, col_major);
    if (L.nmaj == 0 || L.nmin == 0) return GENLIB_OK;
    const int64_t per = std::max<int64_t>(1, std::min<int64_t>(L.nmaj, (int64_t)(d.stage / (L.nmin * sizeof(O)))));
    int rc = staged_d2h(st, cst, reinterpret_cast<O *>(stage_base), reinterpret_cast<O *>(stage_base + d.stage), L.nmaj, per, "gc fetch",
        [&](O *stage, int64_t m0, int64_t nb) {
            GcGatherArgs a;
            a.O = Oblk; a.ws = d.ws(); a.tgt_row = tgt_row; a.col = col;
            a.ovf = ovf; a.j0 = d.j0; a.n_pro = P.n_pro; a.tgt_is_pro = P.direction == kGcDescend;
            if (L.cmaj) { a.t0 = 0; a.n_t = (int32_t)L.nmin; a.c0 = (int32_t)m0; a.n_c = (int32_t)nb; }
            else        { a.t0 = (int32_t)m0; a.n_t = (int32_t)nb; a.c0 = 0; a.n_c = (int32_t)L.nmin; }
            dim3 grid((unsigned)((a.n_c + 31) / 32), (unsigned)std::min<int64_t>((a.n_t + 31) / 32, 65535)), block(32, 8);
            if (L.cmaj) gc_gather_kernel<true, E, O><<<grid, block, 0, st>>>(a, stage);
            else        gc_gather_kernel<false, E, O><<<grid, block, 0, st>>>(a, stage);
        },
        [&](const O *stage, int64_t m0, int64_t nb) {
            return cudaMemcpy2DAsync(out + (L.maj_off + m0) * L.ld + L.min_off, (size_t)L.ld * sizeof(O), stage,
                                     (size_t)L.nmin * sizeof(O), (size_t)L.nmin * sizeof(O), (size_t)nb, cudaMemcpyDeviceToHost, cst);
        });
    if (rc == GENLIB_OK) d.d2h += L.nmaj * L.nmin * (int64_t)sizeof(O);
    return rc;
}

template <typename Op>
void gc_launch_layer(const GcLayerArgs &a, unsigned gx, cudaStream_t st) {
    const int rpc = kGcThreads >> a.tpr_log2;
    const unsigned gy = (unsigned)std::min<int64_t>(((int64_t)a.n_rows + rpc - 1) / rpc, 65535);
    if (a.tpr_log2 == kGcThreadsLog2) gc_layer_kernel<Op, true><<<dim3(gx, gy), kGcThreads, 0, st>>>(a);
    else                              gc_layer_kernel<Op, false><<<dim3(gx, gy), kGcThreads, 0, st>>>(a);
}

// Every layer of the plan over the share's columns on its device, then its block of `out` (gen.gc, gen.occ's
// matrix) or its part of the reduction (d.red).
int gc_run_share(const GcPlan &P, GcShare &d, void *out, int out_dtype, int col_major) {
    DeviceGuard guard;
    if (int rc = guard.enter(d.device)) return rc;
    struct Res {
        cudaStream_t st = nullptr, cst = nullptr;
        cudaEvent_t ev[2] = {nullptr, nullptr};
        Arena arena;
        ~Res() {
            if (st) cudaStreamSynchronize(st);
            if (cst) cudaStreamSynchronize(cst);
            for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
            if (st) cudaStreamDestroy(st);
            if (cst) cudaStreamDestroy(cst);
            g_arenas.release(arena);
        }
    } res;
    CU(cudaStreamCreateWithFlags(&res.st, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&res.cst, cudaStreamNonBlocking));
    for (cudaEvent_t &e : res.ev) CU(cudaEventCreate(&e));
    if (int rc = acquire_arena(d.device, d.need, res.arena, [&](size_t free_b) {
            char msg[256];
            std::snprintf(msg, sizeof msg, "gen.%s needs %.2f GB on device %d, %.2f GB free (%lld frontier rows x %lld columns): "
                          "split the columns over more devices", kGcFnName[d.fn], d.need / 1e9, d.device, free_b / 1e9,
                          (long long)P.capacity, (long long)(d.hi - d.lo));
            return std::string(msg);
        }))
        return rc;
    const size_t ws = (size_t)d.ws(), R = (size_t)P.rows(), T = (size_t)P.n_targets(), W = (size_t)(d.hi - d.lo);
    const bool reduce = gc_fn_reduces(d.fn), asc = P.direction == kGcAscend;
    unsigned char *cur = static_cast<unsigned char *>(res.arena.base);
    auto take = [&](size_t bytes) { unsigned char *p = cur; cur += pad256(bytes); return p; };
    void *F = take((size_t)P.capacity * ws * 8);
    void *O = take(T * ws * 8);
    DevBuf<int32_t> row_slot, row_seed, row_out, in_slot, tgt_row, col, err;
    DevBuf<int64_t> in_ptr;
    DevBuf<unsigned long long> ovf, m1, m2, red;
    DevBuf<uint32_t> wt;
    row_slot.place(cur, R); row_seed.place(cur, R); row_out.place(cur, R); in_ptr.place(cur, R + 1);
    in_slot.place(cur, (size_t)P.inputs()); tgt_row.place(cur, P.target_uid().size());
    col.place(cur, (size_t)(d.j1 - d.j0)); err.place(cur, 1);
    unsigned char *stage = cur;
    cur += 2 * d.stage;
    if (d.fn != kFnGc) ovf.place(cur, 1);
    // reduction weights: how often the lists name each column (ascend) or each target row (descend)
    std::vector<uint32_t> h_wt;
    std::vector<unsigned long long> h_m1, h_m2;
    if (reduce) {
        if (asc) {
            h_wt.assign(d.fn == kFnRec ? ws * 64 : ws, 0);
            for (int32_t j = d.j0; j < d.j1; j++) h_wt[(size_t)(P.column_uid()[(size_t)j] - d.lo)]++;
            if (d.fn == kFnRec) {
                h_m1.assign(ws, 0); h_m2.assign(ws, 0);
                for (size_t c = 0; c < W; c++) {
                    if (h_wt[c] >= 1) h_m1[c >> 6] |= 1ull << (c & 63);
                    if (h_wt[c] >= 2) h_m2[c >> 6] |= 1ull << (c & 63);
                }
                m1.place(cur, ws); m2.place(cur, ws);
            }
            red.place(cur, T);
        } else {
            h_wt.assign(T, 0);
            for (int32_t t : P.target_uid()) h_wt[(size_t)t]++;
            red.place(cur, W);
        }
        wt.place(cur, h_wt.size());
    }
    if ((size_t)(cur - static_cast<unsigned char *>(res.arena.base)) > d.need) return fail(GENLIB_EINVAL, "internal: gc arena layout overflow");
    std::vector<int32_t> cols((size_t)(d.j1 - d.j0));
    for (int32_t j = d.j0; j < d.j1; j++) cols[(size_t)(j - d.j0)] = P.column_uid()[(size_t)j] - d.lo;
    CU(row_slot.upload(P.row_slot, res.st)); CU(row_seed.upload(P.row_seed, res.st)); CU(row_out.upload(P.row_out, res.st));
    CU(in_ptr.upload(P.in_ptr, res.st)); CU(in_slot.upload(P.in_slot, res.st)); CU(tgt_row.upload(P.target_uid(), res.st));
    CU(col.upload(cols, res.st));
    CU(cudaMemsetAsync(err.p, 0, sizeof(int32_t), res.st));
    if (d.fn != kFnGc) CU(cudaMemsetAsync(ovf.p, 0xff, sizeof(unsigned long long), res.st));
    if (reduce) {
        CU(wt.upload(h_wt, res.st)); CU(m1.upload(h_m1, res.st)); CU(m2.upload(h_m2, res.st));
        if (!asc) CU(cudaMemsetAsync(red.p, 0, W * sizeof(unsigned long long), res.st));
    }
    if (P.n_out_rows < P.n_targets())                       // a target no path reaches: its output row is 0
        CU(cudaMemsetAsync(O, 0, T * ws * 8, res.st));
    GcLayerArgs a;
    a.F = F; a.O = O;
    a.w2 = (int64_t)ws / 2; a.width = d.hi - d.lo; a.col_lo = d.lo;
    a.tpr_log2 = gc_tpr_log2(a.w2);
    a.capacity = P.capacity; a.n_targets = P.n_targets(); a.in_slot = in_slot.p; a.err = err.p;
    const unsigned gx = (unsigned)((a.w2 + ((int64_t)kGcVec << a.tpr_log2) - 1) / ((int64_t)kGcVec << a.tpr_log2));
    CU(cudaEventRecord(res.ev[0], res.st));
    for (int32_t t = 0; t < P.n_layers(); t++) {
        const int64_t r0 = P.layer_begin[(size_t)t];
        a.n_rows = (int32_t)(P.layer_begin[(size_t)t + 1] - r0);
        a.row_slot = row_slot.p + r0; a.row_seed = row_seed.p + r0; a.row_out = row_out.p + r0; a.in_ptr = in_ptr.p + r0;
        if (d.fn == kFnGc) gc_launch_layer<GcOpHalfSum>(a, gx, res.st);
        else if (d.fn == kFnRec) gc_launch_layer<GcOpReach>(a, gx, res.st);
        else gc_launch_layer<GcOpCount>(a, gx, res.st);
        CU(cudaGetLastError());
        d.launches++;
    }
    if (reduce && T > 0) {
        if (asc) {
            GcRowReduceArgs r;
            r.O = static_cast<const ulonglong2 *>(O); r.w2 = (int64_t)ws / 2; r.n_rows = (int32_t)T;
            r.wt = wt.p; r.m1 = m1.p; r.m2 = m2.p; r.out = red.p;
            const unsigned g = (unsigned)((T + 7) / 8);
            if (d.fn == kFnRec) gc_row_reduce_kernel<true><<<g, 256, 0, res.st>>>(r);
            else                gc_row_reduce_kernel<false><<<g, 256, 0, res.st>>>(r);
        } else {
            GcColReduceArgs r;
            r.O = static_cast<const unsigned long long *>(O); r.ws = (int64_t)ws; r.n_rows = (int32_t)T;
            r.width = (int32_t)W; r.wt = wt.p; r.out = red.p;
            // enough CTAs for the whole device: about 8 per SM, at least 64 rows each
            const int64_t gxr = ((int64_t)W + 255) / 256;
            const int64_t gyr = std::max<int64_t>(1, std::min<int64_t>(((int64_t)T + 63) / 64, (148 * 8 + gxr - 1) / gxr));
            r.rows_per_cta = (int32_t)(((int64_t)T + gyr - 1) / gyr);
            const dim3 g((unsigned)gxr, (unsigned)(((int64_t)T + r.rows_per_cta - 1) / r.rows_per_cta));
            if (d.fn == kFnRec) gc_col_reduce_kernel<true><<<g, 256, 0, res.st>>>(r);
            else                gc_col_reduce_kernel<false><<<g, 256, 0, res.st>>>(r);
        }
        CU(cudaGetLastError());
        d.launches++;
    }
    CU(cudaEventRecord(res.ev[1], res.st));
    CU(cudaStreamSynchronize(res.st));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, res.ev[0], res.ev[1]));
    d.ms_kernels = ms;
    int32_t errw = 0;
    CU(cudaMemcpy(&errw, err.p, sizeof errw, cudaMemcpyDeviceToHost));
    if (errw) return fail(GENLIB_ECUDA, "the gc layer kernel reported a bound violated at line " + std::to_string(errw - 100000));
    const double t0 = now_ms();
    int rc = GENLIB_OK;
    if (reduce) {
        d.red.assign(asc ? T : W, 0);
        if (T > 0) CU(cudaMemcpy(d.red.data(), red.p, d.red.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        d.d2h += (int64_t)(d.red.size() * sizeof(unsigned long long));
    } else if (d.fn == kFnOcc) {
        rc = gc_fetch<unsigned long long, int64_t>(P, d, O, tgt_row.p, col.p, static_cast<int64_t *>(out), col_major, stage, ovf.p, res.st, res.cst);
        if (rc == GENLIB_OK) CU(cudaMemcpy(&d.ovf, ovf.p, sizeof d.ovf, cudaMemcpyDeviceToHost));
    } else {
        rc = out_dtype == GENLIB_F64
            ? gc_fetch<double, double>(P, d, O, tgt_row.p, col.p, static_cast<double *>(out), col_major, stage, nullptr, res.st, res.cst)
            : gc_fetch<double, float>(P, d, O, tgt_row.p, col.p, static_cast<float *>(out), col_major, stage, nullptr, res.st, res.cst);
    }
    d.ms_fetch = now_ms() - t0;
    return rc;
}

void gc_fill_stats(const GcPlan &P, genlib_gc_stats *s) {
    std::memset(s, 0, sizeof *s);
    s->n_pro = P.n_pro; s->n_anc = P.n_anc; s->n_layers = P.n_layers(); s->direction = P.direction;
    s->rows = P.rows(); s->inputs = P.inputs(); s->width = P.width(); s->capacity = P.capacity;
    s->alg_bytes = P.alg_bytes(P.width());
    s->n_dev = 1;
}

}  // namespace

extern "C" {

int genlib_gc_plan_create(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                          const int32_t *proband, int32_t n_anc, const int32_t *ancestor, genlib_gc_plan **out) {
    if (!out) return fail(GENLIB_EINVAL, "genlib_gc_plan_create: null argument");
    *out = nullptr;
    std::unique_ptr<genlib_gc_plan> pl(new (std::nothrow) genlib_gc_plan);
    if (!pl) return fail(GENLIB_ENOMEM, "out of host memory");
    const double t0 = now_ms();
    std::string err;
    try {
        if (int rc = build_gc_plan(n, father, mother, n_pro, proband, n_anc, ancestor, -1, pl->p, err)) return fail(rc, err);
    } catch (const std::bad_alloc &) {
        return fail(GENLIB_ENOMEM, "out of host memory while planning");
    }
    pl->ms_plan = now_ms() - t0;
    *out = pl.release();
    return GENLIB_OK;
}

void genlib_gc_plan_destroy(genlib_gc_plan *plan) { delete plan; }

int genlib_gc_plan_info(const genlib_gc_plan *plan, genlib_gc_stats *out) {
    if (!plan || !out) return fail(GENLIB_EINVAL, "genlib_gc_plan_info: null argument");
    gc_fill_stats(plan->p, out);
    GcShare d;
    d.j1 = (int32_t)plan->p.column_uid().size(); d.hi = plan->p.width();
    out->device_bytes = plan->p.width() > 0 && plan->p.n_targets() > 0 ? (int64_t)gc_device_bytes(plan->p, d, 0, 8) : 0;
    return GENLIB_OK;
}

int genlib_gc_plan_layer(const genlib_gc_plan *plan, int32_t layer, int32_t *n_rows, int64_t *n_inputs) {
    if (!plan) return fail(GENLIB_EINVAL, "genlib_gc_plan_layer: null plan");
    const GcPlan &P = plan->p;
    if (layer < 0 || layer >= P.n_layers()) return fail(GENLIB_EINVAL, "layer out of range");
    const int64_t r0 = P.layer_begin[(size_t)layer], r1 = P.layer_begin[(size_t)layer + 1];
    if (n_rows) *n_rows = (int32_t)(r1 - r0);
    if (n_inputs) *n_inputs = P.in_ptr[(size_t)r1] - P.in_ptr[(size_t)r0];
    return GENLIB_OK;
}

int genlib_gc_plan_layer_arrays(const genlib_gc_plan *plan, int32_t layer, int32_t *row_ind, int32_t *row_slot,
                                int32_t *row_seed, int32_t *row_out, int64_t *in_ptr, int32_t *in_slot) {
    if (!plan) return fail(GENLIB_EINVAL, "genlib_gc_plan_layer_arrays: null plan");
    const GcPlan &P = plan->p;
    if (layer < 0 || layer >= P.n_layers()) return fail(GENLIB_EINVAL, "layer out of range");
    const size_t r0 = (size_t)P.layer_begin[(size_t)layer], r1 = (size_t)P.layer_begin[(size_t)layer + 1];
    auto copy = [&](const std::vector<int32_t> &v, int32_t *o) { if (o) std::copy(v.begin() + (long)r0, v.begin() + (long)r1, o); };
    copy(P.row_ind, row_ind); copy(P.row_slot, row_slot); copy(P.row_seed, row_seed); copy(P.row_out, row_out);
    const int64_t e0 = P.in_ptr[r0];
    if (in_ptr) for (size_t r = r0; r <= r1; r++) in_ptr[r - r0] = P.in_ptr[r] - e0;
    if (in_slot) std::copy(P.in_slot.begin() + e0, P.in_slot.begin() + P.in_ptr[r1], in_slot);
    return GENLIB_OK;
}

}  // extern "C"

namespace {

// The first proband list position whose individual descends from (or is) `anc`: the proband an overflowing
// row sum is reported with.  Host only, O(n), on the error path.
int32_t gc_first_descendant(int32_t n, const int32_t *father, const int32_t *mother, int32_t anc, int32_t n_pro,
                            const int32_t *proband) {
    std::vector<uint8_t> down((size_t)n, 0);
    down[(size_t)anc] = 1;
    for (int32_t i = anc + 1; i < n; i++)
        down[(size_t)i] = (father[i] >= 0 && down[(size_t)father[i]]) || (mother[i] >= 0 && down[(size_t)mother[i]]);
    for (int32_t j = 0; j < n_pro; j++) if (down[(size_t)proband[j]]) return j;
    return -1;
}

int gc_overflow(int32_t anc_pos, int32_t anc_rank, int32_t pro_pos, int32_t pro_rank, bool total) {
    char msg[320];
    std::snprintf(msg, sizeof msg, "gen.occ: %s exceeds 2^63 - 1 (Int64) at ancestor position %d (rank %d), "
                  "proband position %d (rank %d)", total ? "a row sum of descent-path counts" : "a descent-path count",
                  anc_pos, anc_rank, pro_pos, pro_rank);
    return fail(GENLIB_EOVERFLOW, msg);
}

// genlib_gc, genlib_occ and genlib_rec: one plan, the column-side list split over the devices, every device
// runs the plan over its columns; the matrices are written block by block into `out`, the reductions are
// combined here.
int gc_driver(int fn, int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
              int32_t n_anc, const int32_t *ancestor, void *out, int out_dtype, int col_major, int32_t n_dev,
              const int32_t *devices, genlib_gc_stats *stats) {
    const std::string who = std::string("genlib_") + kGcFnName[fn];
    if (n_dev < 1 || !devices) return fail(GENLIB_EINVAL, who + ": at least one device");
    genlib_gc_plan *plan = nullptr;
    if (int rc = genlib_gc_plan_create(n, father, mother, n_pro, proband, n_anc, ancestor, &plan)) return rc;
    std::unique_ptr<genlib_gc_plan> owner(plan);
    const GcPlan &P = plan->p;
    genlib_gc_stats st;
    gc_fill_stats(P, &st);
    st.alg_bytes = gc_fn_bytes(P, fn, P.width());
    st.ms_plan = plan->ms_plan;
    st.n_dev = n_dev;
    const bool reduce = gc_fn_reduces(fn);
    if (P.n_pro == 0 || P.n_anc == 0) {                     // an empty matrix (or zero counts): no device needed
        if (reduce && P.n_anc > 0) {
            if (!out) return fail(GENLIB_EINVAL, who + ": out is null");
            std::memset(out, 0, (size_t)P.n_anc * sizeof(int64_t));
        }
        if (stats) *stats = st;
        return GENLIB_OK;
    }
    if (!out) return fail(GENLIB_EINVAL, who + ": out is null");
    std::vector<int> dev;
    if (int rc = resolve_devices(who, n_dev, devices, true, dev)) return rc;
    std::vector<GcShare> share((size_t)n_dev);
    const std::vector<int32_t> &cu = P.column_uid();
    const int64_t m = (int64_t)cu.size();
    const size_t esize = fn == kFnGc ? (out_dtype == GENLIB_F64 ? 8 : 4) : 8;
    for (int g = 0; g < n_dev; g++) {
        GcShare &d = share[(size_t)g];
        d.fn = fn;
        d.device = dev[(size_t)g];
        d.j0 = (int32_t)(m * g / n_dev); d.j1 = (int32_t)(m * (g + 1) / n_dev);
        if (d.j0 == d.j1) continue;                          // more devices than columns: nothing to do here
        d.lo = *std::min_element(cu.begin() + d.j0, cu.begin() + d.j1);
        d.hi = *std::max_element(cu.begin() + d.j0, cu.begin() + d.j1) + 1;
        d.need = gc_device_bytes(P, d, col_major, esize);
    }
    const std::vector<DeviceStatus> r = on_devices(n_dev, [&](int g) {
        GcShare &d = share[(size_t)g];
        return d.j0 == d.j1 ? GENLIB_OK : gc_run_share(P, d, out, out_dtype, col_major);
    });
    for (int g = 0; g < n_dev; g++)
        if (r[(size_t)g].status != GENLIB_OK) return fail(r[(size_t)g].status, "device " + std::to_string(dev[(size_t)g]) + ": " + r[(size_t)g].message);
    if (stats) {
        st.width = 0; st.alg_bytes = 0;
        for (const GcShare &d : share) {
            if (d.j0 == d.j1) continue;
            st.width += d.hi - d.lo;
            st.alg_bytes += gc_fn_bytes(P, fn, d.hi - d.lo);
            st.device_bytes = std::max(st.device_bytes, (int64_t)d.need);
            st.ms_kernels = std::max(st.ms_kernels, d.ms_kernels);
            st.ms_fetch = std::max(st.ms_fetch, d.ms_fetch);
            st.d2h_bytes += d.d2h;
            st.kernel_launches += d.launches;
        }
        *stats = st;
    }
    if (fn == kFnOcc) {                                      // the smallest saturated pair over all devices
        unsigned long long key = ~0ull;
        for (const GcShare &d : share) if (d.j0 != d.j1) key = std::min(key, d.ovf);
        if (key != ~0ull) {
            const int32_t i = (int32_t)(key / (unsigned long long)P.n_pro), j = (int32_t)(key % (unsigned long long)P.n_pro);
            return gc_overflow(i, ancestor[i], j, proband[j], false);
        }
    }
    if (reduce) {                                            // every device's part -> one value per ancestor position
        const bool rec = fn == kFnRec;
        std::vector<unsigned long long> v((size_t)P.n_anc, 0);
        if (P.direction == kGcAscend) {                      // parts per ancestor (the block's rows): add them
            std::vector<unsigned long long> tot((size_t)P.n_targets(), 0);
            for (const GcShare &d : share) {
                if (d.j0 == d.j1) continue;
                for (size_t t = 0; t < tot.size(); t++) {
                    const unsigned long long s = tot[t] + d.red[t];
                    tot[t] = rec ? s : (s < tot[t] || s > kOccSat) ? kOccSat : s;
                }
            }
            for (int32_t i = 0; i < P.n_anc; i++) v[(size_t)i] = tot[(size_t)P.anc_uid[(size_t)i]];
        } else {                                             // parts per ancestor column: place them
            for (const GcShare &d : share)
                for (int32_t j = d.j0; j < d.j1; j++) v[(size_t)j] = d.red[(size_t)(P.anc_uid[(size_t)j] - d.lo)];
        }
        for (int32_t i = 0; i < P.n_anc; i++)
            if (v[(size_t)i] >= kOccSat) {
                const int32_t j = gc_first_descendant(n, father, mother, ancestor[i], n_pro, proband);
                return gc_overflow(i, ancestor[i], j, j >= 0 ? proband[j] : -1, true);
            }
        int64_t *o = static_cast<int64_t *>(out);
        for (int32_t i = 0; i < P.n_anc; i++) o[i] = (int64_t)v[(size_t)i];
    }
    return GENLIB_OK;
}

}  // namespace

extern "C" {

int genlib_gc(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
              int32_t n_anc, const int32_t *ancestor, void *out, int out_dtype, int col_major, int32_t n_dev,
              const int32_t *devices, genlib_gc_stats *stats) {
    if (out_dtype != GENLIB_F32 && out_dtype != GENLIB_F64) return fail(GENLIB_EINVAL, "unknown out_dtype");
    return gc_driver(kFnGc, n, father, mother, n_pro, proband, n_anc, ancestor, out, out_dtype, col_major, n_dev,
                     devices, stats);
}

int genlib_occ(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
               int32_t n_anc, const int32_t *ancestor, int64_t *out, int type, int col_major, int32_t n_dev,
               const int32_t *devices, genlib_gc_stats *stats) {
    if (type != GENLIB_OCC_IND && type != GENLIB_OCC_TOTAL) return fail(GENLIB_EINVAL, "genlib_occ: unknown type");
    return gc_driver(type == GENLIB_OCC_IND ? kFnOcc : kFnOccTotal, n, father, mother, n_pro, proband, n_anc, ancestor,
                     out, 0, col_major, n_dev, devices, stats);
}

int genlib_rec(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
               int32_t n_anc, const int32_t *ancestor, int64_t *out, int32_t n_dev, const int32_t *devices,
               genlib_gc_stats *stats) {
    return gc_driver(kFnRec, n, father, mother, n_pro, proband, n_anc, ancestor, out, 0, 0, n_dev, devices, stats);
}

}  // extern "C"
