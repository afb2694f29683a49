// engine.cu -- the phi engine and the library-wide part of the C ABI of libgenlib_cuda.so (include/genlib_cuda.h):
// plans, engines, the one-shot genlib_phi / genlib_phi_multi / genlib_phi_over / genlib_phi_groups / genlib_phi_product / genlib_f / genlib_phi_pairs, errors and caches.  gen.gc, gen.occ and gen.rec are
// in gc_engine.cu; the host helpers both share are in runtime.hpp.
//
// The ABI stands where the reference's Julia method stands:
//   phi(pedigree, probandIDs; verbose, compute)            src/compute.jl:233-304
// There is no CPU fallback: without a usable CUDA device every compute entry
// point returns GENLIB_ECUDA.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>

#include "kernels.cuh"
#include "layer_kernel.cuh"
#include "plan.hpp"
#include "runtime.hpp"

using namespace genlib;

thread_local std::string genlib::g_err;
ArenaCache genlib::g_arenas;
int genlib::set_error(int code, const std::string &msg) { return fail(code, msg); }

namespace {

// cudaIpcOpenMemHandle / CloseMemHandle of multi-GB arenas cost tens of milliseconds per peer.
// Arenas are cached, so the same handles come back call after call: keep the mappings open.
class PeerMapCache {
    std::mutex mu_;
    struct Entry { unsigned char handle[64]; int device; void *base; };
    std::vector<Entry> open_;
public:
    cudaError_t map(int device, const void *handle64, void **base) {
        std::lock_guard<std::mutex> g(mu_);
        for (const Entry &en : open_)
            if (en.device == device && std::memcmp(en.handle, handle64, 64) == 0) { *base = en.base; return cudaSuccess; }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, handle64, sizeof h);
        cudaError_t ce = cudaIpcOpenMemHandle(base, h, cudaIpcMemLazyEnablePeerAccess);
        if (ce != cudaSuccess) return ce;
        Entry en; std::memcpy(en.handle, handle64, 64); en.device = device; en.base = *base;
        open_.push_back(en);
        return cudaSuccess;
    }
    void close_all() {
        std::lock_guard<std::mutex> g(mu_);
        for (const Entry &en : open_) {
            int prev = -1; cudaGetDevice(&prev);
            cudaSetDevice(en.device); cudaIpcCloseMemHandle(en.base);
            if (prev >= 0) cudaSetDevice(prev);
        }
        open_.clear();
    }
};
PeerMapCache g_peer_maps;

// Frees a call's transient device buffer (the caller's pointer, null until allocated) on every way out of the call.
template <typename T> struct FreeOnExit {
    T *&p;
    ~FreeOnExit() { if (p) cudaFree(p); }
};

}  // namespace

struct genlib_plan {
    Plan p;
    double ms_plan = 0;
    // genlib_plan_create_async: the plan is made on `worker` and handed over through `stream` (PlanStream); whoever
    // needs the whole plan calls settle() first.  The caller's input arrays stay alive until then.
    std::unique_ptr<PlanStream> stream;
    std::thread worker;
    std::mutex settle_mu;
    int worker_rc = GENLIB_OK;
    std::string worker_err;
    // build_plan into `p` (published through `ps` when given), with its status, message and time from t0.  Out of
    // host memory fails the plan like any planner error and closes a streamed one, so that its readers stop waiting.
    void build(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids, int32_t n_pro,
               const int32_t *proband, int32_t world, int schedule, PlanStream *ps, int planners, double t0,
               const PairList &pairs = PairList{}) {
        try {
            adopt_retired_storage(p);        // the arrays of the last destroyed plan, already paged in
            worker_rc = build_plan(n, father, mother, ids, n_pro, proband, world, schedule, p, worker_err, ps, planners, pairs);
        } catch (const std::bad_alloc &) {
            worker_rc = GENLIB_ENOMEM; worker_err = "out of host memory while planning";
            if (ps) { ps->status.store(GENLIB_ENOMEM); ps->stage.store(2); ps->wake(); }
        }
        ms_plan = now_ms() - t0;
    }
    void settle() {
        std::lock_guard<std::mutex> lk(settle_mu);
        if (worker.joinable()) worker.join();
    }
    bool streaming() const {            // layers are still coming and the bounds hold so far
        return stream && stream->streamed.load() && !stream->overflow.load() && stream->stage.load() != 2;
    }
    ~genlib_plan() { if (worker.joinable()) worker.join(); }
};
inline void settle(const genlib_plan *plan) { if (plan) const_cast<genlib_plan *>(plan)->settle(); }

namespace {
// A reader of a plan that is still being made (PlanStream::consumers): the planner waits for its readers to stop
// before it reallocates anything.
struct StreamConsumer {
    PlanStream *ps = nullptr;
    StreamConsumer() = default;
    explicit StreamConsumer(PlanStream &s) : ps(&s) { ps->consumers.fetch_add(1); }
    StreamConsumer(const StreamConsumer &) = delete;
    StreamConsumer &operator=(StreamConsumer &&o) { reset(); ps = o.ps; o.ps = nullptr; return *this; }
    ~StreamConsumer() { reset(); }
    void reset() { if (ps) { ps->consumers.fetch_sub(1); ps->wake(); ps = nullptr; } }
};
}  // namespace

// launch shape of one layer's persistent kernel (layer_kernel.cuh)
struct LayerLaunch {
    StripArgs s{};
    int prod_warps = 4;                    // producer warps per CTA (template parameter of the layer kernel)
    int grid = 0;
    size_t smem = 0;
    size_t sync_off = 0;                   // ints, into the engine's sync region
};

// the plan's index arrays on the device (views into the arena)
struct IndexBufs {
    DevBuf<int32_t> mem_ind, mem_slot, mem_fam, mem_lrow, fam_pf, fam_pm, fam_q, fam_pf_lrow, fam_pm_lrow, fam_start,
        mt_desc, pro_slot, own_pro_row, live_lrow, tile_map, live_tiles;
    DevBuf<int8_t> fam_pf_owner, fam_pm_owner, live_owner, pro_owner;
    DevBuf<int32_t> pro_lrow;
    DevBuf<int32_t> mem_rank;
    DevBuf<uint8_t> flags;
    DevBuf<double> acc;
    DevBuf<double> fam_kin;                // kScheduleF: Psi[father, mother] per couple (couples whose father row is own)
    DevBuf<int8_t> pair_owner;             // kSchedulePairs: per read, the row's owner, local row and column slot,
    DevBuf<int32_t> pair_lrow, pair_col;
    DevBuf<double> pair_kin;               // and Psi[a, b] (reads whose row is own)
};

struct genlib_engine : IndexBufs {
    const genlib_plan *plan = nullptr;
    int numerics = 0, device = 0, sm_count = 148;
    int rank = 0, world = 1;
    bool attached = false;                 // peers' arenas mapped (always true for one rank)
    size_t esize = 4;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    Arena arena;
    void *A = nullptr;                     // this rank's frontier rows: rows_cap x capacity
    void *Q = nullptr;                     // strip buffers: transposed parent-row pairs, pinned in L2
    size_t q_bytes = 0;
    int32_t *sync = nullptr;               // unit counters and strip completion counts of every layer
    size_t sync_ints = 0;
    std::vector<LayerLaunch> launch;
    bool info_ready = false;               // per-layer byte accounting filled in
#ifdef GENLIB_PROFILE
    long long *prof = nullptr;             // 8 cycle counters per CTA of one layer (GENLIB_PROF_LAYER)
#endif
    unsigned *bar_flags = nullptr;
    unsigned char *fetch_stage[2] = {nullptr, nullptr};
    PeerTable peers{};
    BarrierTable bars{};
    unsigned epoch = 0;
    long long barrier_timeout = (long long)20e9;   // cycles an inter-GPU barrier may wait (GENLIB_BARRIER_TIMEOUT_S)
    bool streamed = false;                 // built on a plan that was still being made: sized by its bounds, uploaded layer by layer
    StreamConsumer consuming;              // registered as a reader of that plan's arrays (until the streamed run ends)
    std::vector<int32_t> own_pro;          // proband indices (output rows) this rank owns, ascending
    std::vector<genlib_layer_info> info;
    std::vector<cudaEvent_t> events;
    genlib_stats stats{};
    bool ran = false;
    int32_t layer_limit = -1;
    ~genlib_engine() {
        consuming.reset();
        for (auto e : events) cudaEventDestroy(e);
        if (stream) cudaStreamSynchronize(stream);
        if (copy_stream) cudaStreamSynchronize(copy_stream);
        g_arenas.release(arena);
        if (stream) cudaStreamDestroy(stream);
        if (copy_stream) cudaStreamDestroy(copy_stream);
    }
};

namespace {

void fill_info(const Layer &L, genlib_layer_info *o) {
    std::memset(o, 0, sizeof *o);
    o->n_new = L.n_new; o->n_fam = L.n_fam; o->live_before = L.live_before; o->carried = L.carried;
    o->ref_founders = L.ref_founders; o->ref_probands = L.ref_probands; o->ref_both = L.ref_both;
    o->alg_elems = L.alg_elems;
}

size_t plan_index_bytes(const Plan &P) {
    return (P.mem_ind.size() * 4 + P.mem_rank.size() + P.fam_pf.size() * 6 + P.fam_start.size() + P.mtile_desc.size() +
            P.pro_slot.size() * 2 + P.live_lrow.size() + P.tile_map.size() + P.live_tiles.size() + P.pair_lrow.size() * 2) * sizeof(int32_t) +
           P.fam_pf.size() * 2 + P.live_owner.size() + P.flags.size() + P.pair_owner.size();
}

// The traffic the layers cannot avoid: s (4 n L + 3 n^2) per layer, for kScheduleF 8 bytes per couple with
// both parents (its Psi[father, mother], read once and written once), for kSchedulePairs 8 bytes per read.
double plan_alg_bytes(const Plan &P, size_t es) {
    double b = P.alg_elems * (double)es;
    if (P.schedule == kScheduleF)
        for (size_t k = 0; k < P.fam_pf.size(); k++) b += (P.fam_pf[k] >= 0 && P.fam_pm[k] >= 0) ? 8.0 : 0.0;
    return b + 8.0 * (double)P.pair_pos.size();
}

// Arena layout of rank g.  The first two regions are what peers address (barrier flags, frontier rows).
constexpr size_t kFlagBytes = 256;
size_t total_rows(const Plan &P, int g) { return (size_t)P.rows_cap[g]; }
size_t a_bytes(const Plan &P, size_t es, int g) { return pad256(total_rows(P, g) * (size_t)P.capacity * es); }
size_t off_A() { return kFlagBytes; }

// ---- launch shapes ---------------------------------------------------------------------------
// The strip buffers are meant to stay in the 126 MB L2; what the buffers of a layer may take of it.  Four
// buffers of a full-width C3 strip (20 MB each) measured best: the slack between the producers and the consumers
// is worth more than the part of the oldest buffer that spills to DRAM (C3: 72.3 ms with four or five buffers,
// 84.9 ms with three kept in a persisting access-policy window; profiles/r02/README.md).
constexpr size_t kStripBudget = (size_t)96 << 20;
constexpr int kMaxGangs = 16, kGangItems = 4;    // gangs of CTAs per layer (at most), producer items a strip should bring every CTA

int env_int(const char *name, int dflt) {
    const char *s = std::getenv(name);
    return s && *s ? std::atoi(s) : dflt;
}

LayerLaunch shape_layer(const Plan &P, int t, int rank, size_t es, int sm_count) {
    const Layer &L = P.layers[t];
    LayerLaunch out;
    StripArgs &s = out.s;
    const int32_t *fb = P.fam_base.data() + L.base_off;
    const int64_t own_nf = fb[rank + 1] - fb[rank];
    if (L.n_new == 0 || own_nf <= 0) return out;
    const bool live = L.live_before > 0;
    const int64_t q_rows = live ? (int64_t)L.n_live_tiles * kPTile : 0;     // rows of a strip buffer
    const size_t pair = 2 * es;
    // strip width: the widest one whose buffers fit the persisting part of L2 at least `min_buf` times (and
    // whose staged tile fits shared memory: 128 parent-row segments of sw pairs <= 64 KB).  A wide strip
    // amortises the per-tile work of the consumers; more buffers give the producers more room to run ahead.
    const size_t min_buf = (size_t)std::max(2, env_int("GENLIB_MIN_NBUF", 2));
    const int sw_cap = es == 4 ? kMaxStrip : kMaxStrip / 2;
    const size_t budget = (size_t)std::max(16, env_int("GENLIB_STRIP_BUDGET_MB", (int)(kStripBudget >> 20))) << 20;
    // (a power of two: the consumers index the strip by shifts, the producers split it into whole items)
    int sw = 8;
    while (2 * sw <= std::min(sw_cap, env_int("GENLIB_MAX_SW", kMaxStrip))) sw *= 2;
    while (sw > 8 && (size_t)q_rows * sw * pair * min_buf > budget) sw >>= 1;
    const size_t strip_bytes = std::max<size_t>((size_t)q_rows * sw * pair, 256);
    s.sw = sw;
    // eight producer warps (and four consumer warps) where the producers have the carried columns to write as well
    {
        const int forced = env_int("GENLIB_PROD_WARPS", 0);
        out.prod_warps = forced == 4 || forced == 8 ? forced : (L.carried > 0 && live ? 8 : 4);
    }
    const size_t cons_bytes = layer_consumer_bytes(sw, es, out.prod_warps);
    const size_t smem_cap = (size_t)227 * 1024 - 2048;      // (static shared memory and the driver's share)
    auto stage_bytes = [&](int ft) { return (size_t)2 * ft * (kPTile * es + 16); };
    // couples per producer item: 32 rows of 512 B (float) / 16 rows of 1 KB (double); one or two items per live
    // tile (ft = sw or sw / 2, at most 32), and the ring must hold two stages of items next to the consumers' part
    s.ft = env_int("GENLIB_FT", es == 4 ? 32 : 16) >= sw || sw == 8 ? sw : sw / 2;
    if (s.ft > 32) s.ft = 32;
    if (s.ft == sw && sw > 8 && cons_bytes + 2 * stage_bytes(s.ft) > smem_cap) s.ft = sw / 2;
    s.n_strips = (int)((own_nf + sw - 1) / sw);
    s.qstride = (int64_t)(strip_bytes / pair);
    // producer items: 2 ft parent rows x one live tile; consumer items: the member tiles
    s.n_pitems = live ? (sw / s.ft) * L.n_live_tiles : 0;
    s.n_citems = L.n_mtiles;
    s.discard = env_int("GENLIB_DISCARD", 1) != 0;     // 0: off
    // One CTA per SM: four producer warps and eight consumer warps (eight and four with carried columns, below).
    // Every CTA of a gang takes part in the hand-over of each of the gang's strips, whether it has an item there or
    // not, and a switch of strips costs a CTA some microseconds of dependent loads: a strip should bring every CTA
    // several items.  Layers with short strips (few live tiles) therefore split the CTAs into G gangs that work on
    // G strips side by side (profiles/r02/README.md: C5 245 -> ... ms, genea140 7.3 -> ... ms); C3-sized layers stay
    // with one gang.
    const int max_buf = (int)std::max<size_t>(2, budget / strip_bytes);
    int G = 1;
    if (live) {
        const int forced = env_int("GENLIB_GANGS", 0);
        const int want_items = std::max(1, env_int("GENLIB_GANG_ITEMS", kGangItems));
        if (forced > 0) G = forced;
        else while (G < kMaxGangs && (int64_t)s.n_pitems * G < (int64_t)want_items * sm_count) G *= 2;
        while (G > 1 && (2 * G > max_buf || s.n_strips < 2 * G || G > sm_count / 4)) G /= 2;
    }
    // (one gang) layers with few items per strip run faster on 7/8 of the SMs (C5: 148 CTAs 246 ms, 128 to 136 CTAs
    // 148 ms; genea140: 8.9 -> 6.4 ms); layers with several items per CTA and strip want every SM (C3: 70.8 ms on
    // 148, 74.3 ms on 132).
    const int few = G == 1 && (sw / s.ft) * L.n_live_tiles < 3 * sm_count / 2 ? sm_count - sm_count / 8 : sm_count;
    const int role_ctas = std::max(1, std::min(sm_count, env_int("GENLIB_CTAS_PER_ROLE", few)));
    while (G > 1 && G > role_ctas) G /= 2;                  // every gang has a CTA of each role
    s.gangs = G;
    // (at most eight buffers per gang: the producer warps of a CTA count themselves off in eight slots by strip)
    s.nbuf = std::min(8 * G, std::max(2 * G, std::min(std::max(2 * G, env_int("GENLIB_MAX_NBUF", 8)), max_buf)) / G * G);
    const int ctas = role_ctas / G;                         // per gang
    s.n_prod = G * std::min(ctas, s.n_pitems);
    s.n_cons = G * std::min(ctas, s.n_citems);
    const size_t stage = stage_bytes(s.ft);                 // (two of them fit: ft above)
    s.stages = (int)std::max<size_t>(2, std::min<size_t>((size_t)std::min(kMaxStages, env_int("GENLIB_STAGES", kMaxStages)), (smem_cap - cons_bytes) / stage));
    s.ring_off = (int32_t)cons_bytes;
    out.smem = cons_bytes + (size_t)s.stages * stage;
    out.grid = std::max(s.n_prod, s.n_cons);
    s.timeout_cycles = (long long)4e9;                     // ~2 s: a lost dependency becomes GENLIB_ECUDA, not a hang
    return out;
}

size_t strip_buffer_bytes(const LayerLaunch &ll, size_t es) { return (size_t)ll.s.nbuf * (size_t)ll.s.qstride * 2 * es; }

// Places the plan's index arrays behind `cur` (a null cursor just measures).  A streamed plan (PlanStream) is
// sized by what its arrays have RESERVED: their final sizes are not known yet, the reserves are upper bounds.
unsigned char *place_arrays(IndexBufs &B, const Plan &P, bool streamed, unsigned char *cur) {
    auto cnt = [&](const auto &v) { return streamed ? v.capacity() : v.size(); };
    const size_t npro = P.pro_ind.size();
    B.mem_ind.place(cur, cnt(P.mem_ind)); B.mem_slot.place(cur, cnt(P.mem_slot)); B.mem_fam.place(cur, cnt(P.mem_fam));
    B.mem_lrow.place(cur, cnt(P.mem_lrow)); B.mem_rank.place(cur, cnt(P.mem_rank));
    B.fam_pf.place(cur, cnt(P.fam_pf)); B.fam_pm.place(cur, cnt(P.fam_pm));
    B.fam_q.place(cur, cnt(P.fam_q));
    B.fam_pf_lrow.place(cur, cnt(P.fam_pf_lrow)); B.fam_pm_lrow.place(cur, cnt(P.fam_pm_lrow));
    B.fam_start.place(cur, cnt(P.fam_start));
    B.mt_desc.place(cur, cnt(P.mtile_desc));
    B.pro_slot.place(cur, npro); B.own_pro_row.place(cur, npro);
    B.live_lrow.place(cur, cnt(P.live_lrow)); B.tile_map.place(cur, cnt(P.tile_map));
    B.live_tiles.place(cur, cnt(P.live_tiles));
    B.fam_pf_owner.place(cur, cnt(P.fam_pf_owner)); B.fam_pm_owner.place(cur, cnt(P.fam_pm_owner));
    B.live_owner.place(cur, cnt(P.live_owner));
    B.flags.place(cur, cnt(P.flags)); B.acc.place(cur, 4);
    B.pro_owner.place(cur, npro); B.pro_lrow.place(cur, npro);
    if (P.schedule == kScheduleF) B.fam_kin.place(cur, cnt(P.fam_pf));
    if (P.schedule == kSchedulePairs) {
        const size_t K = P.pair_pos.size();                    // (sized at the list's length before any layer is published)
        B.pair_owner.place(cur, K); B.pair_lrow.place(cur, K); B.pair_col.place(cur, K); B.pair_kin.place(cur, K);
    }
    return cur;
}

// strip buffers and sync words of all layers: exact for a finished plan, bounds for a streamed one (shape_layer
// never takes more: at most max(budget, two buffers of the narrowest strip), 16 words per strip of >= 8 couples)
void scratch_sizes(const Plan &P, size_t es, int g, int sm_count, bool streamed, size_t &q_bytes, size_t &sync_ints) {
    q_bytes = 256;
    sync_ints = (P.layers.size() + 15) / 16 * 16;                             // the layers' error words come first
    if (streamed) {
        const size_t budget = (size_t)std::max(16, env_int("GENLIB_STRIP_BUDGET_MB", (int)(kStripBudget >> 20))) << 20;
        q_bytes = std::max(budget, (size_t)2 * (size_t)P.capacity * 8 * 2 * es) + 256;
        sync_ints += 16 * (P.fam_pf.capacity() / 8 + 2 * P.layers.size());
        return;
    }
    for (int t = 0; t < (int)P.layers.size(); t++) {
        const LayerLaunch ll = shape_layer(P, t, g, es, sm_count);
        if (ll.grid == 0) continue;
        q_bytes = std::max(q_bytes, strip_buffer_bytes(ll, es));
        sync_ints += 16 * (size_t)ll.s.n_strips;
    }
}

size_t engine_bytes(const Plan &P, int numerics, int g, int sm_count = 148, bool streamed = false) {
    const size_t es = numerics == GENLIB_NUMERICS_FP64 ? 8 : 4;
    size_t q, sync_ints;
    scratch_sizes(P, es, g, sm_count, streamed, q, sync_ints);
    size_t b = kFlagBytes + a_bytes(P, es, g) + pad256(q) + pad256(sync_ints * sizeof(int32_t));
    b += 2 * pad256(kFetchStageBytes);                                         // proband staging
    IndexBufs dummy;
    b += (size_t)(place_arrays(dummy, P, streamed, nullptr) - (unsigned char *)nullptr);
    return b;
}

LayerArgs layer_args(const genlib_engine &E, int t) {
    const Plan &P = E.plan->p;
    const Layer &L = P.layers[t];
    LayerArgs a;
    std::memset(&a, 0, sizeof a);
    a.n_new = L.n_new; a.n_fam = L.n_fam; a.rt_lo = L.rt_lo;
    a.any_carried = L.carried > 0;
    const int32_t *fb = P.fam_base.data() + L.base_off, *mb = P.mem_base.data() + L.base_off;
    a.own_f0 = fb[E.rank]; a.own_nf = fb[E.rank + 1] - fb[E.rank];
    a.own_m0 = mb[E.rank]; a.own_nm = mb[E.rank + 1] - mb[E.rank];
    a.mem_ind = E.mem_ind.p + L.mem_off; a.mem_slot = E.mem_slot.p + L.mem_off; a.mem_fam = E.mem_fam.p + L.mem_off;
    a.mem_lrow = E.mem_lrow.p + L.mem_off;
    a.fam_pf = E.fam_pf.p + L.fam_off; a.fam_pm = E.fam_pm.p + L.fam_off;
    a.fam_q = reinterpret_cast<const int2 *>(E.fam_q.p) + L.fam_off;
    a.fam_pf_owner = E.fam_pf_owner.p + L.fam_off; a.fam_pm_owner = E.fam_pm_owner.p + L.fam_off;
    a.fam_pf_lrow = E.fam_pf_lrow.p + L.fam_off; a.fam_pm_lrow = E.fam_pm_lrow.p + L.fam_off;
    a.fam_start = E.fam_start.p + L.fam_off + t;
    a.flags = E.flags.p + L.flag_off;
    a.live_owner = E.live_owner.p + L.flag_off; a.live_lrow = E.live_lrow.p + L.flag_off;
    a.mt_desc = reinterpret_cast<const int4 *>(E.mt_desc.p) + L.mtile_off;
    a.n_mtiles = L.n_mtiles;
    return a;
}

int launch_barrier(genlib_engine &E) {
    if (E.world == 1) return GENLIB_OK;
    E.epoch++;
    barrier_kernel<<<1, 32, 0, E.stream>>>(E.bars, E.rank, E.world, E.epoch, E.barrier_timeout);
    return GENLIB_OK;
}

template <typename T>
auto layer_function(const Plan &P, int prod_warps) {
    const bool stored = sparse_schedule(P.schedule);           // sparse_phi's arithmetic (Float32 halves of stored values)
    if (prod_warps == 8) return stored ? layer_kernel<T, true, 8> : layer_kernel<T, false, 8>;
    return stored ? layer_kernel<T, true, 4> : layer_kernel<T, false, 4>;
}

template <typename T>
int prepare_launches(genlib_engine &E, size_t smem_max) {
    for (int pw : {4, 8}) {
        auto layer_fn = layer_function<T>(E.plan->p, pw);
        CU(cudaFuncSetAttribute(layer_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
        CU(cudaFuncSetAttribute(layer_fn, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    }
    CU(cudaMemsetAsync(E.sync, 0, std::max<size_t>(E.sync_ints, 1) * sizeof(int32_t), E.stream));
    return GENLIB_OK;
}

// kSchedulePairs: the reads of layer t (t == S: after the last layer and its barrier), while their rows hold them
// (such a plan's engine stores Float64: create_engine refuses any other numerics)
void launch_pair_reads(genlib_engine &E, int t, int &launches) {
    const Plan &P = E.plan->p;
    if (P.schedule != kSchedulePairs) return;
    const int64_t i0 = P.pair_start[(size_t)t], nr = P.pair_start[(size_t)t + 1] - i0;
    if (nr == 0) return;
    pair_kinship_kernel<<<(unsigned)((nr + kThreads - 1) / kThreads), kThreads, 0, E.stream>>>(
        static_cast<const double *>(E.A), P.capacity, E.pair_owner.p + i0, E.pair_lrow.p + i0, E.pair_col.p + i0, nr, E.rank,
        E.pair_kin.p + i0);
    launches++;
}

// one generation step: the layer kernel (and sparse_phi's misfiled pairs), then the inter-GPU barrier
template <typename T>
int launch_layer(genlib_engine &E, int t, bool timed, size_t &ev, int &launches) {
    const Plan &P = E.plan->p;
    const Layer &L = P.layers[t];
    launch_pair_reads(E, t, launches);                          // the pairs read before this layer
    if (L.n_new == 0) return GENLIB_OK;
    T *A = static_cast<T *>(E.A);
    const int64_t ld = P.capacity;
    LayerArgs a = layer_args(E, t);
    LayerLaunch &ll = E.launch[t];
    auto layer_fn = layer_function<T>(P, ll.prod_warps);
    if (P.schedule == kScheduleF && L.n_fam > 0) {              // the parents' kinships, while both rows are live
        couple_kinship_kernel<T><<<(unsigned)((L.n_fam + kThreads - 1) / kThreads), kThreads, 0, E.stream>>>(
            A, ld, E.fam_pf_owner.p + L.fam_off, E.fam_pf_lrow.p + L.fam_off, E.fam_pm.p + L.fam_off, L.n_fam, E.rank,
            E.fam_kin.p + L.fam_off);
        launches++;
    }
    if (timed) CU(cudaEventRecord(E.events[ev++], E.stream));
    if (ll.grid > 0) {
        ll.s.Q = E.Q;
        ll.s.sync = E.sync + ll.sync_off;
        ll.s.err = E.sync + t;
        ll.s.live_tiles = E.live_tiles.p + L.ltile_off;
#ifdef GENLIB_PROFILE
        ll.s.prof = (t == env_int("GENLIB_PROF_LAYER", 5)) ? E.prof : nullptr;
#else
        ll.s.prof = nullptr;
#endif
        layer_fn<<<ll.grid, kLayerThreads, ll.smem, E.stream>>>(A, ld, E.peers, a, ll.s);
        launches++;
        if (P.schedule == kScheduleSparsePhi && L.n_new > 1 && a.own_nm > 0) {   // the reference's misfiled kinships read as 0
            dim3 mgrid((unsigned)a.own_nm, (unsigned)std::min<int64_t>((L.n_new + 4 * kThreads - 1) / (4 * kThreads), 65535));
            misfile_kernel<T><<<mgrid, kThreads, 0, E.stream>>>(A, ld, E.mem_rank.p + L.mem_off, a);
            launches++;
        }
    }
    if (timed) CU(cudaEventRecord(E.events[ev++], E.stream));
    launch_barrier(E);                 // all new rows (and mirrored columns) exist everywhere before the next layer reads them
    if (timed) CU(cudaEventRecord(E.events[ev++], E.stream));
    return GENLIB_OK;
}

template <typename T>
int launch_layers(genlib_engine &E, bool timed) {
    const Plan &P = E.plan->p;
    size_t smem_max = 0;
    for (const LayerLaunch &ll : E.launch) smem_max = std::max(smem_max, ll.smem);
    if (int rc = prepare_launches<T>(E, smem_max)) return rc;
    int launches = 0;
    size_t ev = 0;
    const int S = (int)P.layers.size();
    for (int t = 0; t < S; t++) {
        if (E.layer_limit >= 0 && t >= E.layer_limit) break;
        if (int rc = launch_layer<T>(E, t, timed, ev, launches)) return rc;
    }
    if (E.layer_limit < 0 || E.layer_limit >= S) launch_pair_reads(E, S, launches);   // the pairs read after the last layer
    CU(cudaGetLastError());
    E.stats.kernel_launches = launches;
#ifdef GENLIB_PROFILE
    {
        CU(cudaStreamSynchronize(E.stream));
        std::vector<long long> h(8 * 2 * 160);                      // [CTA][role][phase]
        CU(cudaMemcpy(h.data(), E.prof, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
        const LayerLaunch &pl = E.launch[env_int("GENLIB_PROF_LAYER", 5)];
        double acc[2][8] = {};
        for (int b = 0; b < pl.grid; b++) for (int r = 0; r < 2; r++) for (int i = 0; i < 8; i++) acc[r][i] += (double)h[((size_t)b * 2 + r) * 8 + i];
        std::fprintf(stderr, "[prof] producers %d consumers %d strips %d (avg kcycles per CTA)\n", pl.s.n_prod, pl.s.n_cons, pl.s.n_strips);
        std::fprintf(stderr, "[prof] producer: other %.0f wait_consumers %.0f mbar %.0f issue %.0f transpose %.0f member_rows %.0f mirror %.0f\n",
                     acc[0][0] / pl.s.n_prod / 1e3, acc[0][1] / pl.s.n_prod / 1e3, acc[0][2] / pl.s.n_prod / 1e3, acc[0][3] / pl.s.n_prod / 1e3, acc[0][4] / pl.s.n_prod / 1e3, acc[0][5] / pl.s.n_prod / 1e3, acc[0][6] / pl.s.n_prod / 1e3);
        std::fprintf(stderr, "[prof] consumer: other %.0f wait_producers %.0f switch %.0f stage_wait %.0f compute %.0f stage_issue %.0f expand %.0f mirror %.0f\n",
                     acc[1][0] / pl.s.n_cons / 1e3, acc[1][1] / pl.s.n_cons / 1e3, acc[1][2] / pl.s.n_cons / 1e3, acc[1][3] / pl.s.n_cons / 1e3, acc[1][4] / pl.s.n_cons / 1e3, acc[1][5] / pl.s.n_cons / 1e3, acc[1][6] / pl.s.n_cons / 1e3, acc[1][7] / pl.s.n_cons / 1e3);
    }
#endif
    return GENLIB_OK;
}

int upload_layers(genlib_engine &E, int t0, int t1);
int upload_probands(genlib_engine &E);
int upload_pair_reads(genlib_engine &E, int64_t i0, int64_t i1);

// what the kernels of a run left in their error words
int check_device_errors(genlib_engine &E) {
    int32_t errw = 0;                                     // a dependency inside a layer kernel timed out
    std::vector<int32_t> words(E.launch.size(), 0);
    if (!words.empty()) CU(cudaMemcpy(words.data(), E.sync, words.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
    for (int32_t w : words) if (w) { errw = w; break; }
    if (errw) return fail(GENLIB_ECUDA, "the layer kernel reported error " + std::to_string(errw) + " (1: a strip dependency did not arrive, 2: a bulk copy did not complete)");
    if (E.world > 1) {
        unsigned berr = 0;
        CU(cudaMemcpy(&berr, E.bar_flags + kMaxWorld, sizeof berr, cudaMemcpyDeviceToHost));
        if (berr) return fail(GENLIB_ECOMM, "a rank did not reach the inter-GPU barrier within the time limit");
    }
    return GENLIB_OK;
}

constexpr int kRestart = -1000;      // internal: a bound of the streamed plan did not hold, run again on the finished plan

// The layers of a plan that is still being made (PlanStream): wait for a layer, upload its slice of the index
// arrays, shape and launch it, while the planner works on the next ones.  The caller has registered as a consumer.
template <typename T>
int run_streamed(genlib_engine &E, PlanStream &ps) {
    const Plan &P = E.plan->p;
    const int S = (int)P.layers.size();
    const size_t nev = E.events.size();
    CU(cudaEventRecord(E.events[nev - 2], E.stream));
    if (int rc = prepare_launches<T>(E, (size_t)227 * 1024 - 2048)) return rc;
    int launches = 0, done = 0;
    size_t ev = 0, sync_at = (P.layers.size() + 15) / 16 * 16;
    while (done < S) {
        ps.wait([&] { return ps.layers_done.load(std::memory_order_acquire) > done || ps.overflow.load() || ps.stage.load() == 2; });
        // (after `overflow` nothing more is published: every consumer then launches the same layers, so the
        //  inter-GPU barriers of a sharded run still pair up before it is abandoned)
        const bool overflow = ps.overflow.load();
        const int avail = ps.layers_done.load(std::memory_order_acquire);
        if (avail == done && !overflow)
            return ps.status.load() != GENLIB_OK ? ps.status.load() : fail(GENLIB_EINVAL, "internal: the planner ended before the last layer");
        bool too_small = false;
        if (int rc = upload_layers(E, done, avail)) return rc;
        for (int t = done; t < avail; t++) {
            LayerLaunch &ll = E.launch[(size_t)t];
            ll = shape_layer(P, t, E.rank, E.esize, E.sm_count);
            if (ll.grid > 0) {
                ll.sync_off = sync_at;
                sync_at += 16 * (size_t)ll.s.n_strips;
                if (strip_buffer_bytes(ll, E.esize) > E.q_bytes || sync_at > E.sync_ints) too_small = true;   // (the bounds of scratch_sizes)
            }
            if (too_small && E.world == 1) break;
            if (too_small) return fail(GENLIB_EINVAL, "internal: scratch bounds of a streamed, sharded plan");
            fill_info(P.layers[(size_t)t], &E.info[(size_t)t]);
            if (int rc = launch_layer<T>(E, t, false, ev, launches)) return rc;
        }
        done = avail;
        if (overflow || too_small) { cudaStreamSynchronize(E.stream); return kRestart; }
    }
    ps.wait([&] { return ps.stage.load() == 2; });              // the probands' homes close the plan
    if (ps.status.load() != GENLIB_OK) return ps.status.load();
    if (ps.overflow.load()) { cudaStreamSynchronize(E.stream); return kRestart; }
    if (int rc = upload_probands(E)) return rc;
    launch_pair_reads(E, S, launches);                          // the pairs read after the last layer
    CU(cudaGetLastError());
    E.stats.kernel_launches = launches;
    CU(cudaEventRecord(E.events[nev - 1], E.stream));
    CU(cudaStreamSynchronize(E.stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, E.events[nev - 2], E.events[nev - 1]));
    E.stats.ms_kernels = ms;                                    // first launch to last: includes waiting for the planner
    E.stats.row_updates = P.row_updates; E.stats.alg_bytes = plan_alg_bytes(P, E.esize);
    E.stats.h2d_bytes = (int64_t)plan_index_bytes(P);
    return GENLIB_OK;
}

// Rows of this rank's probands (own_pro order), all proband columns, streamed to host memory.
template <typename T, typename O>
int fetch_rows(genlib_engine &E, O *out) {
    const Plan &P = E.plan->p;
    const int32_t n = P.n_unique, nown = (int32_t)E.own_pro.size();
    if (n == 0 || nown == 0) return GENLIB_OK;
    const size_t row_bytes = (size_t)n * sizeof(O);
    int32_t rows_per = (int32_t)std::max<size_t>(1, std::min<size_t>((size_t)nown, kFetchStageBytes / row_bytes));
    if ((size_t)rows_per * row_bytes > kFetchStageBytes) return fail(GENLIB_EINVAL, "proband row does not fit the staging buffer");
    rows_per = std::min(rows_per, 65535);
    int rc = staged_d2h(E.stream, E.copy_stream, reinterpret_cast<O *>(E.fetch_stage[0]), reinterpret_cast<O *>(E.fetch_stage[1]),
                        nown, rows_per, "proband fetch",
        [&](O *stage, int64_t r0, int64_t nr) {
            dim3 grid((unsigned)std::min<int32_t>((n + 255) / 256, 64), (unsigned)nr);
            gather_kernel<T, O><<<grid, 256, 0, E.stream>>>(static_cast<const T *>(E.A), P.capacity, E.own_pro_row.p, E.pro_slot.p,
                                                           n, (int32_t)r0, (int32_t)nr, stage);
        },
        [&](const O *stage, int64_t r0, int64_t nr) {
            return cudaMemcpyAsync(out + (size_t)r0 * n, stage, (size_t)nr * row_bytes, cudaMemcpyDeviceToHost, E.copy_stream);
        });
    if (rc == GENLIB_OK) E.stats.d2h_bytes += (int64_t)nown * (int64_t)row_bytes;
    return rc;
}

// Output rows [u0, u1) of the proband matrix, whoever owns them (peer reads), to host memory at their
// final place: out + u * n.  Used when one process drives all devices (genlib_phi_multi).
template <typename T, typename O>
int fetch_block(genlib_engine &E, int32_t u0, int32_t u1, O *out) {
    const Plan &P = E.plan->p;
    const int32_t n = P.n_unique;
    if (n == 0 || u1 <= u0) return GENLIB_OK;
    const size_t row_bytes = (size_t)n * sizeof(O);
    int32_t rows_per = (int32_t)std::max<size_t>(1, std::min<size_t>((size_t)(u1 - u0), kFetchStageBytes / row_bytes));
    if ((size_t)rows_per * row_bytes > kFetchStageBytes) return fail(GENLIB_EINVAL, "proband row does not fit the staging buffer");
    rows_per = std::min(rows_per, 65535);
    int rc = staged_d2h(E.stream, E.copy_stream, reinterpret_cast<O *>(E.fetch_stage[0]), reinterpret_cast<O *>(E.fetch_stage[1]),
                        u1 - u0, rows_per, "proband fetch",
        [&](O *stage, int64_t i0, int64_t nr) {
            dim3 grid((unsigned)std::min<int32_t>((n + 255) / 256, 64), (unsigned)nr);
            gather_peer_kernel<T, O><<<grid, 256, 0, E.stream>>>(E.peers, P.capacity, E.pro_owner.p, E.pro_lrow.p, E.pro_slot.p, n,
                                                                u0 + (int32_t)i0, (int32_t)nr, stage);
        },
        [&](const O *stage, int64_t i0, int64_t nr) {
            return cudaMemcpyAsync(out + (size_t)(u0 + i0) * n, stage, (size_t)nr * row_bytes, cudaMemcpyDeviceToHost, E.copy_stream);
        });
    if (rc == GENLIB_OK) E.stats.d2h_bytes += (int64_t)(u1 - u0) * (int64_t)row_bytes;
    return rc;
}

// ---- gen.phiOver (genlib_phi_over) ----------------------------------------------------------------------
// One device's share of the selection: its own proband rows (own_pro order), their per-row counts and then offsets,
// and on the device the same offsets, the rows' positions in the proband list and the rows that have pairs.
struct OverRows {
    int device = -1;
    const std::vector<int32_t> *own = nullptr;   // the engine's own_pro
    std::vector<int64_t> off;                    // nown + 1: the counts after the first pass, exclusive offsets after
    int64_t base = 0;                            // (several devices) where this device's pairs start in the scratch
    int64_t *d_off = nullptr;                    // one allocation: d_off (nown + 1), d_index (nown), d_sel (nown)
    int32_t *d_index = nullptr, *d_sel = nullptr;
    OverRows() = default;
    OverRows(const OverRows &) = delete;
    ~OverRows() {
        if (!d_off) return;
        DeviceGuard guard;
        guard.enter(device);
        cudaFree(d_off);
    }
};

// First pass: each own row's count of columns j > i with M[i, j] >= threshold, to R.off.
template <typename T, typename O>
int phi_over_count(genlib_engine &E, OverRows &R, double threshold) {
    const Plan &P = E.plan->p;
    const int32_t nown = (int32_t)E.own_pro.size();
    R.device = E.device;
    R.own = &E.own_pro;
    R.off.assign((size_t)nown + 1, 0);
    if (nown == 0) return GENLIB_OK;
    CU(cudaMalloc(&R.d_off, (size_t)(nown + 1) * sizeof(int64_t) + 2 * (size_t)nown * sizeof(int32_t)));
    R.d_index = reinterpret_cast<int32_t *>(R.d_off + nown + 1);
    R.d_sel = R.d_index + nown;
    CU(cudaMemcpyAsync(R.d_index, E.own_pro.data(), (size_t)nown * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    phi_over_count_kernel<T, O><<<(unsigned)nown, kThreads, 0, E.stream>>>(static_cast<const T *>(E.A), P.capacity, E.own_pro_row.p,
                                                                           R.d_index, E.pro_slot.p, P.n_unique, threshold, R.d_off);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(R.off.data(), R.d_off, (size_t)nown * sizeof(int64_t), cudaMemcpyDeviceToHost, E.stream));
    CU(cudaStreamSynchronize(E.stream));
    E.stats.d2h_bytes += (int64_t)nown * (int64_t)sizeof(int64_t);
    return GENLIB_OK;
}

// Second pass (R.off holds the offsets by now): the device's pairs in its own row order to col / val in host memory,
// through the staging buffers, in blocks of rows whose pairs fit one buffer (columns first, then the values).
template <typename T, typename O>
int phi_over_select(genlib_engine &E, OverRows &R, double threshold, int32_t *col, O *val) {
    const Plan &P = E.plan->p;
    const int32_t nown = (int32_t)E.own_pro.size();
    std::vector<int32_t> sel;                                    // own rows with at least one pair
    for (int32_t r = 0; r < nown; r++)
        if (R.off[(size_t)r + 1] > R.off[(size_t)r]) sel.push_back(r);
    if (sel.empty()) return GENLIB_OK;
    const int64_t cap = (int64_t)(kFetchStageBytes / (sizeof(int32_t) + sizeof(O))) / 2 * 2;   // (values 8-byte aligned)
    auto first = [&](size_t k) { return R.off[(size_t)sel[k]]; };
    auto last = [&](size_t k) { return R.off[(size_t)sel[k] + 1]; };
    std::vector<size_t> blk{0};                                  // blocks of sel: [blk[b], blk[b + 1])
    for (size_t k = 0; k < sel.size(); k++) {
        if (last(k) - first(k) > cap) return fail(GENLIB_EINVAL, "the pairs of one proband row do not fit the staging buffer");
        if (last(k) - first(blk.back()) > cap) blk.push_back(k);
    }
    blk.push_back(sel.size());
    CU(cudaMemcpyAsync(R.d_off, R.off.data(), ((size_t)nown + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, E.stream));
    CU(cudaMemcpyAsync(R.d_sel, sel.data(), sel.size() * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    auto cols_of = [](unsigned char *s) { return reinterpret_cast<int32_t *>(s); };
    auto vals_of = [&](unsigned char *s) { return reinterpret_cast<O *>(s + (size_t)cap * sizeof(int32_t)); };
    int rc = staged_d2h(E.stream, E.copy_stream, E.fetch_stage[0], E.fetch_stage[1], (int64_t)blk.size() - 1, 1, "phiOver fetch",
        [&](unsigned char *stage, int64_t b, int64_t) {
            const size_t k0 = blk[(size_t)b], k1 = blk[(size_t)b + 1];
            phi_over_select_kernel<T, O><<<(unsigned)(k1 - k0), kThreads, 0, E.stream>>>(
                static_cast<const T *>(E.A), P.capacity, E.own_pro_row.p, R.d_index, E.pro_slot.p, P.n_unique, threshold,
                R.d_sel + k0, R.d_off, first(k0), cols_of(stage), vals_of(stage));
        },
        [&](unsigned char *stage, int64_t b, int64_t) {
            const int64_t a = first(blk[(size_t)b]), m = last(blk[(size_t)b + 1] - 1) - a;
            cudaError_t ce = cudaMemcpyAsync(col + a, cols_of(stage), (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToHost, E.copy_stream);
            if (ce == cudaSuccess) ce = cudaMemcpyAsync(val + a, vals_of(stage), (size_t)m * sizeof(O), cudaMemcpyDeviceToHost, E.copy_stream);
            return ce;
        });
    if (rc == GENLIB_OK) E.stats.d2h_bytes += R.off[(size_t)nown] * (int64_t)(sizeof(int32_t) + sizeof(O));
    return rc;
}

// ---- gen.phiMeanGroups (genlib_phi_groups) --------------------------------------------------------------------
// The grouped column list (phi_groups_kernel): the probands' frontier slots in group-major order (list order within a
// group), where each group starts, and where each list position went.
struct GroupColumns {
    std::vector<int32_t> gcol, gptr, gat;
};

// This device's S rows (own_pro order) to host rows dst[0, nown) of G doubles each, in blocks of rows that fit one
// staging buffer.
template <typename T>
int phi_groups_rows(genlib_engine &E, const GroupColumns &C, double *dst) {
    const Plan &P = E.plan->p;
    const int32_t np = P.n_unique, nown = (int32_t)E.own_pro.size(), G = (int32_t)C.gptr.size() - 1;
    if (nown == 0) return GENLIB_OK;
    const size_t row_bytes = (size_t)G * sizeof(double);
    if (row_bytes > kFetchStageBytes) return fail(GENLIB_EINVAL, "the group means of one proband do not fit the staging buffer");
    const int64_t rows_per = (int64_t)std::min<size_t>((size_t)nown, kFetchStageBytes / row_bytes);
    int32_t *d = nullptr;                                        // d_index (nown), gcol (np), gat (np), gptr (G + 1)
    FreeOnExit<int32_t> free_d{d};
    CU(cudaMalloc(&d, ((size_t)nown + 2 * (size_t)np + (size_t)G + 1) * sizeof(int32_t)));
    int32_t *d_index = d, *d_gcol = d + nown, *d_gat = d_gcol + np, *d_gptr = d_gat + np;
    CU(cudaMemcpyAsync(d_index, E.own_pro.data(), (size_t)nown * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    CU(cudaMemcpyAsync(d_gcol, C.gcol.data(), (size_t)np * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    CU(cudaMemcpyAsync(d_gat, C.gat.data(), (size_t)np * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    CU(cudaMemcpyAsync(d_gptr, C.gptr.data(), ((size_t)G + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    const int rc = staged_d2h(E.stream, E.copy_stream, reinterpret_cast<double *>(E.fetch_stage[0]),
                              reinterpret_cast<double *>(E.fetch_stage[1]), nown, rows_per, "phiMeanGroups fetch",
        [&](double *stage, int64_t r0, int64_t nr) {
            phi_groups_kernel<T><<<(unsigned)nr, kThreads, 0, E.stream>>>(static_cast<const T *>(E.A), P.capacity, E.own_pro_row.p,
                                                                          d_index, d_gcol, d_gat, d_gptr, G, np, (int32_t)r0, stage);
        },
        [&](const double *stage, int64_t r0, int64_t nr) {
            return cudaMemcpyAsync(dst + (size_t)r0 * G, stage, (size_t)nr * row_bytes, cudaMemcpyDeviceToHost, E.copy_stream);
        });
    if (rc == GENLIB_OK) E.stats.d2h_bytes += (int64_t)nown * (int64_t)row_bytes;
    return rc;
}

// ---- gen.phiProduct (genlib_phi_product, genlib_engine_phi_product) ---------------------------------------------
// This device's rows of Y = M X (own_pro order) to host rows dst[0, nown) of k doubles each, and M[i, i] to diag[0,
// nown) when diag is not null, in blocks of rows that fit one staging buffer (each block's Y rows, then its diagonal).
// X (P x k, list order) is on the device for the call only, outside the arena.
template <typename T>
int phi_product_rows(genlib_engine &E, const double *X, int32_t k, double *dst, double *diag) {
    const Plan &P = E.plan->p;
    const int32_t np = P.n_unique, nown = (int32_t)E.own_pro.size();
    if (nown == 0 || (k == 0 && !diag)) return GENLIB_OK;
    const size_t row_bytes = ((size_t)k + (diag ? 1 : 0)) * sizeof(double);
    if (row_bytes > kFetchStageBytes) return fail(GENLIB_EINVAL, "phiProduct: one proband's row of the product does not fit the staging buffer");
    const int64_t rows_per = (int64_t)std::min<size_t>((size_t)nown, kFetchStageBytes / row_bytes);
    const size_t x_bytes = (size_t)np * (size_t)k * sizeof(double);
    double *d_x = nullptr;                                       // X (P k), then d_index (nown)
    FreeOnExit<double> free_x{d_x};
    if (cudaMalloc(&d_x, x_bytes + (size_t)nown * sizeof(int32_t)) != cudaSuccess) {
        cudaGetLastError();
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        return fail(GENLIB_ENOMEM, "phiProduct: X needs " + std::to_string(x_bytes) + " bytes on the device next to the engine's arena, " +
                                   std::to_string(free_b) + " bytes are free");
    }
    int32_t *d_index = reinterpret_cast<int32_t *>(reinterpret_cast<unsigned char *>(d_x) + x_bytes);
    if (k > 0) CU(cudaMemcpyAsync(d_x, X, x_bytes, cudaMemcpyHostToDevice, E.stream));
    CU(cudaMemcpyAsync(d_index, E.own_pro.data(), (size_t)nown * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    const int rc = staged_d2h(E.stream, E.copy_stream, reinterpret_cast<double *>(E.fetch_stage[0]),
                              reinterpret_cast<double *>(E.fetch_stage[1]), nown, rows_per, "phiProduct fetch",
        [&](double *stage, int64_t r0, int64_t nr) {
            const T *A = static_cast<const T *>(E.A);
            double *d = diag ? stage + (size_t)nr * k : nullptr;
            // One column: one row per CTA, as rowsum_kernel reads the block.  Several: 4 rows per CTA share each X load.
            if (k <= 1)
                phi_product_kernel<T, 1, 1><<<(unsigned)nr, kThreads, 0, E.stream>>>(A, P.capacity, E.own_pro_row.p, d_index, E.pro_slot.p,
                                                                                   np, d_x, k, (int32_t)r0, (int32_t)nr, stage, d);
            else
                phi_product_kernel<T, 8, 4><<<(unsigned)((nr + 3) / 4) * (unsigned)((k + 7) / 8), kThreads, 0, E.stream>>>(
                    A, P.capacity, E.own_pro_row.p, d_index, E.pro_slot.p, np, d_x, k, (int32_t)r0, (int32_t)nr, stage, d);
        },
        [&](const double *stage, int64_t r0, int64_t nr) {
            cudaError_t ce = cudaSuccess;
            if (k > 0) ce = cudaMemcpyAsync(dst + (size_t)r0 * k, stage, (size_t)nr * k * sizeof(double), cudaMemcpyDeviceToHost, E.copy_stream);
            if (ce == cudaSuccess && diag)
                ce = cudaMemcpyAsync(diag + r0, stage + (size_t)nr * k, (size_t)nr * sizeof(double), cudaMemcpyDeviceToHost, E.copy_stream);
            return ce;
        });
    if (rc == GENLIB_OK) {
        E.stats.h2d_bytes += (int64_t)x_bytes;
        E.stats.d2h_bytes += (int64_t)nown * (int64_t)row_bytes;
    }
    return rc;
}

// Several devices of one process copy their own proband rows to a list-ordered output, device after device in own_pro
// order (one device: row i lands at row i); afterwards the host moves the rows to list order in place.
struct ListOrderRows {
    std::vector<int64_t> base;      // device g's rows land at [base[g], base[g + 1])
    std::vector<int32_t> at;        // at[p]: the list position of the row landed at p
    void prepare(const Plan &P, int n_dev) {
        const int32_t np = P.n_unique;        // (no duplicates: the plan's proband u is list position u)
        base.assign((size_t)n_dev + 1, 0);
        for (int32_t u = 0; u < np; u++) base[(size_t)P.pro_owner[(size_t)u] + 1]++;
        for (int g = 0; g < n_dev; g++) base[(size_t)g + 1] += base[(size_t)g];
        at.resize((size_t)np);
        std::vector<int64_t> fill(base.begin(), base.end() - 1);
        for (int32_t u = 0; u < np; u++) at[(size_t)fill[(size_t)P.pro_owner[(size_t)u]]++] = u;   // own_pro: ascending
    }
    // every output (rows of `width` doubles; a null one is skipped) moved by the same permutation; runs once
    void to_list_order(std::initializer_list<std::pair<double *, size_t>> outs) {
        for (int32_t p = 0; p < (int32_t)at.size(); p++)
            while (at[(size_t)p] != p) {
                const int32_t q = at[(size_t)p];
                for (const auto &o : outs)
                    if (o.first && o.second)
                        std::swap_ranges(o.first + (size_t)p * o.second, o.first + (size_t)(p + 1) * o.second, o.first + (size_t)q * o.second);
                std::swap(at[(size_t)p], at[(size_t)q]);
            }
    }
};

// Compulsory traffic of every layer on this rank (genlib_layer_info), from the plan.
void account_layers(genlib_engine &E) {
    if (E.info_ready) return;
    const Plan &P = E.plan->p;
    const double es = (double)E.esize;
    for (size_t t = 0; t < P.layers.size(); t++) {
        const Layer &L = P.layers[t];
        genlib_layer_info &o = E.info[t];
        if (L.n_new == 0) continue;
        const int32_t *fb = P.fam_base.data() + L.base_off, *mb = P.mem_base.data() + L.base_off;
        const int64_t f0 = fb[E.rank], f1 = fb[E.rank + 1], own_nm = mb[E.rank + 1] - mb[E.rank];
        int64_t rows_local = 0, rows_remote = 0;
        for (int64_t F = f0; F < f1; F++) {
            const int8_t of = P.fam_pf_owner[L.fam_off + F], om = P.fam_pm_owner[L.fam_off + F];
            if (of >= 0) (of == E.rank ? rows_local : rows_remote)++;
            if (om >= 0) (om == E.rank ? rows_local : rows_remote)++;
        }
        int64_t parents_all = 0;
        for (int64_t F = 0; F < L.n_fam; F++) parents_all += (P.fam_pf[L.fam_off + F] >= 0) + (P.fam_pm[L.fam_off + F] >= 0);
        int64_t carried_remote = 0;
        if (E.world > 1 && L.carried > 0)
            for (int32_t r = 0; r < L.rt_rows; r++)
                if ((P.flags[L.flag_off + r] & kFlagCarried) && P.live_owner[L.flag_off + r] != E.rank) carried_remote++;
        const double live = L.live_before, carried = L.carried;
        const LayerLaunch &ll = E.launch[t];
        o.strip_width = ll.s.sw;
        // DRAM: the parent rows of own couples over the live columns, read once; own members' rows
        // (new x new, new x carried) and their columns in the carried rows, written once
        o.dram_read_bytes = (double)rows_local * live * es;
        o.dram_write_bytes = (double)own_nm * ((double)L.n_new + carried) * es + ((double)(L.carried - carried_remote)) * (double)own_nm * es;
        // L2: the strip buffers, written once and read back per couple of the layer
        o.l2_bytes = (double)(rows_local + rows_remote > 0 ? (f1 - f0) : 0) * live * 2 * es +
                     (double)parents_all * (double)(ll.s.n_strips * (int64_t)ll.s.sw) * 2 * es;
        // NVLink: remote parent rows read, own members' columns pushed into carried rows that live elsewhere
        o.nvlink_bytes = (double)rows_remote * live * es + (double)carried_remote * (double)own_nm * es;
    }
    E.info_ready = true;
}

// this rank's probands in output order, and where their rows and columns are, and the pair reads after the last
// layer (needs the finished plan)
int upload_probands(genlib_engine &E) {
    const Plan &P = E.plan->p;
    if (P.schedule == kSchedulePairs) {
        const size_t S = P.layers.size();
        if (int rc = upload_pair_reads(E, P.pair_start[S], P.pair_start[S + 1])) return rc;
    }
    std::vector<int32_t> own_rows;
    E.own_pro.clear();
    for (size_t u = 0; u < P.pro_owner.size(); u++)            // (empty for kScheduleF: no proband matrix)
        if (P.pro_owner[u] == E.rank) { E.own_pro.push_back((int32_t)u); own_rows.push_back(P.pro_lrow[u]); }
    CU(E.pro_slot.upload(P.pro_slot, E.stream));
    CU(E.own_pro_row.upload(own_rows, E.stream));
    CU(E.pro_owner.upload(P.pro_owner, E.stream));
    CU(E.pro_lrow.upload(P.pro_lrow, E.stream));
    CU(cudaStreamSynchronize(E.stream));                       // (own_rows is a local)
    return GENLIB_OK;
}

// reads [i0, i1) of a kSchedulePairs plan -> device
int upload_pair_reads(genlib_engine &E, int64_t i0, int64_t i1) {
    const Plan &P = E.plan->p;
    if (i1 <= i0) return GENLIB_OK;
    const size_t a = (size_t)i0, k = (size_t)(i1 - i0);
    CU(cudaMemcpyAsync(E.pair_owner.p + a, P.pair_owner.data() + a, k * sizeof(int8_t), cudaMemcpyHostToDevice, E.stream));
    CU(cudaMemcpyAsync(E.pair_lrow.p + a, P.pair_lrow.data() + a, k * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    CU(cudaMemcpyAsync(E.pair_col.p + a, P.pair_col_slot.data() + a, k * sizeof(int32_t), cudaMemcpyHostToDevice, E.stream));
    return GENLIB_OK;
}

// the index arrays of layers [t0, t1) -> device (the whole plan: t0 = 0, t1 = layers)
int upload_layers(genlib_engine &E, int t0, int t1) {
    const Plan &P = E.plan->p;
    if (t1 <= t0) return GENLIB_OK;
    const Layer &A = P.layers[(size_t)t0], &Z = P.layers[(size_t)t1 - 1];
    auto up = [&](auto &dev, const auto &host, size_t a, size_t b) -> cudaError_t {
        if (b <= a) return cudaSuccess;
        return cudaMemcpyAsync(dev.p + a, host.data() + a, (b - a) * sizeof(*dev.p), cudaMemcpyHostToDevice, E.stream);
    };
    CU(up(E.mem_ind, P.mem_ind, A.mem_off, Z.mem_end)); CU(up(E.mem_slot, P.mem_slot, A.mem_off, Z.mem_end));
    CU(up(E.mem_fam, P.mem_fam, A.mem_off, Z.mem_end)); CU(up(E.mem_lrow, P.mem_lrow, A.mem_off, Z.mem_end));
    if (sparse_schedule(P.schedule)) CU(up(E.mem_rank, P.mem_rank, A.mem_off, Z.mem_end));
    CU(up(E.fam_pf, P.fam_pf, A.fam_off, Z.fam_end)); CU(up(E.fam_pm, P.fam_pm, A.fam_off, Z.fam_end));
    CU(up(E.fam_q, P.fam_q, 2 * A.fam_off, 2 * Z.fam_end));
    CU(up(E.fam_pf_lrow, P.fam_pf_lrow, A.fam_off, Z.fam_end)); CU(up(E.fam_pm_lrow, P.fam_pm_lrow, A.fam_off, Z.fam_end));
    CU(up(E.fam_pf_owner, P.fam_pf_owner, A.fam_off, Z.fam_end)); CU(up(E.fam_pm_owner, P.fam_pm_owner, A.fam_off, Z.fam_end));
    CU(up(E.fam_start, P.fam_start, A.fam_off + (size_t)t0, Z.fam_end + (size_t)t1));   // a layer holds couples + 1 entries
    CU(up(E.mt_desc, P.mtile_desc, 4 * A.mtile_off, 4 * Z.mtile_end));
    CU(up(E.flags, P.flags, A.flag_off, Z.flag_end));
    CU(up(E.live_owner, P.live_owner, A.flag_off, Z.flag_end)); CU(up(E.live_lrow, P.live_lrow, A.flag_off, Z.flag_end));
    CU(up(E.tile_map, P.tile_map, A.tile_off, Z.tile_end)); CU(up(E.live_tiles, P.live_tiles, A.ltile_off, Z.ltile_end));
    if (P.schedule == kSchedulePairs)
        if (int rc = upload_pair_reads(E, P.pair_start[(size_t)t0], P.pair_start[(size_t)t1])) return rc;
    return GENLIB_OK;
}

int create_engine(const genlib_plan *plan, int numerics, int device, int rank, genlib_engine **out, bool streamed = false) {
    if (!plan || !out) return fail(GENLIB_EINVAL, "genlib_engine_create: null argument");
    *out = nullptr;
    if (numerics != GENLIB_NUMERICS_REFERENCE && numerics != GENLIB_NUMERICS_FP64) return fail(GENLIB_EINVAL, "unknown numerics mode");
    const Plan &P = plan->p;
    if (sparse_schedule(P.schedule) && numerics != GENLIB_NUMERICS_REFERENCE)
        return fail(GENLIB_EINVAL, "the sparse_phi schedule stores Float32 (numerics must be GENLIB_NUMERICS_REFERENCE)");
    if ((P.schedule == kScheduleF || P.schedule == kSchedulePairs) && numerics != GENLIB_NUMERICS_FP64)
        return fail(GENLIB_EINVAL, "the gen.f and gen.phi_pairs schedules store Float64 (numerics must be GENLIB_NUMERICS_FP64)");
    if (rank < 0 || rank >= P.world) return fail(GENLIB_EINVAL, "rank outside the plan's world");
    if (P.world > kMaxWorld) return fail(GENLIB_EINVAL, "the engine supports at most 16 ranks");
    if (P.n_unique == 0) return fail(GENLIB_EINVAL, "empty proband list: nothing to run");
    if (P.capacity >= ((int64_t)1 << 24)) return fail(GENLIB_EINVAL, "frontier wider than 2^24 slots: shard the probands");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(GENLIB_ECUDA, "no CUDA device: libgenlib_cuda has no CPU fallback");
    DeviceGuard guard;
    if (int rc = guard.enter(device)) return rc;
    std::unique_ptr<genlib_engine> E(new (std::nothrow) genlib_engine);
    if (!E) return fail(GENLIB_ENOMEM, "out of host memory");
    E->plan = plan; E->numerics = numerics; E->rank = rank; E->world = P.world;
    E->esize = numerics == GENLIB_NUMERICS_FP64 ? 8 : 4;
    CU(cudaGetDevice(&E->device));
    CU(cudaDeviceGetAttribute(&E->sm_count, cudaDevAttrMultiProcessorCount, E->device));
    {
        const char *env = std::getenv("GENLIB_BARRIER_TIMEOUT_S");       // inter-GPU barrier: seconds before GENLIB_ECOMM
        const double sec = env ? std::atof(env) : 10.0;
        E->barrier_timeout = (long long)(std::max(sec, 0.001) * 2e9);
    }
    const double t0 = now_ms();
    // launch shapes, strip buffers, sync words (a streamed plan: the shapes follow layer by layer)
    E->streamed = streamed;
    E->launch.resize(P.layers.size());
    scratch_sizes(P, E->esize, rank, E->sm_count, streamed, E->q_bytes, E->sync_ints);
    if (!streamed) {
        size_t at = (P.layers.size() + 15) / 16 * 16;
        for (int t = 0; t < (int)P.layers.size(); t++) {
            LayerLaunch &ll = E->launch[t];
            ll = shape_layer(P, t, rank, E->esize, E->sm_count);
            if (ll.grid == 0) continue;
            ll.sync_off = at;
            at += 16 * (size_t)ll.s.n_strips;
        }
    }
    const size_t need = engine_bytes(P, numerics, rank, E->sm_count, streamed);
    CU(cudaStreamCreateWithFlags(&E->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&E->copy_stream, cudaStreamNonBlocking));
    {
        if (int rc = acquire_arena(E->device, need, E->arena, [&](size_t free_b) {
                char msg[256];
                std::snprintf(msg, sizeof msg, "rank %d needs %.2f GB on the device, %.2f GB free (capacity %lld slots, %lld rows): shard over more GPUs",
                              rank, need / 1e9, free_b / 1e9, (long long)P.capacity, (long long)P.rows_cap[rank]);
                return std::string(msg);
            }))
            return rc;
        unsigned char *base = static_cast<unsigned char *>(E->arena.base), *cur = base;
        auto take = [&](size_t bytes) { unsigned char *p = cur; cur += pad256(bytes); return p; };
        E->bar_flags = reinterpret_cast<unsigned *>(take(kFlagBytes));
        E->A = take(total_rows(P, rank) * (size_t)P.capacity * E->esize);
        E->Q = take(E->q_bytes);
        E->sync = reinterpret_cast<int32_t *>(take(E->sync_ints * sizeof(int32_t)));
        E->fetch_stage[0] = take(kFetchStageBytes);
        E->fetch_stage[1] = take(kFetchStageBytes);
        cur = place_arrays(*E, P, streamed, cur);
        if ((size_t)(cur - base) > need) return fail(GENLIB_EINVAL, "internal: arena layout overflow");
        if ((size_t)(static_cast<unsigned char *>(E->A) - base) != off_A())
            return fail(GENLIB_EINVAL, "internal: peer-visible arena offsets drifted");
    }
    CU(cudaMemsetAsync(E->bar_flags, 0, kFlagBytes, E->stream));
    if (!streamed) {
        if (int rc = upload_layers(*E, 0, (int)P.layers.size())) return rc;
        if (int rc = upload_probands(*E)) return rc;
    }
    CU(cudaStreamSynchronize(E->stream));
#ifdef GENLIB_PROFILE
    CU(cudaMalloc(&E->prof, 8 * 2 * 160 * sizeof(long long)));
    CU(cudaMemset(E->prof, 0, 8 * 2 * 160 * sizeof(long long)));
#endif
    E->peers.A[rank] = E->A; E->bars.flags[rank] = E->bar_flags;
    E->attached = P.world == 1;
    E->info.resize(P.layers.size());
    if (!streamed) for (size_t t = 0; t < P.layers.size(); t++) fill_info(P.layers[t], &E->info[t]);
    E->events.resize(P.layers.size() * 3 + 2);
    for (auto &e : E->events) CU(cudaEventCreate(&e));
    genlib_stats &s = E->stats;
    s.n_unique = P.n_unique; s.n_layers = (int32_t)P.layers.size(); s.row_updates = P.row_updates;
    s.capacity = P.capacity; s.device_bytes = (int64_t)need;
    s.alg_bytes = streamed ? P.alg_elems * (double)E->esize : plan_alg_bytes(P, E->esize);   // (streamed: final in run_streamed)
    s.ms_plan = plan->ms_plan; s.ms_upload = now_ms() - t0;
    s.h2d_bytes = (int64_t)plan_index_bytes(P);
    *out = E.release();
    return GENLIB_OK;
}

}  // namespace

// ------------------------------------------------------------------------------ ABI
extern "C" {

int genlib_version(void) { return GENLIB_ABI_VERSION; }
const char *genlib_last_error(void) { return g_err.c_str(); }

int genlib_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { g_err = "cudaGetDeviceCount failed (no driver / no device)"; return -GENLIB_ECUDA; }
    return n;
}

int genlib_release_cache(void) {
    g_peer_maps.close_all();
    g_arenas.release_device(-1);
    release_plan_cache();
    return GENLIB_OK;
}

int genlib_pinned_alloc(size_t bytes, void **out) {
    if (!out) return fail(GENLIB_EINVAL, "null argument");
    *out = nullptr;
    CU(cudaHostAlloc(out, std::max<size_t>(bytes, 16), cudaHostAllocDefault));
    return GENLIB_OK;
}

int genlib_pinned_free(void *ptr) {
    if (ptr) CU(cudaFreeHost(ptr));
    return GENLIB_OK;
}

int genlib_plan_create(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                       const int32_t *proband, int32_t world, genlib_plan **out) {
    return genlib_plan_create_scheduled(n, father, mother, n_pro, proband, world, GENLIB_SCHEDULE_PHI, out);
}

int genlib_plan_create_scheduled(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                                 const int32_t *proband, int32_t world, int schedule, genlib_plan **out) {
    return genlib_plan_create_ex(n, father, mother, nullptr, n_pro, proband, world, schedule, out);
}

static int plan_create(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids, int32_t n_pro,
                       const int32_t *proband, int32_t world, int schedule, const PairList &pairs, genlib_plan **out) {
    if (!out) return fail(GENLIB_EINVAL, "genlib_plan_create: out is null");
    *out = nullptr;
    std::unique_ptr<genlib_plan> pl(new (std::nothrow) genlib_plan);
    if (!pl) return fail(GENLIB_ENOMEM, "out of host memory");
    pl->build(n, father, mother, ids, n_pro, proband, world, schedule, nullptr, 0, now_ms(), pairs);
    if (pl->worker_rc != GENLIB_OK) return fail(pl->worker_rc, pl->worker_err);
    *out = pl.release();
    return GENLIB_OK;
}

int genlib_plan_create_ex(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids, int32_t n_pro,
                          const int32_t *proband, int32_t world, int schedule, genlib_plan **out) {
    return plan_create(n, father, mother, ids, n_pro, proband, world, schedule, PairList{}, out);
}

// a plan made on a worker thread and published layer by layer (the caller's arrays stay alive until it is settled)
static int plan_create_async(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids, int32_t n_pro,
                             const int32_t *proband, int32_t world, int schedule, const PairList &pairs, genlib_plan **out) {
    if (!out) return fail(GENLIB_EINVAL, "genlib_plan_create: out is null");
    *out = nullptr;
    if (env_int("GENLIB_STREAM", 1) == 0) return plan_create(n, father, mother, ids, n_pro, proband, world, schedule, pairs, out);
    std::unique_ptr<genlib_plan> pl(new (std::nothrow) genlib_plan);
    if (!pl) return fail(GENLIB_ENOMEM, "out of host memory");
    pl->stream.reset(new (std::nothrow) PlanStream);
    if (!pl->stream) return fail(GENLIB_ENOMEM, "out of host memory");
    genlib_plan *raw = pl.get();
    const double t0 = now_ms();
    try {
        raw->worker = std::thread([=] { raw->build(n, father, mother, ids, n_pro, proband, world, schedule, raw->stream.get(), 0, t0, pairs); });
    } catch (...) {                              // no thread to be had
        pl.reset();
        return plan_create(n, father, mother, ids, n_pro, proband, world, schedule, pairs, out);
    }
    PlanStream &ps = *raw->stream;
    ps.wait([&] { return ps.stage.load() >= 1; });
    if (ps.stage.load() == 2) {                  // finished already: an error of the pre-pass, or nothing to stream
        raw->settle();
        if (raw->worker_rc != GENLIB_OK) return fail(raw->worker_rc, raw->worker_err);
    }
    *out = pl.release();
    return GENLIB_OK;
}

int genlib_plan_create_async(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids, int32_t n_pro,
                             const int32_t *proband, int32_t world, int schedule, genlib_plan **out) {
    return plan_create_async(n, father, mother, ids, n_pro, proband, world, schedule, PairList{}, out);
}

int genlib_plan_create_pairs(int32_t n, const int32_t *father, const int32_t *mother, int64_t n_pairs, const int32_t *a,
                             const int32_t *b, int32_t world, int stream, genlib_plan **out) {
    const PairList pairs{n_pairs, a, b};
    return stream ? plan_create_async(n, father, mother, nullptr, 0, nullptr, world, GENLIB_SCHEDULE_PAIRS, pairs, out)
                  : plan_create(n, father, mother, nullptr, 0, nullptr, world, GENLIB_SCHEDULE_PAIRS, pairs, out);
}

int64_t genlib_plan_pair_reads(const genlib_plan *plan, int32_t layer, int64_t *pos, int32_t *row_slot, int32_t *col_slot,
                               int32_t *owner, int32_t *lrow) {
    settle(plan);
    if (!plan || plan->p.schedule != kSchedulePairs || plan->p.pair_start.empty() || layer < 0 || layer > (int32_t)plan->p.layers.size())
        { fail(GENLIB_EINVAL, "genlib_plan_pair_reads: not a GENLIB_SCHEDULE_PAIRS plan, or no such layer"); return -1; }
    const Plan &P = plan->p;
    const int64_t i0 = P.pair_start[(size_t)layer], i1 = P.pair_start[(size_t)layer + 1];
    for (int64_t i = i0; i < i1; i++) {
        const size_t k = (size_t)(i - i0), j = (size_t)i;
        if (pos) pos[k] = P.pair_pos[j];
        if (row_slot) row_slot[k] = P.pair_row_slot[j];
        if (col_slot) col_slot[k] = P.pair_col_slot[j];
        if (owner) owner[k] = P.pair_owner[j];
        if (lrow) lrow[k] = P.pair_lrow[j];
    }
    return i1 - i0;
}

void genlib_plan_destroy(genlib_plan *plan) {
    if (!plan) return;
    plan->settle();
    try { retire_storage(plan->p); } catch (...) {}
    delete plan;
}
uint64_t genlib_plan_digest(const genlib_plan *plan, int with_bounds) { settle(plan); return plan ? plan_digest(plan->p, with_bounds != 0) : 0; }
int32_t genlib_plan_n_unique(const genlib_plan *plan) { return plan ? plan->p.n_unique : -1; }
int32_t genlib_plan_schedule(const genlib_plan *plan) { return plan ? plan->p.schedule : -1; }
int32_t genlib_plan_n_layers(const genlib_plan *plan) { settle(plan); return plan ? (int32_t)plan->p.layers.size() : -1; }
int64_t genlib_plan_capacity(const genlib_plan *plan) { settle(plan); return plan ? plan->p.capacity : -1; }
int64_t genlib_plan_row_updates(const genlib_plan *plan) { settle(plan); return plan ? plan->p.row_updates : -1; }

int genlib_plan_layer_info(const genlib_plan *plan, int32_t layer, genlib_layer_info *out) {
    settle(plan);
    if (!plan || !out || layer < 0 || layer >= (int32_t)plan->p.layers.size()) return fail(GENLIB_EINVAL, "bad layer");
    fill_info(plan->p.layers[layer], out);
    return GENLIB_OK;
}

int64_t genlib_plan_device_bytes(const genlib_plan *plan, int numerics, int32_t rank) {
    settle(plan);
    if (!plan || rank < 0 || rank >= plan->p.world || plan->p.n_unique == 0) return plan ? 0 : -1;
    return (int64_t)engine_bytes(plan->p, numerics, rank);      // strip buffers sized for 148 SMs
}

int genlib_plan_launch_shape(const genlib_plan *plan, int32_t layer, int numerics, int32_t rank, int32_t sm_count,
                             genlib_launch_shape *out) {
    settle(plan);
    if (!plan || !out || layer < 0 || layer >= (int32_t)plan->p.layers.size()) return fail(GENLIB_EINVAL, "bad layer");
    if (numerics != GENLIB_NUMERICS_REFERENCE && numerics != GENLIB_NUMERICS_FP64) return fail(GENLIB_EINVAL, "unknown numerics mode");
    if (rank < 0 || rank >= plan->p.world || sm_count < 1) return fail(GENLIB_EINVAL, "genlib_plan_launch_shape: bad rank or SM count");
    const size_t es = numerics == GENLIB_NUMERICS_FP64 ? 8 : 4;
    const LayerLaunch ll = shape_layer(plan->p, layer, rank, es, sm_count);
    const StripArgs &s = ll.s;
    std::memset(out, 0, sizeof *out);
    if (s.sw == 0) return GENLIB_OK;                             // (no couple of the rank in this layer)
    out->sw = s.sw; out->ft = s.ft; out->prod_warps = ll.prod_warps; out->gangs = s.gangs; out->nbuf = s.nbuf;
    out->stages = s.stages; out->n_strips = s.n_strips; out->n_pitems = s.n_pitems; out->n_citems = s.n_citems;
    out->n_prod = s.n_prod; out->n_cons = s.n_cons; out->grid = ll.grid;
    out->fast_transpose = s.n_pitems > 0 && fast_transpose_shape((int)es, s.sw, s.ft);
    out->smem = (int64_t)ll.smem;
    return GENLIB_OK;
}

int genlib_plan_layer_arrays(const genlib_plan *plan, int32_t layer, int32_t *member_ind,
                             int32_t *member_slot, int32_t *member_fam, int32_t *fam_father_slot,
                             int32_t *fam_mother_slot, int32_t *member_owner) {
    settle(plan);
    if (!plan || layer < 0 || layer >= (int32_t)plan->p.layers.size()) return fail(GENLIB_EINVAL, "bad layer");
    const Plan &P = plan->p;
    const Layer &L = P.layers[layer];
    for (int32_t q = 0; q < L.n_new; q++) {
        if (member_ind) member_ind[q] = P.mem_ind[L.mem_off + q];
        if (member_slot) member_slot[q] = P.mem_slot[L.mem_off + q];
        if (member_fam) member_fam[q] = P.mem_fam[L.mem_off + q];
        if (member_owner) {
            int g = 0;
            while (g + 1 < P.world && q >= P.mem_base[L.base_off + g + 1]) g++;
            member_owner[q] = g;
        }
    }
    for (int32_t f = 0; f < L.n_fam; f++) {
        if (fam_father_slot) fam_father_slot[f] = P.fam_pf[L.fam_off + f];
        if (fam_mother_slot) fam_mother_slot[f] = P.fam_pm[L.fam_off + f];
    }
    return GENLIB_OK;
}

int genlib_plan_layer_ranks(const genlib_plan *plan, int32_t layer, int32_t *member_rank) {
    settle(plan);
    if (!plan || !member_rank || layer < 0 || layer >= (int32_t)plan->p.layers.size()) return fail(GENLIB_EINVAL, "bad layer");
    const Plan &P = plan->p;
    const Layer &L = P.layers[layer];
    for (int32_t q = 0; q < L.n_new; q++)
        member_rank[q] = P.mem_rank.empty() ? P.mem_ind[L.mem_off + q] : P.mem_rank[L.mem_off + q];
    return GENLIB_OK;
}

int genlib_plan_layer_shard(const genlib_plan *plan, int32_t layer, int32_t *fam_base, int32_t *mem_base,
                            int32_t *member_lrow, int32_t *fam_father_owner, int32_t *fam_father_lrow,
                            int32_t *fam_mother_owner, int32_t *fam_mother_lrow) {
    settle(plan);
    if (!plan || layer < 0 || layer >= (int32_t)plan->p.layers.size()) return fail(GENLIB_EINVAL, "bad layer");
    const Plan &P = plan->p;
    const Layer &L = P.layers[layer];
    for (int32_t g = 0; g <= P.world; g++) {
        if (fam_base) fam_base[g] = P.fam_base[L.base_off + g];
        if (mem_base) mem_base[g] = P.mem_base[L.base_off + g];
    }
    for (int32_t q = 0; q < L.n_new; q++)
        if (member_lrow) member_lrow[q] = P.mem_lrow[L.mem_off + q];
    for (int32_t f = 0; f < L.n_fam; f++) {
        if (fam_father_owner) fam_father_owner[f] = P.fam_pf_owner[L.fam_off + f];
        if (fam_father_lrow) fam_father_lrow[f] = P.fam_pf_lrow[L.fam_off + f];
        if (fam_mother_owner) fam_mother_owner[f] = P.fam_pm_owner[L.fam_off + f];
        if (fam_mother_lrow) fam_mother_lrow[f] = P.fam_pm_lrow[L.fam_off + f];
    }
    return GENLIB_OK;
}

int genlib_plan_layer_live_rows(const genlib_plan *plan, int32_t layer, int32_t *live_owner, int32_t *live_lrow) {
    settle(plan);
    if (!plan || !live_owner || !live_lrow || layer < 0 || layer >= (int32_t)plan->p.layers.size()) return fail(GENLIB_EINVAL, "bad layer");
    const Plan &P = plan->p;
    const Layer &L = P.layers[layer];
    for (int64_t s = 0; s < P.capacity; s++) { live_owner[s] = -1; live_lrow[s] = -1; }
    for (int32_t r = 0; r < L.rt_rows; r++)
        if (P.flags[L.flag_off + r] & kFlagLive) {
            live_owner[L.rt_lo + r] = P.live_owner[L.flag_off + r];
            live_lrow[L.rt_lo + r] = P.live_lrow[L.flag_off + r];
        }
    return GENLIB_OK;
}

int64_t genlib_plan_rank_rows(const genlib_plan *plan, int32_t rank) {
    settle(plan);
    if (!plan || rank < 0 || rank >= plan->p.world) return -1;
    return plan->p.rows_cap.empty() ? 0 : (int64_t)total_rows(plan->p, rank);
}

int32_t genlib_plan_world(const genlib_plan *plan) { return plan ? plan->p.world : -1; }

int genlib_plan_proband_rows(const genlib_plan *plan, int32_t *owner, int32_t *lrow) {
    settle(plan);
    if (!plan || !owner || !lrow) return fail(GENLIB_EINVAL, "null argument");
    for (size_t u = 0; u < plan->p.pro_owner.size(); u++) { owner[u] = plan->p.pro_owner[u]; lrow[u] = plan->p.pro_lrow[u]; }
    return GENLIB_OK;
}

int genlib_plan_layer_flags(const genlib_plan *plan, int32_t layer, uint8_t *live_flags) {
    settle(plan);
    if (!plan || !live_flags || layer < 0 || layer >= (int32_t)plan->p.layers.size()) return fail(GENLIB_EINVAL, "bad layer");
    const Plan &P = plan->p;
    const Layer &L = P.layers[layer];
    std::memset(live_flags, 0, (size_t)P.capacity);
    for (int32_t r = 0; r < L.rt_rows; r++) live_flags[L.rt_lo + r] = P.flags[L.flag_off + r];
    return GENLIB_OK;
}

int genlib_plan_proband_slots(const genlib_plan *plan, int32_t *slots) {
    settle(plan);
    if (!plan || !slots) return fail(GENLIB_EINVAL, "null argument");
    std::copy(plan->p.pro_slot.begin(), plan->p.pro_slot.end(), slots);
    return GENLIB_OK;
}

// An engine on a plan that is still being made registers as a reader of its arrays before it looks at them.
static int create_engine_public(const genlib_plan *plan, int numerics, int device, int rank, genlib_engine **out) {
    if (out) *out = nullptr;
    if (plan && plan->p.schedule == kScheduleF)                  // (set before genlib_plan_create* returns)
        return fail(GENLIB_EINVAL, "a GENLIB_SCHEDULE_F plan has no matrix to fetch: call genlib_f");
    if (plan && plan->p.schedule == kSchedulePairs)
        return fail(GENLIB_EINVAL, "a GENLIB_SCHEDULE_PAIRS plan has no matrix to fetch: call genlib_phi_pairs");
    if (plan && plan->streaming()) {
        PlanStream &ps = *plan->stream;
        StreamConsumer reader(ps);
        if (!ps.overflow.load() && ps.stage.load() != 2) {
            int rc = create_engine(plan, numerics, device, rank, out, true);
            if (rc == GENLIB_OK) { (*out)->consuming = std::move(reader); return rc; }
            if (rc != GENLIB_ENOMEM) return rc;             // (the bounds did not fit: size by the finished plan)
        }
    }
    settle(plan);
    if (plan && plan->worker_rc != GENLIB_OK) return fail(plan->worker_rc, plan->worker_err);
    return create_engine(plan, numerics, device, rank, out);
}

int genlib_engine_create(const genlib_plan *plan, int numerics, int device, genlib_engine **out) {
    return create_engine_public(plan, numerics, device, 0, out);
}

int genlib_engine_create_dist(const genlib_plan *plan, int numerics, int device, int32_t rank, genlib_engine **out) {
    return create_engine_public(plan, numerics, device, rank, out);
}

int genlib_engine_ipc_export(genlib_engine *eng, void *handle64) {
    if (!eng || !handle64) return fail(GENLIB_EINVAL, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DeviceGuard guard;
    if (int rc = guard.enter(eng->device)) return rc;
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, eng->arena.base));
    eng->arena.exported = true;
    std::memcpy(handle64, &h, sizeof h);
    return GENLIB_OK;
}

int genlib_engine_ipc_attach(genlib_engine *eng, const void *handles, size_t stride) {
    if (!eng || !handles || stride < 64) return fail(GENLIB_EINVAL, "null argument");
    if (eng->attached) return GENLIB_OK;
    DeviceGuard guard;
    if (int rc = guard.enter(eng->device)) return rc;
    for (int g = 0; g < eng->world; g++) {
        if (g == eng->rank) continue;
        void *base = nullptr;
        cudaError_t ce = g_peer_maps.map(eng->device, static_cast<const unsigned char *>(handles) + (size_t)g * stride, &base);
        if (ce != cudaSuccess) {
            cudaGetLastError();
            return fail(GENLIB_ECOMM, std::string("cudaIpcOpenMemHandle(rank ") + std::to_string(g) + "): " + cudaGetErrorString(ce));
        }
        unsigned char *b = static_cast<unsigned char *>(base);
        eng->bars.flags[g] = reinterpret_cast<unsigned *>(b);
        eng->peers.A[g] = b + off_A();
    }
    eng->attached = true;
    return GENLIB_OK;
}

int32_t genlib_engine_own_probands(const genlib_engine *eng, int32_t *index) {
    if (!eng) return -1;
    if (index) std::copy(eng->own_pro.begin(), eng->own_pro.end(), index);
    return (int32_t)eng->own_pro.size();
}

void genlib_engine_destroy(genlib_engine *eng) {
    if (!eng) return;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(eng->device);
    delete eng;
    if (prev >= 0) cudaSetDevice(prev);
}

int genlib_engine_run(genlib_engine *eng, int time_layers) {
    if (!eng) return fail(GENLIB_EINVAL, "null engine");
    DeviceGuard guard;
    if (int rc = guard.enter(eng->device)) return rc;
    genlib_engine &E = *eng;
    if (!E.attached) return fail(GENLIB_ECOMM, "genlib_engine_run before genlib_engine_ipc_attach");
    if (E.streamed && !E.ran) {                                 // first run on a plan that is still being made
        if (!E.consuming.ps) return fail(GENLIB_ERESTART, "the streamed plan's bounds did not hold: create the engine again");
        PlanStream &ps = *E.consuming.ps;
        int rc = E.numerics == GENLIB_NUMERICS_FP64 ? run_streamed<double>(E, ps) : run_streamed<float>(E, ps);
        E.consuming.reset();
        settle(E.plan);
        if (rc == kRestart) return fail(GENLIB_ERESTART, "a size bound of the streamed plan did not hold: destroy this engine, create it again and run");
        if (rc != GENLIB_OK) return rc == E.plan->worker_rc ? fail(rc, E.plan->worker_err) : rc;
        if (int rc2 = check_device_errors(E)) return rc2;
        E.stats.ms_plan = E.plan->ms_plan;
        E.ran = true;
        return GENLIB_OK;
    }
    const size_t nev = E.events.size();
    CU(cudaEventRecord(E.events[nev - 2], E.stream));
    int rc = E.numerics == GENLIB_NUMERICS_FP64 ? launch_layers<double>(E, time_layers != 0)
                                                : launch_layers<float>(E, time_layers != 0);
    if (rc != GENLIB_OK) return rc;
    CU(cudaEventRecord(E.events[nev - 1], E.stream));
    CU(cudaStreamSynchronize(E.stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, E.events[nev - 2], E.events[nev - 1]));
    E.stats.ms_kernels = ms;
    if (time_layers) {
        size_t ev = 0;
        for (size_t t = 0; t < E.info.size(); t++) {
            if (E.info[t].n_new == 0) continue;
            if (E.layer_limit >= 0 && (int32_t)t >= E.layer_limit) break;
            float a = 0, w = 0;
            CU(cudaEventElapsedTime(&a, E.events[ev], E.events[ev + 1]));
            CU(cudaEventElapsedTime(&w, E.events[ev + 1], E.events[ev + 2]));
            ev += 3;
            E.info[t].ms_layer = a; E.info[t].ms_wait = w;
        }
    }
    if (int rc2 = check_device_errors(E)) return rc2;
    E.ran = true;
    return GENLIB_OK;
}

int genlib_engine_layer_info(genlib_engine *eng, int32_t layer, genlib_layer_info *out) {
    if (eng) settle(eng->plan);
    if (!eng || !out || layer < 0 || layer >= (int32_t)eng->info.size()) return fail(GENLIB_EINVAL, "bad layer");
    account_layers(*eng);
    *out = eng->info[layer];
    return GENLIB_OK;
}

int genlib_engine_stats(const genlib_engine *eng, genlib_stats *out) {
    if (!eng || !out) return fail(GENLIB_EINVAL, "null argument");
    *out = eng->stats;
    return GENLIB_OK;
}

int genlib_engine_fetch(genlib_engine *eng, void *out, int out_dtype) {
    if (!eng || (!out && eng->plan->p.n_unique > 0)) return fail(GENLIB_EINVAL, "null argument");
    if (!eng->ran) return fail(GENLIB_EINVAL, "genlib_engine_fetch before genlib_engine_run");
    if (out_dtype != GENLIB_F32 && out_dtype != GENLIB_F64) return fail(GENLIB_EINVAL, "unknown out_dtype");
    DeviceGuard guard;
    if (int rc = guard.enter(eng->device)) return rc;
    const double t0 = now_ms();
    int rc;
    if (eng->numerics == GENLIB_NUMERICS_FP64)
        rc = out_dtype == GENLIB_F64 ? fetch_rows<double, double>(*eng, (double *)out) : fetch_rows<double, float>(*eng, (float *)out);
    else
        rc = out_dtype == GENLIB_F64 ? fetch_rows<float, double>(*eng, (double *)out) : fetch_rows<float, float>(*eng, (float *)out);
    eng->stats.ms_fetch = now_ms() - t0;
    return rc;
}

int genlib_engine_row_sums(genlib_engine *eng, double *out) {
    if (!eng || (!out && !eng->own_pro.empty())) return fail(GENLIB_EINVAL, "null argument");
    if (!eng->ran) return fail(GENLIB_EINVAL, "genlib_engine_row_sums before genlib_engine_run");
    DeviceGuard guard;
    if (int rc = guard.enter(eng->device)) return rc;
    const Plan &P = eng->plan->p;
    const int32_t n = P.n_unique, nown = (int32_t)eng->own_pro.size();
    if (nown == 0) return GENLIB_OK;
    double *dsum = nullptr;
    int32_t *didx = nullptr;
    FreeOnExit<double> free_sum{dsum};
    FreeOnExit<int32_t> free_idx{didx};
    CU(cudaMalloc(&dsum, (size_t)nown * 2 * sizeof(double)));
    if (cudaMalloc(&didx, (size_t)nown * sizeof(int32_t)) != cudaSuccess) return fail(GENLIB_ENOMEM, "out of device memory");
    cudaError_t ce = cudaMemcpyAsync(didx, eng->own_pro.data(), (size_t)nown * sizeof(int32_t), cudaMemcpyHostToDevice, eng->stream);
    if (ce == cudaSuccess) {
        if (eng->numerics == GENLIB_NUMERICS_FP64)
            rowsum_kernel<double><<<(unsigned)nown, kThreads, 0, eng->stream>>>((const double *)eng->A, P.capacity, eng->own_pro_row.p, didx, eng->pro_slot.p, n, dsum);
        else
            rowsum_kernel<float><<<(unsigned)nown, kThreads, 0, eng->stream>>>((const float *)eng->A, P.capacity, eng->own_pro_row.p, didx, eng->pro_slot.p, n, dsum);
        ce = cudaMemcpyAsync(out, dsum, (size_t)nown * 2 * sizeof(double), cudaMemcpyDeviceToHost, eng->stream);
    }
    const cudaError_t e2 = cudaStreamSynchronize(eng->stream);
    if (ce != cudaSuccess || e2 != cudaSuccess) return fail(GENLIB_ECUDA, std::string("row sums: ") + cudaGetErrorString(ce != cudaSuccess ? ce : e2));
    return GENLIB_OK;
}

int genlib_engine_phi_product(genlib_engine *eng, int32_t k, const double *X, double *out, double *diag) {
    if (!eng || k < 0) return fail(GENLIB_EINVAL, "genlib_engine_phi_product: null engine or k < 0");
    if (!eng->ran) return fail(GENLIB_EINVAL, "genlib_engine_phi_product before genlib_engine_run");
    if (k > 0 && (!X || (!out && !eng->own_pro.empty()))) return fail(GENLIB_EINVAL, "genlib_engine_phi_product: null argument");
    DeviceGuard guard;
    if (int rc = guard.enter(eng->device)) return rc;
    return eng->numerics == GENLIB_NUMERICS_FP64 ? phi_product_rows<double>(*eng, X, k, out, diag)
                                                 : phi_product_rows<float>(*eng, X, k, out, diag);
}

int genlib_engine_phi_mean(genlib_engine *eng, double *out) {
    if (!eng || !out) return fail(GENLIB_EINVAL, "null argument");
    if (eng->world != 1) return fail(GENLIB_EINVAL, "genlib_engine_phi_mean: one rank only; sharded engines combine genlib_engine_row_sums in proband order");
    const int32_t n = eng->plan->p.n_unique;
    if (n < 2) { *out = 0.0; return eng->ran ? (int)GENLIB_OK : fail(GENLIB_EINVAL, "genlib_engine_phi_mean before genlib_engine_run"); }
    std::vector<double> sums((size_t)n * 2);
    if (int rc = genlib_engine_row_sums(eng, sums.data())) return rc;
    double total = 0.0, diag = 0.0;
    for (int32_t r = 0; r < n; r++) { total += sums[2 * (size_t)r]; diag += sums[2 * (size_t)r + 1]; }   // proband order: deterministic
    *out = (total - diag) / ((double)n * n - n);
    return GENLIB_OK;
}

int genlib_engine_set_layer_limit(genlib_engine *eng, int32_t n_layers) {
    if (!eng) return fail(GENLIB_EINVAL, "null engine");
    eng->layer_limit = n_layers;
    return GENLIB_OK;
}

int genlib_engine_read_block(genlib_engine *eng, int32_t n_slots, const int32_t *slots, double *out) {
    if (!eng || !slots || !out || n_slots < 0) return fail(GENLIB_EINVAL, "null argument");
    if (eng->world != 1) return fail(GENLIB_EINVAL, "genlib_engine_read_block: single-rank engines only");
    DeviceGuard guard;
    if (int rc = guard.enter(eng->device)) return rc;
    if (n_slots == 0) return GENLIB_OK;
    const Plan &P = eng->plan->p;
    for (int32_t i = 0; i < n_slots; i++)
        if (slots[i] < 0 || slots[i] >= P.capacity) return fail(GENLIB_EINVAL, "slot out of range");
    int32_t *dslots = nullptr;
    double *dout = nullptr;
    FreeOnExit<int32_t> free_slots{dslots};
    FreeOnExit<double> free_out{dout};
    CU(cudaMalloc(&dslots, (size_t)n_slots * sizeof(int32_t)));
    CU(cudaMalloc(&dout, (size_t)n_slots * n_slots * sizeof(double)));
    CU(cudaMemcpyAsync(dslots, slots, (size_t)n_slots * sizeof(int32_t), cudaMemcpyHostToDevice, eng->stream));
    for (int32_t r0 = 0; r0 < n_slots; r0 += 65535) {
        const int32_t nr = std::min(65535, n_slots - r0);
        dim3 grid((unsigned)std::min<int32_t>((n_slots + 255) / 256, 64), (unsigned)nr);
        if (eng->numerics == GENLIB_NUMERICS_FP64)
            gather_kernel<double, double><<<grid, 256, 0, eng->stream>>>((const double *)eng->A, P.capacity, dslots, dslots, n_slots, r0, nr, dout + (size_t)r0 * n_slots);
        else
            gather_kernel<float, double><<<grid, 256, 0, eng->stream>>>((const float *)eng->A, P.capacity, dslots, dslots, n_slots, r0, nr, dout + (size_t)r0 * n_slots);
    }
    CU(cudaMemcpyAsync(out, dout, (size_t)n_slots * n_slots * sizeof(double), cudaMemcpyDeviceToHost, eng->stream));
    CU(cudaStreamSynchronize(eng->stream));
    return GENLIB_OK;
}

// What a one-shot call takes out of the engines once every device has run: `prepare` (may be empty) reads the
// finished plan on the calling thread, then `device(E, g)` runs on device g's host thread.  A fetch that needs what
// every device found first (gen.phiOver's global offsets) adds `combine`, on the calling thread once every `device`
// has returned, and `finish(E, g)`, again on the devices' threads.
struct OneshotFetch {
    std::function<void(const Plan &)> prepare;
    std::function<int(genlib_engine &, int)> device;
    std::function<int()> combine;
    std::function<int(genlib_engine &, int)> finish;
};

// genlib_phi, genlib_phi_multi, genlib_phi_over, genlib_f and genlib_phi_pairs: ONE plan for all devices, made on a worker thread and handed over layer
// by layer (PlanStream), so that the devices run the first generations while the later ones are planned.
// GENLIB_STREAM=0, or a bound of the streamed plan that did not hold, plans first and then runs.  One device runs on
// the calling thread; several get a host thread each and NVLink peer access.  `has_out`: the caller wants a result.
static int oneshot(const std::string &who, int schedule, int32_t n, const int32_t *father, const int32_t *mother,
                   int32_t n_pro, const int32_t *proband, bool has_out, int numerics, int32_t n_dev, const int32_t *devices,
                   genlib_stats *stats, const OneshotFetch &fetch, const PairList &pairs = PairList{}) {
    const bool multi = n_dev > 1;
    std::vector<int> dev(devices, devices + n_dev);              // (one device: a negative one is the current device)
    if (int rc = multi ? resolve_devices(who, n_dev, devices, false, dev) : GENLIB_OK) return rc;
    std::unique_ptr<genlib_plan> plan_owner(new (std::nothrow) genlib_plan);
    if (!plan_owner) return fail(GENLIB_ENOMEM, "out of host memory");
    genlib_plan *plan = plan_owner.get();
    const bool want_stream = env_int("GENLIB_STREAM", 1) != 0 && has_out;
    const double tp0 = now_ms();
    PlanStream ps;
    auto make_plan = [&](PlanStream *stream) {
        plan->build(n, father, mother, nullptr, n_pro, proband, n_dev, schedule, stream, /*planners=*/1, tp0, pairs);
    };
    if (want_stream) { try { plan->worker = std::thread([&] { make_plan(&ps); }); } catch (...) { } }
    const bool streaming = plan->worker.joinable();
    if (!streaming) make_plan(nullptr);                         // (no thread to be had: plan here)
    // (destruction order: consumer registration, engines, worker joined and plan storage retired)
    struct PlanRetire { genlib_plan *p; ~PlanRetire() { p->settle(); try { retire_storage(p->p); } catch (...) {} } } retire{plan};
    std::vector<genlib_engine *> eng((size_t)n_dev, nullptr);
    struct EngGuard { std::vector<genlib_engine *> &e; ~EngGuard() { for (auto *&x : e) { genlib_engine_destroy(x); x = nullptr; } } } eguard{eng};
    struct DevRestore { int d = -1; ~DevRestore() { if (d >= 0) cudaSetDevice(d); } } restore;
    int peer_rc = GENLIB_OK;
    if (multi) {                 // every device sees every other device's memory -- while the planner's pre-pass runs
        cudaGetDevice(&restore.d);
        for (int g = 0; g < n_dev && peer_rc == GENLIB_OK; g++) {
            if (cudaSetDevice(dev[g]) != cudaSuccess) { peer_rc = fail(GENLIB_ECUDA, "cudaSetDevice failed"); break; }
            for (int h = 0; h < n_dev; h++) {
                if (h == g) continue;
                int can = 0;
                cudaDeviceCanAccessPeer(&can, dev[g], dev[h]);
                if (!can) { peer_rc = fail(GENLIB_ECOMM, "devices " + std::to_string(dev[g]) + " and " + std::to_string(dev[h]) + " have no peer access"); break; }
                const cudaError_t ce = cudaDeviceEnablePeerAccess(dev[h], 0);
                if (ce != cudaSuccess && ce != cudaErrorPeerAccessAlreadyEnabled) { peer_rc = fail(GENLIB_ECOMM, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(ce)); break; }
                cudaGetLastError();
            }
        }
    }
    // GENLIB_OK, kRestart (a bound did not hold or did not fit, and nothing worse happened) or the first error
    auto first_error = [&](const std::vector<DeviceStatus> &r, bool restart_is_error) {
        int rc2 = GENLIB_OK;
        for (int g = 0; g < n_dev; g++) {
            const int st = r[(size_t)g].status;
            if (st == GENLIB_OK) continue;
            if ((st == kRestart || st == GENLIB_ENOMEM) && !restart_is_error) { if (rc2 == GENLIB_OK) rc2 = kRestart; continue; }
            return fail(st, multi ? "device " + std::to_string(dev[g]) + ": " + r[(size_t)g].message : r[(size_t)g].message);
        }
        return rc2;
    };
    auto create_all = [&](bool streamed) {
        return on_devices(n_dev, [&](int g) { return create_engine(plan, numerics, dev[g], g, &eng[(size_t)g], streamed); });
    };
    auto wire_peers = [&]() {                                    // plain peer pointers instead of IPC mappings
        if (!multi) return;
        for (int g = 0; g < n_dev; g++) {
            for (int h = 0; h < n_dev; h++) { eng[(size_t)g]->peers.A[h] = eng[(size_t)h]->A; eng[(size_t)g]->bars.flags[h] = eng[(size_t)h]->bar_flags; }
            eng[(size_t)g]->attached = true;
        }
    };
    int rc = GENLIB_OK;
    bool done = false;
    if (streaming) {
        ps.wait([&] { return ps.stage.load() >= 1; });
        if (peer_rc == GENLIB_OK && ps.streamed.load() && plan->p.n_unique > 0) {
            StreamConsumer consumer(ps);                          // one registration for all devices
            if (!ps.overflow.load()) {
                rc = first_error(create_all(true), false);
                if (rc == GENLIB_OK) {
                    wire_peers();
                    rc = first_error(on_devices(n_dev, [&](int g) {
                        genlib_engine &E = *eng[(size_t)g];
                        DeviceGuard guard;
                        if (int r = guard.enter(E.device)) return r;
                        int r = numerics == GENLIB_NUMERICS_FP64 ? run_streamed<double>(E, ps) : run_streamed<float>(E, ps);
                        if (r == GENLIB_OK) r = check_device_errors(E);
                        if (r == GENLIB_OK) E.ran = true;
                        return r;
                    }), false);
                    done = rc == GENLIB_OK;
                }
                if (rc == kRestart) rc = GENLIB_OK;
            }
        }
        plan->settle();
    }
    if (plan->worker_rc != GENLIB_OK) return fail(plan->worker_rc, plan->worker_err);
    if (peer_rc != GENLIB_OK) return peer_rc;
    if (rc != GENLIB_OK) return rc;
    if (plan->p.n_unique == 0) {
        if (stats) { std::memset(stats, 0, sizeof *stats); stats->ms_plan = plan->ms_plan; }
        return GENLIB_OK;                                         // 0 x 0 matrix, like the reference
    }
    if (!has_out) return fail(GENLIB_EINVAL, who + ": out is null");
    if (!done) {                                                // plan first, then run (no streaming, or its bounds did not hold)
        for (auto *&x : eng) { genlib_engine_destroy(x); x = nullptr; }
        if ((rc = first_error(create_all(false), true)) != GENLIB_OK) return rc;
        wire_peers();
        if ((rc = first_error(on_devices(n_dev, [&](int g) { return genlib_engine_run(eng[(size_t)g], 0); }), true)) != GENLIB_OK) return rc;
    }
    for (auto *x : eng) x->stats.ms_plan = plan->ms_plan;
    const double t0 = now_ms();
    if (fetch.prepare) fetch.prepare(plan->p);
    rc = first_error(on_devices(n_dev, [&](int g) { return fetch.device(*eng[(size_t)g], g); }), true);
    if (rc == GENLIB_OK && fetch.combine) rc = fetch.combine();
    if (rc == GENLIB_OK && fetch.finish) rc = first_error(on_devices(n_dev, [&](int g) { return fetch.finish(*eng[(size_t)g], g); }), true);
    if (rc != GENLIB_OK) return rc;
    if (stats) {
        *stats = eng[0]->stats;
        if (multi) stats->ms_fetch = now_ms() - t0;             // (one device: genlib_engine_fetch's own time)
        for (int g = 1; g < n_dev; g++) {
            stats->ms_kernels = std::max(stats->ms_kernels, eng[(size_t)g]->stats.ms_kernels);
            stats->ms_upload = std::max(stats->ms_upload, eng[(size_t)g]->stats.ms_upload);
            stats->device_bytes = std::max(stats->device_bytes, eng[(size_t)g]->stats.device_bytes);
            stats->h2d_bytes += eng[(size_t)g]->stats.h2d_bytes;
            stats->d2h_bytes += eng[(size_t)g]->stats.d2h_bytes;
            stats->kernel_launches += eng[(size_t)g]->stats.kernel_launches;
        }
    }
    return GENLIB_OK;
}

// genlib_phi / genlib_phi_multi: one device fetches the whole matrix (genlib_engine_fetch); several fetch a
// contiguous block of output rows each, over their own PCIe links.
static int phi_oneshot(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                       void *out, int out_dtype, int numerics, int32_t n_dev, const int32_t *devices, genlib_stats *stats) {
    if (out_dtype != GENLIB_F32 && out_dtype != GENLIB_F64) return fail(GENLIB_EINVAL, "unknown out_dtype");
    const bool multi = n_dev > 1;
    int32_t nu = 0;
    OneshotFetch fetch;
    fetch.prepare = [&](const Plan &P) { nu = P.n_unique; };
    fetch.device = [&](genlib_engine &E, int g) {
        if (!multi) return genlib_engine_fetch(&E, out, out_dtype);
        DeviceGuard guard;
        if (int r = guard.enter(E.device)) return r;
        const int32_t u0 = (int32_t)((int64_t)nu * g / n_dev), u1 = (int32_t)((int64_t)nu * (g + 1) / n_dev);
        if (numerics == GENLIB_NUMERICS_FP64)
            return out_dtype == GENLIB_F64 ? fetch_block<double, double>(E, u0, u1, (double *)out) : fetch_block<double, float>(E, u0, u1, (float *)out);
        return out_dtype == GENLIB_F64 ? fetch_block<float, double>(E, u0, u1, (double *)out) : fetch_block<float, float>(E, u0, u1, (float *)out);
    };
    return oneshot(multi ? "genlib_phi_multi" : "genlib_phi", GENLIB_SCHEDULE_PHI, n, father, mother, n_pro, proband,
                   out != nullptr, numerics, n_dev, devices, stats, fetch);
}

int genlib_phi_multi(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                     const int32_t *proband, void *out, int out_dtype, int numerics, int32_t n_dev,
                     const int32_t *devices, genlib_stats *stats) {
    if (n_dev < 1 || n_dev > kMaxWorld || !devices) return fail(GENLIB_EINVAL, "genlib_phi_multi: 1 .. 16 devices");
    return phi_oneshot(n, father, mother, n_pro, proband, out, out_dtype, numerics, n_dev, devices, stats);
}

// genlib_phi_over: the genlib_phi run, then on every device a count of each own row's pairs; the host turns the counts
// into offsets in (row, col) order over all devices and allocates the result; every device then writes its pairs in
// its own row order and the host puts each run of consecutive rows in place (one device: they are in place already).
int genlib_phi_over(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                    double threshold, int64_t max_pairs, int out_dtype, int numerics, int32_t n_dev, const int32_t *devices,
                    genlib_kinship_pairs *out, genlib_stats *stats) {
    if (!out) return fail(GENLIB_EINVAL, "genlib_phi_over: out is null");
    *out = genlib_kinship_pairs{0, nullptr, nullptr, nullptr, out_dtype};
    if (n < 0 || n_pro < 0 || (n > 0 && (!father || !mother)) || (n_pro > 0 && !proband))
        return fail(GENLIB_EINVAL, "genlib_phi_over: null pointer or negative size");
    if (std::isnan(threshold)) return fail(GENLIB_EINVAL, "genlib_phi_over: the threshold is NaN");
    if (out_dtype != GENLIB_F32 && out_dtype != GENLIB_F64) return fail(GENLIB_EINVAL, "unknown out_dtype");
    if (numerics != GENLIB_NUMERICS_REFERENCE && numerics != GENLIB_NUMERICS_FP64) return fail(GENLIB_EINVAL, "unknown numerics mode");
    if (n_dev < 1 || n_dev > kMaxWorld || !devices) return fail(GENLIB_EINVAL, "genlib_phi_over: 1 .. 16 devices");
    std::vector<char> seen((size_t)n, 0);
    int32_t distinct = 0;
    for (int32_t k = 0; k < n_pro; k++) {
        const int32_t x = proband[k];
        if (x < 0 || x >= n) {
            std::string err;
            if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);   // (a broken pedigree is reported first)
            return fail(GENLIB_EKEY, "KeyError: index " + std::to_string(x) + " not in pedigree");
        }
        if (!seen[(size_t)x]) { seen[(size_t)x] = 1; distinct++; }
    }
    if (distinct < 2) {                                          // no pair: no plan, no device
        std::string err;
        if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);
        if (stats) { std::memset(stats, 0, sizeof *stats); stats->n_unique = distinct; }
        return GENLIB_OK;
    }
    const bool multi = n_dev > 1, f64 = out_dtype == GENLIB_F64;
    const size_t es = f64 ? sizeof(double) : sizeof(float);
    std::vector<OverRows> rows((size_t)n_dev);
    std::vector<int64_t> goff;                                   // per proband: where its pairs start in the result
    unsigned char *scratch = nullptr;                            // several devices: their pairs in their own row order
    struct FreeHost { unsigned char *&p; ~FreeHost() { if (p) cudaFreeHost(p); } } free_scratch{scratch};
    double t0 = 0;
    int32_t nu = 0;
    OneshotFetch fetch;
    fetch.prepare = [&](const Plan &P) { t0 = now_ms(); nu = P.n_unique; };
    fetch.device = [&](genlib_engine &E, int g) {
        DeviceGuard guard;
        if (int r = guard.enter(E.device)) return r;
        OverRows &R = rows[(size_t)g];
        if (numerics == GENLIB_NUMERICS_FP64)
            return f64 ? phi_over_count<double, double>(E, R, threshold) : phi_over_count<double, float>(E, R, threshold);
        return f64 ? phi_over_count<float, double>(E, R, threshold) : phi_over_count<float, float>(E, R, threshold);
    };
    fetch.combine = [&]() {
        goff.assign((size_t)nu + 1, 0);
        for (const OverRows &R : rows)
            for (size_t r = 0; r < R.own->size(); r++) goff[(size_t)(*R.own)[r] + 1] = R.off[r];
        for (int32_t u = 0; u < nu; u++) goff[(size_t)u + 1] += goff[(size_t)u];
        const int64_t total = goff[(size_t)nu];
        if (max_pairs >= 0 && total > max_pairs) {
            out->n = total;
            char msg[160];
            std::snprintf(msg, sizeof msg, "genlib_phi_over: %lld pairs reach the threshold %.17g, more than max_pairs = %lld",
                          (long long)total, threshold, (long long)max_pairs);
            return fail(GENLIB_EOVERFLOW, msg);
        }
        int64_t base = 0;
        for (OverRows &R : rows) {                               // counts -> offsets in the device's own row order
            R.base = base;
            for (int64_t &o : R.off) { const int64_t c = o; o = base - R.base; base += c; }
        }
        if (total == 0) return (int)GENLIB_OK;
        void *block = nullptr;
        CU(cudaHostAlloc(&block, (size_t)total * (2 * sizeof(int32_t) + es), cudaHostAllocPortable));
        out->row = static_cast<int32_t *>(block);
        out->col = out->row + total;
        out->value = out->col + total;                           // (8 total bytes in: aligned)
        out->n = total;
        for (int32_t u = 0; u < nu; u++) std::fill(out->row + goff[(size_t)u], out->row + goff[(size_t)u + 1], u);
        if (multi) CU(cudaHostAlloc(reinterpret_cast<void **>(&scratch), (size_t)total * (sizeof(int32_t) + es), cudaHostAllocPortable));
        return (int)GENLIB_OK;
    };
    fetch.finish = [&](genlib_engine &E, int g) {
        DeviceGuard guard;
        if (int r = guard.enter(E.device)) return r;
        OverRows &R = rows[(size_t)g];
        const int64_t total = out->n;
        if (total > 0) {
            // scratch: every device's values, then every device's columns
            unsigned char *val = multi ? scratch + (size_t)R.base * es : static_cast<unsigned char *>(out->value);
            int32_t *col = multi ? reinterpret_cast<int32_t *>(scratch + (size_t)total * es) + R.base : out->col;
            int r;
            if (numerics == GENLIB_NUMERICS_FP64)
                r = f64 ? phi_over_select<double, double>(E, R, threshold, col, (double *)val) : phi_over_select<double, float>(E, R, threshold, col, (float *)val);
            else
                r = f64 ? phi_over_select<float, double>(E, R, threshold, col, (double *)val) : phi_over_select<float, float>(E, R, threshold, col, (float *)val);
            if (r != GENLIB_OK) return r;
            const std::vector<int32_t> &own = *R.own;
            for (size_t a = 0; multi && a < own.size();) {       // runs of consecutive proband rows
                size_t b = a + 1;
                while (b < own.size() && own[b] == own[b - 1] + 1) b++;
                const int64_t from = R.off[a], m = R.off[b] - from, to = goff[(size_t)own[a]];
                if (m > 0) {
                    std::memcpy(out->col + to, col + from, (size_t)m * sizeof(int32_t));
                    std::memcpy(static_cast<unsigned char *>(out->value) + (size_t)to * es, val + (size_t)from * es, (size_t)m * es);
                }
                a = b;
            }
        }
        E.stats.ms_fetch = now_ms() - t0;
        return (int)GENLIB_OK;
    };
    const int rc = oneshot("genlib_phi_over", GENLIB_SCHEDULE_PHI, n, father, mother, n_pro, proband, true, numerics, n_dev,
                           devices, stats, fetch);
    if (rc != GENLIB_OK && rc != GENLIB_EOVERFLOW) {             // (over max_pairs: out->n is the count)
        const std::string msg = g_err;
        genlib_kinship_pairs_free(out);
        g_err = msg;
    }
    return rc;
}

int genlib_kinship_pairs_free(genlib_kinship_pairs *pairs) {
    if (!pairs) return GENLIB_OK;
    if (pairs->row) CU(cudaFreeHost(pairs->row));
    pairs->n = 0;
    pairs->row = pairs->col = nullptr;
    pairs->value = nullptr;
    return GENLIB_OK;
}

// genlib_phi_groups: the genlib_phi run, then every device reduces its own proband rows to S (phi_groups_kernel) and
// copies them into proband_mean, device after device in own_pro order (one device: row i lands at row i); the host
// moves the rows to list order, adds T in list order and divides both outputs in place.
int genlib_phi_groups(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                      const int32_t *group, int32_t n_groups, int numerics, int32_t n_dev, const int32_t *devices,
                      double *proband_mean, double *group_mean, genlib_stats *stats) {
    if (n < 0 || n_pro < 0 || n_groups < 0 || (n > 0 && (!father || !mother)) ||
        (n_pro > 0 && (!proband || !group || !proband_mean || !group_mean)))
        return fail(GENLIB_EINVAL, "genlib_phi_groups: null pointer or negative size");
    if (numerics != GENLIB_NUMERICS_REFERENCE && numerics != GENLIB_NUMERICS_FP64) return fail(GENLIB_EINVAL, "unknown numerics mode");
    if (n_dev < 1 || n_dev > kMaxWorld || !devices) return fail(GENLIB_EINVAL, "genlib_phi_groups: 1 .. 16 devices");
    if (n_pro > 0 && n_groups < 1) return fail(GENLIB_EINVAL, "genlib_phi_groups: probands without groups");
    const int32_t G = n_groups;
    std::vector<int64_t> members((size_t)G, 0);    // n_g
    for (int32_t k = 0; k < n_pro; k++) {
        if (group[k] < 0 || group[k] >= G)
            return fail(GENLIB_EINVAL, "genlib_phi_groups: group index " + std::to_string(group[k]) + " of proband position " +
                                       std::to_string(k) + " is not in [0, " + std::to_string(G) + ")");
        members[(size_t)group[k]]++;
    }
    for (int32_t g = 0; g < G; g++)
        if (members[(size_t)g] == 0) return fail(GENLIB_EINVAL, "genlib_phi_groups: group " + std::to_string(g) + " has no proband");
    std::vector<char> seen((size_t)n, 0);
    for (int32_t k = 0; k < n_pro; k++) {
        const int32_t x = proband[k];
        if (x < 0 || x >= n) {
            std::string err;
            if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);   // (a broken pedigree is reported first)
            return fail(GENLIB_EKEY, "KeyError: index " + std::to_string(x) + " not in pedigree");
        }
        if (seen[(size_t)x]) return fail(GENLIB_EINVAL, "genlib_phi_groups: duplicate proband rank " + std::to_string(x));
        seen[(size_t)x] = 1;
    }
    if (n_pro < 2) {                                             // no pair: no plan, no device
        std::string err;
        if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);
        if (stats) { std::memset(stats, 0, sizeof *stats); stats->n_unique = n_pro; }
        if (n_pro == 1) proband_mean[0] = group_mean[0] = std::nan("");
        return GENLIB_OK;
    }
    GroupColumns cols;
    ListOrderRows rows;                                          // where each device's rows land in proband_mean
    double t0 = 0;
    OneshotFetch fetch;
    fetch.prepare = [&](const Plan &P) {
        t0 = now_ms();
        cols.gptr.assign((size_t)G + 1, 0);                      // (the plan's proband u is list position u: no duplicates)
        for (int32_t g = 0; g < G; g++) cols.gptr[(size_t)g + 1] = cols.gptr[(size_t)g] + (int32_t)members[(size_t)g];
        cols.gcol.resize((size_t)n_pro);
        cols.gat.resize((size_t)n_pro);
        std::vector<int32_t> next(cols.gptr.begin(), cols.gptr.end() - 1);
        for (int32_t u = 0; u < n_pro; u++) {
            const int32_t k = next[(size_t)group[u]]++;
            cols.gcol[(size_t)k] = P.pro_slot[(size_t)u];
            cols.gat[(size_t)u] = k;
        }
        rows.prepare(P, n_dev);
    };
    fetch.device = [&](genlib_engine &E, int g) {
        DeviceGuard guard;
        if (int r = guard.enter(E.device)) return r;
        double *dst = proband_mean + (size_t)rows.base[(size_t)g] * G;
        return numerics == GENLIB_NUMERICS_FP64 ? phi_groups_rows<double>(E, cols, dst) : phi_groups_rows<float>(E, cols, dst);
    };
    fetch.combine = [&]() {
        const size_t Gs = (size_t)G;
        rows.to_list_order({{proband_mean, Gs}});                // (one device: in place already)
        std::fill(group_mean, group_mean + Gs * Gs, 0.0);         // T, in list order
        for (int32_t i = 0; i < n_pro; i++) {
            double *t = group_mean + (size_t)group[i] * Gs;
            const double *s = proband_mean + (size_t)i * Gs;
            for (size_t g = 0; g < Gs; g++) t[g] += s[g];
        }
        const double nan = std::nan("");                       // (no pair to average over)
        for (size_t a = 0; a < Gs; a++)                          // T[a][b], a <= b, to both means
            for (size_t b = a; b < Gs; b++) {
                const int64_t pairs = members[a] * members[b] - (a == b ? members[a] : 0);
                group_mean[a * Gs + b] = group_mean[b * Gs + a] = pairs ? group_mean[a * Gs + b] / (double)pairs : nan;
            }
        for (int32_t i = 0; i < n_pro; i++) {
            double *s = proband_mean + (size_t)i * Gs;
            for (size_t g = 0; g < Gs; g++) {
                const int64_t others = members[g] - ((size_t)group[i] == g ? 1 : 0);
                s[g] = others ? s[g] / (double)others : nan;
            }
        }
        return (int)GENLIB_OK;
    };
    fetch.finish = [&](genlib_engine &E, int) {                  // (one device: stats come from its engine)
        E.stats.ms_fetch = now_ms() - t0;
        return (int)GENLIB_OK;
    };
    return oneshot("genlib_phi_groups", GENLIB_SCHEDULE_PHI, n, father, mother, n_pro, proband, true, numerics, n_dev,
                   devices, stats, fetch);
}

// genlib_phi_product: the genlib_phi run, then every device multiplies its own proband rows by X (phi_product_rows)
// into out and diag, device after device in own_pro order; the host moves the rows to list order in place.
int genlib_phi_product(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                       int32_t k, const double *X, int numerics, int32_t n_dev, const int32_t *devices, double *out,
                       double *diag, genlib_stats *stats) {
    if (n < 0 || n_pro < 0 || k < 0 || (n > 0 && (!father || !mother)) || (n_pro > 0 && (!proband || (k > 0 && (!X || !out)))))
        return fail(GENLIB_EINVAL, "genlib_phi_product: null pointer or negative size");
    if (numerics != GENLIB_NUMERICS_REFERENCE && numerics != GENLIB_NUMERICS_FP64) return fail(GENLIB_EINVAL, "unknown numerics mode");
    if (n_dev < 1 || n_dev > kMaxWorld || !devices) return fail(GENLIB_EINVAL, "genlib_phi_product: 1 .. 16 devices");
    std::vector<char> seen((size_t)n, 0);
    for (int32_t p = 0; p < n_pro; p++) {
        const int32_t x = proband[p];
        if (x < 0 || x >= n) {
            std::string err;
            if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);   // (a broken pedigree is reported first)
            return fail(GENLIB_EKEY, "KeyError: index " + std::to_string(x) + " not in pedigree");
        }
        if (seen[(size_t)x]) return fail(GENLIB_EINVAL, "genlib_phi_product: duplicate proband rank " + std::to_string(x));
        seen[(size_t)x] = 1;
    }
    if (n_pro == 0 || (k == 0 && !diag)) {                       // nothing to compute: no plan, no device
        std::string err;
        if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);
        if (stats) { std::memset(stats, 0, sizeof *stats); stats->n_unique = n_pro; }
        return GENLIB_OK;
    }
    ListOrderRows rows;
    double t0 = 0;
    OneshotFetch fetch;
    fetch.prepare = [&](const Plan &P) { t0 = now_ms(); rows.prepare(P, n_dev); };
    fetch.device = [&](genlib_engine &E, int g) {
        DeviceGuard guard;
        if (int r = guard.enter(E.device)) return r;
        const int64_t b = rows.base[(size_t)g];
        double *dst = k > 0 ? out + (size_t)b * k : nullptr, *d = diag ? diag + b : nullptr;
        return numerics == GENLIB_NUMERICS_FP64 ? phi_product_rows<double>(E, X, k, dst, d) : phi_product_rows<float>(E, X, k, dst, d);
    };
    fetch.combine = [&]() {
        rows.to_list_order({{k > 0 ? out : nullptr, (size_t)k}, {diag, 1}});   // (one device: in place already)
        return (int)GENLIB_OK;
    };
    fetch.finish = [&](genlib_engine &E, int) {                  // (one device: stats come from its engine)
        E.stats.ms_fetch = now_ms() - t0;
        return (int)GENLIB_OK;
    };
    return oneshot("genlib_phi_product", GENLIB_SCHEDULE_PHI, n, father, mother, n_pro, proband, true, numerics, n_dev,
                   devices, stats, fetch);
}

// genlib_f: a GENLIB_SCHEDULE_F plan of the listed individuals with both parents; every device copies its per-couple
// kinships to the host once, and each list position takes the value of its couple from the device that holds the
// couple's father row.
int genlib_f(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_ids, const int32_t *ids,
             void *out, int out_dtype, int32_t n_dev, const int32_t *devices, genlib_stats *stats) {
    if (n < 0 || n_ids < 0 || (n > 0 && (!father || !mother)) || (n_ids > 0 && (!ids || !out)))
        return fail(GENLIB_EINVAL, "genlib_f: null pointer or negative size");
    if (out_dtype != GENLIB_F32 && out_dtype != GENLIB_F64) return fail(GENLIB_EINVAL, "unknown out_dtype");
    if (n_dev < 1 || n_dev > kMaxWorld || !devices) return fail(GENLIB_EINVAL, "genlib_f: 1 .. 16 devices");
    bool any = false;                                            // a listed individual with both parents
    for (int32_t i = 0; i < n_ids; i++) {
        const int32_t x = ids[i];
        if (x < 0 || x >= n) {
            std::string err;
            if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);   // (a broken pedigree is reported first)
            return fail(GENLIB_EKEY, "KeyError: index " + std::to_string(x) + " not in pedigree");
        }
        any = any || (father[x] >= 0 && mother[x] >= 0);
    }
    auto put = [&](int32_t i, double v) {
        if (out_dtype == GENLIB_F64) static_cast<double *>(out)[i] = v;
        else static_cast<float *>(out)[i] = (float)v;
    };
    for (int32_t i = 0; i < n_ids; i++) put(i, 0.0);             // a missing parent: F = 0
    if (!any) {                                                  // no plan, no device
        std::string err;
        if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);
        if (stats) std::memset(stats, 0, sizeof *stats);
        return GENLIB_OK;
    }
    std::vector<int64_t> couple;                                 // per list position: its couple (-1: F = 0)
    OneshotFetch fetch;
    fetch.prepare = [&](const Plan &P) {
        std::vector<int64_t> of((size_t)n, -1);
        for (const Layer &L : P.layers)
            for (int32_t q = 0; q < L.n_new; q++) of[(size_t)P.mem_ind[L.mem_off + q]] = (int64_t)L.fam_off + P.mem_fam[L.mem_off + q];
        couple.assign((size_t)n_ids, -1);
        for (int32_t i = 0; i < n_ids; i++)
            if (father[ids[i]] >= 0 && mother[ids[i]] >= 0) couple[(size_t)i] = of[(size_t)ids[i]];
    };
    fetch.device = [&](genlib_engine &E, int g) {
        DeviceGuard guard;
        if (int r = guard.enter(E.device)) return r;
        const double t0 = now_ms();
        const Plan &P = E.plan->p;
        std::vector<double> kin(P.fam_pf.size());
        CU(cudaMemcpyAsync(kin.data(), E.fam_kin.p, kin.size() * sizeof(double), cudaMemcpyDeviceToHost, E.stream));
        CU(cudaStreamSynchronize(E.stream));
        for (int32_t i = 0; i < n_ids; i++) {
            const int64_t c = couple[(size_t)i];
            if (c >= 0 && P.fam_pf_owner[(size_t)c] == g) put(i, kin[(size_t)c]);
        }
        E.stats.d2h_bytes += (int64_t)(kin.size() * sizeof(double));
        E.stats.ms_fetch = now_ms() - t0;
        return GENLIB_OK;
    };
    return oneshot("genlib_f", kScheduleF, n, father, mother, n_ids, ids, true, GENLIB_NUMERICS_FP64, n_dev, devices,
                   stats, fetch);
}

// genlib_phi_pairs: a GENLIB_SCHEDULE_PAIRS plan of everybody named; every device copies its per-read kinships to the
// host once (all K entries: a device leaves the reads it does not own unwritten, and they are not used), and each
// list position takes the value of its read from the device that holds the read's row.
int genlib_phi_pairs(int32_t n, const int32_t *father, const int32_t *mother, int64_t n_pairs, const int32_t *a,
                     const int32_t *b, void *out, int out_dtype, int32_t n_dev, const int32_t *devices, genlib_stats *stats) {
    if (n < 0 || n_pairs < 0 || (n > 0 && (!father || !mother)) || (n_pairs > 0 && (!a || !b || !out)))
        return fail(GENLIB_EINVAL, "genlib_phi_pairs: null pointer or negative size");
    if (out_dtype != GENLIB_F32 && out_dtype != GENLIB_F64) return fail(GENLIB_EINVAL, "unknown out_dtype");
    if (n_dev < 1 || n_dev > kMaxWorld || !devices) return fail(GENLIB_EINVAL, "genlib_phi_pairs: 1 .. 16 devices");
    for (int64_t k = 0; k < n_pairs; k++)
        for (const int32_t x : {a[k], b[k]})
            if (x < 0 || x >= n) {
                std::string err;
                if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);   // (a broken pedigree is reported first)
                return fail(GENLIB_EKEY, "KeyError: index " + std::to_string(x) + " not in pedigree");
            }
    if (n_pairs == 0) {                                          // no plan, no device
        std::string err;
        if (int rc = check_pedigree(n, father, mother, err)) return fail(rc, err);
        if (stats) std::memset(stats, 0, sizeof *stats);
        return GENLIB_OK;
    }
    auto put = [&](int64_t i, double v) {
        if (out_dtype == GENLIB_F64) static_cast<double *>(out)[i] = v;
        else static_cast<float *>(out)[i] = (float)v;
    };
    OneshotFetch fetch;
    fetch.device = [&](genlib_engine &E, int g) {
        DeviceGuard guard;
        if (int r = guard.enter(E.device)) return r;
        const double t0 = now_ms();
        const Plan &P = E.plan->p;
        std::vector<double> kin(P.pair_pos.size());
        CU(cudaMemcpyAsync(kin.data(), E.pair_kin.p, kin.size() * sizeof(double), cudaMemcpyDeviceToHost, E.stream));
        CU(cudaStreamSynchronize(E.stream));
        for (size_t i = 0; i < kin.size(); i++)
            if (P.pair_owner[i] == g) put(P.pair_pos[i], kin[i]);
        E.stats.d2h_bytes += (int64_t)(kin.size() * sizeof(double));
        E.stats.ms_fetch = now_ms() - t0;
        return GENLIB_OK;
    };
    return oneshot("genlib_phi_pairs", kSchedulePairs, n, father, mother, 0, nullptr, true, GENLIB_NUMERICS_FP64, n_dev,
                   devices, stats, fetch, PairList{n_pairs, a, b});
}

int genlib_phi(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
               const int32_t *proband, void *out, int out_dtype, int numerics, int device,
               genlib_stats *stats) {
    const int32_t dev = device;
    return phi_oneshot(n, father, mother, n_pro, proband, out, out_dtype, numerics, 1, &dev, stats);
}

int genlib_plan_stream_selftest(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                                const int32_t *proband, int32_t world, double slack_pct,
                                int32_t *layers_streamed, int32_t *overflowed) {
    if (layers_streamed) *layers_streamed = 0;
    if (overflowed) *overflowed = 0;
    {
        char buf[64];
        std::snprintf(buf, sizeof buf, "%g", slack_pct);
        setenv("GENLIB_STREAM_SLACK_PCT", buf, 1);
    }
    struct EnvReset { ~EnvReset() { unsetenv("GENLIB_STREAM_SLACK_PCT"); } } env_reset;
    Plan ref, P;
    std::string err;
    int rc = build_plan(n, father, mother, nullptr, n_pro, proband, world, GENLIB_SCHEDULE_PHI, ref, err);
    if (rc != GENLIB_OK) return fail(rc, err);
    PlanStream ps;
    int plan_rc = GENLIB_OK;
    std::string plan_err;
    std::thread worker([&] { plan_rc = build_plan(n, father, mother, nullptr, n_pro, proband, world, GENLIB_SCHEDULE_PHI, P, plan_err, &ps); });
    // the consumer: copies of the published slices, taken when they are published
    std::vector<int32_t> c_mem_slot, c_fam_pf, c_fam_start, c_live_tiles, c_mtile, c_live_lrow;
    std::vector<uint8_t> c_flags;
    int done = 0;
    bool saw_overflow = false;
    int64_t bound = 0;
    ps.wait([&] { return ps.stage.load() >= 1; });
    if (ps.streamed.load()) {
        ps.consumers.fetch_add(1);
        bound = P.capacity;
        const int S = (int)P.layers.size();
        while (done < S) {
            ps.wait([&] { return ps.layers_done.load(std::memory_order_acquire) > done || ps.overflow.load() || ps.stage.load() == 2; });
            const bool ovf = ps.overflow.load();
            const int avail = ps.layers_done.load(std::memory_order_acquire);
            if (avail > done) {
                const Layer &Z = P.layers[(size_t)avail - 1];
                auto grab = [&](auto &copy, const auto &src, size_t end) { copy.insert(copy.end(), src.data() + copy.size(), src.data() + end); };
                grab(c_mem_slot, P.mem_slot, Z.mem_end); grab(c_fam_pf, P.fam_pf, Z.fam_end);
                grab(c_fam_start, P.fam_start, Z.fam_end + (size_t)avail); grab(c_live_tiles, P.live_tiles, Z.ltile_end);
                grab(c_mtile, P.mtile_desc, 4 * Z.mtile_end); grab(c_live_lrow, P.live_lrow, Z.flag_end);
                grab(c_flags, P.flags, Z.flag_end);
                done = avail;
            }
            if (ovf) { saw_overflow = true; break; }
            if (avail < S && ps.stage.load() == 2 && ps.layers_done.load() == avail) break;
        }
        ps.consumers.fetch_sub(1);
        ps.wake();
    }
    worker.join();
    if (plan_rc != GENLIB_OK) return fail(plan_rc, plan_err);
    if (layers_streamed) *layers_streamed = done;
    if (overflowed) *overflowed = saw_overflow ? 1 : 0;
    auto prefix_ok = [](const auto &copy, const auto &fin) { return copy.size() <= fin.size() && std::equal(copy.begin(), copy.end(), fin.begin()); };
    if (!prefix_ok(c_mem_slot, P.mem_slot) || !prefix_ok(c_fam_pf, P.fam_pf) || !prefix_ok(c_fam_start, P.fam_start) ||
        !prefix_ok(c_live_tiles, P.live_tiles) || !prefix_ok(c_mtile, P.mtile_desc) || !prefix_ok(c_live_lrow, P.live_lrow) ||
        !prefix_ok(c_flags, P.flags))
        return fail(GENLIB_EINVAL, "stream selftest: a published slice changed afterwards");
    if (ps.streamed.load() && !saw_overflow && done != (int)P.layers.size()) return fail(GENLIB_EINVAL, "stream selftest: not every layer was published");
    // the streamed plan against the plan made in one piece
    bool same = P.n_unique == ref.n_unique && P.layers.size() == ref.layers.size() && P.row_updates == ref.row_updates &&
                P.mem_ind == ref.mem_ind && P.mem_slot == ref.mem_slot && P.mem_fam == ref.mem_fam && P.mem_lrow == ref.mem_lrow &&
                P.fam_pf == ref.fam_pf && P.fam_pm == ref.fam_pm && P.fam_q == ref.fam_q && P.fam_start == ref.fam_start &&
                P.fam_pf_lrow == ref.fam_pf_lrow && P.fam_pm_lrow == ref.fam_pm_lrow && P.fam_pf_owner == ref.fam_pf_owner &&
                P.fam_pm_owner == ref.fam_pm_owner && P.flags == ref.flags && P.live_owner == ref.live_owner &&
                P.live_lrow == ref.live_lrow && P.tile_map == ref.tile_map && P.live_tiles == ref.live_tiles &&
                P.mtile_desc == ref.mtile_desc && P.fam_base == ref.fam_base && P.mem_base == ref.mem_base &&
                P.pro_slot == ref.pro_slot && P.pro_owner == ref.pro_owner && P.pro_lrow == ref.pro_lrow;
    for (size_t t = 0; same && t < P.layers.size(); t++) {
        const Layer &a = P.layers[t], &b = ref.layers[t];
        same = a.n_new == b.n_new && a.n_fam == b.n_fam && a.rt_lo == b.rt_lo && a.rt_rows == b.rt_rows && a.mem_off == b.mem_off &&
               a.fam_off == b.fam_off && a.flag_off == b.flag_off && a.tile_off == b.tile_off && a.ltile_off == b.ltile_off &&
               a.mtile_off == b.mtile_off && a.n_mtiles == b.n_mtiles && a.n_live_tiles == b.n_live_tiles && a.carried == b.carried;
    }
    if (!same) return fail(GENLIB_EINVAL, "stream selftest: the streamed plan differs from the plan made in one piece");
    const bool kept_bound = ps.streamed.load() && !saw_overflow;
    if (kept_bound ? (P.capacity != bound || P.capacity < ref.capacity) : (P.capacity != ref.capacity))
        return fail(GENLIB_EINVAL, "stream selftest: frontier width " + std::to_string(P.capacity) + " against " + std::to_string(ref.capacity));
    for (int g = 0; g < world; g++)
        if (kept_bound ? P.rows_cap[(size_t)g] < ref.rows_cap[(size_t)g] : P.rows_cap[(size_t)g] != ref.rows_cap[(size_t)g])
            return fail(GENLIB_EINVAL, "stream selftest: rows of rank " + std::to_string(g));
    return GENLIB_OK;
}

}  // extern "C"
