// engine.cu -- device runtime + C ABI of libgenlib_cuda.so (include/genlib_cuda.h).
//
// The ABI stands where the reference's Julia method stands:
//   phi(pedigree, probandIDs; verbose, compute)            src/compute.jl:233-304
// There is no CPU fallback: without a usable CUDA device every compute entry
// point returns GENLIB_ECUDA.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/genlib_cuda.h"
#include "gc_kernel.cuh"
#include "gc_plan.hpp"
#include "kernels.cuh"
#include "layer_kernel.cuh"
#include "plan.hpp"

using namespace genlib;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg) { g_err = msg; return code; }
}  // namespace
int genlib::set_error(int code, const std::string &msg) { return fail(code, msg); }
namespace {

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(e_ == cudaErrorMemoryAllocation ? GENLIB_ENOMEM : GENLIB_ECUDA,       \
                        std::string(#call) + ": " + cudaGetErrorString(e_));                  \
    } while (0)

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

struct DeviceGuard {
    int prev = -1;
    bool active = false;
    int enter(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) return fail(GENLIB_ECUDA, "no usable CUDA device (cudaGetDevice failed)");
        if (dev >= 0 && dev != prev) {
            if (cudaSetDevice(dev) != cudaSuccess) return fail(GENLIB_ECUDA, "cudaSetDevice failed");
            active = true;
        }
        return GENLIB_OK;
    }
    ~DeviceGuard() { if (active) cudaSetDevice(prev); }
};

// ---- device arena: ONE allocation per engine, cached across calls -------------------------
// cudaMalloc / cudaFree of tens of GB cost hundreds of milliseconds; a repeated gen.phi call
// (and the one-shot genlib_phi) reuses the previous arena when it is large enough.
struct Arena {
    void *base = nullptr;
    size_t size = 0;
    int device = -1;
    bool exported = false;      // a CUDA-IPC handle of it was handed out: peer processes may keep it mapped
};

class ArenaCache {
    std::mutex mu_;
    std::vector<Arena> free_;
public:
    cudaError_t acquire(int device, size_t bytes, Arena &out) {
        {
            std::lock_guard<std::mutex> g(mu_);
            int best = -1;
            for (int i = 0; i < (int)free_.size(); i++)
                if (free_[i].device == device && free_[i].size >= bytes && (best < 0 || free_[i].size < free_[best].size)) best = i;
            if (best >= 0) { out = free_[best]; free_.erase(free_.begin() + best); return cudaSuccess; }
        }
        // Nothing cached fits.  The smaller cached arenas of this device are given back first (a long-lived
        // process would otherwise pin one arena per size it ever needed) -- except those a peer process may
        // still have mapped (CUDA IPC: freeing exported memory under an open mapping is undefined); these go
        // only when the device is out of memory.
        release_device(device, /*also_exported=*/false);
        out = Arena{nullptr, bytes, device, false};
        cudaError_t ce = cudaMalloc(&out.base, bytes);
        if (ce == cudaErrorMemoryAllocation) {
            cudaGetLastError();
            release_device(device, true);
            ce = cudaMalloc(&out.base, bytes);
        }
        return ce;
    }
    void release(Arena a) {
        if (!a.base) return;
        std::lock_guard<std::mutex> g(mu_);
        free_.push_back(a);
    }
    void release_device(int device, bool also_exported = true) {
        std::lock_guard<std::mutex> g(mu_);
        for (size_t i = 0; i < free_.size();) {
            if ((device < 0 || free_[i].device == device) && (also_exported || !free_[i].exported)) {
                int prev = -1; cudaGetDevice(&prev);
                cudaSetDevice(free_[i].device); cudaFree(free_[i].base);
                if (prev >= 0) cudaSetDevice(prev);
                free_.erase(free_.begin() + (long)i);
            } else i++;
        }
    }
};
ArenaCache g_arenas;

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

// non-owning typed view into the arena
template <typename T> struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    static size_t padded(size_t count) { return (std::max<size_t>(count, 1) * sizeof(T) + 255) / 256 * 256; }
    void place(unsigned char *&cursor, size_t count) { p = reinterpret_cast<T *>(cursor); n = count; cursor += padded(count); }
    cudaError_t upload(const std::vector<T> &h, cudaStream_t s) {
        if (h.empty()) return cudaSuccess;
        return cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s);
    }
};

constexpr size_t kFetchStageBytes = (size_t)64 << 20;

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
    PlanStream *consuming = nullptr;       // registered as a reader of that plan's arrays (until the streamed run ends)
    void stop_consuming() { if (consuming) { consuming->consumers.fetch_sub(1); consuming->wake(); consuming = nullptr; } }
    std::vector<int32_t> own_pro;          // proband indices (output rows) this rank owns, ascending
    std::vector<genlib_layer_info> info;
    std::vector<cudaEvent_t> events;
    genlib_stats stats{};
    bool ran = false;
    int32_t layer_limit = -1;
    ~genlib_engine() {
        stop_consuming();
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

size_t pad256(size_t b) { return (std::max<size_t>(b, 1) + 255) / 256 * 256; }

size_t plan_index_bytes(const Plan &P) {
    return (P.mem_ind.size() * 4 + P.mem_rank.size() + P.fam_pf.size() * 6 + P.fam_start.size() + P.mtile_desc.size() +
            P.pro_slot.size() * 2 + P.live_lrow.size() + P.tile_map.size() + P.live_tiles.size()) * sizeof(int32_t) + P.fam_pf.size() * 2 + P.live_owner.size() + P.flags.size();
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
    // consumer groups per CTA, each with its own items and shared memory (two only fit with narrower strips)
    const int groups = std::max(1, std::min(kConsGroups, env_int("GENLIB_CONS_GROUPS", kConsGroups)));
    const int sw_cap = (es == 4 ? kMaxStrip : kMaxStrip / 2) / groups;
    const size_t budget = (size_t)std::max(16, env_int("GENLIB_STRIP_BUDGET_MB", (int)(kStripBudget >> 20))) << 20;
    int sw = std::min(sw_cap, std::max(8, env_int("GENLIB_MAX_SW", kMaxStrip)));
    while (sw > 8 && (size_t)q_rows * sw * pair * min_buf > budget) sw >>= 1;
    const size_t strip_bytes = std::max<size_t>((size_t)q_rows * sw * pair, 256);
    s.sw = sw;
    // couples per producer item: 32 rows of 512 B (float) / 16 rows of 1 KB (double); at most two items per live tile
    s.ft = std::max(sw / 2, std::min(sw, std::max(8, env_int("GENLIB_FT", es == 4 ? 32 : 16))));
    if (s.ft > 32) s.ft = 32;
    s.n_strips = (int)((own_nf + sw - 1) / sw);
    s.qstride = (int64_t)(strip_bytes / pair);
    // producer items: 2 ft parent rows x one live tile; consumer items: the member tiles
    s.n_pitems = live ? (sw / s.ft) * L.n_live_tiles : 0;
    s.n_citems = L.n_mtiles;
    s.discard = env_int("GENLIB_DISCARD", 2);     // 0: off, 1: without the release fence (experiments), 2: on
    // One CTA per SM: four producer warps and a consumer group of eight.  Every CTA of a gang takes part in the
    // hand-over of each of the gang's strips, whether it has an item there or not, and a switch of strips costs a
    // CTA some microseconds of dependent loads: a strip should bring every CTA several items.  Layers with short
    // strips (few live tiles) therefore split the CTAs into G gangs that work on G strips side by side
    // (profiles/r02/README.md: C5 245 -> ... ms, genea140 7.3 -> ... ms); C3-sized layers stay with one gang.
    const int max_buf = (int)std::max<size_t>(2, budget / strip_bytes);
    int G = 1;
    if (live) {
        const int forced = env_int("GENLIB_GANGS", 0);
        const int want_items = std::max(1, env_int("GENLIB_GANG_ITEMS", kGangItems));
        if (forced > 0) G = forced;
        else while (G < kMaxGangs && (int64_t)s.n_pitems * G < (int64_t)want_items * sm_count) G *= 2;
        while (G > 1 && (2 * G > max_buf || s.n_strips < 2 * G || G > sm_count / 4)) G /= 2;
    }
    s.gangs = G;
    // (at most eight buffers per gang: the producer warps of a CTA count themselves off in eight slots by strip)
    s.nbuf = std::min(8 * G, std::max(2 * G, std::min(std::max(2 * G, env_int("GENLIB_MAX_NBUF", 8)), max_buf)) / G * G);
    // (one gang) layers with few items per strip run faster on 7/8 of the SMs (C5: 148 CTAs 246 ms, 128 to 136 CTAs
    // 148 ms; genea140: 8.9 -> 6.4 ms); layers with several items per CTA and strip want every SM (C3: 70.8 ms on
    // 148, 74.3 ms on 132).
    const int few = G == 1 && (sw / s.ft) * L.n_live_tiles < 3 * sm_count / 2 ? sm_count - sm_count / 8 : sm_count;
    const int ctas = std::max(1, std::min(sm_count, env_int("GENLIB_CTAS_PER_ROLE", few))) / G;   // per gang
    s.n_prod = G * std::min(ctas, s.n_pitems);
    s.groups = groups;
    s.n_cons = G * std::min(ctas * groups, s.n_citems);
    const size_t stage = (size_t)2 * s.ft * (kPTile * es + 16);
    // eight producer warps (and four consumer warps) where the producers have the carried columns to write as well
    {
        const int forced = env_int("GENLIB_PROD_WARPS", 0);
        out.prod_warps = forced == 4 || forced == 8 ? forced : (L.carried > 0 && live && kConsGroups == 1 ? 8 : 4);
    }
    const size_t cons_bytes = layer_consumer_bytes(sw, es, out.prod_warps);
    const size_t smem_cap = (size_t)227 * 1024 - 2048;      // (static shared memory and the driver's share)
    s.stages = (int)std::max<size_t>(2, std::min<size_t>((size_t)std::min(kMaxStages, env_int("GENLIB_STAGES", kMaxStages)), (smem_cap - groups * cons_bytes) / stage));
    s.cons_bytes = (int32_t)cons_bytes;
    s.ring_off = (int32_t)(groups * cons_bytes);
    out.smem = groups * cons_bytes + (size_t)s.stages * stage;
    out.grid = std::max(s.n_prod, (s.n_cons + groups - 1) / groups);
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
    a.n_new = L.n_new; a.n_fam = L.n_fam; a.rt_lo = L.rt_lo; a.rt_rows = L.live_before > 0 ? L.rt_rows : 0; a.nf_pad = L.nf_pad;
    a.any_carried = L.carried > 0;
    a.rank = E.rank; a.world = E.world;
    const int32_t *fb = P.fam_base.data() + L.base_off, *mb = P.mem_base.data() + L.base_off;
    for (int g = 0; g <= E.world; g++) a.fam_base[g] = fb[g];
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
    a.tile_map = E.tile_map.p + L.tile_off;
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

// one generation step: the layer kernel (and sparse_phi's misfiled pairs), then the inter-GPU barrier
template <typename T>
int launch_layer(genlib_engine &E, int t, bool timed, size_t &ev, int &launches) {
    const Plan &P = E.plan->p;
    const Layer &L = P.layers[t];
    if (L.n_new == 0) return GENLIB_OK;
    T *A = static_cast<T *>(E.A);
    const int64_t ld = P.capacity;
    LayerArgs a = layer_args(E, t);
    LayerLaunch &ll = E.launch[t];
    auto layer_fn = layer_function<T>(P, ll.prod_warps);
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
    for (int t = 0; t < (int)P.layers.size(); t++) {
        if (E.layer_limit >= 0 && t >= E.layer_limit) break;
        if (int rc = launch_layer<T>(E, t, timed, ev, launches)) return rc;
    }
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
    CU(cudaGetLastError());
    E.stats.kernel_launches = launches;
    ps.wait([&] { return ps.stage.load() == 2; });              // the probands' homes close the plan
    if (ps.status.load() != GENLIB_OK) return ps.status.load();
    if (ps.overflow.load()) { cudaStreamSynchronize(E.stream); return kRestart; }
    if (int rc = upload_probands(E)) return rc;
    CU(cudaEventRecord(E.events[nev - 1], E.stream));
    CU(cudaStreamSynchronize(E.stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, E.events[nev - 2], E.events[nev - 1]));
    E.stats.ms_kernels = ms;                                    // first launch to last: includes waiting for the planner
    E.stats.row_updates = P.row_updates; E.stats.alg_bytes = P.alg_elems * (double)E.esize;
    E.stats.h2d_bytes = (int64_t)plan_index_bytes(P);
    return GENLIB_OK;
}

// Rows of this rank's probands (own_pro order), all proband columns, streamed to host memory.
template <typename T, typename O>
int fetch_rows(genlib_engine &E, O *out) {
    const Plan &P = E.plan->p;
    const int32_t n = P.n_unique, nown = (int32_t)E.own_pro.size();
    if (n == 0 || nown == 0) return GENLIB_OK;
    // stream row blocks through two staging buffers so the gather of block b+1
    // overlaps the D2H copy of block b
    const size_t row_bytes = (size_t)n * sizeof(O);
    int32_t rows_per = (int32_t)std::max<size_t>(1, std::min<size_t>((size_t)nown, kFetchStageBytes / row_bytes));
    if ((size_t)rows_per * row_bytes > kFetchStageBytes) return fail(GENLIB_EINVAL, "proband row does not fit the staging buffer");
    rows_per = std::min(rows_per, 65535);
    O *stage[2] = {reinterpret_cast<O *>(E.fetch_stage[0]), reinterpret_cast<O *>(E.fetch_stage[1])};
    cudaEvent_t done[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
    cudaError_t ce = cudaSuccess;
    for (int b = 0; b < 2 && ce == cudaSuccess; b++) {
        ce = cudaEventCreateWithFlags(&done[b], cudaEventDisableTiming);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&copied[b], cudaEventDisableTiming);
    }
    int blk = 0;
    for (int32_t r0 = 0; r0 < nown && ce == cudaSuccess; r0 += rows_per, blk++) {
        const int b = blk & 1;
        const int32_t nr = std::min(rows_per, nown - r0);
        if (blk >= 2 && (ce = cudaStreamWaitEvent(E.stream, copied[b], 0)) != cudaSuccess) break;
        dim3 grid((unsigned)std::min<int32_t>((n + 255) / 256, 64), (unsigned)nr);
        gather_kernel<T, O><<<grid, 256, 0, E.stream>>>(static_cast<const T *>(E.A), P.capacity, E.own_pro_row.p, E.pro_slot.p,
                                                       n, r0, nr, stage[b]);
        cudaEventRecord(done[b], E.stream);
        cudaStreamWaitEvent(E.copy_stream, done[b], 0);
        ce = cudaMemcpyAsync(out + (size_t)r0 * n, stage[b], (size_t)nr * row_bytes, cudaMemcpyDeviceToHost, E.copy_stream);
        cudaEventRecord(copied[b], E.copy_stream);
    }
    const cudaError_t e1 = cudaStreamSynchronize(E.stream), e2 = cudaStreamSynchronize(E.copy_stream);
    for (int b = 0; b < 2; b++) { if (done[b]) cudaEventDestroy(done[b]); if (copied[b]) cudaEventDestroy(copied[b]); }
    if (ce != cudaSuccess || e1 != cudaSuccess || e2 != cudaSuccess)
        return fail(GENLIB_ECUDA, std::string("proband fetch failed: ") + cudaGetErrorString(ce != cudaSuccess ? ce : e1 != cudaSuccess ? e1 : e2));
    E.stats.d2h_bytes += (int64_t)nown * (int64_t)row_bytes;
    return GENLIB_OK;
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
    O *stage[2] = {reinterpret_cast<O *>(E.fetch_stage[0]), reinterpret_cast<O *>(E.fetch_stage[1])};
    cudaEvent_t done[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
    cudaError_t ce = cudaSuccess;
    for (int b = 0; b < 2 && ce == cudaSuccess; b++) {
        ce = cudaEventCreateWithFlags(&done[b], cudaEventDisableTiming);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&copied[b], cudaEventDisableTiming);
    }
    int blk = 0;
    for (int32_t r0 = u0; r0 < u1 && ce == cudaSuccess; r0 += rows_per, blk++) {
        const int b = blk & 1;
        const int32_t nr = std::min(rows_per, u1 - r0);
        if (blk >= 2 && (ce = cudaStreamWaitEvent(E.stream, copied[b], 0)) != cudaSuccess) break;
        dim3 grid((unsigned)std::min<int32_t>((n + 255) / 256, 64), (unsigned)nr);
        gather_peer_kernel<T, O><<<grid, 256, 0, E.stream>>>(E.peers, P.capacity, E.pro_owner.p, E.pro_lrow.p, E.pro_slot.p, n, r0, nr, stage[b]);
        cudaEventRecord(done[b], E.stream);
        cudaStreamWaitEvent(E.copy_stream, done[b], 0);
        ce = cudaMemcpyAsync(out + (size_t)r0 * n, stage[b], (size_t)nr * row_bytes, cudaMemcpyDeviceToHost, E.copy_stream);
        cudaEventRecord(copied[b], E.copy_stream);
    }
    const cudaError_t e1 = cudaStreamSynchronize(E.stream), e2 = cudaStreamSynchronize(E.copy_stream);
    for (int b = 0; b < 2; b++) { if (done[b]) cudaEventDestroy(done[b]); if (copied[b]) cudaEventDestroy(copied[b]); }
    if (ce != cudaSuccess || e1 != cudaSuccess || e2 != cudaSuccess)
        return fail(GENLIB_ECUDA, std::string("proband fetch failed: ") + cudaGetErrorString(ce != cudaSuccess ? ce : e1 != cudaSuccess ? e1 : e2));
    E.stats.d2h_bytes += (int64_t)(u1 - u0) * (int64_t)row_bytes;
    return GENLIB_OK;
}

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

// this rank's probands in output order, and where their rows and columns are (needs the finished plan)
int upload_probands(genlib_engine &E) {
    const Plan &P = E.plan->p;
    std::vector<int32_t> own_rows;
    E.own_pro.clear();
    for (size_t u = 0; u < P.pro_ind.size(); u++)
        if (P.pro_owner[u] == E.rank) { E.own_pro.push_back((int32_t)u); own_rows.push_back(P.pro_lrow[u]); }
    CU(E.pro_slot.upload(P.pro_slot, E.stream));
    CU(E.own_pro_row.upload(own_rows, E.stream));
    CU(E.pro_owner.upload(P.pro_owner, E.stream));
    CU(E.pro_lrow.upload(P.pro_lrow, E.stream));
    CU(cudaStreamSynchronize(E.stream));                       // (own_rows is a local)
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
    return GENLIB_OK;
}

int create_engine(const genlib_plan *plan, int numerics, int device, int rank, genlib_engine **out, bool streamed = false) {
    if (!plan || !out) return fail(GENLIB_EINVAL, "genlib_engine_create: null argument");
    *out = nullptr;
    if (numerics != GENLIB_NUMERICS_REFERENCE && numerics != GENLIB_NUMERICS_FP64) return fail(GENLIB_EINVAL, "unknown numerics mode");
    const Plan &P = plan->p;
    if (sparse_schedule(P.schedule) && numerics != GENLIB_NUMERICS_REFERENCE)
        return fail(GENLIB_EINVAL, "the sparse_phi schedule stores Float32 (numerics must be GENLIB_NUMERICS_REFERENCE)");
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
        cudaError_t ce = g_arenas.acquire(E->device, need, E->arena);
        if (ce != cudaSuccess) {
            E->arena = Arena();
            cudaGetLastError();
            size_t free_b = 0, total_b = 0;
            cudaMemGetInfo(&free_b, &total_b);
            char msg[256];
            std::snprintf(msg, sizeof msg, "rank %d needs %.2f GB on the device, %.2f GB free (capacity %lld slots, %lld rows): shard over more GPUs",
                          rank, need / 1e9, free_b / 1e9, (long long)P.capacity, (long long)P.rows_cap[rank]);
            return fail(GENLIB_ENOMEM, msg);
        }
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
    // Optional (GENLIB_L2_PERSIST=1): a persisting access-policy window for the strip buffers on the engine's
    // stream.  Off by default: it limits the buffers to the 79 MB that can persist and measured slower.
    {
        int max_persist = 0, max_window = 0;
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, E->device);
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, E->device);
        const char *env = std::getenv("GENLIB_L2_PERSIST");                // "1": persisting window (measured slower, see kStripBudget)
        if (max_persist > 0 && max_window > 0 && env && env[0] == '1') {
            cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)max_persist);
            cudaStreamAttrValue attr;
            std::memset(&attr, 0, sizeof attr);
            attr.accessPolicyWindow.base_ptr = E->Q;
            attr.accessPolicyWindow.num_bytes = std::min<size_t>(E->q_bytes, (size_t)max_window);
            attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)max_persist / (double)std::max<size_t>(E->q_bytes, 1));
            attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
            if (cudaStreamSetAttribute(E->stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
        }
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
    s.capacity = P.capacity; s.device_bytes = (int64_t)need; s.alg_bytes = P.alg_elems * (double)E->esize;
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

int genlib_plan_create_ex(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids, int32_t n_pro,
                          const int32_t *proband, int32_t world, int schedule, genlib_plan **out) {
    if (!out) return fail(GENLIB_EINVAL, "genlib_plan_create: out is null");
    *out = nullptr;
    std::unique_ptr<genlib_plan> pl(new (std::nothrow) genlib_plan);
    if (!pl) return fail(GENLIB_ENOMEM, "out of host memory");
    const double t0 = now_ms();
    std::string err;
    int rc;
    try {
        adopt_retired_storage(pl->p);        // the arrays of the last destroyed plan, already paged in
        rc = build_plan(n, father, mother, ids, n_pro, proband, world, schedule, pl->p, err);
    } catch (const std::bad_alloc &) {
        return fail(GENLIB_ENOMEM, "out of host memory while planning");
    }
    if (rc != GENLIB_OK) return fail(rc, err);
    pl->ms_plan = now_ms() - t0;
    *out = pl.release();
    return GENLIB_OK;
}

int genlib_plan_create_async(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids, int32_t n_pro,
                             const int32_t *proband, int32_t world, int schedule, genlib_plan **out) {
    if (!out) return fail(GENLIB_EINVAL, "genlib_plan_create: out is null");
    *out = nullptr;
    if (env_int("GENLIB_STREAM", 1) == 0) return genlib_plan_create_ex(n, father, mother, ids, n_pro, proband, world, schedule, out);
    std::unique_ptr<genlib_plan> pl(new (std::nothrow) genlib_plan);
    if (!pl) return fail(GENLIB_ENOMEM, "out of host memory");
    pl->stream.reset(new (std::nothrow) PlanStream);
    if (!pl->stream) return fail(GENLIB_ENOMEM, "out of host memory");
    genlib_plan *raw = pl.get();
    const double t0 = now_ms();
    try {
        raw->worker = std::thread([=] {
            try {
                adopt_retired_storage(raw->p);
                raw->worker_rc = build_plan(n, father, mother, ids, n_pro, proband, world, schedule, raw->p, raw->worker_err, raw->stream.get());
            } catch (const std::bad_alloc &) {
                raw->worker_rc = GENLIB_ENOMEM; raw->worker_err = "out of host memory while planning";
                raw->stream->status.store(GENLIB_ENOMEM); raw->stream->stage.store(2); raw->stream->wake();
            }
            raw->ms_plan = now_ms() - t0;
        });
    } catch (...) {                              // no thread to be had
        pl.reset();
        return genlib_plan_create_ex(n, father, mother, ids, n_pro, proband, world, schedule, out);
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

void genlib_plan_destroy(genlib_plan *plan) {
    if (!plan) return;
    plan->settle();
    try { retire_storage(plan->p); } catch (...) {}
    delete plan;
}
uint64_t genlib_plan_digest(const genlib_plan *plan, int with_bounds) {
    settle(plan);
    if (!plan) return 0;
    const Plan &P = plan->p;
    uint64_t h = 1469598103934665603ULL;
    auto bytes = [&h](const void *p, size_t nb) { const unsigned char *c = (const unsigned char *)p; for (size_t i = 0; i < nb; i++) { h ^= c[i]; h *= 1099511628211ULL; } };
    auto vec = [&bytes](const auto &v) { const uint64_t s = v.size(); bytes(&s, 8); if (s) bytes(v.data(), s * sizeof(v[0])); };
    const int64_t hdr[6] = {P.n, P.n_unique, P.world, P.schedule, with_bounds ? P.capacity : 0, P.row_updates};
    bytes(hdr, sizeof hdr); bytes(&P.alg_elems, 8);
    for (const Layer &L : P.layers) {
        const int64_t f[] = {L.n_new, L.n_fam, L.live_before, L.carried, L.ref_founders, L.ref_probands, L.ref_both, L.rt_lo, L.rt_rows,
                             L.n_live_tiles, (int64_t)L.tile_off, (int64_t)L.ltile_off, L.nf_pad, L.n_mtiles, L.max_tile_fam,
                             (int64_t)L.mem_off, (int64_t)L.fam_off, (int64_t)L.flag_off, (int64_t)L.mtile_off, (int64_t)L.base_off,
                             (int64_t)L.mem_end, (int64_t)L.fam_end, (int64_t)L.flag_end, (int64_t)L.tile_end, (int64_t)L.ltile_end,
                             (int64_t)L.mtile_end};
        bytes(f, sizeof f); bytes(&L.alg_elems, 8);
    }
    vec(P.pro_ind); vec(P.pro_slot); vec(P.mem_ind); vec(P.mem_slot); vec(P.mem_fam); vec(P.mem_rank); vec(P.fam_pf); vec(P.fam_pm);
    vec(P.fam_start); vec(P.fam_q); vec(P.flags); vec(P.tile_map); vec(P.live_tiles); vec(P.mtile_desc); vec(P.fam_base); vec(P.mem_base);
    vec(P.mem_lrow); vec(P.fam_pf_owner); vec(P.fam_pm_owner); vec(P.fam_pf_lrow); vec(P.fam_pm_lrow); vec(P.live_owner); vec(P.live_lrow);
    vec(P.pro_owner); vec(P.pro_lrow);
    if (with_bounds) vec(P.rows_cap);
    return h;
}
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
    for (size_t u = 0; u < plan->p.pro_ind.size(); u++) { owner[u] = plan->p.pro_owner[u]; lrow[u] = plan->p.pro_lrow[u]; }
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
    if (plan && plan->streaming()) {
        PlanStream &ps = *plan->stream;
        ps.consumers.fetch_add(1);
        if (!ps.overflow.load() && ps.stage.load() != 2) {
            int rc = create_engine(plan, numerics, device, rank, out, true);
            if (rc == GENLIB_OK) { (*out)->consuming = &ps; return rc; }
            ps.consumers.fetch_sub(1); ps.wake();
            if (rc != GENLIB_ENOMEM) return rc;             // (the bounds did not fit: size by the finished plan)
        } else { ps.consumers.fetch_sub(1); ps.wake(); }
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
        if (!E.consuming) return fail(GENLIB_ERESTART, "the streamed plan's bounds did not hold: create the engine again");
        PlanStream &ps = *E.consuming;
        int rc = E.numerics == GENLIB_NUMERICS_FP64 ? run_streamed<double>(E, ps) : run_streamed<float>(E, ps);
        E.stop_consuming();
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
    CU(cudaMalloc(&dsum, (size_t)nown * 2 * sizeof(double)));
    if (cudaMalloc(&didx, (size_t)nown * sizeof(int32_t)) != cudaSuccess) { cudaFree(dsum); return fail(GENLIB_ENOMEM, "out of device memory"); }
    cudaError_t ce = cudaMemcpyAsync(didx, eng->own_pro.data(), (size_t)nown * sizeof(int32_t), cudaMemcpyHostToDevice, eng->stream);
    if (ce == cudaSuccess) {
        if (eng->numerics == GENLIB_NUMERICS_FP64)
            rowsum_kernel<double><<<(unsigned)nown, kThreads, 0, eng->stream>>>((const double *)eng->A, P.capacity, eng->own_pro_row.p, didx, eng->pro_slot.p, n, dsum);
        else
            rowsum_kernel<float><<<(unsigned)nown, kThreads, 0, eng->stream>>>((const float *)eng->A, P.capacity, eng->own_pro_row.p, didx, eng->pro_slot.p, n, dsum);
        ce = cudaMemcpyAsync(out, dsum, (size_t)nown * 2 * sizeof(double), cudaMemcpyDeviceToHost, eng->stream);
    }
    const cudaError_t e2 = cudaStreamSynchronize(eng->stream);
    cudaFree(dsum); cudaFree(didx);
    if (ce != cudaSuccess || e2 != cudaSuccess) return fail(GENLIB_ECUDA, std::string("row sums: ") + cudaGetErrorString(ce != cudaSuccess ? ce : e2));
    return GENLIB_OK;
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
    cudaFree(dslots); cudaFree(dout);
    return GENLIB_OK;
}

int genlib_phi_multi(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                     const int32_t *proband, void *out, int out_dtype, int numerics, int32_t n_dev,
                     const int32_t *devices, genlib_stats *stats) {
    if (n_dev < 1 || n_dev > kMaxWorld || !devices) return fail(GENLIB_EINVAL, "genlib_phi_multi: 1 .. 16 devices");
    if (out_dtype != GENLIB_F32 && out_dtype != GENLIB_F64) return fail(GENLIB_EINVAL, "unknown out_dtype");
    if (n_dev == 1) return genlib_phi(n, father, mother, n_pro, proband, out, out_dtype, numerics, devices[0], stats);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(GENLIB_ECUDA, "no CUDA device: libgenlib_cuda has no CPU fallback");
    for (int g = 0; g < n_dev; g++) {
        if (devices[g] < 0 || devices[g] >= ndev) return fail(GENLIB_EINVAL, "genlib_phi_multi: no such device");
        for (int h = 0; h < g; h++) if (devices[h] == devices[g]) return fail(GENLIB_EINVAL, "genlib_phi_multi: a device is listed twice");
    }
    // ONE plan for all ranks, made on a worker thread and handed over layer by layer (see genlib_phi)
    std::unique_ptr<genlib_plan> plan_owner(new (std::nothrow) genlib_plan);
    if (!plan_owner) return fail(GENLIB_ENOMEM, "out of host memory");
    genlib_plan *plan = plan_owner.get();
    const bool want_stream = env_int("GENLIB_STREAM", 1) != 0 && out != nullptr;
    const double tp0 = now_ms();
    PlanStream ps;
    int plan_rc = GENLIB_OK;
    std::string plan_err;
    auto make_plan = [&](PlanStream *stream) {
        try {
            adopt_retired_storage(plan->p);
            plan_rc = build_plan(n, father, mother, nullptr, n_pro, proband, n_dev, GENLIB_SCHEDULE_PHI, plan->p, plan_err, stream, /*planners=*/1);
        } catch (const std::bad_alloc &) {
            plan_rc = GENLIB_ENOMEM; plan_err = "out of host memory while planning";
            if (stream) { stream->status.store(plan_rc); stream->stage.store(2); stream->wake(); }
        }
        plan->ms_plan = now_ms() - tp0;
    };
    std::thread worker;
    if (want_stream) { try { worker = std::thread([&] { make_plan(&ps); }); } catch (...) { } }
    const bool streaming = worker.joinable();
    if (!streaming) make_plan(nullptr);
    // (destruction order: consumer registration, engines, worker joined, plan storage retired)
    struct PlanRetire { genlib_plan *p; ~PlanRetire() { try { retire_storage(p->p); } catch (...) {} } } retire{plan};
    struct Joiner { std::thread &t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{worker};   // (joins before the plan is retired)
    std::vector<genlib_engine *> eng((size_t)n_dev, nullptr);
    struct EngGuard { std::vector<genlib_engine *> &e; ~EngGuard() { for (auto *&x : e) { genlib_engine_destroy(x); x = nullptr; } } } eguard{eng};
    int prev_dev = -1;
    cudaGetDevice(&prev_dev);
    struct DevRestore { int d; ~DevRestore() { if (d >= 0) cudaSetDevice(d); } } restore{prev_dev};
    // every device sees every other device's memory (NVLink peer access) -- while the planner's pre-pass runs
    int peer_rc = GENLIB_OK;
    for (int g = 0; g < n_dev && peer_rc == GENLIB_OK; g++) {
        if (cudaSetDevice(devices[g]) != cudaSuccess) { peer_rc = fail(GENLIB_ECUDA, "cudaSetDevice failed"); break; }
        for (int h = 0; h < n_dev; h++) {
            if (h == g) continue;
            int can = 0;
            cudaDeviceCanAccessPeer(&can, devices[g], devices[h]);
            if (!can) { peer_rc = fail(GENLIB_ECOMM, "devices " + std::to_string(devices[g]) + " and " + std::to_string(devices[h]) + " have no peer access"); break; }
            const cudaError_t ce = cudaDeviceEnablePeerAccess(devices[h], 0);
            if (ce != cudaSuccess && ce != cudaErrorPeerAccessAlreadyEnabled) { peer_rc = fail(GENLIB_ECOMM, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(ce)); break; }
            cudaGetLastError();
        }
    }
    // one host thread per device
    std::vector<int> status((size_t)n_dev, GENLIB_OK);
    std::vector<std::string> message((size_t)n_dev);
    auto run_all = [&](auto &&fn) {                              // statuses stay in `status`
        std::vector<std::thread> th;
        for (int g = 0; g < n_dev; g++)
            th.emplace_back([&, g] { status[(size_t)g] = fn(g); if (status[(size_t)g] != GENLIB_OK) message[(size_t)g] = g_err; });
        for (auto &t : th) t.join();
    };
    auto first_error = [&](bool restart_is_error) {              // GENLIB_OK, kRestart (nothing worse happened) or an error
        int rc2 = GENLIB_OK;
        for (int g = 0; g < n_dev; g++) {
            const int st = status[(size_t)g];
            if (st == GENLIB_OK) continue;
            if ((st == kRestart || st == GENLIB_ENOMEM) && !restart_is_error) { if (rc2 == GENLIB_OK) rc2 = kRestart; continue; }
            return fail(st, "device " + std::to_string(devices[g]) + ": " + message[(size_t)g]);
        }
        return rc2;
    };
    auto on_all = [&](auto &&fn) { run_all(fn); return first_error(true); };
    auto wire_peers = [&]() {                                    // plain peer pointers instead of IPC mappings
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
            struct Consumer {                                     // one registration for all device threads
                PlanStream &s;
                explicit Consumer(PlanStream &st) : s(st) { s.consumers.fetch_add(1); }
                ~Consumer() { s.consumers.fetch_sub(1); s.wake(); }
            } consumer(ps);
            if (!ps.overflow.load()) {
                run_all([&](int g) { return create_engine(plan, numerics, devices[g], g, &eng[(size_t)g], true); });
                rc = first_error(false);
                if (rc == GENLIB_OK) {
                    wire_peers();
                    run_all([&](int g) {
                        genlib_engine &E = *eng[(size_t)g];
                        DeviceGuard guard;
                        if (int r = guard.enter(E.device)) return r;
                        int r = numerics == GENLIB_NUMERICS_FP64 ? run_streamed<double>(E, ps) : run_streamed<float>(E, ps);
                        if (r == GENLIB_OK) r = check_device_errors(E);
                        if (r == GENLIB_OK) E.ran = true;
                        return r;
                    });
                    rc = first_error(false);
                    done = rc == GENLIB_OK;
                }
                if (rc == kRestart) rc = GENLIB_OK;
            }
        }
        worker.join();
    }
    if (plan_rc != GENLIB_OK) return fail(plan_rc, plan_err);
    if (peer_rc != GENLIB_OK) return peer_rc;
    if (rc != GENLIB_OK) return rc;
    if (plan->p.n_unique == 0) {
        if (stats) { std::memset(stats, 0, sizeof *stats); stats->ms_plan = plan->ms_plan; }
        return GENLIB_OK;
    }
    if (!out) return fail(GENLIB_EINVAL, "genlib_phi_multi: out is null");
    if (!done) {                                                // plan first, then run (no streaming, or its bounds did not hold)
        for (auto *&x : eng) { genlib_engine_destroy(x); x = nullptr; }
        rc = on_all([&](int g) { return create_engine(plan, numerics, devices[g], g, &eng[(size_t)g]); });
        if (rc != GENLIB_OK) return rc;
        wire_peers();
        rc = on_all([&](int g) { return genlib_engine_run(eng[(size_t)g], 0); });
        if (rc != GENLIB_OK) return rc;
    }
    for (auto *x : eng) x->stats.ms_plan = plan->ms_plan;
    const int32_t nu = plan->p.n_unique;
    const double t0 = now_ms();
    rc = on_all([&](int g) {                                    // contiguous row blocks, one PCIe link each
        genlib_engine &E = *eng[(size_t)g];
        DeviceGuard guard;
        if (int r = guard.enter(E.device)) return r;
        const int32_t u0 = (int32_t)((int64_t)nu * g / n_dev), u1 = (int32_t)((int64_t)nu * (g + 1) / n_dev);
        if (numerics == GENLIB_NUMERICS_FP64)
            return out_dtype == GENLIB_F64 ? fetch_block<double, double>(E, u0, u1, (double *)out) : fetch_block<double, float>(E, u0, u1, (float *)out);
        return out_dtype == GENLIB_F64 ? fetch_block<float, double>(E, u0, u1, (double *)out) : fetch_block<float, float>(E, u0, u1, (float *)out);
    });
    if (rc != GENLIB_OK) return rc;
    if (stats) {
        *stats = eng[0]->stats;
        stats->ms_fetch = now_ms() - t0;
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

int genlib_phi(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
               const int32_t *proband, void *out, int out_dtype, int numerics, int device,
               genlib_stats *stats) {
    if (out_dtype != GENLIB_F32 && out_dtype != GENLIB_F64) return fail(GENLIB_EINVAL, "unknown out_dtype");
    // The plan is made on a worker thread and handed over layer by layer (PlanStream): the device runs the first
    // generations while the later ones are planned.  GENLIB_STREAM=0: plan first, then run.
    std::unique_ptr<genlib_plan> pl(new (std::nothrow) genlib_plan);
    if (!pl) return fail(GENLIB_ENOMEM, "out of host memory");
    const bool want_stream = env_int("GENLIB_STREAM", 1) != 0 && out != nullptr;
    const double t0 = now_ms();
    PlanStream ps;
    int plan_rc = GENLIB_OK;
    std::string plan_err;
    auto make_plan = [&](PlanStream *stream) {
        try {
            adopt_retired_storage(pl->p);        // the arrays of the last destroyed plan, already paged in
            plan_rc = build_plan(n, father, mother, nullptr, n_pro, proband, 1, GENLIB_SCHEDULE_PHI, pl->p, plan_err, stream);
        } catch (const std::bad_alloc &) {
            plan_rc = GENLIB_ENOMEM; plan_err = "out of host memory while planning";
            if (stream) { stream->status.store(plan_rc); stream->stage.store(2); stream->wake(); }
        }
        pl->ms_plan = now_ms() - t0;
    };
    genlib_engine *eng = nullptr;
    struct EngGuard { genlib_engine *&e; ~EngGuard() { genlib_engine_destroy(e); e = nullptr; } } eguard{eng};
    int rc = GENLIB_OK;
    bool done = false;
    if (want_stream) {
        std::thread worker;
        try { worker = std::thread([&] { make_plan(&ps); }); } catch (...) { }
        if (!worker.joinable()) make_plan(nullptr);               // no thread to be had: plan here
        else {
            struct Joiner { std::thread &t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{worker};
            ps.wait([&] { return ps.stage.load() >= 1; });
            if (ps.streamed.load() && pl->p.n_unique > 0) {
                struct Consumer {                                 // the planner waits for us before it reallocates anything
                    PlanStream &s;
                    explicit Consumer(PlanStream &st) : s(st) { s.consumers.fetch_add(1); }
                    ~Consumer() { s.consumers.fetch_sub(1); s.wake(); }
                } consumer(ps);
                if (!ps.overflow.load()) {
                    rc = create_engine(pl.get(), numerics, device, 0, &eng, true);
                    if (rc == GENLIB_OK) {
                        DeviceGuard guard;
                        rc = guard.enter(eng->device);
                        if (rc == GENLIB_OK) rc = numerics == GENLIB_NUMERICS_FP64 ? run_streamed<double>(*eng, ps) : run_streamed<float>(*eng, ps);
                        if (rc == GENLIB_OK) rc = check_device_errors(*eng);
                        if (rc == GENLIB_OK) { eng->ran = true; done = true; }
                    }
                    if (rc == kRestart || rc == GENLIB_ENOMEM) rc = GENLIB_OK;   // the bounds did not hold (or did not fit): run on the finished plan
                }
            }
        }                                                         // (consumer released, worker joined)
    } else make_plan(nullptr);
    if (plan_rc != GENLIB_OK) return fail(plan_rc, plan_err);
    if (rc != GENLIB_OK) return rc;
    if (pl->p.n_unique == 0) {
        if (stats) { std::memset(stats, 0, sizeof *stats); stats->ms_plan = pl->ms_plan; }
        return GENLIB_OK;                       // 0 x 0 matrix, like the reference
    }
    if (!out) return fail(GENLIB_EINVAL, "genlib_phi: out is null");
    if (!done) {
        genlib_engine_destroy(eng); eng = nullptr;
        rc = create_engine(pl.get(), numerics, device, 0, &eng);
        if (rc != GENLIB_OK) return rc;
        rc = genlib_engine_run(eng, 0);
        if (rc != GENLIB_OK) return rc;
    }
    eng->stats.ms_plan = pl->ms_plan;
    rc = genlib_engine_fetch(eng, out, out_dtype);
    if (rc == GENLIB_OK && stats) *stats = eng->stats;
    genlib_engine_destroy(eng); eng = nullptr;                    // before the plan it refers to
    try { retire_storage(pl->p); } catch (...) {}
    return rc;
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

// ------------------------------------------------------------------------------ gen.gc, gen.occ, gen.rec (DESIGN.md 2b, 2c)
struct genlib_gc_plan {
    GcPlan p;
    double ms_plan = 0;
};

namespace {

// What a run of the gc plan computes: gen.gc's matrix, gen.occ's matrix or row sums, gen.rec's counts.
enum GcFn { kFnGc = 0, kFnOcc, kFnOccTotal, kFnRec };
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
    O *stage[2] = {reinterpret_cast<O *>(stage_base), reinterpret_cast<O *>(stage_base + d.stage)};
    cudaEvent_t done[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
    cudaError_t ce = cudaSuccess;
    for (int b = 0; b < 2 && ce == cudaSuccess; b++) {
        ce = cudaEventCreateWithFlags(&done[b], cudaEventDisableTiming);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&copied[b], cudaEventDisableTiming);
    }
    int blk = 0;
    for (int64_t m0 = 0; m0 < L.nmaj && ce == cudaSuccess; m0 += per, blk++) {      // gather of block b+1 overlaps the D2H of block b
        const int b = blk & 1;
        const int64_t nb = std::min(per, L.nmaj - m0);
        if (blk >= 2 && (ce = cudaStreamWaitEvent(st, copied[b], 0)) != cudaSuccess) break;
        GcGatherArgs a;
        a.O = Oblk; a.ws = d.ws(); a.tgt_row = tgt_row; a.col = col;
        a.ovf = ovf; a.j0 = d.j0; a.n_pro = P.n_pro; a.tgt_is_pro = P.direction == kGcDescend;
        if (L.cmaj) { a.t0 = 0; a.n_t = (int32_t)L.nmin; a.c0 = (int32_t)m0; a.n_c = (int32_t)nb; }
        else        { a.t0 = (int32_t)m0; a.n_t = (int32_t)nb; a.c0 = 0; a.n_c = (int32_t)L.nmin; }
        dim3 grid((unsigned)((a.n_c + 31) / 32), (unsigned)std::min<int64_t>((a.n_t + 31) / 32, 65535)), block(32, 8);
        if (L.cmaj) gc_gather_kernel<true, E, O><<<grid, block, 0, st>>>(a, stage[b]);
        else        gc_gather_kernel<false, E, O><<<grid, block, 0, st>>>(a, stage[b]);
        if ((ce = cudaGetLastError()) != cudaSuccess) break;
        cudaEventRecord(done[b], st);
        cudaStreamWaitEvent(cst, done[b], 0);
        ce = cudaMemcpy2DAsync(out + (L.maj_off + m0) * L.ld + L.min_off, (size_t)L.ld * sizeof(O), stage[b],
                               (size_t)L.nmin * sizeof(O), (size_t)L.nmin * sizeof(O), (size_t)nb, cudaMemcpyDeviceToHost, cst);
        cudaEventRecord(copied[b], cst);
    }
    const cudaError_t e1 = cudaStreamSynchronize(st), e2 = cudaStreamSynchronize(cst);
    for (int b = 0; b < 2; b++) { if (done[b]) cudaEventDestroy(done[b]); if (copied[b]) cudaEventDestroy(copied[b]); }
    if (ce != cudaSuccess || e1 != cudaSuccess || e2 != cudaSuccess)
        return fail(GENLIB_ECUDA, std::string("gc fetch failed: ") + cudaGetErrorString(ce != cudaSuccess ? ce : e1 != cudaSuccess ? e1 : e2));
    d.d2h += L.nmaj * L.nmin * (int64_t)sizeof(O);
    return GENLIB_OK;
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
    static const char *const kName[] = {"gen.gc", "gen.occ", "gen.occ", "gen.rec"};
    if (g_arenas.acquire(d.device, d.need, res.arena) != cudaSuccess) {
        res.arena = Arena();
        cudaGetLastError();
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        char msg[256];
        std::snprintf(msg, sizeof msg, "%s needs %.2f GB on device %d, %.2f GB free (%lld frontier rows x %lld columns): "
                      "split the columns over more devices", kName[d.fn], d.need / 1e9, d.device, free_b / 1e9,
                      (long long)P.capacity, (long long)(d.hi - d.lo));
        return fail(GENLIB_ENOMEM, msg);
    }
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
    static const char *const kEntry[] = {"genlib_gc", "genlib_occ", "genlib_occ", "genlib_rec"};
    const std::string who = kEntry[fn];
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
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(GENLIB_ECUDA, "no CUDA device: libgenlib_cuda has no CPU fallback");
    std::vector<GcShare> share((size_t)n_dev);
    const std::vector<int32_t> &cu = P.column_uid();
    const int64_t m = (int64_t)cu.size();
    const size_t esize = fn == kFnGc ? (out_dtype == GENLIB_F64 ? 8 : 4) : 8;
    for (int g = 0; g < n_dev; g++) {
        GcShare &d = share[(size_t)g];
        d.fn = fn;
        d.device = devices[g];
        if (d.device < 0 && cudaGetDevice(&d.device) != cudaSuccess) return fail(GENLIB_ECUDA, "no usable CUDA device (cudaGetDevice failed)");
        if (d.device >= ndev) return fail(GENLIB_EINVAL, who + ": no such device");
        for (int h = 0; h < g; h++) if (share[(size_t)h].device == d.device) return fail(GENLIB_EINVAL, who + ": a device is listed twice");
        d.j0 = (int32_t)(m * g / n_dev); d.j1 = (int32_t)(m * (g + 1) / n_dev);
        if (d.j0 == d.j1) continue;                          // more devices than columns: nothing to do here
        d.lo = *std::min_element(cu.begin() + d.j0, cu.begin() + d.j1);
        d.hi = *std::max_element(cu.begin() + d.j0, cu.begin() + d.j1) + 1;
        d.need = gc_device_bytes(P, d, col_major, esize);
    }
    std::vector<int> status((size_t)n_dev, GENLIB_OK);
    std::vector<std::string> message((size_t)n_dev);
    auto run = [&](int g) {
        GcShare &d = share[(size_t)g];
        if (d.j0 == d.j1) return;
        status[(size_t)g] = gc_run_share(P, d, out, out_dtype, col_major);
        if (status[(size_t)g] != GENLIB_OK) message[(size_t)g] = g_err;
    };
    if (n_dev == 1) run(0);
    else {                                                   // one host thread per device, as genlib_phi_multi
        std::vector<std::thread> th;
        for (int g = 0; g < n_dev; g++) th.emplace_back(run, g);
        for (auto &t : th) t.join();
    }
    for (int g = 0; g < n_dev; g++)
        if (status[(size_t)g] != GENLIB_OK) return fail(status[(size_t)g], "device " + std::to_string(share[(size_t)g].device) + ": " + message[(size_t)g]);
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
