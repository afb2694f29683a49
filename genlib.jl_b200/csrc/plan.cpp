// plan.cpp -- see plan.hpp.  Pure host C++17.
#include "plan.hpp"

#include <algorithm>
#include <climits>
#include <cstdlib>
#include <atomic>
#include <memory>
#include <mutex>
#include <thread>

#include "../../include/genlib_cuda.h"
#include <chrono>
#include <cstdio>

namespace genlib {

namespace {

inline int32_t round_up(int64_t x, int64_t m) { return (int32_t)(((x + m - 1) / m) * m); }

// (father, mother) -> family id of the current layer.  Open addressing with a
// generation stamp so the table is never cleared.
struct FamilyTable {
    struct Bucket { uint64_t key; int32_t val, stamp; };      // 16 bytes: one cache line touch per probe
    std::vector<Bucket> b;
    uint64_t mask = 0;
    int32_t tick = 0;             // stamp of the current layer; never repeats while the table lives
    void next_layer(size_t n) {   // empties the table (by stamp) and makes room for n keys
        size_t cap = 64;
        while (cap < 2 * n + 2) cap <<= 1;
        if (cap > b.size() || tick == INT32_MAX) { b.assign(std::max(cap, b.size()), Bucket{0, 0, -1}); tick = 0; }
        else tick++;
        mask = b.size() - 1;
    }
    static uint64_t mix(uint64_t x) {
        x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33;
        x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33; return x;
    }
    void prefetch(uint64_t k) const { __builtin_prefetch(&b[mix(k) & mask], 1); }
    // returns the bucket of `k` (existing or fresh); *found tells which
    Bucket &find(uint64_t k, bool *found) {
        size_t h = mix(k) & mask;
        while (b[h].stamp == tick && b[h].key != k) h = (h + 1) & mask;
        *found = b[h].stamp == tick;
        if (!*found) { b[h].stamp = tick; b[h].key = k; }
        return b[h];
    }
};

// where an individual's row lives while it is in the frontier; one record so that the planner's
// random accesses (by individual) cost one cache miss each
struct Pre {
    int32_t h = -1, minch = INT_MAX, rl = INT_MAX - 1;
};

struct Home {
    int32_t slot = -1, lrow = -1;
    int8_t owner = 0;
};

// The same for the individuals in the frontier, kept as a list in the order they entered it: the pass over the live
// individuals of every layer (their flags, who leaves) then reads sequentially instead of one home per individual.
struct LiveRec {
    int32_t slot, lrow;
    int32_t last;                // last layer that reads the row (INT_MAX for probands: kept to the end)
    int32_t owner;
};

// Local rows of one rank: any free row will do (a row index only selects a row), so freed rows go on
// a stack -- the sorted free list this replaces cost a third of the planning time at 8 ranks.  Rows
// freed in a layer are still read by that layer, so they become available at its end.
struct Alloc {
    std::vector<int32_t> stack;
    int32_t next_fresh = 0;
    void reset() { stack.clear(); next_fresh = 0; }
    int32_t take() {
        if (stack.empty()) return next_fresh++;
        const int32_t r = stack.back();
        stack.pop_back();
        return r;
    }
    void end_layer(std::vector<int32_t> &freed) {
        stack.insert(stack.end(), freed.rbegin(), freed.rend());
        freed.clear();
    }
};

// Column slots are handed out in whole LINES of kSlotLine consecutive slots (128 bytes of a float
// row): the members of a layer fill free lines in ascending order, so every group of four members
// sits in four consecutive, 16-byte aligned columns (the 128-bit row stores of the layer kernel's consumers) and
// the 4-byte column writes into the carried rows (its producers' mirror pass) fill whole 32-byte sectors.  A line returns to the
// free list only when every individual in it has been evicted (lowest free line first).
struct LineAlloc {
    std::vector<int32_t> freelist, merged;     // free lines, ascending
    std::vector<int32_t> live;                 // per line: individuals still in the frontier
    int32_t next_fresh = 0;                    // first line never used
    size_t cursor = 0;
    int32_t cur = -1, pos = kSlotLine;
    void reset() { freelist.clear(); live.clear(); next_fresh = 0; cursor = 0; cur = -1; pos = kSlotLine; }
    int32_t take() {
        if (pos == kSlotLine) {
            cur = cursor < freelist.size() ? freelist[cursor++] : next_fresh++;
            pos = 0;
            if ((size_t)cur >= live.size()) live.resize((size_t)cur + 1024, 0);
        }
        live[cur]++;
        return cur * kSlotLine + pos++;
    }
    // `slot` was evicted; its line goes to `freed_lines` when it was the last one
    void release(int32_t slot, std::vector<int32_t> &freed_lines) {
        if (--live[slot / kSlotLine] == 0) freed_lines.push_back(slot / kSlotLine);
    }
    void end_layer(std::vector<int32_t> &freed_lines_sorted) {
        pos = kSlotLine;                           // the next layer starts a new line
        freelist.erase(freelist.begin(), freelist.begin() + (ptrdiff_t)cursor);
        cursor = 0;
        if (!freed_lines_sorted.empty()) {
            merged.resize(freelist.size() + freed_lines_sorted.size());
            std::merge(freelist.begin(), freelist.end(), freed_lines_sorted.begin(), freed_lines_sorted.end(), merged.begin());
            freelist.swap(merged);
            freed_lines_sorted.clear();
        }
    }
};

// The planner's temporaries; kept between calls for the same reason as the plan's arrays.
struct Scratch {
    std::vector<uint8_t> is_pro;
    std::vector<Pre> pre;
    std::vector<int32_t> seq_order, orient, cstart, clist, depth;   // sparse_phi schedule
    std::vector<int32_t> hist, count, by_layer, cut_size, both_size;
    std::vector<Home> home;
    std::vector<size_t> lstart, pos;
    std::vector<int64_t> d_cut, d_both;
    std::vector<LiveRec> live, next_live;
    std::vector<int32_t> last_of;
    std::vector<int32_t> dead_slots;                            // kScheduleF: slots / rows (per owner) of the members that no
    std::vector<std::vector<int32_t>> dead_rows;                // later layer reads, freed at the end of their own layer
    std::vector<int32_t> read_last;                             // kSchedulePairs: per individual, its last read layer (-1: none)
    std::vector<int32_t> fam_of, fam_count, fam_first, fam_key, fam_n;   // couples of every layer (grouped ahead by helper threads)
    std::vector<int32_t> order, newid, nf_of, load, freed, evicted[2], cnt, cnt_order, ipos;   // order / newid: by member / couple of every layer
    std::vector<FamilyTable> tables;          // one per planning thread
    std::vector<int8_t> fam_own, owner_of;
    std::vector<std::vector<int32_t>> freed_rows[2];
    LineAlloc slots;
    std::vector<Alloc> rows;
};

std::mutex g_pool_mu;
std::unique_ptr<Scratch> g_scratch;
std::unique_ptr<Plan> g_retired;

std::unique_ptr<Scratch> take_scratch() {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    return g_scratch ? std::move(g_scratch) : std::unique_ptr<Scratch>(new Scratch);
}
void give_scratch(std::unique_ptr<Scratch> s) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (!g_scratch) g_scratch = std::move(s);
}

constexpr int32_t kPf = 24;      // software prefetch distance of the planner's random accesses
constexpr int32_t kKeys = 64;    // couple order keys: layers until the couple's longest-lived member leaves (capped)

// Threads of one planner: min(3, cores / planners sharing the host) once `work` reaches `threshold` (small plans are not
// worth the threads), at most 16.  GENLIB_PLAN_THREADS overrides (also for small plans: the tests run those with helpers).
int plan_threads(int64_t work, int64_t threshold, int planners, int32_t world) {
    const char *env = std::getenv("GENLIB_PLAN_THREADS");
    const int hw = (int)std::thread::hardware_concurrency();
    return std::max(1, std::min(env ? std::atoi(env) : (work >= threshold ? std::min(3, hw / std::max(planners > 0 ? planners : world, 1)) : 1), 16));
}

// GENLIB_PLAN_TIMING (a debugging aid): times on stderr, per phase or summed into sum[] per piece of a lane; off without it.
struct PhaseTimer {
    using clock = std::chrono::steady_clock;
    const bool on = std::getenv("GENLIB_PLAN_TIMING") != nullptr;
    clock::time_point last = clock::now();
    double sum[6] = {0, 0, 0, 0, 0, 0};
    double lap() { const auto t = last; last = clock::now(); return std::chrono::duration<double, std::milli>(last - t).count(); }
    void start() { if (on) last = clock::now(); }
    void add(int k) { if (on) sum[k] += lap(); }
    void phase(const char *name) { if (on) std::fprintf(stderr, "[plan] %-12s %.2f ms\n", name, lap()); }
};

// kSchedulePairs: both slots of every read hold the pair's members when it is read.  Before layer t (t < S) they are
// live there, and the row side is where the live list says; after the last layer (t == S) the slots' last members are
// the pair's own (no one born later took them), and an earlier-born member's row was carried through the last layer
// (only carried rows receive the columns of the last layer's members).
int verify_pair_reads(const Plan &P, const PairList &pairs, std::string &err) {
    const int32_t S = (int32_t)P.layers.size();
    if ((int64_t)P.pair_pos.size() != pairs.n || (int32_t)P.pair_start.size() != S + 2 || P.pair_start[(size_t)S + 1] != pairs.n)
        { err = "verify: the pair reads do not cover the list"; return GENLIB_EINVAL; }
    std::vector<int32_t> last_in((size_t)P.capacity, -1);            // slot -> its last member (mem_ind is the rank)
    std::vector<uint8_t> born_last((size_t)P.capacity, 0);           // slot of a member of the last layer
    for (int32_t t = 0; t < S; t++) {
        const Layer &L = P.layers[(size_t)t];
        for (int32_t q = 0; q < L.n_new; q++) {
            last_in[(size_t)P.mem_slot[L.mem_off + q]] = P.mem_ind[L.mem_off + q];
            if (t == S - 1) born_last[(size_t)P.mem_slot[L.mem_off + q]] = 1;
        }
    }
    for (int32_t t = 0; t <= S; t++)
        for (int64_t i = P.pair_start[(size_t)t]; i < P.pair_start[(size_t)t + 1]; i++) {
            const int64_t p = P.pair_pos[(size_t)i];
            const int32_t x = pairs.a[p], y = pairs.b[p], slots[2] = {P.pair_row_slot[(size_t)i], P.pair_col_slot[(size_t)i]};
            const std::string at = " of list position " + std::to_string(p) + " read in layer " + std::to_string(t);
            if (t < S) {
                const Layer &L = P.layers[(size_t)t];
                for (int32_t s : slots)
                    if (s < L.rt_lo || s >= L.rt_lo + L.rt_rows || !(P.flags[L.flag_off + (size_t)(s - L.rt_lo)] & kFlagLive))
                        { err = "verify: a slot" + at + " is not live"; return GENLIB_EINVAL; }
                const size_t r = L.flag_off + (size_t)(slots[0] - L.rt_lo);
                if (P.live_owner[r] != P.pair_owner[(size_t)i] || P.live_lrow[r] != P.pair_lrow[(size_t)i])
                    { err = "verify: the row" + at + " is not where the live list has it"; return GENLIB_EINVAL; }
            } else {
                if (last_in[(size_t)slots[0]] != std::max(x, y) || last_in[(size_t)slots[1]] != std::min(x, y))
                    { err = "verify: a slot" + at + " was handed to someone born later"; return GENLIB_EINVAL; }
                const Layer &L = P.layers[(size_t)S - 1];
                for (int32_t s : slots) {
                    const bool carried = s >= L.rt_lo && s < L.rt_lo + L.rt_rows && (P.flags[L.flag_off + (size_t)(s - L.rt_lo)] & kFlagCarried);
                    if (!born_last[(size_t)s] && !carried) { err = "verify: a row" + at + " was not carried through the last layer"; return GENLIB_EINVAL; }
                }
            }
        }
    return GENLIB_OK;
}

// GENLIB_PLAN_VERIFY (a debugging aid): the index ranges the layer kernel relies on.
int verify_plan(const Plan &P, std::string &err) {
    for (int32_t t = 0; t < (int32_t)P.layers.size(); t++) {
        const Layer &L = P.layers[t];
        const int64_t qrows = (int64_t)L.n_live_tiles * kPTile;
        for (int32_t f = 0; f < L.n_fam; f++)
            for (int s2 = 0; s2 < 2; s2++) {
                const int32_t q0 = P.fam_q[2 * (L.fam_off + (size_t)f) + s2], q = q0 >= 0 ? (q0 & ~kSoleReader) : q0;
                const int32_t slot = s2 ? P.fam_pm[L.fam_off + f] : P.fam_pf[L.fam_off + f];
                if (q < -1 || q >= qrows || (q < 0) != (slot < 0)) { err = "verify: fam_q out of range in layer " + std::to_string(t) + " couple " + std::to_string(f) + " q " + std::to_string(q) + " qrows " + std::to_string(qrows) + " slot " + std::to_string(slot) + " rt_lo " + std::to_string(L.rt_lo); return GENLIB_EINVAL; }
                // a parent's row is live in its child's layer (for kScheduleF: the engine reads Psi[father, mother] there)
                if (slot >= 0 && (slot < L.rt_lo || slot >= L.rt_lo + L.rt_rows || !(P.flags[L.flag_off + (size_t)(slot - L.rt_lo)] & kFlagLive)))
                    { err = "verify: a parent of couple " + std::to_string(f) + " is not live in layer " + std::to_string(t); return GENLIB_EINVAL; }
            }
        for (int32_t j = 0; j < L.n_mtiles; j++) {
            const int32_t *d = &P.mtile_desc[4 * (L.mtile_off + (size_t)j)];
            if (d[0] < 0 || d[1] < 1 || d[1] > kMaxTileFam || d[0] + d[1] > L.n_fam || d[2] < 0 || d[3] < 1 || d[3] > kMTile || d[2] + d[3] > L.n_new || (d[2] & 7))
                { err = "verify: tile descriptor in layer " + std::to_string(t) + " tile " + std::to_string(j) + ": " + std::to_string(d[0]) + " " + std::to_string(d[1]) + " " + std::to_string(d[2]) + " " + std::to_string(d[3]); return GENLIB_EINVAL; }
        }
        // kSoleReader: the consumer item that stages such a strip-buffer row drops it from L2 afterwards, so it
        // must be the ONLY item that stages it -- count the (member tile, couple, parent) triples per row
        std::vector<int32_t> staged((size_t)std::max<int64_t>(qrows, 1), 0);
        std::vector<uint8_t> marked((size_t)std::max<int64_t>(qrows, 1), 0);
        for (int32_t j = 0; j < L.n_mtiles; j++) {
            const int32_t *d = &P.mtile_desc[4 * (L.mtile_off + (size_t)j)];
            for (int32_t f = d[0]; f < d[0] + d[1]; f++)
                for (int s2 = 0; s2 < 2; s2++) {
                    const int32_t q0 = P.fam_q[2 * (L.fam_off + (size_t)f) + s2];
                    if (q0 < 0) continue;
                    staged[(size_t)(q0 & ~kSoleReader)]++;
                    if (q0 & kSoleReader) marked[(size_t)(q0 & ~kSoleReader)] = 1;
                }
        }
        for (int64_t q = 0; q < qrows; q++)
            if (marked[(size_t)q] && staged[(size_t)q] != 1) { err = "verify: strip-buffer row " + std::to_string(q) + " of layer " + std::to_string(t) + " is marked sole-reader but staged " + std::to_string(staged[(size_t)q]) + " times"; return GENLIB_EINVAL; }
        // every couple with members must be covered by the tiles (its rows are computed by somebody)
        for (int32_t j = 0, next = 0; j < L.n_mtiles; j++) {
            const int32_t *d = &P.mtile_desc[4 * (L.mtile_off + (size_t)j)];
            if (d[2] != next) { err = "verify: member tiles of layer " + std::to_string(t) + " do not tile the members"; return GENLIB_EINVAL; }
            next = d[2] + d[3];
            if (j == L.n_mtiles - 1 && next != L.n_new) { err = "verify: member tiles of layer " + std::to_string(t) + " end early"; return GENLIB_EINVAL; }
        }
    }
    return GENLIB_OK;
}

// One plan in the making: the inputs, the scratch and what one phase hands to the next.  The hot loops of the
// pre-pass read the inputs through locals (members could alias the stores of the loop and be reloaded every time).
struct Planner {
    Scratch &W; Plan &P; std::string &err; PlanStream *ps;
    const int32_t n, *father, *mother; const int64_t *ids; const int32_t n_pro, *proband, world; const int schedule, planners;
    const PairList &pairs;                                      // kSchedulePairs
    const bool by_seq = sparse_schedule(schedule);              // members of a layer in processing order
    const bool reads = schedule == kSchedulePairs;              // rows read by pairs (pair_* arrays)
    const bool by_depth = by_seq || schedule == kScheduleF || reads;     // layers by depth below the founders
    const bool short_rows = schedule == kScheduleF || reads;    // rows that no later layer reads (childless members)
    PhaseTimer clock{};
    std::vector<uint8_t> &is_pro = W.is_pro;
    std::vector<Pre> &pre = W.pre;
    std::vector<Home> &home = W.home;
    std::vector<size_t> &lstart = W.lstart;
    std::vector<int32_t> &hist = W.hist, &count = W.count, &by_layer = W.by_layer, &last_of = W.last_of, &seq_order = W.seq_order,
                         &orient = W.orient, &cut_size = W.cut_size, &both_size = W.both_size, &load = W.load, &freed = W.freed;
    std::vector<int64_t> d_occ{};                               // individuals in the frontier per step (streamed plans: bounds)
    std::vector<LiveRec> &live = W.live, &next_live = W.next_live;   // individuals live before the current step (lane B's)
    LineAlloc &slots = W.slots; std::vector<Alloc> &rows = W.rows;   // allocators: column slots, local rows per rank
    std::vector<int8_t> &owner_of = W.owner_of;
    int32_t hmax = 0, S = 0, rr = 0;
    int kC = 1, chunk = 0;                                      // threads of the bucket pass; its range c = [c * chunk, (c + 1) * chunk)
    bool streaming = false;
    int64_t bound_slots = 0, bound_rows = 0;
    int32_t live_lo = INT_MAX, live_hi = -1;                    // lowest / highest slot on the live list (lane B's)

    int run() {
        P.reset();
        if (schedule != kSchedulePhi && !sparse_schedule(schedule) && schedule != kScheduleF && !reads) { err = "unknown schedule"; return GENLIB_EINVAL; }
        P.schedule = schedule;
        if (n < 0 || n_pro < 0 || world < 1 || (n > 0 && (!father || !mother)) || (n_pro > 0 && !proband) ||
            pairs.n < 0 || (pairs.n > 0 && (!pairs.a || !pairs.b)))
            { err = "genlib_plan_create: null pointer or negative size"; return GENLIB_EINVAL; }
        if (reads ? n_pro > 0 : pairs.n > 0)
            { err = "genlib_plan_create: a GENLIB_SCHEDULE_PAIRS plan takes pairs and no probands, the other schedules no pairs"; return GENLIB_EINVAL; }
        P.n = n; P.world = world;
        if (int rc = probands()) return rc;
        if (P.n_unique == 0) return check_pedigree(n, father, mother, err);     // nothing to plan
        clock.phase("probands");
        if (int rc = sweep()) return rc;
        if (int rc = by_seq ? queue_order() : GENLIB_OK) return rc;
        if (by_depth && !by_seq) depth_layers();
        if (reads) read_layers();
        clock.phase("heights");
        buckets();
        clock.phase("buckets");
        if (world > 127) { err = "at most 127 ranks"; return GENLIB_EINVAL; }
        bounds();
        run_layers();
        clock.phase("layers");
        return finish();
    }

    // probands: first occurrence wins (intersect/union keep first-argument order, compute.jl:247,251); kScheduleF
    // leaves out the listed individuals with a missing parent (their F is 0 without a plan)
    // (kSchedulePairs: everybody named in a pair, in list order, a before b)
    int probands() {
        is_pro.assign((size_t)n + 1, 0);
        auto add = [&](int32_t x) {
            if (x < 0 || x >= n) {
                if (int rc = check_pedigree(n, father, mother, err)) return rc;   // (a broken pedigree is reported first)
                err = "KeyError: proband index " + std::to_string(x) + " not in pedigree";
                return (int)GENLIB_EKEY;
            }
            if (schedule == kScheduleF && (father[x] < 0 || mother[x] < 0)) return (int)GENLIB_OK;
            if (!is_pro[x]) { is_pro[x] = 1; P.pro_ind.push_back(x); }
            return (int)GENLIB_OK;
        };
        for (int32_t t = 0; t < n_pro; t++)
            if (int rc = add(proband[t])) return rc;
        for (int64_t k = 0; k < pairs.n; k++) {
            if (int rc = add(pairs.a[k])) return rc;
            if (int rc = add(pairs.b[k])) return rc;
        }
        P.n_unique = (int32_t)P.pro_ind.size();
        return GENLIB_OK;
    }

    // One reverse sweep (children have larger ranks, so an individual is final when it is visited; check_pedigree says
    // what is wrong when a parent does not precede its child):
    //   h     height above the probands = longest downward path to one (compute.jl:236-241 builds
    //         the same levels by repeated _previous_generation); layer = first raw level = S-1-h
    //   minch lowest height among the children: the last child is born in layer S-1-minch, after
    //         which the engine evicts the row
    //   rl    S-1 - (last raw level): the reference keeps the individual in its cuts until then
    int sweep() {
        const int32_t n = this->n, *father = this->father, *mother = this->mother;
        std::vector<Pre> &pre = this->pre; pre.assign((size_t)n, Pre());
        for (int32_t x : P.pro_ind) { pre[x].h = 0; pre[x].rl = 0; }
        int32_t hmax = 0;
        bool bad_pedigree = false;
        // Threads of the bucket pass (buckets()): it works on equal ranges of ranks, and this sweep counts the heights
        // per range for it (hist[h * kC + c]).
        const int kC = this->kC = by_depth ? 1 : plan_threads(n, 400000, planners, world);
        const int32_t chunk = this->chunk = n / kC + 1;
        std::vector<int32_t> &hist = this->hist; hist.clear();
        int32_t c_of_x = kC - 1, c_lo = (kC - 1) * chunk;
        for (int32_t x = n - 1; x >= 0; x--) {
            while (x < c_lo) { c_of_x--; c_lo -= chunk; }
            if (x >= kPf) {
                const int32_t y = x - kPf, fy = father[y], my = mother[y];
                if ((uint32_t)fy < (uint32_t)n) __builtin_prefetch(&pre[fy], 1);      // (not validated yet)
                if ((uint32_t)my < (uint32_t)n) __builtin_prefetch(&pre[my], 1);
            }
            // parents are -1 or precede the child (create.jl:234-254 orders them so): one unsigned compare each
            const int32_t fx = father[x], mx = mother[x];
            if ((uint32_t)fx + 1u > (uint32_t)x || (uint32_t)mx + 1u > (uint32_t)x) { bad_pedigree = true; continue; }
            const Pre px = pre[x];
            if (px.h < 0) continue;
            if ((size_t)px.h * kC >= hist.size()) hist.resize(((size_t)px.h + 64) * kC, 0);
            hist[(size_t)px.h * kC + c_of_x]++;
            hmax = std::max(hmax, px.h);
            const int32_t par[2] = {fx, mx};
            for (int32_t p : par) {
                if (p < 0) continue;
                Pre &pp = pre[p];                                      // (unconditional stores: the compares do not predict)
                pp.h = std::max(pp.h, px.h + 1);
                pp.minch = std::min(pp.minch, px.h);
                pp.rl = std::min(pp.rl, px.rl + 1);
            }
        }
        this->hmax = hmax;
        return bad_pedigree ? check_pedigree(n, father, mother, err) : GENLIB_OK;
    }

    // Layers by depth below the founders (sparse_phi's schedule and kScheduleF): the sweep marked the ancestors of
    // the probands; re-label them so that layer = S-1-h = depth, and the last child is the deepest one.
    void depth_layers() {
        const int32_t n = this->n, *father = this->father, *mother = this->mother;
        std::vector<int32_t> &depth = W.depth;
        depth.assign((size_t)n, 0);
        int32_t dmax = 0;
        for (int32_t x = 0; x < n; x++) {                       // parents precede children
            if (pre[x].h < 0) continue;
            const int32_t f = father[x], m = mother[x];
            int32_t d = 0;
            if (f >= 0) d = std::max(d, depth[f] + 1);
            if (m >= 0) d = std::max(d, depth[m] + 1);
            depth[x] = d; dmax = std::max(dmax, d);
        }
        std::fill(hist.begin(), hist.end(), 0);
        hist.resize((size_t)dmax + 1, 0);
        hmax = dmax;
        for (int32_t x = 0; x < n; x++) {
            if (pre[x].h < 0) continue;
            pre[x].h = dmax - depth[x];                          // layer = S-1-h = depth
            pre[x].minch = INT_MAX;
            pre[x].rl = pre[x].h;                                // the reference's cut counts do not apply
            hist[(size_t)pre[x].h]++;
        }
        for (int32_t x = 0; x < n; x++) {                       // last child: the deepest one
            if (pre[x].h < 0) continue;
            const int32_t par[2] = {father[x], mother[x]};
            for (int32_t p : par) if (p >= 0 && pre[p].minch > pre[x].h) pre[p].minch = pre[x].h;
        }
    }

    // kSchedulePairs: the read layer of every pair, r = max(depth a, depth b) + 1 in [1, S] -- just before layer r
    // both rows hold the pair's kinship (the later-born member's row got the other one's column, the other row the
    // mirror of it) and nobody has written over it.  The reads are bucketed by r with a counting sort, list order
    // kept, and each named individual learns its last read layer.  A pair read after the last layer (r == S) keeps
    // its rows through that layer as CARRIED rows: only carried rows receive the columns of a layer's members.
    void read_layers() {
        const int32_t S = hmax + 1, *a = pairs.a, *b = pairs.b;
        const int64_t K = pairs.n;
        const std::vector<int32_t> &depth = W.depth;
        std::vector<int32_t> &read_last = W.read_last;
        read_last.assign((size_t)n, -1);
        std::vector<int64_t> &start = P.pair_start;
        start.assign((size_t)S + 2, 0);
        for (int64_t k = 0; k < K; k++) {
            const int32_t r = std::max(depth[a[k]], depth[b[k]]) + 1;
            start[(size_t)r + 1]++;
            read_last[a[k]] = std::max(read_last[a[k]], r);
            read_last[b[k]] = std::max(read_last[b[k]], r);
        }
        for (int32_t t = 0; t <= S; t++) start[(size_t)t + 1] += start[(size_t)t];
        P.pair_pos.resize((size_t)K);
        std::vector<int64_t> at(start.begin(), start.end() - 1);
        for (int64_t k = 0; k < K; k++) P.pair_pos[(size_t)at[(size_t)std::max(depth[a[k]], depth[b[k]]) + 1]++] = k;
        // (exactly K entries each, sized before the first layer is published: a streamed plan never outgrows them)
        P.pair_row_slot.resize((size_t)K); P.pair_col_slot.resize((size_t)K);
        P.pair_owner.resize((size_t)K); P.pair_lrow.resize((size_t)K);
    }

    // kSchedulePairs, lane A: where the reads of layer t (t == S: after the last layer) find their two slots -- every
    // member was born before t, and a home does not move while its row is live
    void pair_reads(int32_t t) {
        for (int64_t i = P.pair_start[(size_t)t]; i < P.pair_start[(size_t)t + 1]; i++) {
            const int64_t k = P.pair_pos[(size_t)i];
            const int32_t hi = std::max(pairs.a[k], pairs.b[k]), lo = std::min(pairs.a[k], pairs.b[k]);
            const Home hr = home[hi];
            P.pair_row_slot[(size_t)i] = hr.slot; P.pair_col_slot[(size_t)i] = home[lo].slot;
            P.pair_owner[(size_t)i] = hr.owner; P.pair_lrow[(size_t)i] = hr.lrow;
        }
    }

    // Schedule of sparse_phi (compute.jl:335-439): individuals are processed in the order of a queue
    // that starts with the founders and receives a child when its last parent has been processed --
    // i.e. by depth below the founders, ties in queue order -- and of a pair, the one processed LATER
    // is climbed.  The layer is then the depth, `seq` (the position in that queue) replaces the rank
    // wherever the kernels decide who is climbed, and eviction is sparse_phi's own rule (:400-430).
    int queue_order() {
        const int32_t n = this->n, *father = this->father, *mother = this->mother;
        std::vector<int32_t> &cstart = W.cstart, &clist = W.clist, &depth = W.depth;
        depth_layers();
        seq_order.clear();
        cstart.assign((size_t)n + 2, 0);
        for (int32_t x = 0; x < n; x++) {
            if (pre[x].h < 0) continue;
            const int32_t f = father[x], m = mother[x];
            if (f >= 0) cstart[(size_t)f + 2]++;
            if (m >= 0 && m != f) cstart[(size_t)m + 2]++;
        }
        for (int32_t x = 0; x < n; x++) cstart[(size_t)x + 2] += cstart[(size_t)x + 1];
        clist.resize((size_t)cstart[(size_t)n + 1]);
        for (int32_t x = 0; x < n; x++) {                       // children lists in rank order (_index_pedigree, :176-183)
            if (pre[x].h < 0) continue;
            const int32_t f = father[x], m = mother[x];
            if (f >= 0) clist[(size_t)cstart[(size_t)f + 1]++] = x;
            if (m >= 0 && m != f) clist[(size_t)cstart[(size_t)m + 1]++] = x;
        }                                                       // now children of p = clist[cstart[p] .. cstart[p+1])
        orient.assign((size_t)n, -1);
        seq_order.reserve((size_t)n);
        for (int32_t x = 0; x < n; x++)                         // founder(isolated_pedigree) (:335-339) ...
            if (pre[x].h >= 0 && father[x] < 0 && mother[x] < 0) seq_order.push_back(x);
        if (ids)                                                // ... is sorted by ID (identify.jl:15-19)
            std::sort(seq_order.begin(), seq_order.end(), [ids = ids](int32_t a, int32_t b) {
                return ids[a] != ids[b] ? ids[a] < ids[b] : a < b;
            });
        for (size_t head = 0; head < seq_order.size(); head++) {
            const int32_t i = seq_order[head];
            orient[i] = (int32_t)head;                          // processed: founder_index != 0 from here on
            for (int32_t k = cstart[i]; k < cstart[(size_t)i + 1]; k++) {
                const int32_t c = clist[(size_t)k], f = father[c], m = mother[c];
                if (f >= 0 && m >= 0 && f != m) { if (orient[f] >= 0 && orient[m] >= 0) seq_order.push_back(c); }
                else seq_order.push_back(c);
            }
        }
        int32_t last_depth = 0;
        for (int32_t i : seq_order) {                           // the queue order is sorted by depth (asserted, not assumed)
            if (depth[i] < last_depth) { err = "sparse_phi schedule: queue order is not sorted by depth"; return GENLIB_EINVAL; }
            last_depth = depth[i];
        }
        return GENLIB_OK;
    }

    // members of each layer in rank order, where each row is read for the last time, and the
    // reference's cut sizes (verbose lines, compute.jl:254-261)
    void buckets() {
        S = hmax + 1;
        hist.resize((size_t)S * kC, 0);                               // (by_seq: kC == 1)
        count.assign((size_t)S + 1, 0);
        for (int32_t k = 0; k < S; k++) for (int c = 0; c < kC; c++) count[S - 1 - k] += hist[(size_t)k * kC + c];
        lstart.assign((size_t)S + 1, 0);
        for (int32_t t = 0; t < S; t++) lstart[t + 1] = lstart[t] + count[t];
        by_layer.resize(lstart[S]);
        std::vector<int64_t> &d_cut = W.d_cut, &d_both = W.d_both;
        d_cut.assign((size_t)S + 2, 0); d_both.assign((size_t)S + 2, 0);
        d_occ.assign((size_t)S + 2, 0);
        home.resize((size_t)n);                                       // filled when a slot is assigned; entries outside the plan are never read
        last_of.resize((size_t)n);                                    // last layer that reads the row (a sequential write here)
        // One range of visits: its members go to their layers from `pos` on, its share of the difference arrays to d[0..2].
        auto bucket_range = [&](int32_t v0, int32_t v1, size_t *pos, int64_t *occ, int64_t *cut, int64_t *both) {
            const int32_t S = this->S; const bool by_seq = this->by_seq, short_rows = this->short_rows, reads = this->reads;   // (copies: not reloaded after every store below)
            for (int32_t v = v0; v < v1; v++) {
                const int32_t x = by_seq ? seq_order[(size_t)v] : v;
                const Pre px = pre[x];
                if (px.h < 0) continue;
                const int32_t lx = S - 1 - px.h, ref_last = S - 1 - px.rl;
                by_layer[pos[lx]++] = x;
                // probands stay to the end (kScheduleF, kSchedulePairs: nobody does); a row without children leaves after
                // its own layer; kSchedulePairs: not before its last read (S: carried through the last layer)
                int32_t last = is_pro[x] && !short_rows ? INT_MAX : px.minch == INT_MAX ? lx : S - 1 - px.minch;
                if (reads) last = std::max(last, W.read_last[x]);
                last_of[x] = last;
                occ[(size_t)std::min<int64_t>(std::max(last, lx), S - 1) + 1]--;   // born in or before, read in or after
                cut[ref_last + 1]--;                                   // in cut[k] for layer <= k <= ref_last
                if (ref_last > lx) { both[lx]++; both[ref_last]--; }   // in cut[k] and cut[k+1]
            }
        };
        std::vector<size_t> &pos = W.pos;
        if (kC > 1 && (std::getenv("GENLIB_PLAN_THREADS") || lstart[S] >= 200000)) {
            // ranges of ranks side by side: range c starts, in layer t, after the members that the ranges below it
            // hold there (counted by the sweep); the difference arrays are summed afterwards
            const size_t D = (size_t)S + 2;
            pos.assign((size_t)kC * S, 0);
            for (int32_t t = 0; t < S; t++) {
                size_t at = lstart[t];
                for (int c = 0; c < kC; c++) { pos[(size_t)c * S + t] = at; at += (size_t)hist[(size_t)(S - 1 - t) * kC + c]; }
            }
            std::vector<int64_t> dd((size_t)kC * 3 * D, 0);
            auto range = [&](int c) {
                bucket_range(std::min(n, c * chunk), std::min(n, (c + 1) * chunk), pos.data() + (size_t)c * S,
                             dd.data() + ((size_t)c * 3) * D, dd.data() + ((size_t)c * 3 + 1) * D, dd.data() + ((size_t)c * 3 + 2) * D);
            };
            std::vector<std::thread> th;
            int started = 1;
            try {
                for (int c = 1; c < kC; c++, started++) th.emplace_back(range, c);
            } catch (...) {}                                           // no thread: the ranges left are done here
            range(0);
            for (int c = started; c < kC; c++) range(c);
            for (auto &t : th) t.join();
            for (int c = 0; c < kC; c++)
                for (size_t k = 0; k < D; k++) {
                    d_occ[k] += dd[((size_t)c * 3) * D + k]; d_cut[k] += dd[((size_t)c * 3 + 1) * D + k]; d_both[k] += dd[((size_t)c * 3 + 2) * D + k];
                }
        } else {
            pos.assign(lstart.begin(), lstart.end() - 1);
            bucket_range(0, by_seq ? (int32_t)seq_order.size() : n, pos.data(), d_occ.data(), d_cut.data(), d_both.data());
        }
        for (int32_t t = 0; t < S; t++) { d_occ[t] += count[t]; d_cut[t] += count[t]; }   // everybody enters with its layer
        cut_size.assign((size_t)S, 0); both_size.assign((size_t)S, 0);
        int64_t a = 0, b = 0;
        for (int32_t k = 0; k < S; k++) { a += d_cut[k]; b += d_both[k]; cut_size[k] = (int32_t)a; both_size[k] = (int32_t)b; }
    }

    // upper bounds of the plan's arrays (untouched reserve costs nothing): members + alignment padding, couples + rank
    // padding; a streamed plan: upper bounds for what the engine sizes before the first layer exists
    void bounds() {
        P.layers.resize(S);
        const size_t mcap = lstart[S] + 4 * (size_t)S, fcap = lstart[S] + 4 * (size_t)world * (size_t)S;
        for (auto *v : {&P.mem_ind, &P.mem_slot, &P.mem_fam, &P.mem_lrow}) v->reserve(mcap);
        if (by_seq) P.mem_rank.reserve(mcap);
        for (auto *v : {&P.fam_pf, &P.fam_pm, &P.fam_pf_lrow, &P.fam_pm_lrow}) v->reserve(fcap);
        P.fam_q.reserve(2 * fcap);
        P.fam_pf_owner.reserve(fcap); P.fam_pm_owner.reserve(fcap); P.fam_start.reserve(fcap + (size_t)S);
        streaming = ps != nullptr;
        if (streaming) {
            // most individuals in the frontier during one step (counted in the bucket pass)
            int64_t occ = 0, occ_max = 0;
            for (int32_t k = 0; k < S; k++) { occ += d_occ[k]; occ_max = std::max(occ_max, occ); }
            // slack: lines of kSlotLine slots shared by individuals that leave in different layers (the member order
            // keeps those to a few per cohort and rank), and a layer always starts on a fresh line
            const char *env = std::getenv("GENLIB_STREAM_SLACK_PCT");
            const double pct = env ? std::atof(env) : 6.25;
            const int64_t cohorts = std::min<int64_t>(S, 128);
            bound_slots = round_up((int64_t)((double)occ_max * (1.0 + pct / 100.0)) + (pct >= 0 ? 2 * kSlotLine * cohorts * world + 2048 : 0), kPTile);
            bound_slots = std::max<int64_t>(bound_slots, kPTile);
            bound_rows = world == 1 ? bound_slots
                                    : (int64_t)((double)occ_max / world * (1.125 + pct / 100.0)) + (pct >= 0 ? (kMaxFamily + kSlotLine) * cohorts + 1024 : 1);
            if (bound_slots >= ((int64_t)1 << 24) || bound_slots * (int64_t)S > ((int64_t)1 << 31)) streaming = false;   // not worth the arrays
        }
        if (streaming) {
            P.capacity = bound_slots;
            P.rows_cap.assign((size_t)world, bound_rows);
            const size_t fl = (size_t)bound_slots * (size_t)S, tl = fl / kPTile, M8 = lstart[S] / 8 + 2 * (size_t)S;
            P.flags.reserve(fl); P.live_owner.reserve(fl); P.live_lrow.reserve(fl);
            P.tile_map.reserve(tl); P.live_tiles.reserve(tl);
            P.mtile_desc.reserve(4 * M8);
            P.fam_base.reserve((size_t)(world + 1) * (size_t)S); P.mem_base.reserve((size_t)(world + 1) * (size_t)S);
            ps->streamed.store(true);
            ps->stage.store(1);
            ps->wake();
        }
    }

    // A bound does not hold: tell the consumers, wait until none of them reads the arrays any more (they may be
    // reallocated from here on), go on as an ordinary plan.
    void give_up_streaming() {
        streaming = false;
        ps->overflow.store(true);                   // (sequentially consistent, like the consumers' registration)
        ps->wake();
        ps->wait([&] { return ps->consumers.load() == 0; });
    }

    // ---- couples: same (father, mother) => same cross row (compute.jl:111-126 gives full siblings
    //      identical kinship to everybody else), split at kMaxFamily members; and the layer in which the
    //      couple's longest-lived member leaves the frontier.  A layer's couples depend on nothing but
    //      the pre-pass, so helper threads group the layers ahead of the sequential slot assignment. ----
    void group_layer(int32_t t, FamilyTable &table) {
        const int32_t *X = by_layer.data() + lstart[t];
        const int32_t nn = count[t];
        int32_t *fam_of = W.fam_of.data() + lstart[t], *fam_count = W.fam_count.data() + lstart[t];
        int32_t *fam_first = W.fam_first.data() + lstart[t], *fam_key = W.fam_key.data() + lstart[t];
        table.next_layer((size_t)nn);
        // kScheduleF: the siblings that nobody reads after this layer form couples of their own, so that their lines
        // of slots come back whole at its end (mixed with the carried siblings they would leave holes in the frontier)
        const bool split_dead = short_rows;
        auto couple_key = [&](int32_t x) {
            const uint64_t dead = split_dead && last_of[x] == t ? 1ULL << 63 : 0;     // (father + 1 < 2^31)
            return dead | ((uint64_t)(uint32_t)(father[x] + 1) << 32) | (uint32_t)(mother[x] + 1);
        };
        constexpr int32_t kAhead = 16;
        int32_t nfr = 0;
        for (int32_t q = 0; q < std::min(nn, kAhead); q++) table.prefetch(couple_key(X[q]));
        for (int32_t q = 0; q < nn; q++) {
            if (q + kAhead < nn) table.prefetch(couple_key(X[q + kAhead]));
            bool found;
            FamilyTable::Bucket &bk = table.find(couple_key(X[q]), &found);
            const int32_t key = std::min(last_of[X[q]] - t, kKeys - 1);   // >= 1: somebody is born later, or proband; 0: nobody (kScheduleF)
            if (found && fam_count[bk.val] < kMaxFamily) {
                fam_of[q] = bk.val;
                fam_key[bk.val] = std::max(fam_key[bk.val], key);
            } else {
                fam_of[q] = nfr;
                bk.val = nfr;
                fam_count[nfr] = 0;
                fam_first[nfr] = q;
                fam_key[nfr] = key;
                nfr++;
            }
            fam_count[fam_of[q]]++;
        }
        W.fam_n[t] = nfr;
    }

    void begin_layer(int32_t t) {
        Layer &L = P.layers[t];
        L.n_new = count[t];
        L.ref_founders = t > 0 ? cut_size[t - 1] : 0;
        L.ref_probands = cut_size[t];
        L.ref_both = t > 0 ? both_size[t - 1] : 0;
        // member arrays of a layer start 16-byte aligned (the layer kernel copies them in 16-byte chunks)
        while (P.mem_ind.size() % 4) {
            P.mem_ind.push_back(0); P.mem_slot.push_back(0); P.mem_fam.push_back(0); P.mem_lrow.push_back(0);
            if (by_seq) P.mem_rank.push_back(0);
        }
        L.mem_off = P.mem_ind.size();              // (the offsets into lane B's arrays are set there)
        L.mtile_off = P.mtile_desc.size() / 4;
    }

    // lane B, first piece: the members of the previous layer join the live list (in rank order, after those carried);
    // live range and flags (state BEFORE the step); who stays
    void live_flags(int32_t t) {
        Layer &L = P.layers[t];
        if (t > 0) {
            const int32_t *Xp = by_layer.data() + lstart[t - 1];
            const int32_t np = count[t - 1];
            for (int32_t q = 0; q < np; q++) {             // (ranks ascend: nearly sequential reads)
                const int32_t x = Xp[q];
                if (short_rows && last_of[x] < t) continue;    // nobody reads the row after its own layer
                const Home hx = home[x];
                live.push_back(LiveRec{hx.slot, hx.lrow, last_of[x], hx.owner});
                live_lo = std::min(live_lo, hx.slot); live_hi = std::max(live_hi, hx.slot);
            }
        }
        L.live_before = (int32_t)live.size();
        L.flag_off = P.flags.size();
        L.tile_off = P.tile_map.size();
        L.ltile_off = P.live_tiles.size();
        std::vector<int32_t> &evicted = W.evicted[t & 1];
        std::vector<std::vector<int32_t>> &freed_rows = W.freed_rows[t & 1];
        evicted.clear();
        next_live.clear();
        L.flag_end = L.flag_off; L.tile_end = L.tile_off; L.ltile_end = L.ltile_off;
        if (live.empty()) return;
        // (lowest and highest live slot: kept up to date by the pass below for those who stay, above for those who join)
        L.rt_lo = (live_lo / kPTile) * kPTile;
        L.rt_rows = round_up(live_hi + 1, kPTile) - L.rt_lo;
        P.flags.resize(L.flag_off + (size_t)L.rt_rows, 0);
        P.live_owner.resize(L.flag_off + (size_t)L.rt_rows, 0);
        P.live_lrow.resize(L.flag_off + (size_t)L.rt_rows, 0);
        uint8_t *fl = P.flags.data() + L.flag_off;
        int8_t *lown = P.live_owner.data() + L.flag_off;
        int32_t *llrow = P.live_lrow.data() + L.flag_off;
        const int32_t rt_lo = L.rt_lo, rt_rows = L.rt_rows;
        int32_t carried = 0, lo = INT_MAX, hi = -1;
        for (const LiveRec &rec : live) {
            const bool stays = rec.last > t;      // read for the last time in step `last`
            const int32_t r = rec.slot - rt_lo;
            fl[r] = (uint8_t)(kFlagLive | (stays ? kFlagCarried : 0));
            lown[r] = (int8_t)rec.owner;
            llrow[r] = rec.lrow;
            if (stays) { next_live.push_back(rec); carried++; lo = std::min(lo, rec.slot); hi = std::max(hi, rec.slot); }
            else if (world > 1) freed_rows[(size_t)rec.owner].push_back(rec.lrow);
        }
        live_lo = lo; live_hi = hi;
        L.carried = carried;
        for (int32_t r = 0; r < rt_rows; r++)          // evicted slots in ascending order -> freed lines, ascending
            if (fl[r] == kFlagLive) evicted.push_back(rt_lo + r);
        // the strip buffers of the layer kernel hold the live tiles only (holes of a fragmented range cost nothing)
        P.tile_map.resize(L.tile_off + (size_t)(rt_rows / kPTile), -1);
        int32_t n_live_tiles = 0;
        for (int32_t tl = 0; tl < rt_rows / kPTile; tl++) {
            uint8_t any = 0;
            for (int32_t r = tl * kPTile; r < (tl + 1) * kPTile; r++) any |= fl[r];
            if (any) {
                P.tile_map[L.tile_off + (size_t)tl] = n_live_tiles++;
                P.live_tiles.push_back(tl | ((any & kFlagCarried) ? kTileCarried : 0));
            }
        }
        L.n_live_tiles = n_live_tiles;
        L.flag_end = P.flags.size(); L.tile_end = P.tile_map.size(); L.ltile_end = P.live_tiles.size();
        live.swap(next_live);                              // those carried; the members of this layer follow at the next one
    }

    // row owners, couple order, member order: a chain of its own from layer to layer (the owner rule reads the owners of
    // the parents), independent of the slots -- run ahead by whoever is free (see order_one in run_layers)
    void owners_order(int32_t t) {
        Layer &L = P.layers[t];
        const int32_t *X = by_layer.data() + lstart[t];
        const int32_t nn = count[t];
        const int32_t *fam_of = W.fam_of.data() + lstart[t], *fam_count = W.fam_count.data() + lstart[t];
        const int32_t *fam_first = W.fam_first.data() + lstart[t], *fam_key = W.fam_key.data() + lstart[t];
        const int32_t nf_real = W.fam_n[t];
        int8_t *fam_own = W.fam_own.data() + lstart[t];
        int32_t *newid = W.newid.data() + lstart[t], *order = W.order.data() + lstart[t];
        L.base_off = P.fam_base.size();
        // ---- row owners: a couple's children live with one of their parents' rows (the other
        //      parent row is read through NVLink); spill to the least loaded rank past +12.5 %.
        //      Couples are renumbered rank-major; every rank's range starts at a multiple of 4
        //      (16-byte aligned couple columns), the gaps are empty dummy couples. ----
        std::fill(fam_own, fam_own + nf_real, (int8_t)0);
        P.fam_base.resize(L.base_off + (size_t)world + 1, 0);
        P.mem_base.resize(L.base_off + (size_t)world + 1, 0);
        int32_t *fbase = P.fam_base.data() + L.base_off, *mbase = P.mem_base.data() + L.base_off;
        int32_t nf = nf_real;
        if (world > 1) {
            std::fill(load.begin(), load.end(), 0);
            const int32_t cap = (nn + world - 1) / world + (nn + world - 1) / world / 8 + kMaxFamily;
            for (int32_t f = 0; f < nf_real; f++) {
                if (f + kPf < nf_real) {
                    const int32_t y = X[fam_first[f + kPf]], fy = father[y], my = mother[y];
                    if (fy >= 0) __builtin_prefetch(&owner_of[fy]);
                    if (my >= 0) __builtin_prefetch(&owner_of[my]);
                }
                const int32_t x = X[fam_first[f]];
                const int32_t fa = father[x], mo = mother[x];
                int32_t g;
                if (fa >= 0 && mo >= 0) {
                    const int32_t of = owner_of[fa], om = owner_of[mo];
                    g = load[om] < load[of] ? om : of;
                } else if (fa >= 0) g = owner_of[fa];
                else if (mo >= 0) g = owner_of[mo];
                else g = rr++ % world;
                if (load[g] + fam_count[f] > cap) g = (int32_t)(std::min_element(load.begin(), load.end()) - load.begin());
                fam_own[f] = (int8_t)g;
                load[g] += fam_count[f];
            }
            for (int32_t q = 0; q < nn; q++) owner_of[X[q]] = fam_own[fam_of[q]];   // (ranks ascend: sequential writes)
        }
        // ---- couple order inside a rank's range: by the layer in which the couple's longest-lived
        //      member leaves the frontier, then by rank (stable).  A line of column slots then holds
        //      individuals that are evicted together, so whole lines come back (LineAlloc) and the
        //      live slot range stays dense in pedigrees with overlapping generations.  When all
        //      couples of the layer leave together (discrete generations) this is the rank order. ----
        int32_t key_lo = kKeys, key_hi = -1;
        for (int32_t f = 0; f < nf_real; f++) { key_lo = std::min(key_lo, fam_key[f]); key_hi = std::max(key_hi, fam_key[f]); }
        if (world > 1 || key_lo != key_hi) {
            std::vector<int32_t> &cnt = W.cnt_order; cnt.assign((size_t)world * kKeys, 0);
            for (int32_t f = 0; f < nf_real; f++) cnt[(size_t)fam_own[f] * kKeys + fam_key[f]]++;
            for (int32_t g = 0; g < world; g++) {
                int32_t at = fbase[g];
                for (int32_t k = 0; k < kKeys; k++) { const int32_t c = cnt[(size_t)g * kKeys + k]; cnt[(size_t)g * kKeys + k] = at; at += c; }
                // every rank's range starts at a multiple of 4 (16-byte aligned couple columns); the
                // gaps are empty dummy couples
                fbase[g + 1] = world > 1 ? round_up(at, 4) : at;
            }
            nf = fbase[world];
            for (int32_t f = 0; f < nf_real; f++) newid[f] = cnt[(size_t)fam_own[f] * kKeys + fam_key[f]]++;   // stable
        } else {
            fbase[1] = nf;
            for (int32_t f = 0; f < nf_real; f++) newid[f] = f;
        }
        L.n_fam = nf;
        L.nf_pad = round_up(std::max(nf, 1), 32);
        // couple-major member order (couples rank-major, then by first member's rank; members by rank)
        size_t fs0 = P.fam_start.size();
        P.fam_start.resize(fs0 + (size_t)nf + 1);
        int32_t *fstart = P.fam_start.data() + fs0;
        std::fill(fstart, fstart + nf + 1, 0);
        for (int32_t f = 0; f < nf_real; f++) fstart[newid[f] + 1] = fam_count[f];
        for (int32_t f = 0; f < nf; f++) fstart[f + 1] += fstart[f];
        for (int32_t g = 0; g <= world; g++) mbase[g] = fstart[fbase[g]];
        {
            std::vector<int32_t> &pos = W.ipos; pos.assign(fstart, fstart + nf);
            for (int32_t q = 0; q < nn; q++) order[pos[newid[fam_of[q]]]++] = q;
        }
        W.nf_of[t] = nf;
    }

    // lane A: column slots (global, in lines) and local rows (per owner)
    void assign_slots(int32_t t) {
        Layer &L = P.layers[t];
        const int32_t *X = by_layer.data() + lstart[t];
        const int32_t nn = count[t];
        const int32_t *fam_of = W.fam_of.data() + lstart[t];
        const int8_t *fam_own = W.fam_own.data() + lstart[t];
        const int32_t *newid = W.newid.data() + lstart[t], *order = W.order.data() + lstart[t];
        P.mem_ind.resize(L.mem_off + (size_t)nn); P.mem_slot.resize(L.mem_off + (size_t)nn);
        P.mem_fam.resize(L.mem_off + (size_t)nn); P.mem_lrow.resize(L.mem_off + (size_t)nn);
        if (by_seq) P.mem_rank.resize(L.mem_off + (size_t)nn);
        int32_t *mi = P.mem_ind.data() + L.mem_off, *ms = P.mem_slot.data() + L.mem_off;
        int32_t *mf = P.mem_fam.data() + L.mem_off, *ml = P.mem_lrow.data() + L.mem_off;
        for (int32_t q = 0; q < nn; q++) {
            if (q + kPf < nn) __builtin_prefetch(&home[X[order[q + kPf]]], 1);
            if (q + 2 * kPf < nn) { __builtin_prefetch(&X[order[q + 2 * kPf]]); __builtin_prefetch(&fam_of[order[q + 2 * kPf]]); }
            const int32_t oq = order[q], x = X[oq], f = fam_of[oq];
            const int32_t g = fam_own[f];
            const int32_t s = slots.take(), lr = world > 1 ? rows[g].take() : s;   // one rank: row == slot
            if (streaming && (s >= bound_slots || lr >= bound_rows)) give_up_streaming();
            Home &hx = home[x];
            hx.slot = s; hx.lrow = lr; hx.owner = (int8_t)g;
            if (short_rows && last_of[x] == t) {          // read by nobody after this layer: never joins the live list
                W.dead_slots.push_back(s);
                if (world > 1) W.dead_rows[(size_t)g].push_back(lr);
            }
            mi[q] = by_seq ? orient[x] : x; ms[q] = s; mf[q] = newid[f]; ml[q] = lr;
            if (by_seq) P.mem_rank[L.mem_off + (size_t)q] = x;
        }
    }

    // lane B, second piece: the couples' parents -- slots, owners, local rows, rows of the strip buffers
    void couples(int32_t t) {
        Layer &L = P.layers[t];
        const int32_t *X = by_layer.data() + lstart[t];
        const int32_t *fam_first = W.fam_first.data() + lstart[t];
        const int32_t nf = W.nf_of[t], nf_real = W.fam_n[t];
        const int32_t *newid = W.newid.data() + lstart[t];
        L.fam_off = P.fam_pf.size();
        P.fam_pf.resize(L.fam_off + (size_t)nf, -1); P.fam_pm.resize(L.fam_off + (size_t)nf, -1);
        P.fam_pf_owner.resize(L.fam_off + (size_t)nf, -1); P.fam_pm_owner.resize(L.fam_off + (size_t)nf, -1);
        P.fam_pf_lrow.resize(L.fam_off + (size_t)nf, -1); P.fam_pm_lrow.resize(L.fam_off + (size_t)nf, -1);
        P.fam_q.resize(2 * (L.fam_off + (size_t)nf), -1);
        for (int32_t f = 0; f < nf_real; f++) {
            if (f + kPf < nf_real) {
                const int32_t y = X[fam_first[f + kPf]], fy = father[y], my = mother[y];
                if (fy >= 0) __builtin_prefetch(&home[fy]);
                if (my >= 0) __builtin_prefetch(&home[my]);
            }
            if (f + 2 * kPf < nf_real) { const int32_t y = X[fam_first[f + 2 * kPf]]; __builtin_prefetch(&father[y]); __builtin_prefetch(&mother[y]); }
            const int32_t x = X[fam_first[f]], fa = father[x], mo = mother[x];
            const size_t k = L.fam_off + (size_t)newid[f];
            int32_t *ps[2] = {&P.fam_pf[k], &P.fam_pm[k]};
            int8_t *po[2] = {&P.fam_pf_owner[k], &P.fam_pm_owner[k]};
            int32_t *pl[2] = {&P.fam_pf_lrow[k], &P.fam_pm_lrow[k]};
            int32_t *pq[2] = {&P.fam_q[2 * k], &P.fam_q[2 * k + 1]};
            const int32_t par[2] = {fa, mo};
            for (int s = 0; s < 2; s++) {
                const int32_t p = par[s];
                if (p < 0) { *ps[s] = -1; *po[s] = -1; *pl[s] = -1; *pq[s] = -1; continue; }
                const Home hp = home[p];
                *ps[s] = hp.slot; *po[s] = hp.owner; *pl[s] = hp.lrow;
                const int32_t rel = hp.slot - L.rt_lo;             // the parent is live: its tile is in the map
                *pq[s] = P.tile_map[L.tile_off + (size_t)(rel / kPTile)] * kPTile + rel % kPTile;
            }
        }
        L.fam_end = P.fam_pf.size();
    }

    // lane A: member tiles, sole-reader marks, the layer is complete
    void finish_layer(int32_t t) {
        Layer &L = P.layers[t];
        const int32_t nn = count[t], nf = W.nf_of[t];
        // member tiles = the column blocks the layer kernel writes at a time: at most kMTile members and at
        // most kMaxTileFam couples (bounds the staged couple tile), cut at multiples of 8 members (whole
        // 32-byte sectors of a float row on both sides of the cut)
        L.n_mtiles = 0;
        for (int32_t q0 = 0; q0 < nn;) {
            const int32_t *mf = P.mem_fam.data() + L.mem_off;
            int32_t q1 = std::min(nn, q0 + kMTile);
            while (q1 > q0 + 8 && mf[q1 - 1] - mf[q0] >= kMaxTileFam) q1 = std::max(q0 + 8, (q1 - 1) & ~7);
            const int32_t f0 = mf[q0], f1 = mf[q1 - 1];
            for (int32_t v : {f0, f1 - f0 + 1, q0, q1 - q0}) P.mtile_desc.push_back(v);
            L.max_tile_fam = std::max(L.max_tile_fam, f1 - f0 + 1);
            L.n_mtiles++;
            q0 = q1;
        }
        {   // Parents of ONE couple of the layer whose members lie in ONE member tile: their strip-buffer rows are read
            // by a single consumer item (kSoleReader).  A couple whose members straddle a tile cut counts twice.
            std::vector<int32_t> &readers = W.cnt; readers.assign((size_t)std::max(L.n_live_tiles, 1) * kPTile, 0);
            int32_t *fq = P.fam_q.data() + 2 * L.fam_off;
            for (int32_t k = 0; k < 2 * nf; k++) if (fq[k] >= 0) readers[(size_t)fq[k]]++;
            const int32_t *md = P.mtile_desc.data() + 4 * L.mtile_off;
            for (int32_t j = 1; j < L.n_mtiles; j++)
                if (md[4 * j] == md[4 * (j - 1)] + md[4 * (j - 1) + 1] - 1)           // first couple == the previous tile's last
                    for (int32_t k = 2 * md[4 * j]; k < 2 * md[4 * j] + 2; k++) if (fq[k] >= 0) readers[(size_t)fq[k]]++;
            for (int32_t k = 0; k < 2 * nf; k++) if (fq[k] >= 0 && readers[(size_t)fq[k]] == 1) fq[k] |= kSoleReader;
        }
        L.alg_elems = 4.0 * nn * (double)L.live_before + 3.0 * (double)nn * nn;
        P.alg_elems += L.alg_elems;
        P.row_updates += nn;
        if (reads) pair_reads(t);                  // (published with the layer)

        L.mem_end = P.mem_ind.size(); L.mtile_end = P.mtile_desc.size() / 4;     // (lane B has set the ends of its arrays)
        if (streaming) { ps->layers_done.store(t + 1, std::memory_order_release); ps->wake(); }
    }

    // lane A: after the step, evicted slots / rows become reusable from the next layer on (and those of the layer's
    // members that no later layer reads)
    void end_layer(int32_t t) {
        freed.clear();
        for (int32_t s : W.evicted[t & 1]) slots.release(s, freed);
        if (!W.dead_slots.empty()) {
            const size_t mid = freed.size();
            for (int32_t s : W.dead_slots) slots.release(s, freed);      // (slots of one layer ascend)
            std::inplace_merge(freed.begin(), freed.begin() + (ptrdiff_t)mid, freed.end());
            W.dead_slots.clear();
        }
        slots.end_layer(freed);
        for (int32_t g = 0; g < world && world > 1; g++) {
            rows[g].end_layer(W.freed_rows[t & 1][(size_t)g]);
            rows[g].end_layer(W.dead_rows[(size_t)g]);
        }
    }

    // ---- the layers, as a pipeline.  What is sequential in planning is the slot assignment: the members of layer t
    //      take the lines that the evictions of layer t-1 gave back.  The rest hangs off it:
    //        lane A (the planning thread)  column slots and rows (t), member tiles (t), end of the layer (evicted
    //                                      lines and rows return to the allocators)
    //        lane B (a helper thread)      the live list, live range, flags and live tiles BEFORE step t, who is
    //                                      evicted by it; the parents of the couples (t)
    //        ahead of both, by whoever is free: couples grouped (group_layer, any layer) and the ordering chain
    //                                      (owners_order: owners, couple and member order, layer after layer)
    //      Lane B of layer t reads the homes of individuals born before t, so it may start as soon as lane A has
    //      assigned the slots of layer t-1 (`slotted`), and needs the couple order of t for the parents (`ordered`);
    //      lane A needs the order of t for the slots and both pieces of lane B before it closes layer t (`coupled`).
    //      Each array of the plan, and each field of a Layer, is written by one lane only; what lane B hands back
    //      for the end of a layer (evicted slots, freed rows) exists twice, because lane B is by then at work on the
    //      next layer.  Without a helper thread lane A runs everything itself, in the same order. ----
    void run_layers() {
        live.clear(); next_live.clear();
        // allocators: global column slots (lines, lowest free first) and local rows per rank (stack)
        slots.reset(); rows.resize((size_t)world);
        for (Alloc &a : rows) a.reset();
        // (two sets: lane B fills those of layer t+1 while lane A still returns those of layer t)
        for (auto &fr : W.freed_rows) { fr.resize((size_t)world); for (auto &v : fr) v.clear(); }
        W.dead_slots.clear(); W.dead_rows.resize((size_t)world);
        for (auto &v : W.dead_rows) v.clear();
        if (!streaming) P.rows_cap.assign((size_t)world, 0);
        load.assign((size_t)world, 0);
        // the owners once more, one byte per individual: the owner rule reads two parents per couple, and a generation of
        // these stays in cache where the 16-byte homes do not
        if (world > 1) owner_of.resize((size_t)n);
        const size_t M = lstart[S];
        W.fam_of.resize(M); W.fam_count.resize(M); W.fam_first.resize(M); W.fam_key.resize(M);
        W.order.resize(M); W.newid.resize(M); W.fam_own.resize(M); W.nf_of.assign((size_t)S, 0);   // (owners_order, per layer)
        W.fam_n.assign((size_t)S, 0);
        // the planning thread, one helper that runs lane B, one that groups couples ahead (with two threads, lane B's does both)
        const int n_threads = plan_threads((int64_t)M, 200000, planners, world);
        if (W.tables.size() < (size_t)n_threads) W.tables.resize((size_t)n_threads);
        std::vector<std::atomic<int>> grouped((size_t)S);
        for (auto &g : grouped) g.store(0, std::memory_order_relaxed);
        std::atomic<int32_t> next_job{0};
        std::atomic<bool> group_failed{false};
        auto run_job = [&](int32_t t, int id) {
            try { group_layer(t, W.tables[(size_t)id]); } catch (...) { group_failed.store(true); }
            grouped[(size_t)t].store(1, std::memory_order_release);
        };
        // a grouping job, if one is left; false when there was none
        auto group_one = [&](int id) {
            const int32_t j = next_job.load(std::memory_order_relaxed) < S ? next_job.fetch_add(1) : S;
            if (j >= S) return false;
            run_job(j, id);
            return true;
        };
        PhaseTimer lane_a, lane_b;                 // time of each piece, summed over the layers

        // hand-over between the lanes: layer numbers + 1.  A lane that has to wait groups couples ahead; with none left it
        // spins politely (the other lane may run on the sibling hardware thread) and yields now and then
        auto idle = [](unsigned &spins) {
#if defined(__x86_64__) || defined(__i386__)
            for (int i = 0; i < 16; i++) __builtin_ia32_pause();
#elif defined(__aarch64__)
            for (int i = 0; i < 16; i++) asm volatile("yield");
#endif
            if ((++spins & 15) == 0) std::this_thread::yield();   // (every few microseconds: ranks of a job share the host's cores)
        };
        std::atomic<int32_t> slotted{0}, ordered{0}, coupled{0};
        std::atomic<bool> stop{false}, lane_failed{false};
        // The ordering chain (owners_order, layer after layer) belongs to nobody: whoever is free and finds the next
        // layer grouped takes it (one at a time), so it runs ahead of the slots on a helper when there is one and on
        // the planning thread when there is not.  Returns false when there was nothing to take.
        std::atomic<bool> order_busy{false};
        int32_t order_next = 0;                              // (guarded by order_busy)
        auto order_one = [&]() {
            if (ordered.load(std::memory_order_relaxed) >= S) return false;
            if (order_busy.exchange(true, std::memory_order_acquire)) return false;
            bool did = false;
            const int32_t t = order_next;
            if (t < S && grouped[(size_t)t].load(std::memory_order_acquire) && !group_failed.load()) {
                try { owners_order(t); } catch (...) { lane_failed.store(true); }
                order_next = t + 1;
                ordered.store(t + 1, std::memory_order_release);
                did = true;
            }
            order_busy.store(false, std::memory_order_release);
            return did;
        };
        // what a waiting thread does meanwhile: the ordering chain first (it is on the way of both lanes), else grouping
        auto side_job = [&](int id) { return order_one() || group_one(id); };
        struct Helpers {
            std::vector<std::thread> th;
            std::atomic<bool> *stop = nullptr;
            void join_all() { if (stop) stop->store(true); for (auto &t : th) if (t.joinable()) t.join(); th.clear(); }
            ~Helpers() { join_all(); }
        } helpers;
        helpers.stop = &stop;
        bool piped = false;
        for (int id = 1; id < n_threads; id++) {
            try {
                if (id == 1) {
                    helpers.th.emplace_back([&, id] {                 // lane B; groups couples ahead whenever it has to wait
                        unsigned spins0 = 0;
                        try {
                            for (int32_t t = 0; t < S; t++) {
                                unsigned spins = 0;
                                while (slotted.load(std::memory_order_acquire) < t) {      // the homes of layer t-1
                                    if (stop.load(std::memory_order_relaxed)) return;
                                    if (!side_job(id)) idle(spins);
                                }
                                lane_b.start();
                                live_flags(t);
                                lane_b.add(0);
                                while (ordered.load(std::memory_order_acquire) <= t) {
                                    if (stop.load(std::memory_order_relaxed)) return;
                                    if (!side_job(id)) idle(spins);
                                }
                                lane_b.start();
                                couples(t);
                                lane_b.add(1);
                                coupled.store(t + 1, std::memory_order_release);
                            }
                            while (!stop.load(std::memory_order_relaxed) && ordered.load(std::memory_order_acquire) < S) { if (!side_job(id)) idle(spins0); }
                        } catch (...) {
                            lane_failed.store(true);
                            coupled.store(INT32_MAX, std::memory_order_release);
                        }
                    });
                    piped = true;
                } else {
                    helpers.th.emplace_back([&, id] {             // grouping and the ordering chain, until both are through
                        unsigned spins = 0;
                        while (!stop.load(std::memory_order_relaxed) && ordered.load(std::memory_order_acquire) < S) { if (!side_job(id)) idle(spins); }
                    });
                }
            } catch (...) { break; }                 // no thread: the planning thread does the jobs itself
        }

        for (int32_t t = 0; t < S; t++) {
            lane_a.add(5);
            begin_layer(t);
            if (!piped) live_flags(t);
            lane_a.add(0);
            // ---- couples of the layer grouped (group_layer) and ordered (owners_order), here or on a helper thread ----
            unsigned spins = 0;
            while (ordered.load(std::memory_order_acquire) <= t) {
                if (group_failed.load() || lane_failed.load()) { helpers.join_all(); throw std::bad_alloc(); }
                if (!side_job(0)) idle(spins);
            }
            if (group_failed.load() || lane_failed.load()) { helpers.join_all(); throw std::bad_alloc(); }
            lane_a.add(1);
            assign_slots(t);
            if (piped) slotted.store(t + 1, std::memory_order_release);
            lane_a.add(2);
            if (piped) {
                while (coupled.load(std::memory_order_acquire) <= t)
                    if (!side_job(0)) idle(spins);
                if (lane_failed.load() || group_failed.load()) { helpers.join_all(); throw std::bad_alloc(); }
            } else couples(t);
            lane_a.add(3);
            finish_layer(t);
            lane_a.add(4);
            end_layer(t);
        }
        helpers.join_all();
        if (group_failed.load() || lane_failed.load()) throw std::bad_alloc();
        if (lane_a.on) {
            const double *a = lane_a.sum;
            std::fprintf(stderr, "[plan]   lane A: %s %.2f  order: own share or wait %.2f  slots %.2f  %s %.2f  tiles %.2f  end %.2f\n",
                         piped ? "begin" : "live/flags", a[0], a[1], a[2], piped ? "wait-B" : "couples", a[3], a[4], a[5]);
            if (piped) std::fprintf(stderr, "[plan]   lane B: live/flags %.2f  couples %.2f\n", lane_b.sum[0], lane_b.sum[1]);
        }
    }

    // capacities (a streamed plan keeps the bounds its engine was sized with) and the probands' homes
    int finish() {
        if (!streaming) {
            P.capacity = round_up(std::max<int64_t>((int64_t)slots.next_fresh * kSlotLine, 1), kPTile);
            P.rows_cap.resize((size_t)world);
            for (int32_t g = 0; g < world; g++) P.rows_cap[g] = world > 1 ? std::max(rows[g].next_fresh, 1) : P.capacity;
        }
        if (reads) pair_reads(S);                  // after the last layer (published with the finished plan)
        if (int rc = std::getenv("GENLIB_PLAN_VERIFY") ? verify_plan(P, err) : GENLIB_OK) return rc;
        if (int rc = reads && std::getenv("GENLIB_PLAN_VERIFY") ? verify_pair_reads(P, pairs, err) : GENLIB_OK) return rc;
        const size_t np = short_rows ? 0 : P.pro_ind.size();    // (kScheduleF, kSchedulePairs: no proband matrix)
        P.pro_slot.resize(np); P.pro_owner.resize(np); P.pro_lrow.resize(np);
        for (size_t u = 0; u < np; u++) {
            const Home &hu = home[P.pro_ind[u]];
            P.pro_slot[u] = hu.slot; P.pro_owner[u] = hu.owner; P.pro_lrow[u] = hu.lrow;
        }
        return GENLIB_OK;
    }
};

}  // namespace

void adopt_retired_storage(Plan &into) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (g_retired) { into = std::move(*g_retired); g_retired.reset(); }
}
void retire_storage(Plan &from) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (!g_retired) { from.reset(); g_retired.reset(new Plan(std::move(from))); }
}
void release_plan_cache() {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    g_retired.reset(); g_scratch.reset();
}

int check_pedigree(int32_t n, const int32_t *father, const int32_t *mother, std::string &err) {
    for (int32_t i = 0; i < n; i++) {
        const int32_t f = father[i], m = mother[i];
        if (f < -1 || f >= n || m < -1 || m >= n) { err = "KeyError: parent index out of range at rank " + std::to_string(i); return GENLIB_EKEY; }
        if (f >= i || m >= i) { err = "parent does not precede child at rank " + std::to_string(i); return GENLIB_EORDER; }
    }
    return GENLIB_OK;
}

uint64_t plan_digest(const Plan &P, bool with_bounds) {
    uint64_t h = 1469598103934665603ULL;
    auto bytes = [&h](const void *p, size_t nb) { const unsigned char *c = (const unsigned char *)p; for (size_t i = 0; i < nb; i++) { h ^= c[i]; h *= 1099511628211ULL; } };
    auto vec = [&bytes](const auto &v) { const uint64_t s = v.size(); bytes(&s, 8); if (s) bytes(v.data(), s * sizeof(v[0])); };
    const int64_t hdr[6] = {P.n, P.n_unique, P.world, P.schedule, with_bounds ? P.capacity : 0, P.row_updates};
    bytes(hdr, sizeof hdr); bytes(&P.alg_elems, 8);
    for (const Layer &L : P.layers) {
        const int64_t f[] = {L.n_new, L.n_fam, L.live_before, L.carried, L.ref_founders, L.ref_probands, L.ref_both, L.rt_lo, L.rt_rows,
                             L.n_live_tiles, (int64_t)L.tile_off, (int64_t)L.ltile_off, L.nf_pad, L.n_mtiles, L.max_tile_fam, (int64_t)L.mem_off,
                             (int64_t)L.fam_off, (int64_t)L.flag_off, (int64_t)L.mtile_off, (int64_t)L.base_off, (int64_t)L.mem_end, (int64_t)L.fam_end,
                             (int64_t)L.flag_end, (int64_t)L.tile_end, (int64_t)L.ltile_end, (int64_t)L.mtile_end};
        bytes(f, sizeof f); bytes(&L.alg_elems, 8);
    }
    vec(P.pro_ind); vec(P.pro_slot); vec(P.mem_ind); vec(P.mem_slot); vec(P.mem_fam); vec(P.mem_rank); vec(P.fam_pf); vec(P.fam_pm);
    vec(P.fam_start); vec(P.fam_q); vec(P.flags); vec(P.tile_map); vec(P.live_tiles); vec(P.mtile_desc); vec(P.fam_base); vec(P.mem_base);
    vec(P.mem_lrow); vec(P.fam_pf_owner); vec(P.fam_pm_owner); vec(P.fam_pf_lrow); vec(P.fam_pm_lrow); vec(P.live_owner); vec(P.live_lrow);
    vec(P.pro_owner); vec(P.pro_lrow);
    if (with_bounds) vec(P.rows_cap);
    if (P.schedule == kSchedulePairs) {        // (the other schedules' digests stay what they were)
        vec(P.pair_start); vec(P.pair_pos); vec(P.pair_row_slot); vec(P.pair_col_slot); vec(P.pair_owner); vec(P.pair_lrow);
    }
    return h;
}

int build_plan(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids, int32_t n_pro,
               const int32_t *proband, int32_t world, int schedule, Plan &P, std::string &err, PlanStream *ps, int planners,
               const PairList &pairs) {
    int rc;
    try {
        std::unique_ptr<Scratch> W = take_scratch();
        rc = Planner{*W, P, err, ps, n, father, mother, ids, n_pro, proband, world, schedule, planners, pairs}.run();
        give_scratch(std::move(W));
    } catch (const std::bad_alloc &) {
        if (!ps) throw;
        rc = GENLIB_ENOMEM; err = "out of host memory while planning";
    }
    if (ps) {                                  // whatever happened, the consumers must not wait for ever
        if (rc != GENLIB_OK) { ps->err = err; ps->status.store(rc, std::memory_order_release); }
        ps->stage.store(2, std::memory_order_release);
        ps->wake();
    }
    return rc;
}

}  // namespace genlib
