// plan.hpp -- host-side schedule of the level-synchronous kinship sweep.
//
// Replaces, on flat arrays, what gen.phi does serially before and inside its
// step loop (reference, relative to /root/reference):
//   src/compute.jl:193-207,236-241  raw levels by upward BFS from the probands
//   src/compute.jl:243-251          cut vertices (who is live in which step)
//   src/compute.jl:165-186          _index_pedigree
//   src/compute.jl:287-289          founder_index (here: a slot in the frontier matrix)
// plus the Kirkpatrick-2019 eviction rule the reference states in sparse_phi
// (src/compute.jl:400-430): a row is dropped once its last child is born.
//
// No CUDA in this file: the plan is testable without a GPU.
#pragma once
#include <atomic>
#include <condition_variable>
#include <cstddef>
#include <cstdint>
#include <mutex>
#include <string>
#include <vector>

namespace genlib {

constexpr int kPTile = 128;      // frontier columns per producer tile (and slot-range alignment)
constexpr int kFTile = 32;       // couples per producer tile (upper bound)
constexpr int kMTile = 128;      // member columns per consumer tile (4 per lane)
constexpr int kMaxFamily = 32;   // sibships larger than this are split (bounds per-tile work)
constexpr int kSlotLine = 32;     // column slots are allocated and recycled in lines of this many (128 B of a float row)
constexpr int kMaxTileFam = 64;  // couples per member tile (bounds the couple tile staged by the layer kernel)

// Which reference function's floating-point schedule the plan reproduces:
//   phi        (compute.jl:233-304)  layers by height above the probands, the higher RANK is climbed,
//                                    one Float32 rounding per step (unrounded Float64 inside a step)
//   sparse_phi (compute.jl:321-447)  layers by depth below the founders, the individual processed
//                                    later by its queue is climbed, every stored entry is Float32
//   sparse_phi, symmetric            the same schedule, but every kinship is filed where it is looked up:
//                                    the reference files phi[earlier][later] and reads phi[lower rank][higher
//                                    rank] (compute.jl:393 vs :367-389), losing the pairs whose queue order
//                                    inverts their rank order; kScheduleSparsePhi reproduces that loss
//   f                                gen.f for many individuals: the members are the ancestors-or-self of the listed
//                                    individuals that have both parents, layered by depth below the founders (a
//                                    childless member of generation 3 is born in layer 3, not with the last one),
//                                    with phi's arithmetic (the higher RANK is climbed, mem_ind is the rank).  No
//                                    row is kept to the end: a row leaves after the layer of its last child, a row
//                                    without children after its own layer (the layer still writes it).  The engine
//                                    reads Psi[father, mother] of every couple just before its layer; there is no
//                                    proband matrix (pro_slot / pro_owner / pro_lrow are empty).
//   pairs                            gen.phi_pairs: f's layers, arithmetic and short rows, over the ancestors-or-self
//                                    of everybody named in a pair (a, b).  The pair is read in layer
//                                    r = max(depth a, depth b) + 1, just before that layer's kernel (r == S: once after
//                                    the last layer), from the row of the higher-ranked member; both rows live until
//                                    then (a row's last layer is the later of its last child and its last read).
//                                    pro_ind = the distinct named individuals; no proband matrix either.
constexpr int kSchedulePhi = 0, kScheduleSparsePhi = 1, kScheduleSparsePhiSymmetric = 2, kScheduleF = 3, kSchedulePairs = 4;
inline bool sparse_schedule(int s) { return s == kScheduleSparsePhi || s == kScheduleSparsePhiSymmetric; }

constexpr int32_t kTileCarried = 1 << 30;   // live_tiles entry: the tile has a carried column
constexpr int32_t kSoleReader = 1 << 30;    // fam_q entry (>= 0): no other couple of the layer has this parent -- whoever reads its row of a
                                            // strip buffer is the only one to do so (and may drop it from L2 afterwards)
constexpr uint8_t kFlagLive = 1;     // slot holds an individual that is live before the step
constexpr uint8_t kFlagCarried = 2;  // ... and stays live after it

struct Layer {
    int32_t n_new = 0, n_fam = 0;
    int32_t live_before = 0, carried = 0;
    int32_t ref_founders = 0, ref_probands = 0, ref_both = 0;
    int32_t rt_lo = 0, rt_rows = 0;   // live slots lie in [rt_lo, rt_lo + rt_rows), both multiples of kPTile
    int32_t n_live_tiles = 0;         // tiles of kPTile slots in that range that hold a live individual
    size_t tile_off = 0;              // into tile_map (rt_rows / kPTile entries)
    size_t ltile_off = 0;             // into live_tiles (n_live_tiles entries)
    int32_t nf_pad = 0;               // row stride of the transposed cross block (families, multiple of 32)
    int32_t n_mtiles = 0;
    int32_t max_tile_fam = 0;         // most couples in one member tile
    size_t mem_off = 0;               // into mem_* arrays
    size_t fam_off = 0;               // into fam_pf / fam_pm; fam_start uses fam_off + layer index
    size_t flag_off = 0;              // into flags
    size_t mtile_off = 0;             // into mtile_* arrays
    size_t base_off = 0;              // into fam_base / mem_base (world + 1 entries each)
    // sizes of the concatenated arrays once the layer is complete (a streamed plan is uploaded layer by layer)
    size_t mem_end = 0, fam_end = 0, flag_end = 0, tile_end = 0, ltile_end = 0, mtile_end = 0;
    double alg_elems = 0;             // 4 n L + 3 n^2
};

struct Plan {
    int32_t n = 0, n_unique = 0, world = 1, schedule = kSchedulePhi;
    int64_t capacity = 0;             // W, multiple of kPTile; also the leading dimension
    int64_t row_updates = 0;
    double alg_elems = 0;
    std::vector<Layer> layers;
    std::vector<int32_t> pro_ind, pro_slot;          // kScheduleF: pro_ind = the distinct listed individuals with both parents
    // concatenated per-layer arrays
    std::vector<int32_t> mem_ind, mem_slot, mem_fam;   // family-major order inside a layer
    std::vector<int32_t> mem_rank;                     // sparse_phi schedules: the members' pedigree ranks (mem_ind = queue position)
    std::vector<int32_t> fam_pf, fam_pm, fam_start;    // parents as slots (-1 = none)
    std::vector<int32_t> fam_q;                        // 2 per couple: father, mother as rows of the layer kernel's strip buffers (-1 = none), | kSoleReader
    std::vector<uint8_t> flags;
    std::vector<int32_t> tile_map;                     // per tile of a layer's live range: its index among the live tiles (-1: hole)
    std::vector<int32_t> live_tiles;                   // the inverse: live tiles in order, | kTileCarried if a column is carried
    std::vector<int32_t> mtile_desc;                   // 4 per member tile: first couple, couples, first member, members
    // ---- row sharding (world ranks; world == 1 puts everything on rank 0) ----
    // Couples are numbered rank-major inside a layer: rank g owns couples
    // [fam_base[g], fam_base[g+1]) and members [mem_base[g], mem_base[g+1]), and holds the
    // full-width rows of those members at local row indices mem_lrow.
    std::vector<int32_t> fam_base, mem_base;           // per layer, world + 1 entries
    std::vector<int32_t> mem_lrow;                     // parallel to mem_ind
    std::vector<int8_t> fam_pf_owner, fam_pm_owner;    // parallel to fam_pf (-1 = no such parent)
    std::vector<int32_t> fam_pf_lrow, fam_pm_lrow;
    std::vector<int8_t> live_owner;                    // parallel to flags
    std::vector<int32_t> live_lrow;
    std::vector<int8_t> pro_owner;
    std::vector<int32_t> pro_lrow;
    std::vector<int64_t> rows_cap;                     // per rank: rows of the frontier it holds
    // ---- kSchedulePairs: one read per list position, bucketed by read layer (list order inside a bucket).  The
    //      reads of layer t are [pair_start[t], pair_start[t + 1]) for t in [0, S]; t == S: after the last layer.
    //      Sized at the list's length before the first layer is published, filled layer by layer. ----
    std::vector<int64_t> pair_start, pair_pos;         // pair_pos: the read's list position
    std::vector<int32_t> pair_row_slot, pair_col_slot; // the higher-ranked member's slot (its row), the other one's (the column)
    std::vector<int8_t> pair_owner;                    // the rank that holds the row, and its local row there
    std::vector<int32_t> pair_lrow;

    // Every array above, for reset(): the storage of a destroyed plan is handed to the next
    // genlib_plan_create, because first-touch page faults on a few hundred MB of fresh vectors
    // cost more than the planning itself.
    template <class F> void each_array(F &&f) {
        f(layers); f(pro_ind); f(pro_slot); f(mem_ind); f(mem_rank); f(mem_slot); f(mem_fam); f(fam_pf); f(fam_pm);
        f(fam_q);
        f(fam_start); f(flags); f(tile_map); f(live_tiles);
        f(mtile_desc); f(fam_base); f(mem_base); f(mem_lrow);
        f(fam_pf_owner); f(fam_pm_owner); f(fam_pf_lrow); f(fam_pm_lrow); f(live_owner); f(live_lrow);
        f(pro_owner); f(pro_lrow); f(rows_cap);
        f(pair_start); f(pair_pos); f(pair_row_slot); f(pair_col_slot); f(pair_owner); f(pair_lrow);
    }
    void reset() {                     // empty plan, capacities kept
        each_array([](auto &v) { v.clear(); });
        n = n_unique = 0; world = 1; schedule = kSchedulePhi; capacity = row_updates = 0; alg_elems = 0;
    }
};

// Hand-over of a plan that is still being built: the planner publishes the layers one by one, an engine on
// another thread uploads and launches them while the later layers are planned (planning is otherwise the
// largest host-side part of a call).  What the engine must know before the first layer -- the frontier width
// (leading dimension of the frontier matrix), the rows per rank, the sizes of the index arrays -- exists only
// as an UPPER BOUND then: the planner derives it from the pre-pass (most individuals in the frontier at once,
// plus slack for the line-granular slot allocator), reserves every array at its bound (no reallocation under
// the reader) and keeps the bound as Plan::capacity.  Should a layer need more, it raises `overflow`, waits
// until the consumer has stopped, and finishes as an ordinary plan with exact sizes.
struct PlanStream {
    std::atomic<int32_t> stage{0};         // 0: pre-pass; 1: bounds set, arrays reserved, layers are coming; 2: finished
    std::atomic<int32_t> layers_done{0};   // layers [0, layers_done) are final in the plan's arrays
    std::atomic<int32_t> status{0};        // a GENLIB_E* code once the planner has failed
    std::atomic<bool> streamed{false};     // set with stage 1: the plan carries bounds and is published layer by layer
    std::atomic<bool> overflow{false};     // a bound was too small: consumers stop, the plan ends with exact sizes
    std::atomic<int32_t> consumers{0};     // consumers still reading the arrays (the planner waits for 0 on overflow)
    std::string err;                       // the planner's message (read after stage == 2)
    std::mutex mu;
    std::condition_variable cv;
    void wake() { { std::lock_guard<std::mutex> lk(mu); } cv.notify_all(); }
    template <class Pred> void wait(Pred &&pred) { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, pred); }
};

// Recycling of plan storage across calls (bounded: one retired plan, one set of planner scratch).
void adopt_retired_storage(Plan &into);   // moves a retired plan's (empty, reserved) arrays into `into`
void retire_storage(Plan &from);          // keeps `from`'s arrays for the next adopt_retired_storage
void release_plan_cache();                // frees what is kept (genlib_release_cache)

inline int32_t pad32(int32_t x) { return ((x > 0 ? x : 1) + 31) / 32 * 32; }

// Records `msg` as the calling thread's last error (genlib_last_error) and returns `code`.
int set_error(int code, const std::string &msg);

// Returns 0 or a GENLIB_E* status; `err` receives a message.
// `ids` (nullable, by rank) orders the founders in sparse_phi's queue (founder() sorts by ID,
// identify.jl:15-19); without it they are taken in rank order.
// With `stream` the plan is published layer by layer (see PlanStream); stage 2 is always reached.
// `planners`: how many planners share this host's cores while this one runs -- `world` when every rank is a process
// of its own that plans for itself (0: assume that), 1 when one process plans for all its devices; the planner
// takes up to three threads out of cores / planners (GENLIB_PLAN_THREADS overrides).
// The pairs of a kSchedulePairs plan: ranks a[k], b[k] for k in [0, n), in list order.
struct PairList {
    int64_t n = 0;
    const int32_t *a = nullptr, *b = nullptr;
};

int build_plan(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids, int32_t n_pro,
               const int32_t *proband, int32_t world, int schedule, Plan &plan, std::string &err,
               PlanStream *stream = nullptr, int planners = 0, const PairList &pairs = PairList{});

// Internal to the library (hidden: not exported).
// The pedigree's own errors, the first offending rank: a parent index out of range (GENLIB_EKEY) or a parent that
// does not precede its child (GENLIB_EORDER).  Returns 0 or that status; `err` receives the message.
__attribute__((visibility("hidden"))) int check_pedigree(int32_t n, const int32_t *father, const int32_t *mother, std::string &err);
// FNV-1a over the header, every Layer field and every array of the plan, in a fixed order (genlib_plan_digest);
// `with_bounds` adds Plan::capacity and Plan::rows_cap.  A new array of Plan belongs here as well as in each_array.
__attribute__((visibility("hidden"))) uint64_t plan_digest(const Plan &P, bool with_bounds);

}  // namespace genlib
