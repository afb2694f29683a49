/*
 * genlib_cuda.h -- C ABI of libgenlib_cuda.so, the B200 kinship engine that sits
 * behind GenLib.jl's `gen.phi(ped)` / `gen.phi(ped, probandIDs)`.
 *
 * The reference has no FFI boundary: the path is the Julia method
 *     phi(pedigree::Pedigree, probandIDs::Vector{Int} = pro(pedigree);
 *         verbose::Bool = false, compute::Bool = true)      src/compute.jl:233-304
 * so these entry points are what a `ccall` shim (genlib.jl_b200/julia/GenLibCUDA.jl,
 * INTEGRATION.md) binds in its place.  Everything is plain pointers and sizes;
 * the caller owns every buffer (except the result of genlib_phi_over, whose
 * size only the device knows: the library allocates it, genlib_kinship_pairs_free
 * releases it); no call throws, exits or keeps a pointer after it returns
 * (handles excepted).
 *
 * Pedigree encoding (what `values(pedigree)` yields, src/create.jl:234-254):
 *   individuals are numbered by 0-based rank (Individual.rank - 1); father[i] /
 *   mother[i] are the rank of the parent or -1 for `nothing`; every parent
 *   precedes its children.  Probands are ranks, in the order the output matrix
 *   must have (src/compute.jl:303); duplicates collapse onto their first
 *   occurrence (the `intersect` at src/compute.jl:251).
 */
#ifndef GENLIB_CUDA_H
#define GENLIB_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GENLIB_ABI_VERSION 2

/* status codes (0 = ok) */
#define GENLIB_OK 0
#define GENLIB_EINVAL 1    /* malformed arguments (null pointer, bad dtype ...)          */
#define GENLIB_EKEY 2      /* proband or parent index out of range: Julia's KeyError,   */
                           /* src/create.jl:70 reached from src/compute.jl:196          */
#define GENLIB_EORDER 3    /* a parent does not precede its child (create.jl:240)       */
#define GENLIB_ECUDA 4     /* CUDA runtime / driver error, no usable device             */
#define GENLIB_ENOMEM 5    /* working set does not fit the device(s)                    */
#define GENLIB_ECOMM 6     /* NCCL / peer-memory set-up failed                          */
#define GENLIB_ERESTART 7  /* genlib_engine_run on an engine of a plan that was still    */
                           /* being made (genlib_plan_create_async): a size bound did    */
                           /* not hold; destroy the engine, create it again (the plan is */
                           /* finished by then) and run                                  */
#define GENLIB_EOVERFLOW 8 /* genlib_occ: a path count or row sum does not fit an Int64;  */
                           /* genlib_phi_over: more pairs than max_pairs (out->n = count) */

/* numerics: how the frontier is stored between generation steps */
#define GENLIB_NUMERICS_REFERENCE 0 /* Float32 storage, Float64 arithmetic, one RN32 per   */
                                    /* cut-vertex step: bit-identical to src/compute.jl:   */
                                    /* 105-158,291-301                                      */
#define GENLIB_NUMERICS_FP64 1      /* Float64 storage, no intermediate rounding           */

/* output element type */
#define GENLIB_F32 0 /* Matrix{Float32}: what gen.phi returns (src/compute.jl:271,291)      */
#define GENLIB_F64 1

typedef struct genlib_plan genlib_plan;     /* host-side schedule; needs no GPU */
typedef struct genlib_engine genlib_engine; /* device-side state of one rank    */

/* One generation step (= one cut-vertex step of src/compute.jl:276-302). */
typedef struct genlib_layer_info {
    int32_t n_new;        /* individuals born in this layer (row-updates)               */
    int32_t n_fam;        /* distinct (father, mother) couples among them               */
    int32_t live_before;  /* L: individuals whose rows are live when the step starts    */
    int32_t carried;      /* of those, how many stay live after the step                */
    int32_t ref_founders; /* |cut[k]|   -- "founders" of the verbose line, compute.jl:258 */
    int32_t ref_probands; /* |cut[k+1]| -- "probands", compute.jl:259                     */
    int32_t ref_both;     /* |cut[k] n cut[k+1]|, compute.jl:260                          */
    int32_t strip_width;  /* engine: couples per strip of the layer kernel               */
    double alg_elems;     /* 4*n*L + 3*n^2 (SURVEY.md 8d); bytes = elems * sizeof(storage) */
    double ms_layer;      /* engine: device time of the layer kernel (when timed)        */
    double ms_wait;       /* ... spent in the inter-GPU barrier that ends the layer      */
    /* engine, this rank: the traffic the step cannot avoid, from the plan */
    double dram_read_bytes;  /* parent rows of own couples over the live columns, once   */
    double dram_write_bytes; /* own members' rows and their columns in carried rows, once */
    double l2_bytes;         /* strip buffers written and read back (L2-resident scratch) */
    double nvlink_bytes;     /* parent rows / carried rows that live on another GPU      */
} genlib_layer_info;

typedef struct genlib_stats {
    int32_t n_unique;      /* side of the output matrix                                  */
    int32_t n_layers;      /* generation layers including the top one                    */
    int64_t row_updates;   /* individuals born = sum of n_new                            */
    int64_t capacity;      /* W: slots (rows/columns) of the frontier matrix             */
    int64_t device_bytes;  /* device memory the engine allocated on this rank            */
    double alg_bytes;      /* sum over layers of s*(4nL+3n^2)                             */
    double ms_plan;        /* host planning (on a worker thread, beside the device, when */
                           /* the plan is streamed: genlib_phi, genlib_plan_create_async) */
    double ms_upload;      /* engine set-up + plan H2D (a streamed plan is uploaded      */
                           /* layer by layer inside ms_kernels instead)                  */
    double ms_kernels;     /* all layers, CUDA events on the engine's stream; with a     */
                           /* streamed plan: first launch to last, waits for the planner */
                           /* included                                                   */
    double ms_fetch;       /* proband gather + D2H                                       */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    int32_t kernel_launches;
    int32_t reserved;
} genlib_stats;

int genlib_version(void);
/* Thread-local, human-readable description of the last failure on this thread. */
const char *genlib_last_error(void);
/* Number of visible CUDA devices, or a negative status. */
int genlib_device_count(void);

/* The library keeps the device arena of the last engine per device for reuse (cudaMalloc of
 * tens of GB costs hundreds of ms).  This frees every cached arena. */
int genlib_release_cache(void);

/* Page-locked host memory for `out` buffers (D2H at full PCIe speed).  Optional:
 * every entry point also accepts pageable memory. */
int genlib_pinned_alloc(size_t bytes, void **out);
int genlib_pinned_free(void *ptr);

/* ---- input side (host only): the `gen.genealogy` ordering on flat arrays --------------------
 * Replaces genealogy(::String) / genealogy(::DataFrame), src/create.jl:131-189, with the stable
 * depth ordering of :196-227 and the rank assignment of :234-254 (SURVEY.md 8(f) N4: 5 M-row
 * files must not become the bottleneck).  IDs are arbitrary non-zero integers, 0 = unknown
 * parent; `sort = 0` keeps the file order and requires parents to come first (KeyError else). */
typedef struct genlib_pedigree genlib_pedigree;
int genlib_genealogy_csv(const char *path, int sort, genlib_pedigree **out);
int genlib_genealogy_arrays(int64_t n, const int64_t *ind, const int64_t *father, const int64_t *mother,
                            const int32_t *sex /* may be NULL */, int sort, genlib_pedigree **out);
void genlib_pedigree_destroy(genlib_pedigree *ped);
int64_t genlib_pedigree_n(const genlib_pedigree *ped);
/* Number of generations (gen.depth, src/describe.jl:60-66 = largest _max_depth). */
int32_t genlib_pedigree_depth(const genlib_pedigree *ped);
/* Rank-ordered view: IDs, 0-based parent ranks (-1 = none), sex.  Any pointer may be NULL. */
int genlib_pedigree_arrays(const genlib_pedigree *ped, int64_t *ids, int32_t *father, int32_t *mother, int32_t *sex);
/* gen.pro (src/identify.jl:35-39): IDs without children, ascending; returns the count. */
int64_t genlib_pedigree_pro(const genlib_pedigree *ped, int64_t *out);
/* IDs -> 0-based ranks; GENLIB_EKEY (Julia's KeyError) on an unknown ID. */
int genlib_pedigree_ranks(const genlib_pedigree *ped, int64_t n, const int64_t *ids, int32_t *ranks);

/* ---- planning (host only): levels, Kirkpatrick frontier, slots -------------
 * Replaces src/compute.jl:236-251 (cut vertices), :165-186 (_index_pedigree)
 * and :287-289 (founder_index).  `world` > 1 prepares the row-sharded schedule
 * for that many ranks. */
int genlib_plan_create(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                       const int32_t *proband, int32_t world, genlib_plan **out);
/* The same plan for the floating-point schedule of another reference function (SURVEY.md 8(f) N2):
 *   GENLIB_SCHEDULE_PHI         phi, src/compute.jl:233-304 (= genlib_plan_create)
 *   GENLIB_SCHEDULE_SPARSE_PHI  sparse_phi, src/compute.jl:321-447: individuals are processed by a
 *       queue from the founders (:335-339, :431-439), of a pair the one processed later is climbed
 *       (:363-395), every stored kinship is a Float32 (:331), rows are evicted when the last child has
 *       been processed (:400-430).  The engine then returns, densely, the values `sparse_phi` keeps
 *       for the probands; numerics must be GENLIB_NUMERICS_REFERENCE.
 *   GENLIB_SCHEDULE_SPARSE_PHI_SYMMETRIC  the same schedule with every kinship filed where it is looked
 *       up.  The reference files phi[rank of the earlier processed][rank of the later] (:393) and reads
 *       phi[lower rank][higher rank] (:36-40, :367-389); when the queue order of two individuals of the
 *       same depth inverts their rank order the value is never found again and the reference carries on
 *       as if they were unrelated.  GENLIB_SCHEDULE_SPARSE_PHI reproduces that (bit-identical to the
 *       reference's KinshipMatrix look-ups); this variant keeps those kinships.
 *   GENLIB_SCHEDULE_F  the schedule of genlib_f: the members are the ancestors-or-self of the listed individuals
 *       that have both parents (the others never reach the plan), layered by depth below the founders, with
 *       phi's arithmetic; no row is kept to the end (a row leaves after the layer of its last child, or after
 *       its own layer when it has none).  Such a plan has no proband matrix: it can be inspected with the
 *       genlib_plan_* calls, genlib_engine_create* refuses it (GENLIB_EINVAL). *
 *   GENLIB_SCHEDULE_PAIRS  the schedule of genlib_phi_pairs (made by genlib_plan_create_pairs, which takes pairs
 *       instead of probands): GENLIB_SCHEDULE_F's layers and arithmetic over the ancestors-or-self of everybody
 *       named in a pair.  The pair (a, b) is read in layer r = max(depth a, depth b) + 1, just before that layer
 *       (r == the number of layers: once after the last one), from the row of the higher-ranked member; a row
 *       leaves after the later of its last child and its last read.  No proband matrix either. */
#define GENLIB_SCHEDULE_PHI 0
#define GENLIB_SCHEDULE_SPARSE_PHI 1
#define GENLIB_SCHEDULE_SPARSE_PHI_SYMMETRIC 2
#define GENLIB_SCHEDULE_F 3
#define GENLIB_SCHEDULE_PAIRS 4
int genlib_plan_create_scheduled(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                                 const int32_t *proband, int32_t world, int schedule, genlib_plan **out);
/* The same with the individuals' IDs (by rank; may be NULL).  sparse_phi seeds its queue with
 * founder(isolated_pedigree), which is sorted by ID (src/identify.jl:15-19 via src/compute.jl:335-339):
 * the sparse_phi schedules need the IDs to process the founders in that order.  Without them the
 * founders are taken in rank order, which is the reference's order only when founder IDs ascend with
 * the rank.  Ignored by GENLIB_SCHEDULE_PHI. */
int genlib_plan_create_ex(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids,
                          int32_t n_pro, const int32_t *proband, int32_t world, int schedule, genlib_plan **out);
/* The same, made on a worker thread: the call returns when the pre-pass is done (validation errors are reported
 * here, like above) and the layers follow one by one.  An engine created on such a plan is sized by upper bounds
 * and genlib_engine_run uploads and launches every layer as soon as it is planned -- planning overlaps the device
 * (it is otherwise the largest host-side part of a call; genlib_phi does the same internally).  If a bound turns
 * out too small, genlib_engine_run returns GENLIB_ERESTART (see there).  father / mother / ids / proband must
 * stay valid until the plan is finished: until genlib_engine_run, any genlib_plan_* query other than n_unique /
 * world / schedule, or genlib_plan_destroy returns.  In a multi-rank job every rank takes the same decisions. */
int genlib_plan_create_async(int32_t n, const int32_t *father, const int32_t *mother, const int64_t *ids,
                             int32_t n_pro, const int32_t *proband, int32_t world, int schedule, genlib_plan **out);
int32_t genlib_plan_schedule(const genlib_plan *plan);
void genlib_plan_destroy(genlib_plan *plan);
int32_t genlib_plan_n_unique(const genlib_plan *plan);
int32_t genlib_plan_n_layers(const genlib_plan *plan);
int64_t genlib_plan_capacity(const genlib_plan *plan);
int64_t genlib_plan_row_updates(const genlib_plan *plan);
int genlib_plan_layer_info(const genlib_plan *plan, int32_t layer, genlib_layer_info *out);
/* Device bytes rank `rank` needs for the given numerics. */
int64_t genlib_plan_device_bytes(const genlib_plan *plan, int numerics, int32_t rank);
/* The launch shape of one layer's kernel, as an engine of `rank` with the given numerics would launch it on a
 * device with `sm_count` SMs (host only: no device is needed).  It follows the GENLIB_* tuning variables of the
 * environment like the engine does.  All zero for a layer in which the rank has no couple. */
typedef struct genlib_launch_shape {
    int32_t sw;             /* couples per strip: 8, 16, 32 or 64 (at most 32 with Float64 storage)  */
    int32_t ft;             /* couples per producer item: sw or sw / 2, and 8, 16 or 32             */
    int32_t prod_warps;     /* producer warps per CTA, 4 or 8 (the other warps of 12 consume)      */
    int32_t gangs;          /* independent gangs of CTAs, each on its own strips                    */
    int32_t nbuf;           /* strip buffers in rotation (a multiple of gangs)                      */
    int32_t stages;         /* stages of the producers' shared-memory ring                          */
    int32_t n_strips;       /* strips of the rank's couples                                         */
    int32_t n_pitems;       /* producer items per strip: (sw / ft) x live tiles                     */
    int32_t n_citems;       /* consumer items per strip: the layer's member tiles                   */
    int32_t n_prod;         /* CTAs with producer items                                             */
    int32_t n_cons;         /* CTAs with consumer items                                             */
    int32_t grid;           /* CTAs launched: max(n_prod, n_cons); 0: the layer kernel is skipped   */
    int32_t fast_transpose; /* 1: the producers take the Float32 transpose with immediate offsets   */
    int32_t reserved;
    int64_t smem;           /* dynamic shared memory per CTA, bytes                                 */
} genlib_launch_shape;
int genlib_plan_launch_shape(const genlib_plan *plan, int32_t layer, int numerics, int32_t rank, int32_t sm_count,
                             genlib_launch_shape *out);
/* Schedule export (tests replay it on the CPU to check the planner).  Arrays
 * may be NULL; sizes come from genlib_plan_layer_info.  member_*: n_new
 * entries in family-major order; fam_*: n_fam entries; slots are columns of
 * the frontier matrix; parents are given as slots (-1 = none). */
int genlib_plan_layer_arrays(const genlib_plan *plan, int32_t layer, int32_t *member_ind,
                             int32_t *member_slot, int32_t *member_fam, int32_t *fam_father_slot,
                             int32_t *fam_mother_slot, int32_t *member_owner);
/* Pedigree rank of each member (n_new entries).  For GENLIB_SCHEDULE_PHI this equals member_ind; for
 * the sparse_phi schedules member_ind is the position in sparse_phi's queue. */
int genlib_plan_layer_ranks(const genlib_plan *plan, int32_t layer, int32_t *member_rank);
/* Row sharding of a layer (plans built with world > 1; world == 1 puts everything on rank 0):
 * fam_base / mem_base have world + 1 entries (rank g owns couples [fam_base[g], fam_base[g+1])
 * and members [mem_base[g], mem_base[g+1])); member_lrow is the local row of each member on
 * its owner; the parents of each couple are given as (rank, local row), -1 = none. */
int genlib_plan_layer_shard(const genlib_plan *plan, int32_t layer, int32_t *fam_base, int32_t *mem_base,
                            int32_t *member_lrow, int32_t *fam_father_owner, int32_t *fam_father_lrow,
                            int32_t *fam_mother_owner, int32_t *fam_mother_lrow);
/* Owner rank and local row of whoever is live in each slot before the step (capacity entries). */
int genlib_plan_layer_live_rows(const genlib_plan *plan, int32_t layer, int32_t *live_owner, int32_t *live_lrow);
/* Local rows rank `rank` needs. */
int64_t genlib_plan_rank_rows(const genlib_plan *plan, int32_t rank);
int32_t genlib_plan_world(const genlib_plan *plan);
int genlib_plan_proband_rows(const genlib_plan *plan, int32_t *owner, int32_t *lrow);
/* live_flags: capacity bytes; bit0 = live before the step, bit1 = still live after it. */
int genlib_plan_layer_flags(const genlib_plan *plan, int32_t layer, uint8_t *live_flags);
int genlib_plan_proband_slots(const genlib_plan *plan, int32_t *slots);
/* A 64-bit digest (FNV-1a) of everything the plan holds: the layer table and every index array the engine uploads.
 * Two plans with equal digests run the same schedule; the planner's helper threads (environment
 * GENLIB_PLAN_THREADS) and the streamed hand-over must not change it.  with_bounds = 0 leaves out the frontier
 * width and the rows per rank (a streamed plan keeps the upper bounds its engine was sized with).  CPU only. */
uint64_t genlib_plan_digest(const genlib_plan *plan, int with_bounds);
/* A GENLIB_SCHEDULE_PAIRS plan of the pairs (a[k], b[k]), k < n_pairs (ranks; duplicates and a == b allowed), for
 * `world` ranks.  stream != 0: made on a worker thread and published layer by layer, like genlib_plan_create_async
 * (a, b, father and mother stay valid until the plan is finished).  An index out of range gives GENLIB_EKEY. */
int genlib_plan_create_pairs(int32_t n, const int32_t *father, const int32_t *mother, int64_t n_pairs, const int32_t *a,
                             const int32_t *b, int32_t world, int stream, genlib_plan **out);
/* The reads of a GENLIB_SCHEDULE_PAIRS plan in layer `layer` (just before it), or after the last layer
 * (layer == n_layers), in list order: the list position, the row's slot (the higher-ranked member), the column's slot,
 * the rank that holds the row and its local row there.  Returns their number (any pointer may be NULL), -1 on error. */
int64_t genlib_plan_pair_reads(const genlib_plan *plan, int32_t layer, int64_t *pos, int32_t *row_slot,
                               int32_t *col_slot, int32_t *owner, int32_t *lrow);

/* ---- one-shot: the `gen.phi(ped, probandIDs)` call -------------------------
 * out: n_unique^2 elements of out_dtype (row-major == column-major: symmetric),
 * host memory (pinned or pageable).  n_unique <= n_pro; query it with
 * genlib_plan_n_unique or read stats->n_unique.  device < 0 = current device. */
int genlib_phi(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
               const int32_t *proband, void *out, int out_dtype, int numerics, int device,
               genlib_stats *stats);

/* genlib_phi and genlib_phi_multi plan on a worker thread and hand the layers to the device one by one while the
 * later ones are still being planned (the planner is otherwise the largest host-side part of a call; environment
 * GENLIB_STREAM=0 plans first and runs afterwards).  This diagnostic runs that hand-over WITHOUT a device: a
 * consumer thread copies every layer's slice of the index arrays when it is published, and at the end the copies
 * must equal the finished plan, which in turn must equal the plan made in one piece (only the frontier width
 * differs: a streamed plan keeps the upper bound its engine was sized with).  slack_pct < 0 makes the bound too
 * small on purpose (the planner must then notice, wait for the consumer and finish with exact sizes).
 * layers_streamed / overflowed (nullable) report what happened.  CPU only. */
int genlib_plan_stream_selftest(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                                const int32_t *proband, int32_t world, double slack_pct,
                                int32_t *layers_streamed, int32_t *overflowed);

/* The same call on SEVERAL devices of one box, from one process (SURVEY.md 8(b): `n_dev, devices`):
 * one plan, the frontier's rows sharded over the devices, one host thread per device, NVLink peer
 * access between all of them (cudaDeviceEnablePeerAccess), no MPI / IPC.  Every device assembles a
 * contiguous block of output rows and copies it into `out` over its own PCIe link.  The result is
 * bitwise the single-device one.  n_dev = 1 is genlib_phi on devices[0]. */
int genlib_phi_multi(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                     const int32_t *proband, void *out, int out_dtype, int numerics, int32_t n_dev,
                     const int32_t *devices, genlib_stats *stats);

/* ---- gen.f: inbreeding coefficients (src/compute.jl:500-511) ---------------------------------------------------
 * F[i] = Psi[father(ids[i]), mother(ids[i])], 0 when a parent is missing.  One sweep of the engine over the IDs'
 * ancestors-or-self (GENLIB_SCHEDULE_F, Float64 storage) reads each couple's Psi[father, mother] on the device just
 * before the couple's layer; nothing quadratic in the number of IDs is formed or leaves the device (8 bytes per
 * couple are copied back).  The value is read directly, not as 2 Psi[i, i] - 1.  While kinships fit 53 bits (about
 * 26 generations) every value is exact and equals the reference's Float64 recursion; deeper pedigrees are summed in
 * the depth-layered order of this schedule, so their last Float64 bits may differ.
 * out: n_ids elements of out_dtype in list order (duplicates kept).  An index out of range gives GENLIB_EKEY.  A list
 * without an individual that has both parents gives zeros without a device.  devices[0] < 0 = the current device
 * (one device); several devices shard the frontier rows as genlib_phi_multi does, with the same result bitwise.
 * GENLIB_ENOMEM names the bytes one device needs.  stats->n_unique counts the distinct IDs with both parents. */
int genlib_f(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_ids, const int32_t *ids,
             void *out, int out_dtype, int32_t n_dev, const int32_t *devices, genlib_stats *stats);

/* ---- gen.phi_pairs: the kinship of each pair of a list (src/compute.jl:66-95, one value per pair) --------------
 * out[k] = Psi[a[k], b[k]] for k < n_pairs, in list order (duplicates and reversed pairs kept; Psi[a, a] = 1/2 + 1/2 F_a).
 * One sweep of the engine over the ancestors-or-self of everybody named (GENLIB_SCHEDULE_PAIRS, Float64 storage)
 * reads each pair on the device in the layer after its later-born member's; no matrix is formed.  Every device
 * copies its per-read array back once, 8 bytes per pair, and the host takes each entry from the device that holds the
 * pair's row (stats->d2h_bytes = 8 * n_pairs * n_dev; entries of reads a device does not own are not used).  Both rows of a pair stay in the frontier until it is read, so pairs whose members are born
 * generations apart widen it (GENLIB_ENOMEM, naming the bytes one device needs, when it does not fit).  While
 * kinships fit 53 bits every value is exact; deeper pedigrees follow the depth-layered order of the sums, like
 * genlib_f (genlib_phi_pairs of a couple equals genlib_f of its child bitwise).  An index out of range gives
 * GENLIB_EKEY (a broken pedigree is reported first); n_pairs == 0 returns without a device.  devices as in genlib_f.
 * stats->n_unique counts the distinct individuals named. */
int genlib_phi_pairs(int32_t n, const int32_t *father, const int32_t *mother, int64_t n_pairs, const int32_t *a,
                     const int32_t *b, void *out, int out_dtype, int32_t n_dev, const int32_t *devices,
                     genlib_stats *stats);

/* ---- gen.phiOver: the proband pairs whose kinship reaches a threshold (GENLIB's phiOver(phiMatrix, threshold)) ---
 * M is the matrix genlib_phi returns for the same arguments (numerics, out_dtype); rows and columns are positions in
 * the deduplicated proband list.  (i, j) is selected when i < j and M[i, j] >= threshold, M[i, j] compared as a binary64
 * number (a Float32 entry is widened exactly): the diagonal never, threshold <= 0 every pair, +inf none.  The pairs come
 * in (row, col) order with the stored M[i, j] bit for bit, the same for every number of devices.  The genlib_phi plan
 * runs unchanged (streamed, several devices as genlib_phi_multi); then every device selects from the proband rows it
 * holds, counts per row first, and copies back only its per-row counts and its pairs: no matrix leaves the device.
 *   THE LIBRARY ALLOCATES the result (host memory, exactly n entries of each array, page-locked); release it with
 *   genlib_kinship_pairs_free and nothing else.  n == 0 leaves the pointers NULL.
 *   max_pairs >= 0 and more pairs than that: GENLIB_EOVERFLOW with out->n = the count and nothing allocated or copied.
 *   A NaN threshold gives GENLIB_EINVAL, an index out of range GENLIB_EKEY (a broken pedigree is reported first);
 *   fewer than two distinct probands give n = 0 without a device.  devices[0] < 0 = the current device (one device).
 *   stats as genlib_phi's, but ms_fetch = the selection and the copy back, d2h_bytes = the bytes copied (8 per own
 *   row and device, 4 + element size per pair). */
typedef struct genlib_kinship_pairs {
    int64_t n;            /* pairs selected (or, with GENLIB_EOVERFLOW, pairs that would have been)       */
    int32_t *row, *col;   /* positions in the deduplicated proband list, row < col, (row, col) ascending   */
    void *value;          /* n elements of value_dtype (GENLIB_F32 / GENLIB_F64): M[row, col]              */
    int value_dtype;
} genlib_kinship_pairs;
int genlib_phi_over(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                    double threshold, int64_t max_pairs /* < 0: no limit */, int out_dtype, int numerics,
                    int32_t n_dev, const int32_t *devices, genlib_kinship_pairs *out, genlib_stats *stats);
/* Frees what genlib_phi_over allocated and zeroes the struct (NULL or an empty result: nothing to do). */
int genlib_kinship_pairs_free(genlib_kinship_pairs *pairs);

/* ---- gen.phiMeanGroups: mean kinship within and between groups of probands ---------------------------------------
 * proband[0 .. n_pro) are distinct ranks in list order, group[k] in [0, n_groups) the group of proband[k]; every group
 * has at least one member (n_g of them).  M is the matrix genlib_phi returns for the same list and numerics (Float32
 * or Float64 storage), each entry widened exactly to binary64:
 *   S[i][g]            = sum of M[i, j] over j in group g, j != i (the diagonal is skipped, not subtracted)
 *   proband_mean[i][g] = S[i][g] / (n_g - [group[i] == g])                       (n_pro x n_groups, row-major)
 *   T[h][g]            = sum of S[i][g] over i in group h, added in list order on the host
 *   group_mean[h][g]   = group_mean[g][h] = T[a][b] / (n_a n_b - [a == b] n_a), a = min(h, g), b = max(h, g)
 * A proband alone in its group gives NaN in its own column, a one-member group NaN on the diagonal.  The order of every
 * sum depends only on the list and the groups, so the result is the same bits on any number of devices; where every
 * partial sum is a binary64 number, each mean is the exact rational rounded once.  The genlib_phi plan runs unchanged
 * (streamed, several devices as genlib_phi_multi); then every device reduces the proband rows it holds and copies back
 * n_groups doubles per row: no matrix leaves the device.  The caller owns both outputs.
 *   GENLIB_EINVAL: a null pointer or negative size, unknown numerics, not 1 .. 16 devices, n_groups < 1 with probands,
 *   a group index out of range, a group without a proband, a rank listed twice.  A rank out of range gives GENLIB_EKEY
 *   (a broken pedigree is reported first).  n_pro == 0 writes nothing, n_pro == 1 writes NaN to both outputs, neither
 *   with a device.  devices[0] < 0 = the current device (one device).
 *   stats as genlib_phi's, but ms_fetch = the reduction, the copy back and the host's part, d2h_bytes = 8 n_pro n_groups. */
int genlib_phi_groups(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                      const int32_t *group, int32_t n_groups, int numerics, int32_t n_dev, const int32_t *devices,
                      double *proband_mean, double *group_mean, genlib_stats *stats);

/* ---- gen.phiProduct: the proband kinship matrix times a block of vectors, Y = M X ---------------------------------
 * proband[0 .. n_pro) are distinct ranks in list order; X is n_pro x k binary64, row-major (X[j k + c]), its rows in
 * list order.  M is the matrix genlib_phi returns for the same list and numerics (Float32 or Float64 storage), each
 * entry widened exactly to binary64:
 *   out[i k + c] = sum over ALL j of M[i, j] X[j][c]       (the diagonal included: a true matrix product)
 *   diag[i]      = M[i, i]      (when diag is not null: the sum over j != i is then out[i k + c] - diag[i] X[i][c])
 * both n_pro rows in list order.  Every out[i k + c] is accumulated in binary64 with one FMA per term, in an order that
 * depends only on n_pro: column j goes to partial j mod 256, each partial ascending in j, the 256 partials combined
 * by a fixed tree (genlib_engine_row_sums' order).  So a column of a k-column call is the same bits as a one-column
 * call on that column, and the result does not depend on the number of devices, on which device holds a row or on
 * genlib_engine_phi_product against this call.  Where every product and every partial sum is a binary64 number
 * (kinships that are multiples of 2^-32 and at most 1 times integers with n_pro max|x| <= 2^21), out is the exact
 * sum.  Non-finite entries of X are not checked; they propagate as in IEEE arithmetic.  The genlib_phi plan runs
 * unchanged (streamed, several devices as genlib_phi_multi); then every device multiplies the proband rows it holds
 * (no peer reads) and copies back k (+ 1) doubles per row: no matrix leaves the device.  X takes 8 n_pro k bytes of
 * device memory for the call, next to the engine's arena.  The caller owns X, out and diag.
 *   GENLIB_EINVAL: a null pointer or negative size (k < 0 included), unknown numerics, not 1 .. 16 devices, a rank
 *   listed twice.  A rank out of range gives GENLIB_EKEY (a broken pedigree is reported first).  GENLIB_ENOMEM when
 *   the device has no room for X (the message names the bytes).  n_pro == 0, or k == 0 with diag == NULL, writes
 *   nothing and touches no device.  devices[0] < 0 = the current device (one device).
 *   stats as genlib_phi's, but ms_fetch = the products, the copies back and the host's part, d2h_bytes = 8 n_pro k
 *   (+ 8 n_pro with diag), h2d_bytes includes X once per device. */
int genlib_phi_product(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                       int32_t k, const double *X, int numerics, int32_t n_dev, const int32_t *devices, double *out,
                       double *diag, genlib_stats *stats);

/* ---- handle API: keep the schedule on the device, run, fetch ---------------
 * (what the benchmark and a multi-call Julia session use) */
int genlib_engine_create(const genlib_plan *plan, int numerics, int device, genlib_engine **out);
void genlib_engine_destroy(genlib_engine *eng);
/* Run every layer on the engine's stream and wait.  time_layers != 0 brackets
 * every layer with CUDA events (per-layer ms in genlib_engine_layer_info). */
int genlib_engine_run(genlib_engine *eng, int time_layers);
int genlib_engine_layer_info(genlib_engine *eng, int32_t layer, genlib_layer_info *out);
int genlib_engine_stats(const genlib_engine *eng, genlib_stats *out);
/* Gather proband rows/columns and stream them to host memory.  A sharded engine writes only
 * the rows of the probands it owns, compactly: n_own x n_unique elements, in the order of
 * genlib_engine_own_probands. */
int genlib_engine_fetch(genlib_engine *eng, void *out, int out_dtype);
/* Output rows (proband indices, ascending) held by this rank; returns their number. */
int32_t genlib_engine_own_probands(const genlib_engine *eng, int32_t *index);

/* ---- several GPUs of one box: one process (rank) per GPU, rows sharded ---------------------
 * Every rank builds the SAME plan with world = N, creates its engine, exports the CUDA-IPC
 * handle of its device arena (64 bytes), exchanges handles with its peers by any means and
 * attaches them (rank-major array, `stride` bytes apart).  run / fetch are then collective:
 * every rank must call them.  Kernels read parent rows and push couple-matrix rows directly
 * through the NVLink peer mappings; ranks meet at in-stream barriers twice per layer. */
int genlib_engine_create_dist(const genlib_plan *plan, int numerics, int device, int32_t rank, genlib_engine **out);
int genlib_engine_ipc_export(genlib_engine *eng, void *handle64);
int genlib_engine_ipc_attach(genlib_engine *eng, const void *handles, size_t stride);
/* Mean off-diagonal kinship of the proband matrix, reduced on the device
 * (consumer of the path: phiMean, src/compute.jl:454-459): binary64 accumulation in a FIXED order
 * (columns ascending per thread, fixed tree per row, rows in proband order), so the value is
 * reproducible.  One rank only; sharded engines combine genlib_engine_row_sums. */
int genlib_engine_phi_mean(genlib_engine *eng, double *out);
/* Per own proband row (genlib_engine_own_probands order): out[2 r] = sum of the row over all proband
 * columns, out[2 r + 1] = its diagonal entry.  Adding the rows of all ranks in proband order gives
 * the same bits whatever the number of ranks. */
int genlib_engine_row_sums(genlib_engine *eng, double *out);
/* gen.phiProduct on an engine that has run: Y = M X for the rows of the probands this rank holds, out[r k + c] and
 * diag[r] (nullable) for its r-th own proband (genlib_engine_own_probands order; one rank: list order).  X is
 * n_unique x k, row-major, its rows in the plan's proband order.  The bits are genlib_phi_product's, whatever the
 * rank.  Not collective, no peer reads; call it any number of times without running the layers again.  Errors as
 * genlib_phi_product's where they apply, and GENLIB_EINVAL before genlib_engine_run. */
int genlib_engine_phi_product(genlib_engine *eng, int32_t k, const double *X, double *out, double *diag);
/* Debug/test: stop genlib_engine_run after `n_layers` layers (< 0: no limit). */
int genlib_engine_set_layer_limit(genlib_engine *eng, int32_t n_layers);
/* Debug/test: copy the frontier entry block [slots x slots] (as double). */
int genlib_engine_read_block(genlib_engine *eng, int32_t n_slots, const int32_t *slots, double *out);

/* ---- gen.gc: the proband x ancestor genetic-contribution matrix (SURVEY.md 2: src/compute.jl:518-595) -----
 *   G[p, a] = sum over descent paths a -> ... -> p of (1/2)^(path length)
 *           = [p == a] + 1/2 G[father(p), a] + 1/2 G[mother(p), a]        (a missing parent adds 0)
 * Rows follow `proband`, columns follow `ancestor`; duplicates are KEPT (a repeated rank gives a repeated
 * row / column).  Every value is a sum of powers of 1/2: while no path from a listed ancestor to a listed
 * proband is longer than 52 edges the result is exact (whatever the order of the sums), deeper pedigrees get
 * the fixed summation order of DESIGN.md 2b.  The engine propagates the narrower side (DIRECTION below;
 * environment GENLIB_GC_DIRECTION=descend|ascend overrides the rule) over the individuals that lie on a path
 * from a listed ancestor to a listed proband. */
#define GENLIB_GC_DESCEND 0 /* columns = unique ancestors, rows go down the generations              */
#define GENLIB_GC_ASCEND 1  /* columns = unique probands, rows go up; the output is the transpose  */
typedef struct genlib_gc_stats {
    int32_t n_pro, n_anc;        /* output shape (duplicates kept)                                  */
    int32_t n_layers, direction;
    int64_t rows, inputs;        /* active rows computed, input edges read                          */
    int64_t width, capacity;     /* columns propagated (all devices), peak live frontier rows       */
    int64_t device_bytes;        /* largest per-device allocation                                   */
    double alg_bytes;            /* required traffic, summed over devices: (input rows read +       */
                                 /* frontier rows written + output rows written) x columns x 8      */
                                 /* (genlib_rec: x 16-byte-padded 64-column words x 8; the row sums */
                                 /* of genlib_occ and genlib_rec add one read of the output block)  */
    double ms_plan, ms_kernels, ms_fetch; /* ms_kernels: CUDA events, slowest device                */
    int64_t d2h_bytes;
    int32_t kernel_launches, n_dev;
} genlib_gc_stats;
/* out: n_pro x n_anc elements of out_dtype, row-major, or column-major when col_major != 0 (what a Julia
 * Matrix is); host memory (pinned or pageable).  The column side's list is split into n_dev contiguous,
 * balanced ranges, one per device (one host thread each, no peer access); every device writes its own
 * rectangular block of `out` and the result is bitwise the one-device result.  devices[g] < 0 = the current
 * device.  An empty list gives an empty matrix without a device.  GENLIB_ENOMEM names the bytes one device
 * needs (more devices need less each). */
int genlib_gc(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
              int32_t n_anc, const int32_t *ancestor, void *out, int out_dtype, int col_major, int32_t n_dev,
              const int32_t *devices, genlib_gc_stats *stats);
/* The schedule alone (host only; tests replay it).  Unique probands / ancestors are numbered in order of
 * first occurrence; `columns` are the unique ancestors (descend) or probands (ascend), the output block holds
 * one row per unique target (the other side).  Per layer: row_ind = pedigree rank, row_slot = frontier slot
 * (-1: nobody reads the row later), row_seed = the row's own column (-1: none), row_out = output-block row
 * (-1: not a target), in_ptr (n_rows + 1 entries, from 0) / in_slot = the frontier slots of the inputs, in
 * the order they are added.  genlib_gc_plan_info reports no timings; device_bytes is for one device. */
typedef struct genlib_gc_plan genlib_gc_plan;
int genlib_gc_plan_create(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro,
                          const int32_t *proband, int32_t n_anc, const int32_t *ancestor, genlib_gc_plan **out);
void genlib_gc_plan_destroy(genlib_gc_plan *plan);
int genlib_gc_plan_info(const genlib_gc_plan *plan, genlib_gc_stats *out);
int genlib_gc_plan_layer(const genlib_gc_plan *plan, int32_t layer, int32_t *n_rows, int64_t *n_inputs);
int genlib_gc_plan_layer_arrays(const genlib_gc_plan *plan, int32_t layer, int32_t *row_ind, int32_t *row_slot,
                                int32_t *row_seed, int32_t *row_out, int64_t *in_ptr, int32_t *in_slot);

/* ---- gen.gcGroups: genetic contributions summed over groups of probands and/or ancestors (DESIGN.md 2i) -------
 * Each side is a list of ranks as in genlib_gc (group pointer null: list order, duplicates kept, one row / column
 * per entry) or GROUPED: distinct ranks, rank k in group pro_group[k] (anc_group[k]) in [0, n_groups), every group
 * non-empty.  With G = genlib_gc's matrix for the same lists,
 *   out[r, c] = sum over p in row r, a in column c of G[p, a]                  (R x C float64)
 * R = n_pro_groups if the probands are grouped, else n_pro; C likewise.  Row-major, or column-major when
 * col_major != 0.  G is linear, so the engine propagates one column per group of the column side (the narrower
 * side, counting a grouped side's groups and an ungrouped side's unique entries; descend on ties;
 * GENLIB_GC_DIRECTION overrides) and, when the other side is grouped, sums its output rows per group on the device
 * (members in list order, no atomics); only R x C doubles leave the devices.  Every G[p, a] is a multiple of 2^-L
 * (L = the longest listed path) and every sum adds non-negative values: while every partial sum is a multiple of
 * 2^-L below 2^(53 - L) the result is the exact sum, in either direction and on any device count; otherwise the
 * order is fixed (the same bits on a repeat and on any device count; the two directions may differ in the last
 * bits).  Devices as genlib_gc.
 *   GENLIB_EINVAL: a null pointer or negative size, neither side grouped (that is genlib_gc), a group index out of
 *   range, an empty group, a rank listed twice on a grouped side, no device.  A rank out of range gives GENLIB_EKEY
 *   (a broken pedigree is reported first).  R == 0 or C == 0 writes nothing, without a device.
 *   stats: n_pro / n_anc = R / C, width = columns propagated, d2h_bytes = 8 R C, alg_bytes = the plan's byte model
 *   plus one read of the output block when the target side is summed per group. */
int genlib_gc_groups(int32_t n, const int32_t *father, const int32_t *mother,
                     int32_t n_pro, const int32_t *proband, const int32_t *pro_group, int32_t n_pro_groups,
                     int32_t n_anc, const int32_t *ancestor, const int32_t *anc_group, int32_t n_anc_groups,
                     double *out, int col_major, int32_t n_dev, const int32_t *devices, genlib_gc_stats *stats);
/* genlib_gc_groups' schedule alone (host only), read with genlib_gc_plan_info / _layer / _layer_arrays.  A grouped
 * column side has one column per group (row_seed = the member's group); a grouped target side keeps one output-block
 * row per member, numbered in list order, and the sums per group follow the layers. */
int genlib_gc_groups_plan_create(int32_t n, const int32_t *father, const int32_t *mother,
                                 int32_t n_pro, const int32_t *proband, const int32_t *pro_group, int32_t n_pro_groups,
                                 int32_t n_anc, const int32_t *ancestor, const int32_t *anc_group, int32_t n_anc_groups,
                                 genlib_gc_plan **out);

/* ---- gen.occ / gen.rec: descent-path counts and proband coverage (SURVEY.md 2: src/describe.jl:133-234) --------
 * The same plan and devices as genlib_gc (GENLIB_GC_DIRECTION applies), with the 1/2 dropped:
 *   O[a, p] = number of descent paths a -> ... -> p (the empty path when a == p)
 *           = [p == a] + O[a, father(p)] + O[a, mother(p)]                (a missing parent adds 0)
 * ROWS ARE ANCESTORS (the transpose of genlib_gc's matrix); duplicates of either list are kept.
 * Counts are added with saturation at 2^63, which is associative and commutative: every result is bitwise
 * independent of the direction, the order of the sums and the number of devices.  A returned count or row
 * sum that does not fit an int64 fails with GENLIB_EOVERFLOW; the message names the smallest offending
 * (ancestor position, proband position) pair in list order (for a row sum: the ancestor and its first
 * listed descendant), the same on every run and for every device count.
 *   GENLIB_OCC_IND:   out = n_anc x n_pro int64, row-major, or column-major when col_major != 0
 *   GENLIB_OCC_TOTAL: out = n_anc int64, the row sums over the proband list (duplicates counted), reduced on
 *                     the devices: the matrix never leaves them (col_major is ignored)
 * genlib_rec: out = n_anc int64, the number of proband list entries that descend from the ancestor, the
 * ancestor itself included (= count(O[a, :] .> 0)); reachability rows of 64 columns per word, reduced on the
 * devices; it cannot overflow.  Empty lists give an empty (or zero) result without a device. */
#define GENLIB_OCC_IND 0
#define GENLIB_OCC_TOTAL 1
int genlib_occ(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
               int32_t n_anc, const int32_t *ancestor, int64_t *out, int type, int col_major, int32_t n_dev,
               const int32_t *devices, genlib_gc_stats *stats);
int genlib_rec(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
               int32_t n_anc, const int32_t *ancestor, int64_t *out, int32_t n_dev, const int32_t *devices,
               genlib_gc_stats *stats);

/* ---- gen.findMRCA / gen.findDistance: most recent common ancestors and minimum meioses ------------------------
 * (SURVEY.md 2: src/identify.jl _findMRCA :101-107, _findMinDistanceMRCA :114-118, GenMatrix :129-133,
 * findMRCA :153-161; src/describe.jl _get_paths :241-258, findDistance :296-300)
 * The reference enumerates every descent path and keeps the shortest; here the same plan and devices as
 * genlib_gc (GENLIB_GC_DIRECTION applies) propagate shortest distances in the (min, +1) semiring:
 *   d(a, p) = number of parent -> child edges on the shortest descent path a -> ... -> p, d(p, p) = 0
 *           = min(d(a, father(p)), d(a, mother(p))) + 1                     (a missing parent: no path)
 * Distances are uint16 on the device; a plan of 0xFFFF layers or more fails with GENLIB_EOVERFLOW before any
 * launch (a distance is below the plan's layer count), so a distance is never confused with "no path".
 * The minimum is order-free: the result is bitwise independent of the direction and the number of devices.
 * genlib_meioses: out = n_pro x n_anc int64, out[i, j] = d(ancestor[j], proband[i]), -1 where proband[i] does
 * not descend from (and is not) ancestor[j]; row-major, or column-major when col_major != 0; duplicates of
 * either list are kept.  Stats and alg_bytes as genlib_gc with 2 bytes per (16-byte padded) column. */
int genlib_meioses(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_pro, const int32_t *proband,
                   int32_t n_anc, const int32_t *ancestor, int64_t *out, int col_major, int32_t n_dev,
                   const int32_t *devices, genlib_gc_stats *stats);
/* genlib_mrca: the most recent common ancestors of the ranks `ids` (duplicates allowed).  A common ancestor is
 * a PROPER ancestor of every distinct ID (an individual is not its own ancestor: for [parent, child] the
 * MRCAs are the parent's parents); an MRCA is a common ancestor none of whose children is common (equivalent
 * to "none of whose descendants is common", DESIGN.md 2d).  `mrca` has room for n ranks; it receives *n_mrca
 * ranks in ascending order.  One genlib_rec pass on the devices (pro = the distinct IDs, anc = their
 * ancestors-or-self) decides who is common; everything else is O(n) on the host.  `stats` are the rec pass's.
 * No ID gives no MRCA without a device. */
int genlib_mrca(int32_t n, const int32_t *father, const int32_t *mother, int32_t n_ids, const int32_t *ids,
                int32_t *mrca, int32_t *n_mrca, int32_t n_dev, const int32_t *devices, genlib_gc_stats *stats);

#ifdef __cplusplus
}
#endif
#endif /* GENLIB_CUDA_H */
