// layer_kernel.cuh -- ONE persistent sm_100a kernel per generation step.
//
// A step (one cut-vertex step of the reference, src/compute.jl:276-302) turns the frontier Psi into
//   phi[i, j] = 1/2 (1/2 Psi[f_hi, f_lo] + 1/2 Psi[f_hi, m_lo]) + 1/2 (1/2 Psi[m_hi, f_lo] + 1/2 Psi[m_hi, m_lo])
// for two new individuals (hi = the one with the larger rank is climbed first, compute.jl:130-147) and
//   phi[i, c] = 1/2 Psi[f_i, c] + 1/2 Psi[m_i, c]    against a carried individual c (compute.jl:111-126).
// Full siblings share everything but the diagonal, so the work is done per COUPLE (F = (f, m)).
//
// The four frontier entries of a couple pair sit at the crossing of two parent ROWS (contiguous) and two
// parent COLUMNS (scattered): the step is a gather along both axes.  It is done as two coalesced passes
// through a transposed scratch -- but the scratch never leaves the 126 MB L2:
//
//   strip     = up to 64 of this rank's couples; the strips are processed in order.
//   CTA       = one per SM, 12 warps: PW PRODUCER warps and 12 - PW CONSUMER warps, 4 + 8 for layers without
//               carried individuals and 8 + 4 for layers with them.
//   PRODUCER  warps read the strip's parent rows -- TMA bulk copies into a shared-memory ring that runs on
//             across strips, from local HBM or a peer's over NVLink, handed from warp to warp with full /
//             empty mbarriers (no CTA barrier) -- and write them transposed and interleaved,
//                 Q[p][F] = (Psi[f_F, p], Psi[m_F, p])          for every live column p,
//             into one of a few strip buffers that stay in L2; where the step carries individuals over they also
//             write, from the same staged rows, the members' rows against the carried columns and the mirror
//             image, the members' columns in the carried individuals' rows.
//   CONSUMER  warps take tiles of couples G (ALL couples of the layer), stage Q[f_G][strip], Q[m_G][strip]
//             -- two contiguous segments per couple, L2 hits -- which hold all four entries of every (F, G)
//             pair in BOTH groupings,
//                 a = (Psi[f_F,f_G], Psi[m_F,f_G]), c = (Psi[f_F,m_G], Psi[m_F,m_G])
//                 F climbed: hs(hs(a.x, c.x), hs(a.y, c.y))     G climbed: hs(hs(a.x, a.y), hs(c.x, c.y))
//             (hs(x, y) = 1/2 x + 1/2 y, one binary64 rounding), round ONCE to the storage type
//             (compute.jl:296) and write the strip members' rows over the tile's member columns, picking
//             the grouping by rank; the diagonal is 1/2 + 1/2 Psi[f, m] (compute.jl:148-155).
//
// Every entry of the step is written exactly once, in contiguous row segments, by the rank that owns the
// row; nothing but stored frontier rows crosses NVLink.  DRAM sees the compulsory traffic only: the parent
// rows once, the new rows once.
//
// Flow control is static: the items of a role (producer: column tiles of a strip, consumer: member tiles) are
// numbered strip after strip and dealt round-robin to the CTAs.  A layer whose strips hold too few items to occupy
// every SM splits the CTAs into GANGS that work on different strips side by side (gang g takes strips g, g + G, ...):
// the hand-over of a strip then involves 1/G of the CTAs, G of them overlap.  Every producer warp and the consumer
// warps of every CTA count themselves off on the strip's counter when their share is done; consumers start a strip
// when all producers have counted off, producers reuse a strip buffer when all consumers of the strip that used it
// before have.  All CTAs are resident (one per SM), and a wait that lasts seconds raises the layer's error word
// instead of hanging the device.
//
// The kernel entry sets up the CTA's shared words (LayerShared) and hands every warp to one of the two roles,
// Producer and Consumer: each is a struct whose run() is its item loop, written as a sequence of named steps.
#pragma once
#include <type_traits>

#include "kernels.cuh"
#if defined(GENLIB_CHECK)
#include <cassert>
#define CHECK(cond) assert(cond)
#elif defined(GENLIB_SOFTCHECK)       // record the source line of the FIRST violated bound in the layer's error word, go on
#define CHECK(cond) do { if (!(cond)) atomicCAS(S.err, 0, 100000 + __LINE__); } while (0)
#else
#define CHECK(cond) do { } while (0)
#endif

namespace genlib {

// A CTA has 12 warps.  How many of them produce is a template parameter of the kernel (PW): 4 producer warps and 8
// consumer warps for layers without carried individuals (C3, C4: the two roles take the same time), 8 and 4
// where the producers also write the members' rows against the carried columns and their mirror image (C5,
// genea140: the producers set the pace there and the consumers mostly wait).
constexpr int kLayerWarps = 12, kLayerThreads = kLayerWarps * 32;
__host__ __device__ constexpr int cons_warps(int pw) { return kLayerWarps - pw; }
constexpr int kMaxStrip = 64;                   // couples per strip (upper bound of StripArgs::sw)
constexpr int kVPitch = kMaxTileFam + 1;        // row pitch of the staged couple tile (65: conflict-free)
constexpr int kMaxStages = 4;
constexpr int kSyncStride = 16;                 // ints per strip in StripArgs::sync: every counter has its own 32-byte sector
// The shapes whose producers take the Float32 transpose with immediate offsets (Producer::transpose); every other
// shape takes the generic one.
__host__ __device__ constexpr bool fast_transpose_shape(int esize, int sw, int ft) { return esize == 4 && ft == 32 && (sw == 64 || sw == 32); }

struct StripArgs {
    int32_t sw;          // strip width: couples per strip (8, 16, 32 or 64)
    int32_t ft;          // couples per producer item (8, 16 or 32; sw or sw / 2)
    int32_t n_strips;    // strips of this rank's couples
    int32_t nbuf;        // strip buffers in rotation (a multiple of gangs: a buffer stays with one gang)
    int32_t stages;      // ring stages
    int32_t gangs;       // the CTAs work in this many independent gangs: gang g = CTA index mod gangs takes strips g, g + gangs, ...
    int32_t n_prod;      // CTAs whose producer warps have items (0 when nothing is live; a multiple of gangs)
    int32_t n_cons;      // CTAs whose consumer warps have items (a multiple of gangs)
    int32_t n_pitems;    // producer items per strip: (sw / ft) * live tiles
    int32_t n_citems;    // consumer items per strip: the layer's member tiles
    int32_t discard;     // 1: a consumer drops the strip-buffer rows it was the only one to read from L2 (no write-back of dead lines)
    int32_t ring_off;    // byte offset of the producer ring in dynamic shared memory (after the consumer's part)
    int64_t qstride;     // pairs per strip buffer (live tiles * kPTile * sw)
    void *Q;             // strip buffers
    int32_t *sync;       // strip s: [16 s] producer CTAs done, [16 s + 8] consumer CTAs done (a 32-byte sector each)
    int32_t *err;        // the layer's error word
    const int32_t *live_tiles;   // the live tiles of the layer's slot range: index | kTileCarried
    long long timeout_cycles;
    long long *prof;             // -DGENLIB_PROFILE: 8 cycle counters per CTA and role (else unused)
};

// Polls read the counters RELAXED and acquire once when the wait is over: an acquire load invalidates the SM's whole
// L1 (SASS CCTL.IVALL) every time it is issued, which a spinning thread does to every other warp of its SM (ncu: the
// CCTL.IVALL of the wait loops held 17 % of all stall samples of a C5 layer).  The closing acquire is a load, not a
// fence: a fence also waits for the thread's own outstanding row stores.
__device__ __forceinline__ int ld_relaxed_gpu(const int *p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int ld_acquire_gpu(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// Waits (one thread) until *counter reaches target.  A wait that lasts longer than timeout_cycles sets the layer's
// error word (genlib_engine_run then fails with GENLIB_ECUDA); once it is set nobody waits any more, so a broken
// schedule drains in seconds instead of hanging the device.
__device__ __forceinline__ void spin_wait(const int *counter, int target, int *err, long long timeout_cycles) {
    const long long t0 = clock64();
    unsigned polls = 0;
    while (ld_relaxed_gpu(counter) < target) {
        if (clock64() - t0 > timeout_cycles) { atomicCAS(err, 0, 1); break; }
        if ((++polls & 31u) == 0 && ld_relaxed_gpu(err) != 0) break;   // somebody else gave up: drain
        __nanosleep(100);
    }
    ld_acquire_gpu(counter);
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// The two groupings of the four frontier entries of a couple pair (see the header).  hs(x, y) = RN(x/2 + y/2)
// = RN(x + y) / 2 (scaling by a power of two commutes with rounding: binary64 cannot underflow here), so
// hs(hs(a, b), hs(c, d)) = RN(RN(a + b) + RN(c + d)) / 4 bit for bit: three additions and one exact product.
template <typename T, bool STORED>
__device__ __forceinline__ void couple_pair(double ax, double ay, double cx, double cy, T &f_climbed, T &g_climbed) {
    if constexpr (STORED) {      // sparse_phi: every intermediate kinship is a stored Float32 (compute.jl:331, 363-395)
        f_climbed = (T)half_sum_stored((double)(T)half_sum_stored(ax, cx), (double)(T)half_sum_stored(ay, cy));
        g_climbed = (T)half_sum_stored((double)(T)half_sum_stored(ax, ay), (double)(T)half_sum_stored(cx, cy));
    } else {
        f_climbed = (T)__dmul_rn(0.25, __dadd_rn(__dadd_rn(ax, cx), __dadd_rn(ay, cy)));
        g_climbed = (T)__dmul_rn(0.25, __dadd_rn(__dadd_rn(ax, ay), __dadd_rn(cx, cy)));
    }
}

// consumer: staged parent-row segments of a couple tile (2 x kMaxTileFam rows x sw pairs), Va | Vb, a ring of
// three tiles' metadata, the strip's member rows (row descriptors)
inline size_t layer_consumer_bytes(int sw, size_t es, int prod_warps) {
    const size_t b = (size_t)2 * kMaxTileFam * sw * 2 * es + (size_t)2 * sw * kVPitch * es + (size_t)3 * 4 * kMTile * 4 +
                     (size_t)cons_warps(prod_warps) * 32 * 16;
    return (b + 127) / 128 * 128;
}

// Optional cycle accounting per CTA, role and phase (-DGENLIB_PROFILE): one thread's clock64 between phase
// marks (producer warp 0 / consumer thread 0), summed into S.prof[(2 * blockIdx.x + role) * 8 + phase].
#ifdef GENLIB_PROFILE
#define PROF_DECL long long prof_t = clock64(), prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define PROF_MARK(ph) do { const long long now_ = clock64(); prof_acc[ph] += now_ - prof_t; prof_t = now_; } while (0)
#define PROF_FLUSH(role, who) do { if ((who) && S.prof) for (int i_ = 0; i_ < 8; i_++) S.prof[((size_t)blockIdx.x * 2 + (role)) * 8 + i_] = prof_acc[i_]; } while (0)
#else
#define PROF_DECL
#define PROF_MARK(ph) do { } while (0)
#define PROF_FLUSH(role, who) do { } while (0)
#endif

// The items of a role are numbered strip after strip of a gang and dealt round-robin: item n = (s / G) NI + it of
// gang g belongs to participant n mod NP of the gang (a CTA's producer warps, or its consumer warps).
struct Item { int s, it; };                                        // strip, index in the strip
struct ItemOrder {
    int NS, G, NI, NP;                                             // strips, gangs, items per strip, participants per gang
    __device__ __forceinline__ Item first(int gang, int k) const { return settle(Item{gang, k}); }
    __device__ __forceinline__ Item next(Item c) const { c.it += NP; return settle(c); }
    __device__ __forceinline__ Item settle(Item c) const { while (c.s < NS && c.it >= NI) { c.it -= NI; c.s += G; } return c; }
};

// The CTA's static shared memory: what the roles keep besides the dynamic part.
template <int PW>
struct LayerShared {
    unsigned long long full[kMaxStages];    // producer ring: "stage filled" (bulk copies landed)
    unsigned long long empty[kMaxStages];   // producer ring: "stage read by every producer warp"
    unsigned long long cbar;                // consumer: "tile segments landed"
    int ptinfo[PW][kMaxStages];             // producer: live_tiles entry of the item in a ring slot
    int pcount[8];                          // producer: warps of this CTA done with strip s (slot s & 7)
    int cdone;                              // producer: strips below this one are known to be consumed
    int ready;                              // consumer: the strip of the next item is produced
};

// =============== producer warp: parent rows -> Q[p][F] pairs (+ member rows x carried columns) ===============
// The PW warps share the ring and nothing else: warp w issues the copies of rows [w rpw, (w + 1) rpw) of
// every item and transposes columns [w kProdCols, (w + 1) kProdCols) of it.  A dependency that does not
// arrive in time sets the layer's error word.
template <typename T, bool STORED, int PW>
struct Producer {
    using P2 = std::conditional_t<sizeof(T) == 4, float2, double2>;   // a (father, mother) pair of strip-buffer entries
    static constexpr int kProdCols = kPTile / PW;                  // columns of a tile that one producer warp transposes
    static constexpr uint32_t kLive4 = 0x01010101u * kFlagLive;
    static_assert(kProdCols % 4 == 0 && kProdCols <= 32, "role split");
    // members of the couples whose rows this warp writes against carried columns: lane j < npt cpw holds couple
    // (pt = j / cpw, qd = j % cpw) of strip s: its member range and the rows of its first two members
    struct MemInfo { int mb, me, lr0, lr1; };
    // the same members as COLUMNS of the carried individuals' rows (the mirror image of the block above): the members
    // of the ft couples of either half of strip s, in member order (= slot order), one per lane and chunk of 32:
    // column slot | couple within the half << 24 (-1: none); the first two chunks of a half are kept in registers
    // (a strip ahead), halves with more members than 64 look the rest up per item
    struct MirInfo { int e0a, e1a, na, ba, e0b, e1b, nb, bb; };   // chunks 0 / 1, members, first member: halves a / b
    T *const A; const int64_t ld; const PeerTable &PT; const LayerArgs &L; const StripArgs &S; LayerShared<PW> &sh;
    unsigned char *const ring;
    const int lane = threadIdx.x & 31, pw = (int)(threadIdx.x >> 5) - cons_warps(PW);
    const int sw = S.sw, ft = S.ft, NS = S.n_strips, G = S.gangs;
    const int gang = blockIdx.x % G;                               // this CTA is producer blockIdx.x / G of its gang
    const ItemOrder items{NS, G, S.n_pitems, S.n_prod / G};
    int *const err = S.err;
    int *const done_p = S.sync, *const done_c = S.sync + 8;        // done_p[kSyncStride * s], done_c[kSyncStride * s]
    P2 *const Qall = static_cast<P2 *>(S.Q);
    const int npt = sw / ft, lnpt = npt > 1 ? 1 : 0;               // items per live tile: 1 or 2
    const int RB = kPTile * (int)sizeof(T) + 16, STAGE = 2 * ft * RB;
    const unsigned ROWB = kPTile * (unsigned)sizeof(T);
    const unsigned rbase = (unsigned)__cvta_generic_to_shared(ring);
    const unsigned full0 = (unsigned)__cvta_generic_to_shared(&sh.full[0]), empty0 = (unsigned)__cvta_generic_to_shared(&sh.empty[0]);
    const int rpw = 2 * ft / PW;                                   // rows of an item whose copies this warp issues
    const int myrow = pw * rpw + lane;                             // (lanes < rpw) 0 .. 2 ft - 1: fathers, then mothers
    const bool issuer = lane < rpw, mo = myrow >= ft;
    const int myf = mo ? myrow - ft : myrow;
    const unsigned long long read_once = policy_evict_first();     // the parents' rows pass through L2 once
    const int cpw = ft / PW;                                       // couples of an item whose member rows this warp writes
    Item ic = items.first(gang, blockIdx.x / G), wc = ic;          // issue cursor (copies under way), write cursor
    int rs = -1;                                                   // strip whose rows are in rp0 / rp1; strip rs + G: raw in no / nl
    const T *rp0 = nullptr, *rp1 = nullptr;
    int no0 = -1, no1 = -1, nl0 = 0, nl1 = 0;
    int islot = 0;                                                 // ring slot of the next issue ...
    unsigned iuse = 0;                                             // ... and how often it has been filled before
    int itile = ic.s < NS ? S.live_tiles[ic.it >> lnpt] : 0;       // live_tiles entry of the item at the issue cursor
    int cslot = 0;                                                 // ring slot of the item at the write cursor ...
    unsigned cuse = 0;                                             // ... and how often it has been filled before
    int cur = -1;                                                  // strip this warp is writing
    int ms = -1;                                                   // strip of cmi / cmr; nmi / nmr: strip ms + G
    MemInfo cmi = mem_info(NS), nmi = cmi;
    MirInfo cmr = mir_info(NS), nmr = cmr;
    int tinfo = 0;                                                 // live_tiles entry of the item at the write cursor
    uint32_t live8 = 0u;                                           // its flags (tile_flags)
    T *col_row = nullptr;                                          // lane = column of the warp's share: where its row lives
    __device__ __forceinline__ void run() {
        PROF_DECL
        for (int n = 0; n < S.stages - 1; n++) issue();
        tinfo = wc.s < NS ? S.live_tiles[wc.it >> lnpt] : 0;
        live8 = wc.s < NS ? tile_flags(tinfo) : 0u;
        col_row = wc.s < NS ? tile_rows(tinfo) : nullptr;
        while (wc.s < NS) {
            if (wc.s != cur) {
                count_off(wc.s);
                PROF_MARK(0);
                wait_consumed(wc.s - S.nbuf);                      // the strip that used this buffer before
                PROF_MARK(1);
                if (L.any_carried) strip_members();
            }
            if (!mbar_wait(full0 + 8u * cslot, cuse & 1u)) atomicCAS(err, 0, 2);
            PROF_MARK(2);
            issue();                                               // refills the slot everybody left an item ago
            PROF_MARK(3);
            const int pt = wc.it & (npt - 1), lt = wc.it >> lnpt;
            const unsigned char *st = ring + cslot * STAGE;
            transpose(st, Qall + (size_t)(wc.s % S.nbuf) * S.qstride, pt, lt);
            PROF_MARK(4);
            if (tinfo & kTileCarried) carried_rows(st, pt);
            PROF_MARK(5);
            if (tinfo & kTileCarried) mirror_columns(st, pt);
            PROF_MARK(6);
            next_item();
        }
        count_off(NS);
        PROF_MARK(0);
        PROF_FLUSH(0, pw == 0 && lane == 0);
    }
    // Strip t is consumed (the consumer warps of every CTA have counted off; they do so in strip order): lane 0 asks
    // the CTA's note first, then the counter in L2 -- whoever learns it leaves a note for the other producer warps.
    __device__ __forceinline__ void wait_consumed(int t) {
        if (lane == 0 && t >= 0) {
            if (*reinterpret_cast<volatile int *>(&sh.cdone) <= t) {
                spin_wait(done_c + kSyncStride * t, S.n_cons / G, err, S.timeout_cycles);
                atomicMax(&sh.cdone, t + 1);
            }
            __threadfence_block();
        }
        __syncwarp();
    }
    // This warp's share of the strips of its gang below `upto` is done; the CTA's last warp tells everybody.  Lane 0
    // releases the warp's pairs (ordinary stores that the consumers read with bulk copies: ordered against the async
    // proxy by every writer) at gpu scope before it counts, the last warp once more after it has seen the others' counts.
    __device__ __forceinline__ void count_off(int upto) {
        for (int s = cur < 0 ? gang : cur; s < upto; s += G) {
            asm volatile("fence.proxy.async.global;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                __threadfence();
                if (atomicAdd(&sh.pcount[(s / G) & 7], 1) == PW - 1) {
                    sh.pcount[(s / G) & 7] = 0;
                    __threadfence();
                    atomicAdd(done_p + kSyncStride * s, 1);
                }
            }
        }
        cur = upto;
    }
    // the parent row this lane copies for items of strip s, half pt (nullptr: unknown parent, or not an issuer)
    // (fetched raw a strip ahead -- no branch on what is loaded -- and resolved when the strip starts)
    __device__ __forceinline__ void row_raw(int s, int pt, int &o, int &lr) const {
        o = -1; lr = 0;
        const int Fl = s * sw + pt * ft + myf;
        if (issuer && s < NS && Fl < L.own_nf) {
            const int F = L.own_f0 + Fl;
            o = mo ? L.fam_pm_owner[F] : L.fam_pf_owner[F];
            lr = mo ? L.fam_pm_lrow[F] : L.fam_pf_lrow[F];
        }
    }
    __device__ __forceinline__ const T *row_ptr(int o, int lr) const {
        return o >= 0 ? static_cast<const T *>(PT.A[o]) + (int64_t)lr * ld + L.rt_lo : nullptr;
    }
    __device__ __forceinline__ MemInfo mem_info(int s) const {
        MemInfo m; m.mb = 0; m.me = 0; m.lr0 = 0; m.lr1 = 0;
        if (L.any_carried && lane < npt * cpw && s < NS) {
            const int pt = lane / cpw, qd = lane - pt * cpw;
            const int Fl = s * sw + pt * ft + pw * cpw + qd;
            if (Fl < L.own_nf) {
                m.mb = L.fam_start[L.own_f0 + Fl]; m.me = L.fam_start[L.own_f0 + Fl + 1];
                if (m.me > m.mb) m.lr0 = L.mem_lrow[m.mb];
                if (m.me > m.mb + 1) m.lr1 = L.mem_lrow[m.mb + 1];
            }
        }
        return m;
    }
    __device__ __forceinline__ int mir_entry(int F0h, int mb, int nm, int i) const {   // member i of a half that starts at couple F0h, member mb
        return i < nm ? (L.mem_slot[mb + i] | ((L.mem_fam[mb + i] - F0h) << 24)) : -1;
    }
    __device__ __forceinline__ MirInfo mir_info(int s) const {
        MirInfo m; m.e0a = m.e1a = m.e0b = m.e1b = -1; m.na = m.nb = m.ba = m.bb = 0;
        if (L.any_carried && s < NS) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int Fl = s * sw + h * ft;
                if (h < npt && Fl < L.own_nf) {
                    const int F0h = L.own_f0 + Fl, mb = L.fam_start[F0h], nm = L.fam_start[L.own_f0 + min(Fl + ft, L.own_nf)] - mb;
                    const int e0 = mir_entry(F0h, mb, nm, lane), e1 = mir_entry(F0h, mb, nm, 32 + lane);
                    if (h == 0) { m.e0a = e0; m.e1a = e1; m.na = nm; m.ba = mb; } else { m.e0b = e0; m.e1b = e1; m.nb = nm; m.bb = mb; }
                }
            }
        }
        return m;
    }
    // the member info of the strip the warp enters (fetched a strip ahead when it follows the last one) and of its next
    __device__ __forceinline__ void strip_members() {
        const bool seq = ms >= 0 && wc.s == ms + G;
        cmi = seq ? nmi : mem_info(wc.s);
        cmr = seq ? nmr : mir_info(wc.s);
        ms = wc.s;
        nmi = mem_info(wc.s + G);
        nmr = mir_info(wc.s + G);
    }
    // where the rows of the warp's kProdCols columns of a tile live (lane = column): read with the tile's flags
    __device__ __forceinline__ T *tile_rows(int ti) const {
        if ((ti & kTileCarried) && lane < kProdCols) {
            const size_t at = (size_t)(ti & (kTileCarried - 1)) * kPTile + pw * kProdCols + lane;
            return static_cast<T *>(PT.A[__ldg(L.live_owner + at)]) + (int64_t)__ldg(L.live_lrow + at) * ld;
        }
        return nullptr;
    }
    // flags of the warp's kProdCols columns of a tile: lane & 7 holds the word of column group lane & 7
    __device__ __forceinline__ uint32_t tile_flags(int ti) const {
        return __ldg(reinterpret_cast<const uint32_t *>(L.flags + (size_t)(ti & (kTileCarried - 1)) * kPTile) + pw * (kProdCols / 4) + (lane & (kProdCols / 4 - 1)));
    }
    // The bulk copies of the item at the issue cursor into the next ring slot (warp-collective).
    __device__ __forceinline__ void issue() {
        if (ic.s >= NS) return;
        if (rs != ic.s) {                                          // rows of a new strip (fetched a strip ahead)
            if (!(rs >= 0 && ic.s == rs + G)) { row_raw(ic.s, 0, no0, nl0); if (npt > 1) row_raw(ic.s, 1, no1, nl1); }
            rp0 = row_ptr(no0, nl0); rp1 = npt > 1 ? row_ptr(no1, nl1) : nullptr;
            rs = ic.s;
            row_raw(ic.s + G, 0, no0, nl0); if (npt > 1) row_raw(ic.s + G, 1, no1, nl1);
        }
        const unsigned fullb = full0 + 8u * islot;
        // every producer warp has read what the slot held before (they arrive after their last shared load;
        // the bulk copy below may then overwrite it without a proxy fence)
        if (iuse > 0 && !mbar_wait(empty0 + 8u * islot, (iuse - 1) & 1u)) atomicCAS(err, 0, 2);
        if (lane == 0) sh.ptinfo[pw][islot] = itile;
        if (issuer) {
            const T *src = (ic.it & (npt - 1)) ? rp1 : rp0;
            const unsigned dst = rbase + (unsigned)(islot * STAGE + myrow * RB);
            if (src) {
                mbar_arrive_expect_tx(fullb, ROWB);
                bulk_g2s_hint(dst, src + (size_t)(itile & (kTileCarried - 1)) * kPTile, ROWB, fullb, read_once);
            } else {
                zero_row_shared(dst, ROWB);
                mbar_arrive_expect_tx(fullb, 0);
            }
        }
        __syncwarp();
        if (++islot == S.stages) { islot = 0; iuse++; }
        ic = items.next(ic);
        if (ic.s < NS) itile = S.live_tiles[ic.it >> lnpt];        // in flight until the next issue
    }
    // ---- transposed and interleaved: Q[p][F] = (father row, mother row) at column p.  A lane takes one
    //      couple and four columns at a time: two 128-bit shared loads (a quarter warp spans the 32 banks:
    //      rows are padded by 16 bytes), four 8-byte stores that the lanes of a warp lay side by side.
    //      Columns nobody lives in are skipped (their pairs are never read). ----
    __device__ __forceinline__ void transpose(const unsigned char *st, P2 *const Q, int pt, int lt) {
        bool done = false;
        if constexpr (sizeof(T) == 4) {
            if (fast_transpose_shape(4, sw, ft)) {                 // the common shape: lane = couple, offsets are immediates
                auto fast = [&](auto SWC) {
                    constexpr int SW = decltype(SWC)::value;
                    const unsigned char *xr = st + lane * RB + pw * (kProdCols * 4), *yr = xr + 32 * RB;
                    P2 *q = Q + ((size_t)lt * kPTile + pw * kProdCols) * SW + pt * 32 + lane;
#pragma unroll
                    for (int g = 0; g < kProdCols / 4; g++) {
                        const uint32_t lv = __shfl_sync(0xffffffffu, live8, g) & kLive4;
                        if (lv == 0u) continue;
                        const float4 a4 = *reinterpret_cast<const float4 *>(xr + g * 16), b4 = *reinterpret_cast<const float4 *>(yr + g * 16);
                        P2 *qq = q + g * 4 * SW;
                        CHECK(((size_t)lt * kPTile + pw * kProdCols + g * 4 + 3) * SW + pt * 32 + lane < (size_t)S.qstride);
                        if (lv == kLive4) {
                            qq[0] = make_float2(a4.x, b4.x); qq[SW] = make_float2(a4.y, b4.y);
                            qq[2 * SW] = make_float2(a4.z, b4.z); qq[3 * SW] = make_float2(a4.w, b4.w);
                        } else {
                            if (lv & 0x1u) qq[0] = make_float2(a4.x, b4.x);
                            if (lv & 0x100u) qq[SW] = make_float2(a4.y, b4.y);
                            if (lv & 0x10000u) qq[2 * SW] = make_float2(a4.z, b4.z);
                            if (lv & 0x1000000u) qq[3 * SW] = make_float2(a4.w, b4.w);
                        }
                    }
                };
                if (sw == 64) { fast(std::integral_constant<int, 64>{}); done = true; }
                else if (sw == 32) { fast(std::integral_constant<int, 32>{}); done = true; }
            }
        }
        if (!done) {
            const int f = lane % ft, gpi = 32 / ft;                // column groups the warp handles per step
            const unsigned char *xr = st + f * RB, *yr = st + (ft + f) * RB;
            P2 *q = Q + (size_t)lt * kPTile * sw + pt * ft + f;
            for (int g = lane / ft; g < kProdCols / 4; g += gpi) {
                const uint32_t w = __shfl_sync(0xffffffffu, live8, g);
                const int col = pw * kProdCols + g * 4;
                T x[4], y[4];
                if constexpr (sizeof(T) == 4) {
                    const float4 a4 = *reinterpret_cast<const float4 *>(xr + col * 4), b4 = *reinterpret_cast<const float4 *>(yr + col * 4);
                    x[0] = a4.x; x[1] = a4.y; x[2] = a4.z; x[3] = a4.w; y[0] = b4.x; y[1] = b4.y; y[2] = b4.z; y[3] = b4.w;
                } else {
                    const double2 a0 = *reinterpret_cast<const double2 *>(xr + col * 8), a1 = *reinterpret_cast<const double2 *>(xr + col * 8 + 16);
                    const double2 b0 = *reinterpret_cast<const double2 *>(yr + col * 8), b1 = *reinterpret_cast<const double2 *>(yr + col * 8 + 16);
                    x[0] = a0.x; x[1] = a0.y; x[2] = a1.x; x[3] = a1.y; y[0] = b0.x; y[1] = b0.y; y[2] = b1.x; y[3] = b1.y;
                }
#pragma unroll
                for (int c4 = 0; c4 < 4; c4++)
                    if ((w >> (8 * c4)) & kFlagLive) {
                        CHECK(((size_t)lt * kPTile + col + c4) * sw + pt * ft + f < (size_t)S.qstride);
                        P2 v; v.x = x[c4]; v.y = y[c4];
                        q[(size_t)(col + c4) * sw] = v;
                    }
            }
        }
    }
    // ---- rows of the new members against this tile's carried columns (rounded once, compute.jl:296).
    //      Columns that are not carried receive values nobody reads. ----
    __device__ __forceinline__ void carried_rows(const unsigned char *st, int pt) {
        const int tile = tinfo & (kTileCarried - 1);
        T *const Acol = A + (int64_t)L.rt_lo + (int64_t)tile * kPTile + 4 * lane;
        CHECK((int64_t)L.rt_lo + (int64_t)tile * kPTile + 4 * lane + 3 < ld);
        for (int qd = 0; qd < cpw; qd += 2) {                      // two couples per step: their loads and sums overlap
            int cnt[2], lr0[2], lr1[2];
            double rr[2][4];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int j = pt * cpw + qd + u, fi = pw * cpw + qd + u;
                cnt[u] = __shfl_sync(0xffffffffu, cmi.me - cmi.mb, j);
                lr0[u] = __shfl_sync(0xffffffffu, cmi.lr0, j); lr1[u] = __shfl_sync(0xffffffffu, cmi.lr1, j);
                if (qd + u >= cpw) cnt[u] = 0;
                double x[4], y[4];
                lds4(reinterpret_cast<const T *>(st + min(fi, ft - 1) * RB) + 4 * lane, x);
                lds4(reinterpret_cast<const T *>(st + (ft + min(fi, ft - 1)) * RB) + 4 * lane, y);
#pragma unroll
                for (int e = 0; e < 4; e++) rr[u][e] = half_sum_mode<STORED>(x[e], y[e]);
            }
#pragma unroll
            for (int u = 0; u < 2; u++) {
                if (cnt[u] > 0) store4(Acol + (int64_t)lr0[u] * ld, rr[u]);
                if (cnt[u] > 1) store4(Acol + (int64_t)lr1[u] * ld, rr[u]);
                if (cnt[u] > 2) {
                    const int mb = __shfl_sync(0xffffffffu, cmi.mb, pt * cpw + qd + u);
                    CHECK(mb >= 0 && mb + cnt[u] <= L.n_new);
                    for (int m = mb + 2; m < mb + cnt[u]; m++) store4(Acol + (int64_t)L.mem_lrow[m] * ld, rr[u]);
                }
            }
        }
    }
    // ---- and the mirror image: the carried individuals' rows against the columns of the new members.  Lane =
    //      member (32 at a time, in slot order), four columns per shared load as above (members of a quarter warp
    //      belong to at most 8 consecutive couples: no bank conflict); a store lays 32 members side by side in the
    //      carried row: runs of 128 bytes that the halves of a strip and the neighbouring strips complete in L2. ----
    __device__ __forceinline__ void mirror_columns(const unsigned char *st, int pt) {
        const int nm = pt ? cmr.nb : cmr.na, mb = pt ? cmr.bb : cmr.ba;
        for (int ch = 0; ch * 32 < nm; ch += 2) {                  // two chunks of 32 members per pass
            int ea, eb;
            if (ch == 0) { ea = pt ? cmr.e0b : cmr.e0a; eb = pt ? cmr.e1b : cmr.e1a; }
            else {
                const int F0h = L.own_f0 + wc.s * sw + pt * ft;
                ea = mir_entry(F0h, mb, nm, ch * 32 + lane); eb = mir_entry(F0h, mb, nm, ch * 32 + 32 + lane);
            }
            const bool two = (ch + 1) * 32 < nm;                   // (warp-uniform)
            const int sla = ea & 0xffffff, fa = ea >= 0 ? (ea >> 24) : 0, slb = eb & 0xffffff, fb = eb >= 0 ? (eb >> 24) : 0;
            CHECK((ea < 0 || (fa < ft && sla < ld)) && (eb < 0 || (fb < ft && slb < ld)));
            const T *xa = reinterpret_cast<const T *>(st + fa * RB) + pw * kProdCols, *xb = reinterpret_cast<const T *>(st + fb * RB) + pw * kProdCols;
            const int yoff = ft * RB / (int)sizeof(T);             // the mother's row, in elements
#pragma unroll 2
            for (int g = 0; g < kProdCols / 4; g++) {
                const uint32_t w = __shfl_sync(0xffffffffu, live8, g);
                if ((w & (0x01010101u * kFlagCarried)) == 0u) continue;
                T *rp[4];
#pragma unroll
                for (int c4 = 0; c4 < 4; c4++)
                    rp[c4] = reinterpret_cast<T *>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(col_row), 4 * g + c4));
                double x[4], y[4];
                T va[4], vb[4];
                lds4(xa + 4 * g, x); lds4(xa + yoff + 4 * g, y);
#pragma unroll
                for (int c4 = 0; c4 < 4; c4++) va[c4] = (T)half_sum_mode<STORED>(x[c4], y[c4]);
                if (two) {
                    lds4(xb + 4 * g, x); lds4(xb + yoff + 4 * g, y);
#pragma unroll
                    for (int c4 = 0; c4 < 4; c4++) vb[c4] = (T)half_sum_mode<STORED>(x[c4], y[c4]);
                }
#pragma unroll
                for (int c4 = 0; c4 < 4; c4++) {
                    const bool on = ((w >> (8 * c4)) & kFlagCarried) != 0;
                    CHECK(!on || rp[c4] != nullptr);
                    if (on && ea >= 0) __stcs(rp[c4] + sla, va[c4]);
                    if (two && on && eb >= 0) __stcs(rp[c4] + slb, vb[c4]);
                }
            }
        }
    }
    // Every lane has its values: the slot may be refilled.  The next item's tile was noted when its copies were issued.
    __device__ __forceinline__ void next_item() {
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8u * cslot);
        if (++cslot == S.stages) { cslot = 0; cuse++; }
        wc = items.next(wc);
        if (wc.s < NS) {
            tinfo = sh.ptinfo[pw][cslot];
            live8 = tile_flags(tinfo);
            col_row = tile_rows(tinfo);
        }
    }
};

// ===== consumer warps: couple tiles -> the strip members' rows against all new members =====
// Nothing the inner loops need comes from a dependent global load: tile descriptors travel three items
// ahead in registers, a tile's metadata (its couples' strip-buffer rows, its members' couple / rank /
// slot) two items ahead into a shared-memory ring with cp.async, its segments one item ahead, and the
// strip's member rows one strip ahead.
template <typename T, bool STORED, int PW>
struct Consumer {
    using P2 = std::conditional_t<sizeof(T) == 4, float2, double2>;   // a (father, mother) pair of strip-buffer entries
    static constexpr int kConsWarps = cons_warps(PW), kConsThreads = kConsWarps * 32;
    static constexpr int kRowCache = kConsThreads;                 // strip member rows the consumer warps keep in shared memory at a time
    static constexpr int kMetaSlots = 3, kMetaInts = 4 * kMTile;   // per slot: qrow[128] | couple[128] | rank[128] | slot[128]
    static_assert(2 * kMaxTileFam / kConsWarps <= 32, "role split");
    struct RowMeta { unsigned rowoff; int rank; long long bytes; };   // Va row offset, rank, byte offset of the frontier row
    T *const A; const int64_t ld; const PeerTable &PT; const LayerArgs &L; const StripArgs &S; LayerShared<PW> &sh;
    unsigned char *const smem;                                     // staged segments | Va | Vb | metadata | member rows
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int sw = S.sw, NS = S.n_strips, G = S.gangs;
    const int gang = blockIdx.x % G;                               // this CTA is consumer blockIdx.x / G of its gang
    const ItemOrder items{NS, G, S.n_citems, S.n_cons / G};
    int *const err = S.err;
    int *const done_p = S.sync, *const done_c = S.sync + 8;        // done_p[kSyncStride * s], done_c[kSyncStride * s]
    P2 *const Qall = static_cast<P2 *>(S.Q);
    const int prod_arrivals = S.n_prod / G;                        // what done_p[s] reaches when strip s is complete
    P2 *const stg = reinterpret_cast<P2 *>(smem);                  // [2 g + parent][f]
    T *const Va = reinterpret_cast<T *>(smem + (size_t)2 * kMaxTileFam * sw * sizeof(P2));   // [f][g]: the strip couple's member is climbed first
    T *const Vb = Va + (size_t)sw * kVPitch;                       // [f][g]: the tile couple's member is climbed first
    int *const meta = reinterpret_cast<int *>(Vb + (size_t)sw * kVPitch);
    RowMeta *const rowmeta = reinterpret_cast<RowMeta *>(meta + kMetaSlots * kMetaInts);
    const unsigned stg_s = (unsigned)__cvta_generic_to_shared(stg), meta_s = (unsigned)__cvta_generic_to_shared(meta);
    const unsigned va_s = (unsigned)__cvta_generic_to_shared(Va), vb_s = (unsigned)__cvta_generic_to_shared(Vb);
    const int row_bytes = sw * (int)sizeof(P2);
    const unsigned sbar = (unsigned)__cvta_generic_to_shared(&sh.cbar);
    unsigned n_landed = 0;                                         // tiles whose segments were awaited
    // ---- the strip's member rows: prefetched one strip ahead (registers), cached in shared memory ----
    int cur = -1;                                                  // strip the consumer warps are in
    int F0 = 0, nFs = 0, ms0 = 0, ms1 = 0, n_rows = 0;
    int pre_s = -1, pre_ms0 = 0, pre_ms1 = 0, pre_f = 0, pre_rank = 0, pre_lrow = 0;   // strip pre_s: bounds, row ms0 + tid
    int pre2_s = -1, pre2_ms0 = 0, pre2_ms1 = 0;                   // strip pre2_s: bounds only
    Item c0 = items.first(gang, blockIdx.x / G), c1 = items.next(c0), c2 = items.next(c1), c3 = items.next(c2);
    int4 d0 = fetch_desc(c0), d1 = fetch_desc(c1), d2 = fetch_desc(c2);   // descriptors of the item in hand and the next two
    unsigned n_item = 0;                                           // items done: item j's metadata sits in ring slot j % 3
    bool staged = false;                                           // the segments of c0 are on their way (or there)
    __device__ __forceinline__ void run() {
        PROF_DECL
        if (is_tile(c0)) fetch_meta(d0, 0);
        if (is_tile(c1)) fetch_meta(d1, 1);
        cp_async_commit();
        while (c0.s < NS) {
            const int s = c0.s;
            if (s != cur) {
                count_off(s);
                enter_strip(s);
                prefetch_rows(s);
                PROF_MARK(2);
                if (!staged && tid == 0 && prod_arrivals > 0)       // the strip's pairs are complete (in L2)
                    spin_wait(done_p + kSyncStride * s, prod_arrivals, err, S.timeout_cycles);
                sync();
                PROF_MARK(1);
            }
            const P2 *const Q = Qall + (size_t)(s % S.nbuf) * S.qstride;
            const int slot0 = (int)(n_item % kMetaSlots);
            // ---- a member tile: its couples' segments (staged ahead unless the strip was not ready), Va | Vb, expansion ----
            if (!staged) {
                cp_async_wait<0>();
                sync();                                            // the tile's metadata is in the ring
                stage_tile(Q, d0.y, slot0);
                cp_async_commit();
            }
            PROF_MARK(0);
            cp_async_wait<0>();                                    // the next tile's metadata (own copies) ...
            await_tile();                                          // ... and this tile's segments have landed
            sync();                                                // for everybody; the previous item is written
            drop_sole_reads(Q, d0.y, slot0);
            PROF_MARK(3);
            // is the next item's strip produced?  Asked now, answered after the arithmetic (an L2 round trip)
            const bool peek_next = is_tile(c1) && c1.s != s;
            int peek = 0;
            if (tid == 0 && peek_next) peek = ld_relaxed_gpu(done_p + kSyncStride * c1.s);
            couple_tile(d0.y);
            sync();                                                // Va | Vb complete, the staging area is free
            PROF_MARK(4);
            // the pipeline: descriptor of item +3, metadata of item +2, segments of item +1 (if its strip is produced)
            const int4 d3 = fetch_desc(c3);
            if (is_tile(c2)) fetch_meta(d2, (int)((n_item + 2) % kMetaSlots));
            staged = stage_next(s, peek);
            cp_async_commit();
            PROF_MARK(5);
            expand(s, slot0);
            c0 = c1; c1 = c2; c2 = c3; c3 = items.next(c3);
            d0 = d1; d1 = d2; d2 = d3;
            n_item++;
            PROF_MARK(6);
        }
        count_off(NS);
        PROF_MARK(0);
        PROF_FLUSH(1, tid == 0);
    }
    // barrier of the consumer warps only (the producer warps never meet anybody)
    __device__ __forceinline__ void sync() const { asm volatile("bar.sync 1, %0;" ::"n"(kConsThreads) : "memory"); }
    // The consumer warps' share of the strips of their gang below `upto` is done: their copies of those strips' pairs
    // have landed in shared memory (they waited for them), which is all the producers that will overwrite the buffer
    // need to know -- no fence: the rows they wrote are read by the next kernel at the earliest.
    // With discards in flight the count is a release: the producers that overwrite the buffer must find the
    // discards performed (the barrier makes them the counting thread's business, the fence orders them).
    __device__ __forceinline__ void count_off(int upto) {
        for (int t = cur < 0 ? gang : cur; t < upto; t += G) {
            sync();
            if (tid == 0) {
                if (S.discard) __threadfence();
                atomicAdd(done_c + kSyncStride * t, 1);
            }
        }
        cur = upto;
    }
    __device__ __forceinline__ bool is_tile(Item c) const { return c.s < NS && c.it < L.n_mtiles; }
    __device__ __forceinline__ int4 fetch_desc(Item c) const { return is_tile(c) ? __ldg(L.mt_desc + c.it) : make_int4(0, 0, 0, 0); }
    // metadata of tile `d` -> ring slot (cp.async; the caller commits)
    __device__ __forceinline__ void fetch_meta(int4 d, int slot) {
        CHECK(d.y >= 1 && d.y <= kMaxTileFam && d.w >= 1 && d.w <= kMTile && d.x >= 0 && d.x + d.y <= L.n_fam && d.z >= 0 && d.z + d.w <= L.n_new);
        const unsigned base = meta_s + (unsigned)(slot * kMetaInts * (int)sizeof(int));
        if (tid < d.y)                                             // the couples' (father, mother) rows in the strip buffers
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(base + 8u * tid), "l"(L.fam_q + d.x + tid) : "memory");
        const int nchunk = (d.w + 3) >> 2;                         // member columns: couple, rank, slot in 16-byte chunks
        if (tid < 3 * nchunk) {
            const int arr = tid / nchunk, c = tid - arr * nchunk;
            const int32_t *src = (arr == 0 ? L.mem_fam : arr == 1 ? L.mem_ind : L.mem_slot) + d.z + 4 * c;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"(base + (unsigned)((kMTile * (1 + arr) + 4 * c) * 4)), "l"(src) : "memory");
        }
    }
    // the two parent-row segments of every couple of the tile -> stg: one TMA bulk copy per segment, issued by
    // the first lanes of every warp (one each), all completing on one mbarrier phase per tile
    __device__ __forceinline__ void stage_tile(const P2 *Q, int nfJ, int slot) {
        if (lane < 2 * kMaxTileFam / kConsWarps) {                 // the issue is serial per warp
            const int r = warp * (2 * kMaxTileFam / kConsWarps) + lane;
            const int q0 = r < 2 * nfJ ? meta[slot * kMetaInts + r] : -1, q = q0 >= 0 ? (q0 & ~kSoleReader) : -1;
            CHECK(q >= -1 && (long long)q * sw < S.qstride);
            const unsigned dst = stg_s + (unsigned)(r * row_bytes);
            if (q >= 0) {                                          // (write after read of the staging area: no proxy fence)
                mbar_arrive_expect_tx(sbar, (unsigned)row_bytes);
                bulk_g2s(dst, Q + (size_t)q * sw, (unsigned)row_bytes, sbar);
            } else {
                if (r < 2 * nfJ) zero_row_shared(dst, (unsigned)row_bytes);
                mbar_arrive_expect_tx(sbar, 0);
            }
        }
    }
    __device__ __forceinline__ void await_tile() {                 // all threads
        if (!mbar_wait(sbar, n_landed & 1u)) atomicCAS(err, 0, 2);
        n_landed++;
    }
    // The segments are in shared memory.  Those this tile was the only one to read (kSoleReader: the parent has no
    // other couple in the layer) are dead in the strip buffer, but dirty: dropped from L2 now (discard.global.L2),
    // they are neither written back to DRAM nor do they take the room of pairs that have not been read yet.
    __device__ __forceinline__ void drop_sole_reads(const P2 *Q, int nfJ, int slot) const {
        if (S.discard && row_bytes >= 128 && tid < 2 * nfJ) {
            const int q0 = meta[slot * kMetaInts + tid];
            if (q0 >= 0 && (q0 & kSoleReader)) {
                const unsigned char *seg = reinterpret_cast<const unsigned char *>(Q + (size_t)(q0 & ~kSoleReader) * sw);
                for (int b = 0; b < row_bytes; b += 128) asm volatile("discard.global.L2 [%0], 128;" ::"l"(seg + b) : "memory");
            }
        }
    }
    // The segments of the next item are staged now if its strip is the current one or produced (the peek, acquired
    // here); otherwise they are staged when the consumer warps have waited for it.
    __device__ __forceinline__ bool stage_next(int s, int peek) {
        if (!is_tile(c1)) return false;
        bool ready = c1.s == s;
        if (!ready) {                                              // do not wait here, the expansion comes first
            if (tid == 0) {
                sh.ready = peek >= prod_arrivals;
                if (peek >= prod_arrivals) ld_acquire_gpu(done_p + kSyncStride * c1.s);   // (the peek was a relaxed load)
            }
            sync();
            ready = sh.ready != 0;
        }
        if (ready) stage_tile(Qall + (size_t)(c1.s % S.nbuf) * S.qstride, d1.y, (int)((n_item + 1) % kMetaSlots));
        return ready;
    }
    __device__ __forceinline__ void strip_bounds(int st, int &b0, int &b1) const {
        const int f0 = L.own_f0 + st * sw, nf = min(sw, L.own_nf - st * sw);
        b0 = L.fam_start[f0]; b1 = L.fam_start[f0 + nf];
    }
    __device__ __forceinline__ void strip_row(int st, int b0, int b1, int first, int &f, int &rk, int &lr) const {   // row first + tid of strip st
        const int im = min(b0 + first + tid, b1 - 1);
        f = L.mem_fam[im] - (L.own_f0 + st * sw); rk = L.mem_ind[im]; lr = L.mem_lrow[im];
    }
    __device__ __forceinline__ void put_row(int f, int rk, int lr) const {
        RowMeta m; m.rowoff = (unsigned)(f * kVPitch * (int)sizeof(T)); m.rank = rk; m.bytes = (long long)lr * ld * (long long)sizeof(T);
        rowmeta[tid] = m;
    }
    // strip s: its couples, the bounds of its member rows and the first rows' descriptors (prefetched unless the
    // consumer warps did not know the strip a strip ago)
    __device__ __forceinline__ void enter_strip(int s) {
        F0 = L.own_f0 + s * sw;
        nFs = min(sw, L.own_nf - s * sw);
        int rf, rk, rl;
        if (pre_s == s) { ms0 = pre_ms0; ms1 = pre_ms1; rf = pre_f; rk = pre_rank; rl = pre_lrow; }
        else { strip_bounds(s, ms0, ms1); strip_row(s, ms0, ms1, 0, rf, rk, rl); }
        n_rows = ms1 - ms0;
        put_row(rf, rk, rl);                                       // (read after the barriers that follow)
    }
    // the rows of the strip the consumer warps visit next, and the bounds of the one after, are fetched now and used
    // a strip later (the next items are known: c1, c2, c3)
    __device__ __forceinline__ void prefetch_rows(int s) {
        const int ns = c1.s != s ? c1.s : c2.s != s ? c2.s : c3.s != s ? c3.s : s + G;
        const int ns2 = (c1.s != s && c1.s != ns) ? c1.s : (c2.s != s && c2.s != ns) ? c2.s : (c3.s != s && c3.s != ns) ? c3.s : ns + G;
        if (ns < NS) {
            if (pre2_s == ns) { pre_ms0 = pre2_ms0; pre_ms1 = pre2_ms1; } else strip_bounds(ns, pre_ms0, pre_ms1);
            strip_row(ns, pre_ms0, pre_ms1, 0, pre_f, pre_rank, pre_lrow);
            pre_s = ns;
            if (ns2 < NS) { strip_bounds(ns2, pre2_ms0, pre2_ms1); pre2_s = ns2; }
        }
    }
    // Va | Vb: both groupings of every (strip couple, tile couple) pair, rounded once to T
    __device__ __forceinline__ void couple_tile(int nfJ) const {
        const int lsw = 31 - __clz(sw);                            // sw is a power of two
        const int fl = tid & (sw - 1), g0 = tid >> lsw, gstep = kConsThreads >> lsw;
        if (fl < nFs) {
#pragma unroll 4
            for (int g = g0; g < nfJ; g += gstep) {
                const P2 a = stg[(2 * g) * sw + fl], c = stg[(2 * g + 1) * sw + fl];
                T vf, vg;
                couple_pair<T, STORED>((double)a.x, (double)a.y, (double)c.x, (double)c.y, vf, vg);
                Va[fl * kVPitch + g] = vf;
                Vb[fl * kVPitch + g] = vg;
            }
        }
    }
    // ---- expansion: the lane's four member columns, the warp's share of the strip's rows, four rows at a time ----
    __device__ __forceinline__ void expand(int s, int slot0) {
        const int fJ0 = d0.x, mJ0 = d0.z, cntJ = d0.w;
        const int *mcol = meta + slot0 * kMetaInts + kMTile;
        const int4 cg = *reinterpret_cast<const int4 *>(mcol + 4 * lane);
        const int4 cr = *reinterpret_cast<const int4 *>(mcol + kMTile + 4 * lane);
        const int4 cs4 = *reinterpret_cast<const int4 *>(mcol + 2 * kMTile + 4 * lane);
        const int ncol = min(4, cntJ - 4 * lane);
        // columns past the end of the tile repeat the lane's first one (what the ring holds there is stale)
        const int gq[4] = {cg.x, ncol > 1 ? cg.y : cg.x, ncol > 2 ? cg.z : cg.x, ncol > 3 ? cg.w : cg.x};
        const int rj[4] = {cr.x, ncol > 1 ? cr.y : cr.x, ncol > 2 ? cr.z : cr.x, ncol > 3 ? cr.w : cr.x};
        const int sj[4] = {cs4.x, cs4.y, cs4.z, cs4.w};
        unsigned off[4];
#pragma unroll
        for (int q = 0; q < 4; q++) off[q] = ncol > 0 ? (unsigned)((gq[q] - fJ0) * (int)sizeof(T)) : 0u;
        const bool vec = ncol == 4 && ((sj[0] & 3) == 0) && sj[1] == sj[0] + 1 && sj[2] == sj[0] + 2 && sj[3] == sj[0] + 3;
        unsigned char *const Ab = reinterpret_cast<unsigned char *>(A);
        for (int pass0 = 0; pass0 < n_rows; pass0 += kRowCache) {
            if (pass0 > 0 || n_rows > kRowCache) {                 // a strip with more rows than the cache: reload it per pass
                sync();
                int rf, rk, rl;
                strip_row(s, ms0, ms1, pass0, rf, rk, rl);
                put_row(rf, rk, rl);
                sync();
            }
            const int nrp = min(kRowCache, n_rows - pass0);
            const int share = (nrp + kConsWarps - 1) / kConsWarps;
            const int rbeg = warp * share, rend = min(nrp, rbeg + share);
            if (ncol > 0) {
                int r = rbeg;
                for (; r + 4 <= rend; r += 4) {
                    RowMeta m[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        m[u] = rowmeta[r + u];
                        CHECK(m[u].rowoff < (unsigned)(sw * kVPitch * (int)sizeof(T)) && m[u].bytes >= 0);
                    }
                    CHECK(off[0] < kVPitch * sizeof(T) && off[1] < kVPitch * sizeof(T) && off[2] < kVPitch * sizeof(T) && off[3] < kVPitch * sizeof(T));
                    CHECK(sj[0] >= 0 && sj[0] < ld);
                    T v[4][4];
#pragma unroll
                    for (int u = 0; u < 4; u++)
#pragma unroll
                        for (int q = 0; q < 4; q++)                // the higher rank is climbed first (compute.jl:130-147)
                            v[u][q] = lds<T>((m[u].rank > rj[q] ? va_s : vb_s) + m[u].rowoff + off[q]);
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        T *row = reinterpret_cast<T *>(Ab + m[u].bytes);
                        if (vec) store_vec4(row + sj[0], v[u]);
                        else {
#pragma unroll
                            for (int q = 0; q < 4; q++) if (q < ncol) __stcs(row + sj[q], v[u][q]);
                        }
                    }
                }
                for (; r < rend; r++) {
                    const RowMeta m = rowmeta[r];
                    CHECK(m.rowoff < (unsigned)(sw * kVPitch * (int)sizeof(T)) && m.bytes >= 0);
                    T *row = reinterpret_cast<T *>(Ab + m.bytes);
#pragma unroll
                    for (int q = 0; q < 4; q++)
                        if (q < ncol) __stcs(row + sj[q], lds<T>((m.rank > rj[q] ? va_s : vb_s) + m.rowoff + off[q]));
                }
            }
            // own diagonal entries (compute.jl:148-155): rows of this pass that are also columns of this tile,
            // written over the row segments above (__syncwarp orders the warp's stores)
            __syncwarp();
            const int dlo = max(ms0 + pass0 + rbeg, mJ0), dhi = min(ms0 + pass0 + rend, mJ0 + cntJ);
            for (int i = dlo + lane; i < dhi; i += 32) {
                const RowMeta m = rowmeta[i - ms0 - pass0];
                const int F = F0 + (int)(m.rowoff / (unsigned)(kVPitch * (int)sizeof(T)));
                CHECK(F >= 0 && F < L.n_fam && i - mJ0 >= 0 && i - mJ0 < kMTile);
                const int pf = L.fam_pf[F], pm = L.fam_pm[F];
                double d = 0.5;
                if (pf >= 0 && pm >= 0)
                    d = half_sum_mode<STORED>((double)(static_cast<const T *>(PT.A[L.fam_pf_owner[F]]) + (int64_t)L.fam_pf_lrow[F] * ld)[pm], 1.0);
                reinterpret_cast<T *>(Ab + m.bytes)[meta[slot0 * kMetaInts + 3 * kMTile + (i - mJ0)]] = (T)d;
            }
        }
    }
};

template <typename T, bool STORED, int PW>
__global__ void __launch_bounds__(kLayerThreads, 1)
layer_kernel(T *__restrict__ A, int64_t ld, PeerTable PT, LayerArgs L, StripArgs S) {
    extern __shared__ __align__(128) unsigned char dyn_smem[];    // consumer: staged segments | Va | Vb | metadata | rows; then the producer ring
    __shared__ LayerShared<PW> sh;
    if (threadIdx.x < 8) sh.pcount[threadIdx.x] = 0;
    if (threadIdx.x == 0) {
        sh.cdone = 0;
        for (int st = 0; st < kMaxStages; st++) {
            mbar_init((unsigned)__cvta_generic_to_shared(&sh.full[st]), 2 * S.ft);
            mbar_init((unsigned)__cvta_generic_to_shared(&sh.empty[st]), PW);
        }
        mbar_init((unsigned)__cvta_generic_to_shared(&sh.cbar), 2 * kMaxTileFam);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();                                              // the only CTA-wide barrier: the roles part here
    if (threadIdx.x >= cons_warps(PW) * 32) {
        if ((int)blockIdx.x < S.n_prod) Producer<T, STORED, PW>{A, ld, PT, L, S, sh, dyn_smem + S.ring_off}.run();
    } else if ((int)blockIdx.x < S.n_cons) Consumer<T, STORED, PW>{A, ld, PT, L, S, sh, dyn_smem}.run();
}

}  // namespace genlib
