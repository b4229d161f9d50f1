// orlg_rollout.cuh -- T environment steps per launch for DeepRMSA (the headline rollout path).
//
// Same semantics as T iterations of { action = policy(env); obs, reward, done = env.step(action) } through
// orlg_random_actions / orlg_heuristic + orlg_step (deeprmsa_env.py:48-124 on top of rmsa_env.py:163-282,
// 545-597), with every step's action / reward / done / float32 observation written to [T, N, ...] buffers.
// What changes is where the state lives while the T steps run:
//   * a warp owns 32 consecutive envs for the whole launch: their link masks ([link][lane] uint4, E x 512 B)
//     stay in shared memory and the scalar block (clock, pending request, counters, cached block starts)
//     stays in registers; HBM sees them once at entry and once at exit;
//   * for the duration of the launch the release-event tables of the warp's 32 envs are held LANE-INTERLEAVED
//     (rows of 32 16-byte entries: [row][lane], converted at the first launch and kept until another entry point
//     needs the canonical form), so that a thread-per-env pass over "row r of every env" is one coalesced access.
//     The table is consulted through a per-env WINDOW: every ~30 steps the warp rebuilds it -- each thread
//     streams its table once, moves the services that expire before a horizon into a scratch list and compacts
//     the rest in place; the warp then sorts the 32 lists by release time through shuffles (ro_rebuild).  A
//     step then only compares the list head (registers; the following entry is fetched one pop ahead) with
//     the clock: the directory -> group -> payload fetch chain of the per-step kernel is gone.  Services
//     accepted with a release time inside the horizon wait in a 4-entry side buffer in shared memory.  The exact minimum of what is left in
//     the table gates the next rebuild, so the scheme is exact whatever the horizon (which only tunes how
//     often the tables are streamed); rebuilds are taken by the whole warp together (ballot);
//   * the 32 observation rows of a warp are assembled in a shared-memory tile taken from a small per-CTA
//     pool (held only while the rows are written and copied out with coalesced 16-byte stores); the topology
//     tables arrive by one bulk (TMA) copy per CTA;
//   * the window state persists between launches (st_* arrays); ro_canonicalize_kernel puts the window / side
//     entries back and rebuilds the canonical tables and their directory the first time another entry point of
//     the library (per-step kernels, export, heuristics) needs them;
//   * phase C (free-slot masks and features of the candidate paths) is ONE rolled loop over the paths: the loop
//     body of a step has to fit the 32 KB instruction cache that 14 de-synchronised warps share.
// Release order inside a step is irrelevant (masks only, SURVEY.md App. B-9); what must be exact is WHICH
// services are due, and that is decided on the float64 times.
#pragma once
#include "orlg_deeprmsa_fast.cuh"

namespace orlg {

constexpr int RO_WCAP = 64;            // window entries per env
#ifndef ORLG_RO_SIDE
#define ORLG_RO_SIDE 4        // 3 -> 4: no warp takes two rebuilds inside a 20-step launch any more (side-buffer overflow forced them); 5, 6 cost more in the step loop
#endif
constexpr int RO_SIDE = ORLG_RO_SIDE;             // side-buffer entries per env (shared memory)
constexpr int RO_MAX_THREADS = 448;    // 14 warps x 148 SMs >= 65536 envs in one wave
enum { RO_POLICY_RANDOM = 0, RO_POLICY_SP_FF = 1, RO_POLICY_SAP_FF = 2, RO_POLICY_REPLAY = 3, RO_POLICY_LLP_FF = 4, RO_POLICY_SAP_LF = 5 };

// optional cycle accounting per warp (instrumented builds: -DORLG_PHASE_TIMING, tools/rollout_phases.py)
#ifdef ORLG_PHASE_TIMING
#define RPH_INIT() long long rph_t_ = clock64()
#define RPH_MARK(k)                                                                                      \
    do {                                                                                                 \
        long long rph_n_ = clock64();                                                                    \
        if ((threadIdx.x & 31) == 0) atomicAdd(&g_phase_cycles[k], (unsigned long long)(rph_n_ - rph_t_)); \
        rph_t_ = rph_n_;                                                                                 \
    } while (0)
#define RPH_COUNT(k) do { if ((threadIdx.x & 31) == 0) atomicAdd(&g_phase_cycles[k], 1ULL); } while (0)
#else
#define RPH_INIT() do { } while (0)
#define RPH_MARK(k) do { } while (0)
#define RPH_COUNT(k) do { } while (0)
#endif

// per-warp wall-clock timeline of one launch (instrumented builds: -DORLG_RO_TIMELINE, tools/rollout_timeline.py):
// globaltimer (ns) at kernel entry / first step / after the last step / exit, rebuilds taken and the ns spent in them
#ifdef ORLG_RO_TIMELINE
__device__ unsigned long long g_ro_timeline[8 * 4096];
__device__ __forceinline__ unsigned long long ro_gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define RTL_DECL() unsigned long long rtl_[8] = {ro_gtime(), 0, 0, 0, 0, 0, 0, 0}
#define RTL_SET(k) rtl_[k] = ro_gtime()
#define RTL_REBUILD_BEGIN() const unsigned long long rtl_b_ = ro_gtime()
#define RTL_REBUILD_END() do { rtl_[4] += 1; rtl_[5] += ro_gtime() - rtl_b_; rtl_[6] += g_rtl_scan_; rtl_[7] += g_rtl_sort_; } while (0)
#define RTL_IN_REBUILD(var) var = ro_gtime()
#define RTL_FLUSH(w) do { if ((threadIdx.x & 31) == 0 && (w) < 4096) { for (int i_ = 0; i_ < 8; i_++) g_ro_timeline[8 * (w) + i_] = rtl_[i_]; } } while (0)
#else
#define RTL_DECL() do { } while (0)
#define RTL_SET(k) do { } while (0)
#define RTL_REBUILD_BEGIN() do { } while (0)
#define RTL_REBUILD_END() do { } while (0)
#define RTL_IN_REBUILD(var) do { } while (0)
#define RTL_FLUSH(w) do { } while (0)
#endif

struct __align__(16) WinEntry {
    double t;
    unsigned long long p;
};

struct RolloutArgs {
    int T;                       // steps per launch
    int pool_tiles;              // observation tiles shared by the CTA's warps
    int tile_bytes;              // 32 rows x obs_dim floats, rounded up to 128 bytes
    int warp_bytes;              // per-warp shared memory: E x 512 (masks) + RO_SIDE x 512 (side buffer)
    int lpw;                     // envs (lanes in use) per warp: 32, or 8 for small batches -- more warps per SM and less
                                 // divergence per warp when the batch would not fill the machine (fixed per handle)
    double span;                 // window horizon (time units ahead of the clock)
    float *obs;                  // [T][n][obs_dim]   (NULL: skip)
    float *reward;               // [T][n]            (NULL: skip)
    unsigned char *done;         // [T][n]            (NULL: skip)
    int *actions;                // [T][n]            (NULL: skip; RO_POLICY_REPLAY: the INPUT action sequence)
    uint4 *packed;               // [T][n][2]         (NULL: skip) 32-byte record per env-step: the integer pre-image of the
                                 //                   observation + request + action / accepted / done (orlg.h, orlg_expand_packed)
    // launch-private event storage, lane-interleaved per warp of 32 envs: one slab of (heap_cap + 2 * RO_WCAP) rows of 32
    // 16-byte entries (release time, packed service) per warp -- rows [0, heap_cap) the unsorted table, the next RO_WCAP the
    // rebuild's scratch list, the last RO_WCAP the sorted window; element (row r, lane) of warp w at (w * rows + r) * 32 + lane
    WinEntry *ev;
    // window state kept between launches (the event storage stays in the launch-private form until another entry point
    // needs the canonical tables: ro_canonicalize_kernel)
    int resume;                  // 1: continue from the saved window state; 0: convert the canonical tables first
    unsigned *st_ntab, *st_wh, *st_wn, *st_ncanon;      // [n]
    double *st_tmin, *st_hzn;                           // [n]
    double *st_side_t;                                  // [RO_SIDE][n]
    unsigned long long *st_side_p;                      // [RO_SIDE][n]
    long long *info;             // [T][n][8]         the counters orlg_step's info_dev receives, every step (INFO instances)
};

// apply a release / an allocation to the path's links in the warp's shared-memory mask tile
template <bool SET>
__device__ __forceinline__ void ro_path_update(uint4 *sm, unsigned lm, const Bits &rm) {
    while (lm) {                         // two hops per pass: both loads in flight before either store (a repeated hop is harmless)
        const int l0 = __ffs(lm) - 1;
        lm &= lm - 1;
        const int l1 = lm ? __ffs(lm) - 1 : l0;
        lm &= lm - 1;
        uint4 v = sm[l0 * 32], u = sm[l1 * 32];
        if (SET) { v.x |= rm.w[0]; v.y |= rm.w[1]; v.z |= rm.w[2]; v.w |= rm.w[3]; u.x |= rm.w[0]; u.y |= rm.w[1]; u.z |= rm.w[2]; u.w |= rm.w[3]; }
        else { v.x &= ~rm.w[0]; v.y &= ~rm.w[1]; v.z &= ~rm.w[2]; v.w &= ~rm.w[3]; u.x &= ~rm.w[0]; u.y &= ~rm.w[1]; u.z &= ~rm.w[2]; u.w &= ~rm.w[3]; }
        sm[l0 * 32] = v;
        sm[l1 * 32] = u;
    }
}

// The launch-private event storage of a warp is only ever touched by that warp (one SM): ordinary L1-cached loads are coherent.
__device__ __forceinline__ WinEntry win_load(const WinEntry *w) {
    const uint4 v = *reinterpret_cast<const uint4 *>(w);
    WinEntry e;
    e.t = __hiloint2double((int)v.y, (int)v.x);
    e.p = (unsigned long long)v.z | ((unsigned long long)v.w << 32);
    return e;
}

// one observation tile out of the CTA's pool (lane 0 spins on the free mask; the index is broadcast)
__device__ __forceinline__ unsigned ro_tile_acquire(unsigned *pool_free, int lane) {
    unsigned tile = 0;
    if (lane == 0) {
        unsigned got = 0;
        while (!got) {
            const unsigned f = *reinterpret_cast<volatile unsigned *>(pool_free);
            if (f) {
                const unsigned bit = f & (0u - f);
                if (atomicAnd(pool_free, ~bit) & bit) got = bit;
            } else {
                __nanosleep(32);
            }
        }
        tile = (unsigned)__ffs(got) - 1u;
    }
    return __shfl_sync(0xffffffffu, tile, 0);
}
__device__ __forceinline__ void ro_tile_release(unsigned *pool_free, unsigned tile, int lane) {
    __syncwarp();
    if (lane == 0) atomicOr(pool_free, 1u << tile);
}

constexpr int RO_SCAN = 8;          // table rows per batch of the rebuild's streaming pass
__device__ __forceinline__ void prefetch_l1(const void *ptr) { asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr)); }
__device__ __forceinline__ void win_store(WinEntry *w, double t, unsigned long long pl) {
    *reinterpret_cast<uint4 *>(w) = make_uint4((unsigned)__double2loint(t), (unsigned)__double2hiint(t), (unsigned)pl, (unsigned)(pl >> 32));
}
// Window rebuild of a warp's 32 envs on its slab of the lane-interleaved storage (`ev` already includes the lane; row
// stride 32 entries; `cap` = table rows).  Called by ALL 32 lanes together (a lane without an env arrives with an empty
// table, window and side buffer).
// On entry: table = rows [0, n) (unsorted), window = rows win[wh, wn) (sorted), side = up to RO_SIDE entries.
//   1. thread per env: everything goes back to the table (window loads four at a time);
//   2. thread per env: one streaming pass moves the entries with time <= h (at most RO_WCAP) to the scratch rows and
//      compacts the others in place (forward, stable).  Branch-free per entry: the destination ROW is selected (table
//      and scratch share the slab, so that is one 32-bit select), the loads are unpredicated (the table is a multiple
//      of 16 rows: a batch never leaves it) -- lanes extract different entries, and the divergent form cost 3 x the
//      instructions;
//   3. the WARP sorts the 32 scratch lists: lane q takes entry q (and q + 32) of list L -- a strided read of rows the owner
//      just wrote, 8 lists per 128-byte line -- ranks it against the rest of the list through shuffles (no memory in the
//      loop: the thread-per-env rank sort was c * c / 2 dependent L2 round trips) and stores it at its rank in L's
//      window.  Equal release times keep their list order (__match_any_sync gives the tie groups).  Two lists of at
//      most 16 entries are ranked together, one per half-warp.
// Leaves tmin = exact minimum of the table.  If more than RO_WCAP entries lie below the horizon the rest stays in the table
// (the caller retries with a shorter horizon while a table entry is still due).
__device__ __forceinline__ void ro_rebuild(WinEntry *ev, const unsigned cap, double *side_t, unsigned long long *side_p,
                                           unsigned &n, unsigned &wh, unsigned &wn, double &tmin, double &side_min,
                                           const double h, WinEntry &head, WinEntry &nxt, const int lane, unsigned long long &g_rtl_scan_, unsigned long long &g_rtl_sort_) {
    RPH_INIT();
    WinEntry *const win = ev + (cap + RO_WCAP) * 32;
    // the streaming pass below is a chain of dependent round trips (one per 8-row batch): start the first batches' lines
    // now, and every batch asks for the lines two batches ahead
#pragma unroll
    for (int i = 0; i < 2 * RO_SCAN; i++)
        if ((unsigned)i < n) prefetch_l1(ev + i * 32);
    for (unsigned j = wh; j < wn; j += 4) {             // leftover window entries, four loads in flight
        uint4 w[4];
#pragma unroll
        for (int i = 0; i < 4; i++)
            if (j + i < wn) w[i] = *reinterpret_cast<const uint4 *>(win + (j + i) * 32);
#pragma unroll
        for (int i = 0; i < 4; i++)
            if (j + i < wn) { *reinterpret_cast<uint4 *>(ev + n * 32) = w[i]; n++; }
    }
#pragma unroll
    for (int s = 0; s < RO_SIDE; s++) {                 // side buffer
        const double t = side_t[s * 32];
        if (t < ORLG_INF) { win_store(ev + n * 32, t, side_p[s * 32]); n++; side_t[s * 32] = ORLG_INF; }
    }
    side_min = ORLG_INF;
    RPH_MARK(11);                                       // rebuild: window + side back to the table
    unsigned long long rtl_t1_ = 0, rtl_t2_ = 0, rtl_t3_ = 0;
    RTL_IN_REBUILD(rtl_t1_);
    unsigned k = 0, cs = cap;                           // next table row of the compaction, next scratch row
    double mn = ORLG_INF;
    {
        const WinEntry *rd = ev;
        for (unsigned s0 = 0; s0 < n; s0 += RO_SCAN, rd += RO_SCAN * 32) {
            const unsigned rem = n - s0;
            uint4 v[RO_SCAN];
#pragma unroll
            for (int i = 0; i < RO_SCAN; i++)
                if ((unsigned)(2 * RO_SCAN + i) < rem) prefetch_l1(rd + (2 * RO_SCAN + i) * 32);
#pragma unroll
            for (int i = 0; i < RO_SCAN; i++) v[i] = *reinterpret_cast<const uint4 *>(rd + i * 32);
#pragma unroll
            for (int i = 0; i < RO_SCAN; i++) {
                const double t = __hiloint2double((int)v[i].y, (int)v[i].x);
                const bool in = (unsigned)i < rem;
                const bool ext = in && t <= h && cs < cap + (unsigned)RO_WCAP;
                const bool keep = in && !ext;
                const unsigned row = ext ? cs : k;
                if (in) *reinterpret_cast<uint4 *>(ev + row * 32) = v[i];
                cs += ext ? 1u : 0u;
                k += keep ? 1u : 0u;
                mn = (keep && t < mn) ? t : mn;
            }
        }
    }
    n = k;
    tmin = mn;
    const unsigned c = cs - cap;
    RPH_MARK(12);                                       // rebuild: streaming pass
    RTL_IN_REBUILD(rtl_t2_);
    __syncwarp();
    {
        // the lists are read across the lanes below (32-byte sectors of rows this warp just wrote through to L2): pull the
        // rows into L1 whole, every lane asking for its own entries, so that only the first list waits for a round trip
        const unsigned cmax = __reduce_max_sync(0xffffffffu, c);
        for (unsigned q = 0; q < cmax; q++)
            if (q < c) prefetch_l1(ev + (cap + q) * 32);
        const WinEntry *scw = ev + cap * 32 - lane;      // the warp's scratch rows, lane 0
        WinEntry *winw = win - lane;
        const unsigned lt_mask = (1u << lane) - 1u;
        unsigned todo = __ballot_sync(0xffffffffu, c > 0);
        while (todo) {
            const int L = __ffs(todo) - 1;
            todo &= todo - 1;
            const unsigned cL = __shfl_sync(0xffffffffu, c, L);
            const int LB = todo ? __ffs(todo) - 1 : L;
            const unsigned cB = __shfl_sync(0xffffffffu, c, LB);
            if (todo && cL <= 16u && cB <= 16u) {       // two short lists, one per half-warp
                todo &= todo - 1;
                const bool hi = lane >= 16;
                const int q = lane & 15, myL = hi ? LB : L;
                const unsigned myc = hi ? cB : cL;
                uint4 v = make_uint4(0u, 0x7ff00000u, 0u, 0u);
                if ((unsigned)q < myc) v = *reinterpret_cast<const uint4 *>(scw + q * 32 + myL);
                const double t = __hiloint2double((int)v.y, (int)v.x);
                const unsigned cm = cL > cB ? cL : cB;
                const int base = lane & 16;
                unsigned r = 0;
#pragma unroll 4
                for (unsigned i = 0; i < cm; i++) r += (__shfl_sync(0xffffffffu, t, base + (int)i) < t) ? 1u : 0u;
                // equal release times would share a rank: the ranks then do not cover cL + cB window rows (one warp reduction
                // checks it); only then are the tie groups looked up and ordered by list position
                const bool mine = (unsigned)q < myc;
                if (__popc(__reduce_or_sync(0xffffffffu, mine ? 1u << (base + (int)r) : 0u)) != (int)(cL + cB)) {
                    const unsigned same = __match_any_sync(0xffffffffu, (unsigned long long)__double_as_longlong(t));
                    r += __popc(same & lt_mask & (hi ? 0xffff0000u : 0x0000ffffu));
                }
                if (mine) *reinterpret_cast<uint4 *>(winw + r * 32 + myL) = v;
            } else {                                    // one list of up to 64 entries: lane q ranks entries q and q + 32
                const bool h0 = (unsigned)lane < cL, h1 = (unsigned)lane + 32u < cL;
                uint4 v0 = make_uint4(0u, 0x7ff00000u, 0u, 0u), v1 = v0;
                if (h0) v0 = *reinterpret_cast<const uint4 *>(scw + lane * 32 + L);
                if (h1) v1 = *reinterpret_cast<const uint4 *>(scw + (lane + 32) * 32 + L);
                const double t0 = __hiloint2double((int)v0.y, (int)v0.x), t1 = __hiloint2double((int)v1.y, (int)v1.x);
                unsigned r0 = 0, r1 = 0;
                const unsigned c_lo = cL < 32u ? cL : 32u;
#pragma unroll 2
                for (unsigned i = 0; i < c_lo; i++) {   // entries 0..31 against this lane's two (they precede every entry 32..63)
                    const double tr = __shfl_sync(0xffffffffu, t0, (int)i);
                    r0 += (tr < t0) ? 1u : 0u;
                    r1 += (tr <= t1) ? 1u : 0u;
                }
#pragma unroll 2
                for (unsigned i = 32; i < cL; i++) {    // entries 32..63
                    const double tr = __shfl_sync(0xffffffffu, t1, (int)(i - 32u));
                    r0 += (tr < t0) ? 1u : 0u;
                    r1 += (tr < t1) ? 1u : 0u;
                }
                const unsigned lo_bits = (h0 && r0 < 32u ? 1u << r0 : 0u) | (h1 && r1 < 32u ? 1u << r1 : 0u);
                const unsigned hi_bits = (h0 && r0 >= 32u ? 1u << (r0 - 32u) : 0u) | (h1 && r1 >= 32u ? 1u << (r1 - 32u) : 0u);
                if (__popc(__reduce_or_sync(0xffffffffu, lo_bits)) + __popc(__reduce_or_sync(0xffffffffu, hi_bits)) != (int)cL) {
                    r0 += __popc(__match_any_sync(0xffffffffu, (unsigned long long)__double_as_longlong(t0)) & lt_mask);      // ties (see above)
                    r1 += __popc(__match_any_sync(0xffffffffu, (unsigned long long)__double_as_longlong(t1)) & lt_mask);
                }
                if (h0) *reinterpret_cast<uint4 *>(winw + r0 * 32 + L) = v0;
                if (h1) *reinterpret_cast<uint4 *>(winw + r1 * 32 + L) = v1;
            }
        }
    }
    __syncwarp();
    head.t = ORLG_INF; nxt.t = ORLG_INF;
    if (c > 0) head = win_load(win);
    if (c > 1) nxt = win_load(win + 32);
    wh = 0; wn = c;
    RPH_MARK(13);                                       // rebuild: rank sort
    RTL_IN_REBUILD(rtl_t3_);
    g_rtl_scan_ = rtl_t2_ - rtl_t1_; g_rtl_sort_ = rtl_t3_ - rtl_t2_;
}

// packed integer pre-image of one path's features: start (7, 127 = no block) | length (7) | total free (7) | free runs (6) | slots (5)
__device__ __forceinline__ unsigned feat_pack(int st, int len, int total, int runs, int n) {
    return (unsigned)(st < 0 ? 127 : st) | ((unsigned)(len & 127) << 7) | ((unsigned)total << 14) | ((unsigned)runs << 21) | ((unsigned)n << 27);
}

// TRACE: the requests come from the recorded trace (orlg_set_trace) instead of the Philox generator; with
// RO_POLICY_REPLAY (actions given up front) this replays a reference run through the persistent kernel.
// KIND: DeepRMSA-v0 (block-feature observation, path action), RMSA-v0 or RWA-v0 (no tensor observation, (path, slot) action,
// the reference's first-fit heuristics evaluated on the cached free-slot masks of the candidate paths).
// LPW: envs (lanes in use) per warp, 32 or 8 (compile-time: the 32-lane instances are the code they were before the small-batch
// mapping existed -- a run-time lane count cost the headline instance 3 % through register allocation alone).
// INFO: every step's counters go to ra.info (compile-time: a run-time null check slowed the headline instance by 0.7 %).
template <int ET, int POLICY, bool TRACE = false, int KIND = ORLG_DEEPRMSA, int LPW = 32, bool INFO = false>
__global__ void __launch_bounds__(RO_MAX_THREADS, 1)
deeprmsa_rollout_kernel(const Params p, const RolloutArgs ra) {
    constexpr int KM = 5;
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int wpc = blockDim.x >> 5;
    const int gwarp = blockIdx.x * wpc + wid;                      // warp index over the launch = index of its event slab
    const int env0 = gwarp * LPW;                                  // first env of this warp
    const int env = env0 + lane;
    const bool live = (LPW == 32 || lane < LPW) && env < p.n;
    const int nvalid = min(LPW, p.n - env0);
    const int e = live ? env : p.n - 1;
    const int E = ET > 0 ? ET : p.E;
    unsigned char *warp_area = smem + p.tab_vec * 16 + (size_t)wid * ra.warp_bytes;
    uint4 *sm = reinterpret_cast<uint4 *>(warp_area) + lane;                                   // masks: sm[l * 32]
    double *side_t0 = reinterpret_cast<double *>(warp_area + (size_t)E * 512);                 // [RO_SIDE][32 lanes]
    unsigned long long *side_p0 = reinterpret_cast<unsigned long long *>(warp_area + (size_t)E * 512 + RO_SIDE * 256);
    double *side_t = side_t0 + lane;
    unsigned long long *side_p = side_p0 + lane;
    unsigned char *pool = smem + p.tab_vec * 16 + (size_t)wpc * ra.warp_bytes;
    unsigned long long *tab_bar = reinterpret_cast<unsigned long long *>(pool + (size_t)ra.pool_tiles * ra.tile_bytes);
    unsigned *pool_free = reinterpret_cast<unsigned *>(tab_bar + 1);

    pdl_launch_dependents();
    RPH_INIT();
    RTL_DECL();
    // ---------------- tables: one bulk copy per CTA
    if (tid == 0) {
        mbar_init(tab_bar, 1);
        mbar_expect_tx(tab_bar, (unsigned)p.tab_vec * 16u);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(p.tab_blob), "r"((unsigned)p.tab_vec * 16u),
                       "r"((unsigned)__cvta_generic_to_shared(tab_bar)) : "memory");
        *pool_free = ra.pool_tiles >= 32 ? 0xFFFFFFFFu : ((1u << ra.pool_tiles) - 1u);
    }
    const unsigned short *s_pair_first = reinterpret_cast<const unsigned short *>(smem + p.off_pair_first);
    const unsigned char *s_pair_count = smem + p.off_pair_count;
    const unsigned *s_path_lm = reinterpret_cast<const unsigned *>(smem + p.off_path_lm);
    const unsigned char *s_path_se = smem + p.off_path_se;
    const unsigned long long *s_path_ll = reinterpret_cast<const unsigned long long *>(smem + p.off_path_ll);
    const unsigned char *s_nslots = smem + p.off_nslots;
    const unsigned *s_node_thr = reinterpret_cast<const unsigned *>(smem + p.off_node_thr);
    const float *s_pos = reinterpret_cast<const float *>(smem + p.off_pos);
    const float *s_nsl = reinterpret_cast<const float *>(smem + p.off_nsl);
    const float *s_rcp4 = reinterpret_cast<const float *>(smem + p.off_rcp4);
    const unsigned *s_dbl = reinterpret_cast<const unsigned *>(smem + p.off_dbl);
    pdl_wait();                      // state is touched from here on

    // ---------------- state in: masks -> shared memory (cp.async, coalesced 512 B per link and warp), scalars -> registers
    {
        const uint4 *mr = p.masks + e;
        unsigned sdst = (unsigned)__cvta_generic_to_shared(sm);
        for (int l = 0; l < E; l++) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sdst), "l"(mr) : "memory");
            sdst += 32 * 16;
            mr += p.n;
        }
        cp_async_commit();
    }
    double now = p.now[e];
    double hold = p.cur_hold[e];
    const uint2 rq0 = p.cur_req[e];
    int src = rq0.x & 0xff, dst = (rq0.x >> 8) & 0xff, br = (int)(rq0.x >> 16), sid = (int)rq0.y;
    int ep_proc = (int)p.counters[(size_t)2 * p.n + e], ep_acc = (int)p.counters[(size_t)3 * p.n + e];
    int ep_req = (int)p.counters[(size_t)6 * p.n + e], ep_prov = (int)p.counters[(size_t)7 * p.n + e];
    int d_proc = 0, d_acc = 0, d_req = 0, d_prov = 0;        // deltas of the four running totals over this launch
    unsigned ridx = p.req_index[e];
    unsigned nlive = live ? p.nheap[e] : 0u;                  // live services = table + window + side (a lane without an env: none)
    unsigned n_tab = nlive;
    unsigned err = p.errors[e];
    unsigned long long candw = KIND == ORLG_DEEPRMSA ? *reinterpret_cast<const unsigned long long *>(p.cand + (size_t)e * 8) : 0xFFFFFFFFFFFFFFFFULL;
    const size_t gw = (size_t)gwarp;                             // this warp's slab of the launch-private event storage
    WinEntry *const ev = ra.ev + gw * (size_t)(p.heap_cap + 2 * RO_WCAP) * 32 + lane;       // table rows [0, heap_cap)
    WinEntry *const win = ev + (size_t)(p.heap_cap + RO_WCAP) * 32;
#pragma unroll
    for (int s = 0; s < RO_SIDE; s++) side_t[s * 32] = ORLG_INF;
    if (ridx != p.lockstep_ridx) err |= ORLG_ERR_LOCKSTEP;
    unsigned wh = 0, wn = 0;
    double tmin_tab = ORLG_INF, side_min = ORLG_INF, hzn = now + ra.span;
    WinEntry head, nxt;
    head.t = ORLG_INF; head.p = 0; nxt.t = ORLG_INF; nxt.p = 0;
    cp_async_wait<0>();
    __syncthreads();                 // pool word + table barrier initialised by thread 0 ...
    mbar_wait(tab_bar, 0);           // ... and the tables have landed
    if (env0 >= p.n) return;         // a warp without environments (no CTA-wide barrier below)
    if (ra.resume) {
        // ---------------- the previous launch left the window state behind: nothing to convert or rebuild
        if (live) {
            n_tab = ra.st_ntab[e]; wh = ra.st_wh[e]; wn = ra.st_wn[e];
            tmin_tab = ra.st_tmin[e]; hzn = ra.st_hzn[e];
#pragma unroll
            for (int s = 0; s < RO_SIDE; s++) {
                const double ts = ra.st_side_t[(size_t)s * p.n + e];
                side_t[s * 32] = ts; side_p[s * 32] = ra.st_side_p[(size_t)s * p.n + e];
                side_min = dmin(side_min, ts);
            }
            if (wh < wn) head = win_load(win + wh * 32);
            if (wh + 1 < wn) nxt = win_load(win + (wh + 1) * 32);
        }
    } else {
        // ---------------- event tables in: canonical [env][slot] -> lane-interleaved [slot][lane].  Thread per env: the loads
        // walk the env's own rows (one L2 fetch per 128-byte line, the rest are L1 hits), the stores coalesce.
        if (live) {
            ra.st_ncanon[e] = n_tab;
            const double *__restrict__ ct = p.ev_time + (size_t)e * p.heap_cap;
            const unsigned long long *__restrict__ cp = p.ev_pay + (size_t)e * p.heap_cap;
            for (unsigned s0 = 0; s0 < n_tab; s0 += 8) {             // heap_cap is a multiple of 16: the vector loads stay inside the table
                double2 a[4];
                ulonglong2 b[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    a[i] = *reinterpret_cast<const double2 *>(ct + s0 + 2 * i);
                    b[i] = *reinterpret_cast<const ulonglong2 *>(cp + s0 + 2 * i);
                }
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    win_store(ev + (s0 + 2 * i) * 32, a[i].x, b[i].x);
                    win_store(ev + (s0 + 2 * i + 1) * 32, a[i].y, b[i].y);
                }
            }
            if (n_tab) tmin_tab = 0.0;       // "a table entry is due": the first step of the launch builds the window (one rebuild site)
        }
    }
    int npaths_cur = min((int)s_pair_count[src * p.N + dst], KM);       // candidate paths of the pending request

    const unsigned long long gid = (unsigned long long)(p.env_id_base + e);
    const unsigned k0 = (unsigned)p.seed, k1 = (unsigned)(p.seed >> 32);
    const unsigned n_act = (unsigned)(p.k) + (p.allow_rejection ? 1u : 0u);     // path actions (DeepRMSA: j = 1)

    // release of the window head; the entry after it was requested one pop earlier.  (Tried and measured slower: a
    // straight-line "head, then nxt, then a synchronous loop" form that never waits on its own load -- the lanes of a warp
    // then pop in different copies of the release code: 9.4 -> 10.3 us per step.)
#define RO_POP_DUE()                                                                                              \
    while (head.t <= now) {                                                                                      \
        const int rs_ = svc_start(head.p);                                                                       \
        ro_path_update<true>(sm, s_path_lm[svc_row(head.p)], bits_range_short(rs_, svc_slots(head.p)));          \
        nlive--; wh++;                                                                                           \
        head = nxt;                                                                                              \
        if (wh + 1 < wn) nxt = win_load(win + (wh + 1) * 32); else nxt.t = ORLG_INF;                             \
    }

    RPH_MARK(8);                     // entry: state in + first window build
    RTL_SET(1);
    // cached per candidate path of the PENDING request: first-fit start as the policy defines it (candw, one byte per path,
    // CAND_NONE = none), free slots (candt) and hop count (candh) for the least-loaded / fewest-hops heuristics.
    // DeepRMSA-v0 handles keep candw in the canonical state; the other kinds compute it in an extra phase-C pass (t = -1).
    unsigned long long candt = 0;
    unsigned candh = 0;
    for (int t = (KIND == ORLG_DEEPRMSA ? 0 : -1); t < ra.T; t++) {
        bool done = false;
        int npaths = 0;
        unsigned rec_flags = 0;          // action (low 16 bits) | accepted << 28, for the packed record
        if (t < 0) {
            // ---- first pass of a non-DeepRMSA launch: only the candidate cache of the pending request is built
            if (live) {
                npaths = min((int)s_pair_count[src * p.N + dst], KM);
                npaths_cur = npaths;
            }
        } else if (live) {
            // ---- the next request (rmsa_env.py:545-561): a pure function of (seed, global env id, request index)
            double e_iat = 0.0, e_hold = 0.0, t_arrival = now;
            int p_src = 0, p_dst = 1, p_br = KIND == ORLG_RWA ? 0 : p.br_lo;
            if (TRACE) {
                if ((long long)ridx < p.trace_len) {
                    const orlg_request r = p.trace[(size_t)e * p.trace_len + ridx];
                    t_arrival = r.arrival; e_hold = r.holding; p_src = r.src; p_dst = r.dst;
                    p_br = KIND == ORLG_RWA ? 0 : min(max(r.bit_rate, 0), 127);
                    if (KIND != ORLG_RWA && r.bit_rate > 127) err |= ORLG_ERR_TRACE_RANGE;       // beyond the slot-count table of this kernel
                } else {
                    err |= ORLG_ERR_TRACE_EXHAUSTED;
                }
            } else {
                uint32_t rc_[4] = {ridx, 0u, (uint32_t)gid, 0u};
                philox4x32_10(rc_, k0, k1);
                e_iat = __dmul_rn(neg_log_u32(rc_[0]), p.mean_iat);
                e_hold = __dmul_rn(neg_log_u32(rc_[1]), p.mean_holding);
                const int nn = p.N;
                p_src = pick_thr_bsearch(s_node_thr, nn, p.node_top_step, rc_[2]);
                const unsigned lo = p_src ? s_node_thr[p_src - 1] : 0u;
                const unsigned long long hi = (p_src == nn - 1) ? 4294967296ULL : (unsigned long long)s_node_thr[p_src];
                const unsigned long long mass = hi - lo;
                unsigned long long tt = ((unsigned long long)rc_[3] * (4294967296ULL - mass)) >> 32;
                if (tt >= lo) tt += mass;
                p_dst = pick_thr_bsearch(s_node_thr, nn, p.node_top_step, (unsigned)tt);
                if (p_dst == p_src) p_dst = (p_src + 1) % nn;
                if (KIND != ORLG_RWA) {
                    uint32_t rd_[4] = {ridx, 0u, (uint32_t)gid, 1u};
                    philox4x32_10(rd_, k0, k1);
                    p_br = p.br_lo + (int)__umulhi(rd_[0], (unsigned)p.br_span);
                }
            }
            npaths = min((int)s_pair_count[p_src * p.N + p_dst], KM);

            RPH_MARK(0);             // request draw
            // ---- the policy's action on the pending request: DeepRMSA a path index (j = 1), RMSA / RWA (path, slot)
            const int pair = src * p.N + dst;
            const int np_cur = (int)s_pair_count[pair];
            int act = p.k, act_slot = p.S;                       // the reject action
            bool checked = false;                                // the action came with a first-fit start that is known to be free
            if (POLICY == RO_POLICY_RANDOM) {                    // orlg_random_actions: Philox stream 2, same counter
                uint32_t ra_[4] = {ridx, 0u, (uint32_t)gid, 2u};
                philox4x32_10(ra_, k0, k1);
                act = (int)__umulhi(ra_[0], n_act);
                if (KIND != ORLG_DEEPRMSA) act_slot = (int)__umulhi(ra_[1], (unsigned)p.S + (p.allow_rejection ? 1u : 0u));
            } else if (POLICY == RO_POLICY_REPLAY) {             // a recorded action sequence
                if (KIND == ORLG_DEEPRMSA) act = ra.actions[(size_t)t * p.n + env];
                else { act = ra.actions[((size_t)t * p.n + env) * 2]; act_slot = ra.actions[((size_t)t * p.n + env) * 2 + 1]; }
            } else if (KIND == ORLG_DEEPRMSA) {
                if (POLICY == RO_POLICY_SP_FF) {                 // deeprmsa_env.py:135-143
                    act = (!p.allow_rejection || (candw & 0xffu) != CAND_NONE) ? 0 : p.k;
                } else {                                         // deeprmsa_env.py:146-155
                    for (int q = npaths_cur - 1; q >= 0; q--)
                        if (((candw >> (8 * q)) & 0xffu) != CAND_NONE) act = q;
                }
            } else {
                // rmsa_env.py:747-803 / rwa_env.py:425-502 on the cached first-fit starts (which already honour the
                // reference's range(0, S - n) / range(W - 1, 0, -1) scans)
                checked = true;
                if (POLICY == RO_POLICY_SP_FF) {
                    if (npaths_cur > 0 && (candw & 0xffu) != CAND_NONE) { act = 0; act_slot = (int)(candw & 0xffu); }
                } else if (POLICY == RO_POLICY_LLP_FF) {         // most free slots among the paths that fit (first wins ties)
                    int best = KIND == ORLG_RWA ? -1 : 0;
                    for (int q = 0; q < npaths_cur; q++) {
                        const unsigned st = (unsigned)((candw >> (8 * q)) & 0xffu);
                        const int fr = (int)((candt >> (8 * q)) & 0xffu);
                        if (st != CAND_NONE && fr > best) { best = fr; act = q; act_slot = (int)st; }
                    }
                } else if (KIND == ORLG_RWA) {                   // SAP-FF / SAP-LF: fewest hops among the paths with a free wavelength
                    int best_hops = 0x7fffffff;
                    for (int q = 0; q < npaths_cur; q++) {
                        const unsigned st = (unsigned)((candw >> (8 * q)) & 0xffu);
                        const int hops = (int)((candh >> (4 * q)) & 0xfu);
                        if (hops < best_hops && st != CAND_NONE) { best_hops = hops; act = q; act_slot = (int)st; }
                    }
                } else {                                         // RMSA SAP-FF: first path (k order) that fits
                    for (int q = npaths_cur - 1; q >= 0; q--) {
                        const unsigned st = (unsigned)((candw >> (8 * q)) & 0xffu);
                        if (st != CAND_NONE) { act = q; act_slot = (int)st; }
                    }
                }
            }
            if (POLICY != RO_POLICY_REPLAY && ra.actions) {
                if (KIND == ORLG_DEEPRMSA) ra.actions[(size_t)t * p.n + env] = act;
                else *reinterpret_cast<int2 *>(ra.actions + ((size_t)t * p.n + env) * 2) = make_int2(act, act_slot);
            }

            // ---- Phase A (rmsa_env.py:163-209, deeprmsa_env.py:48-58, rwa_env.py:101-136)
            bool accepted = false;
            int a_start = 0;
            if (KIND == ORLG_RWA && p.act_hist) {                // self.actions_output[path, wavelength] += 1 (rwa_env.py:103)
                const int R = p.k + p.allow_rejection, Cn = p.S + p.allow_rejection;
                if (act >= 0 && act < R && act_slot >= 0 && act_slot < Cn) {
                    atomicAdd(p.act_hist + (size_t)act * p.n + env, 1);               // fire-and-forget (RED): nothing waits for it
                    atomicAdd(p.act_hist + (size_t)(R + act_slot) * p.n + env, 1);
                } else {
                    err |= ORLG_ERR_NO_SUCH_PATH;
                }
            }
            if (act >= 0 && act < p.k && (KIND == ORLG_DEEPRMSA || (act_slot >= 0 && act_slot < p.S))) {
                if (act < np_cur) {
                    const int a_row = s_pair_first[pair] + act;
                    const int a_n = KIND == ORLG_RWA ? 1 : s_nslots[s_path_se[a_row] * 128 + br];
                    const unsigned a_lm = s_path_lm[a_row];
                    bool fits;
                    if (KIND == ORLG_DEEPRMSA) {                 // the cached block start decides
                        const unsigned st = (unsigned)((candw >> (8 * act)) & 0xffu);
                        fits = st != CAND_NONE;
                        a_start = (int)st;
                    } else if (checked) {
                        fits = true; a_start = act_slot;
                    } else {                                     // is_path_free (rmsa_env.py:623-636, rwa_env.py:385-400) on the shared-memory masks
                        a_start = act_slot;
                        fits = a_start + a_n <= p.S;
                        if (fits) {
                            Bits F = bits_ones();
                            unsigned m = a_lm;
                            while (m) {
                                const int l = __ffs(m) - 1;
                                m &= m - 1;
                                F = bits_and(F, bits_from(sm[l * 32]));
                            }
                            fits = bits_contains(F, bits_range_short(a_start, a_n));
                        }
                    }
                    if (fits) {
                        if (nlive + 1 > (unsigned)p.heap_cap) {
                            err |= ORLG_ERR_HEAP_OVERFLOW;
                        } else {
                            ro_path_update<false>(sm, a_lm, bits_range_short(a_start, a_n));      // _provision_path
                            const double rel = __dadd_rn(now, hold);
                            const unsigned long long pl = pack_service(a_row, a_start, a_n, 0, sid);
                            bool in_side = false;
                            if (rel <= hzn) {                    // expires inside the window: side buffer
#pragma unroll
                                for (int s = 0; s < RO_SIDE; s++) {
                                    if (!in_side && !(side_t[s * 32] < ORLG_INF)) {
                                        side_t[s * 32] = rel; side_p[s * 32] = pl; in_side = true;
                                    }
                                }
                                if (in_side) side_min = dmin(side_min, rel);
                            }
                            if (!in_side) {                      // table push: two stores
                                win_store(ev + n_tab * 32, rel, pl); n_tab++;
                                tmin_tab = dmin(tmin_tab, rel);
                            }
                            nlive++;
                            d_acc += 1; ep_acc += 1;
                            if (KIND != ORLG_RWA) { d_prov += br; ep_prov += br; }
                            accepted = true;
                        }
                    }
                } else {
                    err |= ORLG_ERR_NO_SUCH_PATH;
                }
            }
            if (KIND == ORLG_RWA) { d_proc += 1; ep_proc += 1; }             // rwa_env.py:135-136: counted in step
            if (ra.reward) ra.reward[(size_t)t * p.n + env] = accepted ? 1.0f : (KIND == ORLG_DEEPRMSA ? -1.0f : 0.0f);
            rec_flags = ((unsigned)act & 0xffffu) | (accepted ? (1u << 28) : 0u);

            RPH_MARK(1);             // action + phase A
            // ---- Phase B: _next_service (rmsa_env.py:545-597, rwa_env.py:258-288)
            now = TRACE ? t_arrival : __dadd_rn(now, e_iat);
            hold = e_hold; src = p_src; dst = p_dst; br = p_br;
            ridx++;
            sid = ep_proc;
            if (KIND != ORLG_RWA) { d_proc += 1; ep_proc += 1; d_req += br; ep_req += br; }
            npaths_cur = npaths;
            RO_POP_DUE();
            if (side_min <= now) {
                double m2 = ORLG_INF;
#pragma unroll
                for (int s = 0; s < RO_SIDE; s++) {
                    const double ts = side_t[s * 32];
                    if (ts <= now) {
                        const unsigned long long pl = side_p[s * 32];
                        const int rs = svc_start(pl);
                        ro_path_update<true>(sm, s_path_lm[svc_row(pl)], bits_range_short(rs, svc_slots(pl)));
                        side_t[s * 32] = ORLG_INF;
                        nlive--;
                    } else {
                        m2 = dmin(m2, ts);
                    }
                }
                side_min = m2;
            }
        }
        RPH_MARK(2);                 // phase B + window / side releases
        // ---- a table entry is due somewhere in the warp: every lane re-centres its window (~1 step in 30)
        for (int tries = 0; t >= 0 && __any_sync(0xffffffffu, live && tmin_tab <= now); tries++) {
            RPH_COUNT(15);
            // a retry means the window filled up before every due service was reached: shorter horizon, down to the clock itself
            hzn = tries < 60 ? __dadd_rn(now, __dmul_rn(ra.span, __longlong_as_double((long long)(1023 - tries) << 52))) : now;
            RTL_REBUILD_BEGIN();
            unsigned long long g_rtl_scan_ = 0, g_rtl_sort_ = 0;
            ro_rebuild(ev, (unsigned)p.heap_cap, side_t, side_p, n_tab, wh, wn, tmin_tab, side_min, hzn, head, nxt, lane, g_rtl_scan_, g_rtl_sort_);
            RO_POP_DUE();
            RTL_REBUILD_END();
        }
        RPH_MARK(3);                 // rebuild
        if (live && t >= 0) {
            done = (ep_proc == p.episode_length);
            if (INFO) {
                // the counters as the reference builds `info` (rmsa_env.py:234-248, rwa_env.py:141-152): before _next_service,
                // so RMSA / DeepRMSA take back the next request that phase B has already counted.  The running totals are
                // the launch-entry values (unchanged in HBM until the exit below) plus this launch's deltas, re-read here
                // rather than held in registers across the step loop.  One env = 64 contiguous bytes, a warp 2 KB.
                const int nq = KIND == ORLG_RWA ? 0 : 1, nbr = KIND == ORLG_RWA ? 0 : br;
                const long long *c = p.counters + env;
                longlong2 *o = reinterpret_cast<longlong2 *>(ra.info + ((size_t)t * p.n + env) * 8);
                o[0] = make_longlong2(c[0] + d_proc - nq, c[(size_t)p.n] + d_acc);
                o[1] = make_longlong2(ep_proc - nq, ep_acc);
                o[2] = make_longlong2(c[(size_t)4 * p.n] + d_req - nbr, c[(size_t)5 * p.n] + d_prov);
                o[3] = make_longlong2(ep_req - nbr, ep_prov);
            }
            if (done && p.auto_reset) {                          // rmsa_env.py:285-330, rwa_env.py:164-179
                ep_acc = 0; ep_prov = 0;
                if (KIND == ORLG_RWA) { ep_proc = 0; ep_req = 0; } else { ep_proc = 1; ep_req = br; }
            }
            if (ra.done) ra.done[(size_t)t * p.n + env] = done ? 1 : 0;
        }

        // ---- Phase C: free-slot mask of every candidate path of the pending request (get_available_slots,
        // rmsa_env.py:638-649), then DeepRMSA's block features (deeprmsa_env.py:60-121) / the heuristics' first-fit starts.
        // One ROLLED loop over the candidate paths (AND over the path's own hops, then its features): the unrolled
        // link-sweep form was ~1300 instructions of straight-line code in a loop body that overflows the 32 KB
        // instruction cache; this one is a quarter of that and executes fewer instructions as well.
        unsigned feat[KM];
#pragma unroll
        for (int q = 0; q < KM; q++) feat[q] = 0;
        if (live) {
            unsigned long long cand_out = 0xFFFFFFFFFFFFFFFFULL, tot_out = 0;
            unsigned hops_out = 0;
            const int first = s_pair_first[src * p.N + dst];
#pragma unroll 1
            for (int q = 0; q < KM; q++) {
                const bool have = q < npaths;
                const int row = have ? first + q : first;
                unsigned lm = have ? s_path_lm[row] : 0u;
                Bits A = have ? bits_ones() : Bits{{0u, 0u, 0u, 0u}};
                while (lm) {                     // four hops per pass, their loads in flight together (AND is idempotent: a short
                    const int l0 = __ffs(lm) - 1;  // path repeats its first hop)
                    lm &= lm - 1;
                    const int l1 = lm ? __ffs(lm) - 1 : l0;
                    lm &= lm - 1;
                    const int l2 = lm ? __ffs(lm) - 1 : l0;
                    lm &= lm - 1;
                    const int l3 = lm ? __ffs(lm) - 1 : l0;
                    lm &= lm - 1;
                    const uint4 v0 = sm[l0 * 32], v1 = sm[l1 * 32], v2 = sm[l2 * 32], v3 = sm[l3 * 32];
                    A.w[0] &= v0.x & v1.x; A.w[1] &= v0.y & v1.y; A.w[2] &= v0.z & v1.z; A.w[3] &= v0.w & v1.w;
                    A.w[0] &= v2.x & v3.x; A.w[1] &= v2.y & v3.y; A.w[2] &= v2.z & v3.z; A.w[3] &= v2.w & v3.w;
                }
                int st;
                unsigned f = 0;
                if (KIND == ORLG_DEEPRMSA) {
                    const int n = s_nslots[s_path_se[row] * 128 + br];
                    const Bits B = bits_runs_ge_sched(A, s_dbl[n]);
                    st = bits_ffs_flat(B);
                    const int fe = bits_ffs_flat(bits_andnot(B, bits_shr1(B)));
                    const int total = bits_popc(A);
                    const int runs = bits_popc(bits_andnot(A, bits_shl1(A)));
                    f = feat_pack(st, fe - st + n, total, runs, n);
                } else {
                    if (KIND == ORLG_RWA) {
                        if (POLICY == RO_POLICY_SAP_LF) { Bits L = A; L.w[0] &= ~1u; st = bits_fls(L); }     // range(W - 1, 0, -1): never wavelength 0
                        else st = bits_ffs_flat(A);
                        if (have) hops_out |= (unsigned)(s_path_ll[row] >> 60) << (4 * q);
                    } else {                                     // first fit over range(0, S - n): the last feasible start is never tried
                        const int n = s_nslots[s_path_se[row] * 128 + br];
                        const Bits B = bits_and(bits_runs_ge_sched(A, s_dbl[n]), bits_range(0, max(p.S - n, 0)));
                        st = bits_ffs_flat(B);
                    }
                    tot_out |= (unsigned long long)(bits_popc(A) & 0xff) << (8 * q);
                }
                cand_out = st >= 0 ? ((cand_out & ~(0xFFULL << (8 * q))) | ((unsigned long long)st << (8 * q))) : cand_out;
#pragma unroll
                for (int i = 0; i < KM; i++) feat[i] = i == q ? f : feat[i];
            }
            if (KIND != ORLG_DEEPRMSA) { candt = tot_out; candh = hops_out; }
            candw = cand_out;
        }
        RPH_MARK(5);                 // features
        if (t < 0) continue;
        if (KIND == ORLG_DEEPRMSA && ra.packed && live) {        // 32 bytes per env-step, 1 KB contiguous per warp
            uint4 *rec = ra.packed + ((size_t)t * p.n + env) * 2;
            rec[0] = make_uint4(feat[0], feat[1], feat[2], feat[3]);
            rec[1] = make_uint4(feat[4], (unsigned)br | ((unsigned)src << 8) | ((unsigned)dst << 16) | ((unsigned)npaths << 24) |
                                             (rec_flags & (1u << 28)) | (done ? (1u << 29) : 0u),
                                rec_flags & 0xffffu, 0u);
        }
        if (KIND == ORLG_DEEPRMSA && ra.obs) {
            // ---- the warp's 32 rows = one contiguous run of obs[t]: written to a pool tile, copied out by one bulk (TMA) store
            const unsigned tile = ro_tile_acquire(pool_free, lane);
            unsigned char *stage = pool + (size_t)tile * ra.tile_bytes;
            RPH_MARK(4);             // tile acquisition
            if (live) {
                // row = [bit rate / 100 | one-hot(min(src, dst)) | one-hot(max(src, dst)) | 5 x 5 features]: 1 + 2N is odd, so the
                // last one-hot element pairs with the first feature and the whole tail goes out as 13 aligned float2 stores
                float *so32 = reinterpret_cast<float *>(stage) + (size_t)lane * p.obs_dim;
                float2 *r2 = reinterpret_cast<float2 *>(so32);
                const int lo_n = min(src, dst), hi_n = max(src, dst);
                for (int q = 0; q < p.N; q++) r2[q] = make_float2(0.0f, 0.0f);
                float v[2 + 5 * KM];
                v[0] = hi_n == p.N - 1 ? 1.0f : 0.0f;
                v[1 + 5 * KM] = 0.0f;
#pragma unroll
                for (int q = 0; q < KM; q++) {
                    const unsigned f = feat[q];
                    const int st = (int)(f & 127u), len = (int)((f >> 7) & 127u), total = (int)((f >> 14) & 127u);
                    const int runs = (int)((f >> 21) & 63u), n = (int)(f >> 27);
                    const bool have = q < npaths, blk = st != 127;
                    v[1 + 5 * q] = blk ? s_pos[blk ? st : 0] : -1.0f;
                    v[2 + 5 * q] = blk ? (float)(len - 8) * 0.125f : -1.0f;
                    v[3 + 5 * q] = have ? s_nsl[n] : -1.0f;
                    v[4 + 5 * q] = have ? s_pos[total] : -1.0f;
                    v[5 + 5 * q] = runs > 0 ? (float)(total - 4 * runs) * s_rcp4[runs] : -1.0f;   // x * fl(1/y): <= 1.5 ulp
                }
#pragma unroll
                for (int i = 0; i < (1 + 5 * KM + 1) / 2; i++) r2[p.N + i] = make_float2(v[2 * i], v[2 * i + 1]);
                so32[0] = __fdiv_rn((float)br, 100.0f);
                so32[1 + lo_n] = 1.0f;
                if (hi_n != p.N - 1) so32[1 + p.N + hi_n] = 1.0f;
            }
            RPH_MARK(6);             // observation rows into the tile
            {
                float *g = ra.obs + ((size_t)t * p.n + env0) * p.obs_dim;
                const int total_el = nvalid * p.obs_dim;
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if ((reinterpret_cast<size_t>(g) & 15) == 0 && (total_el & 3) == 0) {
                    if (lane == 0) {     // one bulk (TMA) store for the warp's rows; the tile is free once it has been read
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                     ::"l"(g), "r"((unsigned)__cvta_generic_to_shared(stage)), "r"((unsigned)total_el * 4u) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    }
                } else {
                    const float *sv = reinterpret_cast<const float *>(stage);
                    for (int q = lane; q < total_el; q += 32) g[q] = sv[q];
                }
            }
            ro_tile_release(pool_free, tile, lane);
        }
        RPH_MARK(7);                 // observation rows: tile write + copy out
    }
#undef RO_POP_DUE
    RTL_SET(2);

    // ---------------- state out: masks, scalars and the window state.  The event storage stays in the launch-private form
    // (the next orlg_rollout resumes from it; ro_canonicalize_kernel rebuilds the canonical tables for everybody else).
    if (live) {
        ra.st_ntab[env] = n_tab; ra.st_wh[env] = wh; ra.st_wn[env] = wn;
        ra.st_tmin[env] = tmin_tab; ra.st_hzn[env] = hzn;
#pragma unroll
        for (int s = 0; s < RO_SIDE; s++) {
            ra.st_side_t[(size_t)s * p.n + env] = side_t[s * 32];
            ra.st_side_p[(size_t)s * p.n + env] = side_p[s * 32];
        }
        uint4 *mw = p.masks + env;
        for (int l = 0; l < E; l++) mw[(size_t)l * p.n] = sm[l * 32];
        p.now[env] = now;
        p.cur_hold[env] = hold;
        p.cur_req[env] = make_uint2((unsigned)src | ((unsigned)dst << 8) | ((unsigned)br << 16), (unsigned)sid);
        {                                // the four running totals: all loads before the first store (one round trip, not four)
            const auto c0 = p.counters[(size_t)0 * p.n + env], c1 = p.counters[(size_t)1 * p.n + env];
            const auto c4 = p.counters[(size_t)4 * p.n + env], c5 = p.counters[(size_t)5 * p.n + env];
            p.counters[(size_t)0 * p.n + env] = c0 + d_proc;
            p.counters[(size_t)1 * p.n + env] = c1 + d_acc;
            p.counters[(size_t)4 * p.n + env] = c4 + d_req;
            p.counters[(size_t)5 * p.n + env] = c5 + d_prov;
        }
        p.counters[(size_t)2 * p.n + env] = ep_proc;
        p.counters[(size_t)3 * p.n + env] = ep_acc;
        p.counters[(size_t)6 * p.n + env] = ep_req;
        p.counters[(size_t)7 * p.n + env] = ep_prov;
        p.req_index[env] = ridx;
        p.nheap[env] = nlive;
        p.errors[env] = err;
        if (KIND == ORLG_DEEPRMSA) *reinterpret_cast<unsigned long long *>(p.cand + (size_t)env * 8) = candw;
    }
    RPH_MARK(9);                     // exit: state out
    RTL_SET(3);
    RTL_FLUSH((unsigned)gwarp);
}

// Launch-private event storage -> canonical release-event tables (orlg_device.cuh): window and side entries go back to the
// table, the table is written out [env][slot] with +INF above, and the directory / tail bound / global bound are rebuilt.
// Thread per env; launched by the host before any entry point other than orlg_rollout touches the events.
__global__ void __launch_bounds__(128) ro_canonicalize_kernel(const Params p, const RolloutArgs ra) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    const int lane = env % ra.lpw;                               // the rollout kernel's mapping: slab env / lpw, lane env % lpw
    const size_t gw = (size_t)(env / ra.lpw);
    WinEntry *const ev = ra.ev + gw * (size_t)(p.heap_cap + 2 * RO_WCAP) * 32 + lane;
    const WinEntry *const win = ev + (size_t)(p.heap_cap + RO_WCAP) * 32;
    unsigned n_tab = ra.st_ntab[env];
    const unsigned wh = ra.st_wh[env], wn = ra.st_wn[env], n_entry = ra.st_ncanon[env];
    unsigned err = 0;
    for (unsigned j = wh; j < wn; j++) {                         // window + side entries back to the table
        const WinEntry w = win_load(win + j * 32);
        win_store(ev + n_tab * 32, w.t, w.p); n_tab++;
    }
#pragma unroll
    for (int s = 0; s < RO_SIDE; s++) {
        const double ts = ra.st_side_t[(size_t)s * p.n + env];
        if (ts < ORLG_INF) { win_store(ev + n_tab * 32, ts, ra.st_side_p[(size_t)s * p.n + env]); n_tab++; }
    }
    if (n_tab != p.nheap[env]) err |= ORLG_ERR_LOCKSTEP;        // internal consistency (never expected)
    // lane-interleaved -> canonical [env][slot]: coalesced loads, each thread writes its own rows (16-byte stores)
    double *ev_t = p.ev_time + (size_t)env * p.heap_cap;
    unsigned long long *ev_p = p.ev_pay + (size_t)env * p.heap_cap;
    float *gmin = p.ev_gmin + (size_t)env * p.ev_groups;
    const unsigned n_fill = max(n_tab, n_entry);                 // "every slot >= n holds +INF"
    for (unsigned s0 = 0; s0 < n_fill; s0 += 8) {
        double tt[8];
        unsigned long long pp[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const bool in = s0 + i < n_tab;
            WinEntry w;
            w.t = ORLG_INF; w.p = 0ULL;
            if (in) w = win_load(ev + (s0 + i) * 32);
            tt[i] = w.t; pp[i] = w.p;
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            *reinterpret_cast<double2 *>(ev_t + s0 + 2 * i) = make_double2(tt[2 * i], tt[2 * i + 1]);
            *reinterpret_cast<ulonglong2 *>(ev_p + s0 + 2 * i) = make_ulonglong2(pp[2 * i], pp[2 * i + 1]);
        }
    }
    // directory: float lower bound per FULL group below the tail group, +INF from the tail group on
    const int tail_g = n_tab ? (int)((n_tab - 1) / EV_GROUP) : 0;
    double all_min = ORLG_INF, tail_min = ORLG_INF;
    for (int g = 0; g <= tail_g && n_tab; g++) {
        double m = ORLG_INF;
#pragma unroll
        for (int q = 0; q < EV_GROUP; q++) {
            const unsigned sl = (unsigned)(g * EV_GROUP + q);
            m = dmin(m, sl < n_tab ? *reinterpret_cast<const double *>(ev + sl * 32) : ORLG_INF);
        }
        if (g < tail_g) gmin[g] = lower_f32(m); else tail_min = m;
        all_min = dmin(all_min, g < tail_g ? (double)lower_f32(m) : m);
    }
    for (int g = tail_g; g < p.ev_groups; g++) gmin[g] = ORLG_INF_F;
    p.heap_min[env] = all_min;
    p.ev_tail[env] = tail_min;
    if (err) p.errors[env] |= err;
}

}  // namespace orlg
