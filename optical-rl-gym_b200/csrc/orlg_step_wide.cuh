// orlg_step_wide.cuh -- step / heuristic / export kernels for topologies beyond the NSFNET class:
// any number of links (path -> link lists in CSR form instead of 32-bit link bitmaps), up to 512 slots
// per link (NWV = 1..4 128-bit word groups per (core, link)), up to 31 cores, k <= 16 candidate paths.
// Covers BASELINE.json configs[3] (RMSA-v0, 100 nodes / 300 links, 320 slots, k = 10) and configs[4]
// (RMCSA-v0, 7 cores x 320 slots).  Same semantics, same state arrays and the same release-event table as
// step_kernel (orlg_kernels.cuh); one thread per environment, masks accessed in place:
//     masks[(env * C * E + core * E + link) * wstride + v]   (uint4; env-major: an entry's words share one DRAM burst,
//     an env's entries one page -- every thread walks its OWN path, so the [link][env] layout of the NSFNET-class kernels
//     would put each of its accesses on a different 2 MB page)
// The hop lists and wide_path_free read both mask layouts (mask_index), so the heuristic kernel here serves every handle.
#pragma once
#include "orlg_kernels.cuh"

namespace orlg {

// get_available_slots (rmsa_env.py:638-649): AND of the path's link masks.  Four hops at a time: the four link indices are
// fetched together, then all 4 x NWV mask words are requested before any is used (2 dependent round trips per 4 hops instead
// of 2 per hop: the kernel is latency-bound, every lane walks its own path).
template <int NWV>
__device__ __forceinline__ WBits<NWV> wide_path_free(const Params &p, int env, int row, int core) {
    WBits<NWV> a = bits_ones<NWV>();
    const int h0 = p.path_link_ptr[row], h1 = p.path_link_ptr[row + 1];
    const size_t vs = p.wstride ? 1 : (size_t)p.n;          // distance between the word groups of one entry (mask_index)
    const uint4 ones = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    for (int h = h0; h < h1; h += 4) {
        int l[4];
#pragma unroll
        for (int i = 0; i < 4; i++) l[i] = h + i < h1 ? (int)p.path_links16[h + i] : -1;
        uint4 x[4][NWV];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint4 *m = p.masks + mask_index(p, core * p.E + max(l[i], 0), 0, env);
#pragma unroll
            for (int v = 0; v < NWV; v++) x[i][v] = l[i] >= 0 ? __ldcg(m + v * vs) : ones;
        }
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int v = 0; v < NWV; v++) {
                a.w[4 * v] &= x[i][v].x; a.w[4 * v + 1] &= x[i][v].y; a.w[4 * v + 2] &= x[i][v].z; a.w[4 * v + 3] &= x[i][v].w;
            }
    }
    return a;
}

// _provision_path / _release_path on the masks: the slot range [start, start + n) of every link of the path is cleared
// (provision) or set (release) with fire-and-forget 32-bit reductions (RED.AND / RED.OR at the L2): no mask word is LOADED for an
// update, so a release -- whose links were last touched many steps ago, i.e. a DRAM miss per link -- costs no round trip at
// all, and updates of different services commute.  Every mask READ of these kernels bypasses the L1 (__ldcg), so a thread
// that reads a link after updating it (DeepRMSA's observation) sees its own reductions.
template <int NWV>
__device__ __forceinline__ void wide_path_update(const Params &p, int env, int row, int core, int start, int n, bool set) {
    const int h0 = p.path_link_ptr[row], h1 = p.path_link_ptr[row + 1];
    const int w0 = start >> 5, w1 = (start + n - 1) >> 5;          // 32-bit words the range touches (n >= 1)
    const size_t vs = p.wstride ? 1 : (size_t)p.n;
    for (int h = h0; h < h1; h += 4) {
        int l[4];
#pragma unroll
        for (int i = 0; i < 4; i++) l[i] = h + i < h1 ? (int)p.path_links16[h + i] : -1;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            if (l[i] < 0) continue;
            unsigned *m = reinterpret_cast<unsigned *>(p.masks + mask_index(p, core * p.E + l[i], 0, env));
            for (int w = w0; w <= w1; w++) {
                const int lo = max(start - 32 * w, 0), hi = min(start + n - 32 * w, 32);
                const unsigned bits = (hi >= 32 ? 0xFFFFFFFFu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
                unsigned *addr = m + ((size_t)(w >> 2) * vs) * 4 + (w & 3);
                if (set) atomicOr(addr, bits); else atomicAnd(addr, ~bits);
            }
        }
    }
}

__device__ __forceinline__ int wide_nslots(const Params &p, int se, int br) { return p.nslots[se * (p.br_max + 1) + br]; }

// ---------------------------------------------------------------- row f1 (float statistics) on the wide layout
__device__ __forceinline__ int wide_hops(const Params &p, int row) { return p.path_link_ptr[row + 1] - p.path_link_ptr[row]; }

// The integer terms of _get_network_compactness (rmsa_env.py:699-744), kept current so that the compactness needs no pass over
// every link.  They live behind sum_nh in the same allocation (orlg_enable_stats on a wide handle other than RWA-v0), which
// leaves the kernel parameter block -- and with it the code of every other kernel -- as it was:
//     int2     [n][C]    per core, the sums over its links: x = occupied (spans), y = free runs inside the spans
//     unsigned [n][C*E]  per (core, link): span | free runs inside the span << 16
__device__ __forceinline__ int2 *nc_totals(const Params &p) { return reinterpret_cast<int2 *>(p.sum_nh + p.n); }
__device__ __forceinline__ unsigned *nc_links(const Params &p) { return reinterpret_cast<unsigned *>(nc_totals(p) + (size_t)p.n * p.C); }

// _get_network_compactness of one core from its kept integer sums (equal to a pass over every link: exact integers)
__device__ __forceinline__ double wide_compactness(const Params &p, int env, int core, long long sum_nh) {
    const int2 t = nc_totals(p)[(size_t)env * p.C + core];
    return compactness_value(p, t.x, t.y, sum_nh);
}

// _provision_path / _release_path with the statistics (rmsa_env.py:381-396, 418-436): links in hop order, each entry loaded,
// modified and stored by the thread that owns it, so _update_link_stats sees the link's new mask.  The link's compactness terms
// (span, free runs inside it) are refreshed from the same shape and the core's sums adjusted by the difference.
template <int KIND, int NWV>
__device__ __forceinline__ void wide_path_update_stats(const Params &p, int env, int row, int core, int start, int n, bool set, double now) {
    const WBits<NWV> rm = bits_range<NWV>(start, start + n);
    const size_t vs = p.wstride ? 1 : (size_t)p.n;
    int d_occ = 0, d_unused = 0;
    for (int h = p.path_link_ptr[row]; h < p.path_link_ptr[row + 1]; h++) {
        const int l = p.path_links16[h];
        uint4 *m = p.masks + mask_index(p, core * p.E + l, 0, env);
        WBits<NWV> b;
#pragma unroll
        for (int v = 0; v < NWV; v++) {
            const uint4 x = __ldcg(m + v * vs);
            b.w[4 * v] = x.x; b.w[4 * v + 1] = x.y; b.w[4 * v + 2] = x.z; b.w[4 * v + 3] = x.w;
        }
#pragma unroll
        for (int i = 0; i < 4 * NWV; i++) b.w[i] = set ? (b.w[i] | rm.w[i]) : (b.w[i] & ~rm.w[i]);
#pragma unroll
        for (int v = 0; v < NWV; v++) m[v * vs] = make_uint4(b.w[4 * v], b.w[4 * v + 1], b.w[4 * v + 2], b.w[4 * v + 3]);
        LinkShape s{};
        if (KIND == ORLG_RWA) {
            s.free_cnt = bits_popc(b);                   // rwa_env.py:365-383: utilisation only
        } else {
            s = link_shape(b, p.S);
            unsigned *t = nc_links(p) + ((size_t)env * p.C + core) * p.E + l;
            const unsigned old = *t;
            d_occ += s.span - (int)(old & 0xFFFFu);
            d_unused += s.free_runs_in - (int)(old >> 16);
            *t = (unsigned)s.span | ((unsigned)s.free_runs_in << 16);
        }
        update_link_stats_with(p, env, l, now, [&] { return s; });
    }
    if (KIND != ORLG_RWA) {
        int2 *t = nc_totals(p) + (size_t)env * p.C + core;
        int2 v = *t;
        v.x += d_occ; v.y += d_unused;
        *t = v;
    }
}

// DeepRMSA's cached block start i of env's pending request exists: 16-bit entries on wide handles, 8-bit otherwise
__device__ __forceinline__ bool cand_found(const Params &p, int env, int i) {
    const size_t at = (size_t)env * p.cand_stride + i;
    return p.cand16 ? p.cand16[at] != 0xFFFFu : p.cand[at] != CAND_NONE;
}

// ---------------------------------------------------------------- heuristic action sources (SURVEY a21), every handle
// The action of env's pending request (src, dst, br) into a[0..3], from the masks of its candidate paths only.  NB the
// reference's first-fit loops run over range(0, S - n): the last feasible start S - n is never tried (SURVEY.md App. B-5).
// Returns true when the action is KNOWN to fit (it was derived from the path's free mask just now), so that the fused step
// does not have to read the masks a second time for is_path_free.
template <int KIND, int NWV>
__device__ __forceinline__ bool wide_heuristic(const Params &p, const int env, const int which, const int src, const int dst, const int br, int *a) {
    const int pair = src * p.N + dst;
    const int first = p.pair_first[pair];
    const int npaths = min((int)p.pair_count[pair], p.k);
    if (KIND == ORLG_DEEPRMSA) {
        // deeprmsa_env.py:135-155 on the cached block starts
        int act = p.k * p.J;
        if (which == ORLG_HEUR_SP_FF) act = (!p.allow_rejection || cand_found(p, env, 0)) ? 0 : p.k * p.J;
        else
            for (int q = 0; q < npaths; q++)
                if (cand_found(p, env, q * p.J)) { act = q * p.J; break; }
        a[0] = act;
        return false;
    } else if (KIND == ORLG_RMSA) {
        // rmsa_env.py:747-803
        int ap = p.k, as = p.S, max_free = 0;
        const int np_ = (which == ORLG_HEUR_SP_FF) ? min(npaths, 1) : npaths;
        for (int q = 0; q < np_; q++) {
            const int n = wide_nslots(p, meta_se(p.path_meta[first + q]), br);
            const WBits<NWV> A = wide_path_free<NWV>(p, env, first + q, 0);
            WBits<NWV> B = bits_runs_ge(A, n);
            const WBits<NWV> lim = bits_range<NWV>(0, max(p.S - n, 0));
#pragma unroll
            for (int i = 0; i < 4 * NWV; i++) B.w[i] &= lim.w[i];
            const int s = bits_ffs(B);
            if (s >= 0) {
                if (which == ORLG_HEUR_LLP_FF) {
                    const int fr = bits_popc(A);
                    if (fr > max_free) { ap = q; as = s; max_free = fr; }
                } else { ap = q; as = s; break; }
            }
        }
        a[0] = ap; a[1] = as;
        return ap < p.k;
    } else if (KIND == ORLG_RWA) {
        // rwa_env.py:425-502
        int ap = p.k, as = p.S;
        if (which == ORLG_HEUR_SP_FF) {
            if (npaths > 0) {
                const int s = bits_ffs(wide_path_free<NWV>(p, env, first, 0));
                if (s >= 0) { ap = 0; as = s; }
            }
        } else if (which == ORLG_HEUR_SAP_FF || which == ORLG_HEUR_SAP_LF) {
            int best_hops = 0x7fffffff;
            for (int q = 0; q < npaths; q++) {
                const int hops = wide_hops(p, first + q);        // = the table's hop count (orlg_create checks them)
                if (hops < best_hops) {
                    WBits<NWV> A = wide_path_free<NWV>(p, env, first + q, 0);
                    int s;
                    if (which == ORLG_HEUR_SAP_FF) s = bits_ffs(A);
                    else { A.w[0] &= ~1u; s = bits_fls(A); }      // range(W-1, 0, -1): wavelength 0 is never tried
                    if (s >= 0) { best_hops = hops; ap = q; as = s; }
                }
            }
        } else {
            int best = -1;
            for (int q = 0; q < npaths; q++) {
                const WBits<NWV> A = wide_path_free<NWV>(p, env, first + q, 0);
                const int cap = bits_popc(A);
                if (cap > best) {
                    const int s = bits_ffs(A);
                    if (s >= 0) { best = cap; ap = q; as = s; }
                }
            }
        }
        a[0] = ap; a[1] = as;
        return ap < p.k;
    } else {
        // rmcsa_env.py:882-911 (reject = 4-tuple (k, M, C, S))
        int a0 = p.k, a1 = p.M, a2 = p.C, a3 = p.S;
        bool found = false;
        for (int q = 0; q < npaths && !found; q++) {
            const int mod = meta_mod(p.path_meta[first + q]);
            const int n = wide_nslots(p, p.mod_se[mod], br);
            const WBits<NWV> lim = bits_range<NWV>(0, max(p.S - n, 0));
            for (int c = 0; c < p.C && !found; c++) {
                WBits<NWV> B = bits_runs_ge(wide_path_free<NWV>(p, env, first + q, c), n);
#pragma unroll
                for (int i = 0; i < 4 * NWV; i++) B.w[i] &= lim.w[i];
                const int s = bits_ffs(B);
                if (s >= 0) { a0 = q; a1 = mod; a2 = c; a3 = s; found = true; }
            }
        }
        a[0] = a0; a[1] = a1; a[2] = a2; a[3] = a3;
        return found;
    }
}

// thread per env; NSFNET-class handles take NWV = 1
template <int KIND, int NWV>
__global__ void heuristic_kernel(const Params p, const int which, int *actions) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    const uint2 rq = p.cur_req[env];
    constexpr int AD = KIND == ORLG_DEEPRMSA ? 1 : (KIND == ORLG_RMCSA ? 4 : 2);
    int a[4];
    wide_heuristic<KIND, NWV>(p, env, which, rq.x & 0xff, (rq.x >> 8) & 0xff, (int)(rq.x >> 16), a);
#pragma unroll
    for (int i = 0; i < AD; i++) actions[AD * env + i] = a[i];
}

// DeepRMSA-v0 invalid-action mask of env's pending request, thread per env: row [k * j + rej] of uint8, action q * j + b valid
// iff path q is a candidate of the pair and its block b exists (exactly when env.step(q * j + b) provisions, deeprmsa_env.py:48-58),
// the reject action always valid.  Any DeepRMSA handle: every step kernel and the persistent rollout kernel keep the block cache.
// Launched with programmatic dependent launch, and every thread waits before it reads or exits: the policy kernel that follows
// waits on this grid only, then reads the observation the step kernel before it wrote.
__global__ void action_mask_kernel(const Params p, unsigned char *mask) {
    pdl_launch_dependents();
    pdl_wait();
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    const unsigned rq = p.cur_req[env].x;
    const int npaths = min((int)p.pair_count[(rq & 0xff) * p.N + ((rq >> 8) & 0xff)], p.k);
    const int kj = p.k * p.J;
    unsigned char *row = mask + (size_t)env * (kj + p.allow_rejection);
    for (int i = 0; i < kj; i++) row[i] = i < npaths * p.J && cand_found(p, env, i) ? 1 : 0;
    if (p.allow_rejection) row[kj] = 1;
}

// Launch shape, A/B-ed on the B200 (profiles/r2_experiments.md): 64-thread CTAs, 8 per SM (128 registers per thread, 16 warps per
// SM); 128 x 3, 128 x 4 and 64 x 6 are within 3 % of it -- the kernel is bound by its dependent loads, not by occupancy.
#ifndef ORLG_WIDE_THREADS
#define ORLG_WIDE_THREADS 64
#endif
#ifndef ORLG_WIDE_MIN_BLOCKS
#define ORLG_WIDE_MIN_BLOCKS 8
#endif
// STATS = true: the float statistics of row f1 (orlg_enable_stats / orlg_enable_link_stats) are kept as well.  That instance
// carries more live state (the shape of a link, the sorted releases) and is given 6 CTAs per SM (up to 168 registers): with 8
// the RMCSA instance of 512 slots spills.
#ifndef ORLG_WIDE_STATS_MIN_BLOCKS
#define ORLG_WIDE_STATS_MIN_BLOCKS 6
#endif
template <int KIND, int NWV, bool STATS>
__global__ void __launch_bounds__(ORLG_WIDE_THREADS, STATS ? ORLG_WIDE_STATS_MIN_BLOCKS : ORLG_WIDE_MIN_BLOCKS) step_wide_kernel(const Params p, const StepIO io, const int mode) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    double now = p.now[env];
    double hold = p.cur_hold[env];
    uint2 rq = p.cur_req[env];
    int src = rq.x & 0xff, dst = (rq.x >> 8) & 0xff, br = (int)(rq.x >> 16), sid = (int)rq.y;
    long long cnt[8];
#pragma unroll
    for (int q = 0; q < 8; q++) cnt[q] = p.counters[(size_t)q * p.n + env];
    unsigned ridx = p.req_index[env];
    unsigned nheap = p.nheap[env];
    double hmin = p.heap_min[env];
    double tailmin = p.ev_tail[env];
    unsigned err = p.errors[env];
    Events ev = {p.ev_time + (size_t)env * p.heap_cap, p.ev_pay + (size_t)env * p.heap_cap, p.ev_gmin + (size_t)env * p.ev_groups};
    if constexpr (STATS) ev.br = p.ev_br + (size_t)env * p.heap_cap;
    bool accepted = false, done = false;

    if (mode == MODE_FULL_RESET) {
        const WBits<NWV> full = bits_range<NWV>(0, p.S);
        for (int l = 0; l < p.C * p.E; l++)
#pragma unroll
            for (int v = 0; v < NWV; v++)
                p.masks[mask_index(p, l, v, env)] = make_uint4(full.w[4 * v], full.w[4 * v + 1], full.w[4 * v + 2], full.w[4 * v + 3]);
        now = 0.0; nheap = 0; hmin = ORLG_INF; tailmin = ORLG_INF; ridx = 0; err = 0;
#pragma unroll
        for (int q = 0; q < 8; q++) cnt[q] = 0;
        if (KIND == ORLG_RMSA) br_hist_clear(p, env);
        if (KIND == ORLG_RWA) act_hist_clear(p, env);
    }

    if (mode == MODE_STEP) {
        const int pair = src * p.N + dst;
        const int first = p.pair_first[pair];
        const int npaths = p.pair_count[pair];
        int row = -1, start = 0, n = 0, core = 0, mod = -1;
        constexpr int AD = KIND == ORLG_DEEPRMSA ? 1 : (KIND == ORLG_RMCSA ? 4 : 2);
        int act[4];
        bool known_free = false;
        if (io.policy >= 0) {                                // fused rollout step: action = heuristic(env), no second launch, and
            known_free = wide_heuristic<KIND, NWV>(p, env, io.policy, src, dst, br, act);      // the path's masks are in L1 / L2 for what follows
            if (io.actions_out) {
#pragma unroll
                for (int i = 0; i < AD; i++) io.actions_out[AD * env + i] = act[i];
            }
        } else {
#pragma unroll
            for (int i = 0; i < AD; i++) act[i] = io.actions[AD * env + i];
        }
        if (KIND == ORLG_DEEPRMSA) {
            const int a = act[0];
            if (a >= 0 && a < p.k * p.J) {
                const int route = a / p.J;
                if (route < npaths) {
                    const unsigned st = p.cand16[(size_t)env * p.cand_stride + a];
                    if (st != 0xFFFFu) {
                        row = first + route;
                        n = wide_nslots(p, meta_se(p.path_meta[row]), br);
                        start = (int)st;
                        accepted = true;
                    }
                } else err |= ORLG_ERR_NO_SUCH_PATH;
            }
        } else if (KIND == ORLG_RMSA || KIND == ORLG_RWA) {
            const int path = act[0], slot = act[1];
            if (KIND == ORLG_RWA) act_hist_bump(p, env, path, slot, err);
            if (path >= 0 && path < p.k && slot >= 0 && slot < p.S) {
                if (path < npaths) {
                    row = first + path;
                    n = (KIND == ORLG_RWA) ? 1 : wide_nslots(p, meta_se(p.path_meta[row]), br);
                    start = slot;
                    if (known_free) accepted = true;
                    else if (start + n <= p.S) accepted = bits_contains(wide_path_free<NWV>(p, env, row, 0), bits_range<NWV>(start, start + n));
                } else err |= ORLG_ERR_NO_SUCH_PATH;
            }
        } else {
            const int path = act[0], am = act[1], ac = act[2], slot = act[3];
            if (path >= 0 && path < p.k && am >= 0 && am < p.M && ac >= 0 && ac < p.C && slot >= 0 && slot < p.S) {
                if (path < npaths) {
                    row = first + path;
                    n = wide_nslots(p, p.mod_se[am], br);
                    start = slot; core = ac; mod = am;
                    if (start + n <= p.S)
                        accepted = (known_free || bits_contains(wide_path_free<NWV>(p, env, row, core), bits_range<NWV>(start, start + n))) &&
                                   (p.path_length[row] < p.reach[am * (p.br_max + 1) + br]);
                } else err |= ORLG_ERR_NO_SUCH_PATH;
            }
        }
        if (accepted && nheap + 1 > (unsigned)p.heap_cap) { accepted = false; err |= ORLG_ERR_HEAP_OVERFLOW; }
        bool info_stats = false;
        long long snh = 0;
        double prev_compactness = 0.0;
        if constexpr (STATS) {
            info_stats = (KIND == ORLG_RMSA || KIND == ORLG_DEEPRMSA) && p.stats_out;
            snh = p.sum_nh[env];
            if (info_stats) prev_compactness = wide_compactness(p, env, 0, snh);     // rmsa_env.py:168-170
        }
        if (accepted) {
            if constexpr (STATS) {
                wide_path_update_stats<KIND, NWV>(p, env, row, core, start, n, false, now);
                snh += (long long)n * wide_hops(p, row);
                p.sum_nh[env] = snh;
                if (KIND != ORLG_RWA) {
                    const long long rb = p.run_br[env] + br;
                    p.run_br[env] = rb;
                    update_network_stats_with(p, env, rb, now, [&] { return wide_compactness(p, env, core, snh); });
                }
                events_push(ev, nheap, hmin, tailmin, __dadd_rn(now, hold), pack_service(row, start, n, core, sid), (unsigned)br);
            } else {
                wide_path_update<NWV>(p, env, row, core, start, n, false);
                events_push(ev, nheap, hmin, tailmin, __dadd_rn(now, hold), pack_service(row, start, n, core, sid));
            }
        }
        count_decision<KIND>(cnt, accepted, br);
        if (KIND == ORLG_RMSA && accepted) br_hist_bump(p, env, 1, br);
        if (io.reward) io.reward[env] = accepted ? 1.0f : (KIND == ORLG_DEEPRMSA ? -1.0f : 0.0f);
        if (io.decision) {
            int *d = io.decision + (size_t)env * 6;
            d[0] = accepted; d[1] = accepted ? row : -1; d[2] = accepted ? start : -1; d[3] = accepted ? n : -1;
            d[4] = accepted ? core : -1; d[5] = accepted ? mod : -1;
        }
        if (io.info) {
#pragma unroll
            for (int q = 0; q < 8; q++) io.info[(size_t)env * 8 + q] = cnt[q];
        }
        if constexpr (STATS) if (info_stats) {              // rmsa_env.py:229-264
            const double cur = wide_compactness(p, env, 0, snh);
            double *so = p.stats_out + (size_t)env * 4;
            so[0] = cur;
            so[1] = __dadd_rn(prev_compactness, -cur);
            so[2] = mean_over_links(p, p.link_comp, env);
            so[3] = mean_over_links(p, p.link_util, env);
        }
    }

    if constexpr (STATS) if (mode == MODE_FULL_RESET) {
        clear_stats(p, env);
        if (KIND != ORLG_RWA) {
            for (int l = 0; l < p.C * p.E; l++) nc_links(p)[(size_t)env * p.C * p.E + l] = 0u;
            for (int c = 0; c < p.C; c++) nc_totals(p)[(size_t)env * p.C + c] = make_int2(0, 0);
        }
    }

    if (mode == MODE_STEP || mode == MODE_FULL_RESET) {
        double arrival, holding;
        int nsrc, ndst, nbr;
        if (p.traffic == ORLG_TRAFFIC_PHILOX) {
            philox_request(p, p.node_thr, env, ridx, now, arrival, holding, nsrc, ndst, nbr);
        } else {
            const orlg_request r = trace_request(p, env, ridx, now, p.br_max, p.br_lo, false, err);
            arrival = r.arrival; holding = r.holding; nsrc = r.src; ndst = r.dst; nbr = r.bit_rate;
        }
        ridx++;
        now = arrival; hold = holding; src = nsrc; dst = ndst; br = nbr;
        sid = (int)cnt[2];
        count_request<KIND>(cnt, br);
        if (KIND == ORLG_RMSA) br_hist_bump(p, env, 0, br);
        if constexpr (STATS)
            release_due_in_order(p, env, ev, nheap, hmin, tailmin, now, err, [&](unsigned long long pl) {
                wide_path_update_stats<KIND, NWV>(p, env, svc_row(pl), svc_core(pl), svc_start(pl), svc_slots(pl), true, now);
                return (long long)svc_slots(pl) * wide_hops(p, svc_row(pl));
            });
        else
        events_release(ev, nheap, hmin, tailmin, now, apply_payload([&](unsigned long long pl) {
            wide_path_update<NWV>(p, env, svc_row(pl), svc_core(pl), svc_start(pl), svc_slots(pl), true);
        }));
        done = (cnt[2] == (long long)p.episode_length);
    }

    if (mode == MODE_EPISODE_RESET || (mode == MODE_STEP && done && p.auto_reset)) reset_episode_counters<KIND>(cnt, br);

    if (KIND == ORLG_DEEPRMSA) {
        // observation of the pending request (deeprmsa_env.py:60-121), path by path, written in place
        const int pair = src * p.N + dst;
        const int first = p.pair_first[pair];
        const int npaths = min((int)p.pair_count[pair], p.k);
        const int W = 2 * p.J + 3, head = 1 + 2 * p.N;
        float *o32 = reinterpret_cast<float *>(io.obs) + (size_t)env * p.obs_dim;
        double *o64 = reinterpret_cast<double *>(io.obs) + (size_t)env * p.obs_dim;
        if (io.obs) {
            for (int q = 0; q < p.obs_dim; q++) {
                if (p.obs_f64) o64[q] = q >= head ? -1.0 : 0.0; else o32[q] = q >= head ? -1.0f : 0.0f;
            }
            if (p.obs_f64) { o64[0] = __ddiv_rn((double)br, 100.0); o64[1 + min(src, dst)] = 1.0; o64[1 + p.N + max(src, dst)] = 1.0; }
            else { o32[0] = __fdiv_rn((float)br, 100.0f); o32[1 + min(src, dst)] = 1.0f; o32[1 + p.N + max(src, dst)] = 1.0f; }
        }
        for (int q = 0; q < p.k; q++) {
            int *oi = io.obs_int ? io.obs_int + ((size_t)env * p.k + q) * W : nullptr;
            if (q >= npaths) {
                for (int b = 0; b < p.J; b++) p.cand16[(size_t)env * p.cand_stride + q * p.J + b] = 0xFFFFu;
                if (oi) for (int b = 0; b < W; b++) oi[b] = -1;
                continue;
            }
            const int row = first + q;
            const int n = wide_nslots(p, meta_se(p.path_meta[row]), br);
            const WBits<NWV> A = wide_path_free<NWV>(p, env, row, 0);
            const WBits<NWV> B = bits_runs_ge(A, n);
            const WBits<NWV> Bl = bits_shl1(B), Al = bits_shl1(A);
            WBits<NWV> starts, arun;
#pragma unroll
            for (int i = 0; i < 4 * NWV; i++) { starts.w[i] = B.w[i] & ~Bl.w[i]; arun.w[i] = A.w[i] & ~Al.w[i]; }
            const int total = bits_popc(A), runs = bits_popc(arun);
            const int ob = head + q * W;
            for (int b = 0; b < p.J; b++) {
                const int st = bits_ffs(starts);
                p.cand16[(size_t)env * p.cand_stride + q * p.J + b] = (unsigned short)(st < 0 ? 0xFFFF : st);
                int len = -1;
                if (st >= 0) {
                    starts = bits_clear_lowest(starts);
                    len = bits_run_length(A, st);
                    if (io.obs) {
                        if (p.obs_f64) {
                            o64[ob + 2 * b] = __ddiv_rn(__dmul_rn(2.0, __dadd_rn((double)st, -__dmul_rn(0.5, (double)p.S))), (double)p.S);
                            o64[ob + 2 * b + 1] = __ddiv_rn(__dadd_rn((double)len, -8.0), 8.0);
                        } else {
                            o32[ob + 2 * b] = __fdiv_rn((float)(2 * st - p.S), (float)p.S);
                            o32[ob + 2 * b + 1] = (float)(len - 8) * 0.125f;
                        }
                    }
                }
                if (oi) { oi[2 * b] = st; oi[2 * b + 1] = len; }
            }
            if (io.obs) {
                if (p.obs_f64) {
                    o64[ob + 2 * p.J] = __ddiv_rn(__dadd_rn((double)n, -5.5), 3.5);
                    o64[ob + 2 * p.J + 1] = __ddiv_rn(__dmul_rn(2.0, __dadd_rn((double)total, -__dmul_rn(0.5, (double)p.S))), (double)p.S);
                    if (runs > 0) o64[ob + 2 * p.J + 2] = __ddiv_rn(__dadd_rn(__ddiv_rn((double)total, (double)runs), -4.0), 4.0);
                } else {
                    o32[ob + 2 * p.J] = __fdiv_rn((float)(2 * n - 11), 7.0f);
                    o32[ob + 2 * p.J + 1] = __fdiv_rn((float)(2 * total - p.S), (float)p.S);
                    if (runs > 0) o32[ob + 2 * p.J + 2] = __fdiv_rn((float)(total - 4 * runs), (float)(4 * runs));
                }
            }
            if (oi) { oi[2 * p.J] = n; oi[2 * p.J + 1] = total; oi[2 * p.J + 2] = runs; }
        }
    }

    if (mode != MODE_OBSERVE) {
        p.now[env] = now;
        p.cur_hold[env] = hold;
        p.cur_req[env] = make_uint2((unsigned)src | ((unsigned)dst << 8) | ((unsigned)br << 16), (unsigned)sid);
#pragma unroll
        for (int q = 0; q < 8; q++) p.counters[(size_t)q * p.n + env] = cnt[q];
        p.req_index[env] = ridx;
        p.nheap[env] = nheap;
        p.heap_min[env] = hmin;
        p.ev_tail[env] = tailmin;
        p.errors[env] = err;
        if (mode == MODE_STEP && io.done) io.done[env] = done ? 1 : 0;
    }
}

// state export for the wide layout: masks uint32 [n][C*E][4*NWV], allocation int32 [n][C][E][S]
__global__ void export_wide_kernel(const Params p, unsigned *masks_out, int *alloc_out) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    const int CE = p.C * p.E, NWV = p.nwv;
    if (masks_out)
        for (int l = 0; l < CE; l++)
            for (int v = 0; v < NWV; v++) {
                const uint4 m = p.masks[mask_index(p, l, v, env)];
                unsigned *o = masks_out + ((size_t)env * CE + l) * (4 * NWV) + 4 * v;
                o[0] = m.x; o[1] = m.y; o[2] = m.z; o[3] = m.w;
            }
    if (alloc_out) {
        int *o = alloc_out + (size_t)env * CE * p.S;
        for (int q = 0; q < CE * p.S; q++) o[q] = -1;
        const unsigned long long *h = p.ev_pay + (size_t)env * p.heap_cap;
        const unsigned nh = p.nheap[env];
        for (unsigned s = 0; s < nh; s++) {
            const unsigned long long pl = h[s];
            const int row = svc_row(pl);
            for (int hh = p.path_link_ptr[row]; hh < p.path_link_ptr[row + 1]; hh++)
                for (int q = 0; q < svc_slots(pl); q++)
                    o[((size_t)svc_core(pl) * p.E + p.path_links16[hh]) * p.S + svc_start(pl) + q] = svc_id(pl);
        }
    }
}

}  // namespace orlg
