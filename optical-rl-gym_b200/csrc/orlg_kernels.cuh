// orlg_kernels.cuh -- the step kernels (thread-per-environment, struct-of-arrays state in HBM).
//
// One thread owns one environment.  All per-env scalars are struct-of-arrays over the env index
// and the spectrum masks are laid out [core*link][env] as 128-bit words, so that every warp-wide
// access to "the same field / the same link of 32 consecutive envs" is one contiguous 128..512-byte
// run.  DESIGN.md explains why this mapping (and not a warp per env) is used for NSFNET-class
// topologies (<= 32 links, <= 128 slots).
#pragma once
#include "orlg_device.cuh"
#include "../../include/orlg.h"

namespace orlg {

constexpr int KMAX = 8;          // candidate paths per pair handled by the in-register observation pass
constexpr int STEP_THREADS = 128;

enum { MODE_STEP = 0, MODE_FULL_RESET = 1, MODE_EPISODE_RESET = 2, MODE_OBSERVE = 3 };

struct Params {
    // ---- configuration
    int kind, n, N, E, C, S, k, J, M;
    int episode_length, allow_rejection, auto_reset, traffic, obs_f64;
    int br_lo, br_span, n_bit_rates, br_max;
    int heap_cap, cand_stride, obs_dim;
    unsigned long long seed;
    long long env_id_base;
    double mean_holding, mean_iat;
    // ---- read-only tables (HBM, L1/L2 resident)
    const int *pair_first;             // [N*N]
    const unsigned char *pair_count;   // [N*N]
    const unsigned *path_linkmask;     // [P]  bit l = link l on the path (E <= 32)
    const unsigned *path_meta;         // [P]  hops | se << 8 | mod << 16
    const double *path_length;         // [P]
    const int *path_link_ptr;          // [P+1] CSR of the hop lists (wide kernels)
    const unsigned short *path_links16;  // link index of every hop
    const unsigned char *nslots;       // [(se or mod-se) * (br_max+1) + bit_rate]  rmsa_env.py:610-621
    const unsigned char *mod_se;       // [M]
    const double *reach;               // [M * (br_max+1)] min(lmax_snr, lmax_xt) of rmcsa_env.py:341-384
    const unsigned *node_thr;          // [N] integer CDF of node_request_probabilities
    const unsigned *br_thr;            // [n_bit_rates]
    const int *bit_rates;              // [n_bit_rates]
    const orlg_request *trace;         // [n * trace_len]
    long long trace_len;
    // packed copy of the small tables, staged in shared memory by the fast kernel (byte offsets)
    const uint4 *tab_blob;
    int tab_vec;                       // size in 16-byte units
    int off_pair_first, off_pair_count, off_path_lm, off_path_se, off_path_ll, off_nslots, off_node_thr, off_pos, off_nsl, off_rcp4, off_dbl, off_br100;
    int node_top_step;                 // highest power of two <= N-1 (binary search over the node CDF)
    int warp_area_bytes;               // fast kernel: shared-memory work area per warp (masks, then observation rows)
    unsigned lockstep_ridx;            // requests drawn so far by EVERY env (all envs reset and step together)
    // ---- per-env state (struct of arrays)
    uint4 *masks;                      // [C*E][n]
    double *now;                       // [n] current_time
    double *cur_hold;                  // [n] holding time of the pending request
    uint2 *cur_req;                    // [n] x = src | dst << 8 | bit_rate << 16, y = service id
    long long *counters;               // [8][n]
    unsigned *req_index;               // [n] requests generated since the last full reset
    unsigned *nheap;                   // [n]
    double *heap_min;                  // [n] earliest release time (+inf if none)
    double *ev_time;                   // [n][heap_cap] release times of the live services (unsorted, orlg_device.cuh)
    unsigned long long *ev_pay;        // [n][heap_cap] packed services
    float *ev_gmin;                    // [n][ev_groups] per-group lower bounds (directory)
    double *ev_tail;                   // [n] lower bound of the open tail group
    int ev_groups;                     // directory stride (multiple of 16)
    unsigned char *cand;               // [n][cand_stride] first-fit block starts of the pending request
    unsigned short *cand16;            // same for the wide layout (S > 128)
    int nwv;                           // 128-bit word groups per (core, link): 1 unless wide
    int wstride;                       // wide layout (env-major): 128-bit words between consecutive (core, link) entries of one env; 0 = [link][env] layout
    unsigned *errors;                  // [n]
    // ---- float statistics of `info` (row f1: rmsa_env.py:439-543, 699-744); allocated by orlg_enable_stats
    int stats;
    double *link_util, *link_comp, *link_last;   // [E][n] time-averaged utilisation / compactness, last update time
    double *link_frag;                 // [E][n] time-averaged external fragmentation (rmsa_env.py:487-524)
    double *graph_stats;               // [3][n] topology.graph["throughput"], ["compactness"], ["last_update"] (rmsa_env.py:439-462)
    long long *run_br;                 // [n] sum of bit_rate over graph["running_services"]
    unsigned short *ev_br;             // [n][heap_cap] bit rate of every live service (parallel to ev_pay)
    long long *sum_nh;                 // [n] sum over running services of number_slots * hops (wide handles: + nc_totals, nc_links)
    double *stats_out;                 // [n][4] network_compactness, its difference, avg link compactness, avg link utilisation
    const int *link_order;             // [E] link indices in topology.edges() order (np.mean over the links)
    // ---- discrete bit-rate selection (row f4: rmsa_env.py:88-110, 217-227, 268-273, 408-415, 579-581)
    int *br_hist;                      // [2][n_bit_rates][n] bit_rate_requested_histogram / bit_rate_provisioned_histogram
    // ---- RWA actions_output (rwa_env.py:52-58, 103): only its marginals reach `info` (rwa_env.py:148-151)
    int *act_hist;                     // [(k + rej) + (S + rej)][n] row sums, then column sums (NULL unless RWA-v0)
};

// index of the 128-bit word group v of (core, link) entry cl of env e in p.masks: [entry][word][env] (a warp's 32 envs read one
// entry as one 512-byte run: the NSFNET-class kernels), or env-major [env][entry][wstride] for the wide kernels (each thread
// walks its own path, so an entry's words should share a DRAM burst and an env's entries a page)
__device__ __forceinline__ size_t mask_index(const Params &p, int cl, int v, int e) {
    return p.wstride ? ((size_t)e * (p.C * p.E) + cl) * p.wstride + v : ((size_t)cl * p.nwv + v) * p.n + e;
}

// position of a bit rate in the discrete list (-1: not one of them, e.g. a foreign trace)
__device__ __forceinline__ int br_index(const Params &p, int br) {
    for (int i = 0; i < p.n_bit_rates; i++)
        if (p.bit_rates[i] == br) return i;
    return -1;
}
__device__ __forceinline__ void br_hist_bump(const Params &p, int env, int which, int br) {
    if (!p.br_hist) return;
    const int i = br_index(p, br);
    if (i >= 0) p.br_hist[((size_t)which * p.n_bit_rates + i) * p.n + env] += 1;
}
// self.actions_output[path, wavelength] += 1 (rwa_env.py:103); an index outside the (k + rej, W + rej) histogram is an
// IndexError in the reference: flagged here, nothing counted
__device__ __forceinline__ void act_hist_bump(const Params &p, int env, int path, int slot, unsigned &err) {
    if (!p.act_hist) return;
    const int R = p.k + p.allow_rejection, Cn = p.S + p.allow_rejection;
    if (path >= 0 && path < R && slot >= 0 && slot < Cn) {
        p.act_hist[(size_t)path * p.n + env] += 1;
        p.act_hist[(size_t)(R + slot) * p.n + env] += 1;
    } else {
        err |= ORLG_ERR_NO_SUCH_PATH;
    }
}
__device__ __forceinline__ void act_hist_clear(const Params &p, int env) {
    if (!p.act_hist) return;
    const int rows = p.k + p.S + 2 * p.allow_rejection;
    for (int i = 0; i < rows; i++) p.act_hist[(size_t)i * p.n + env] = 0;
}
__device__ __forceinline__ void br_hist_clear(const Params &p, int env) {
    if (!p.br_hist) return;
    for (int i = 0; i < 2 * p.n_bit_rates; i++) p.br_hist[(size_t)i * p.n + env] = 0;
}

struct StepIO {
    const int *actions;
    void *obs;
    float *reward;
    unsigned char *done;
    int *decision;
    long long *info;
    int *obs_int;
    int policy;          // wide kernels, MODE_STEP: >= 0 = this ORLG_HEUR_* is evaluated in the step kernel's prologue (fused), else -1
    int *actions_out;    // ... and the action it took is stored here (may be null)
};

__device__ __forceinline__ int meta_hops(unsigned m) { return m & 0xff; }
__device__ __forceinline__ int meta_se(unsigned m) { return (m >> 8) & 0xff; }
__device__ __forceinline__ int meta_mod(unsigned m) { return (m >> 16) & 0xff; }

// get_available_slots (rmsa_env.py:638-649): AND of the path's link masks, straight from HBM/L2
__device__ __forceinline__ Bits path_free(const Params &p, int env, unsigned lm, int core) {
    Bits a = bits_ones();
    const uint4 *base = p.masks + (size_t)core * p.E * p.n + env;
    while (lm) {
        int l = __ffs(lm) - 1;
        lm &= lm - 1;
        a = bits_and(a, bits_from(base[(size_t)l * p.n]));
    }
    return a;
}

// _provision_path / _release_path on the masks (rmsa_env.py:381-385, 419-424)
__device__ __forceinline__ void path_update(const Params &p, int env, unsigned lm, int core, const Bits &rm, bool set) {
    uint4 *base = p.masks + (size_t)core * p.E * p.n + env;
    while (lm) {
        int l = __ffs(lm) - 1;
        lm &= lm - 1;
        Bits m = bits_from(base[(size_t)l * p.n]);
        m = set ? bits_or(m, rm) : bits_andnot(m, rm);
        base[(size_t)l * p.n] = bits_to(m);
    }
}

__device__ __forceinline__ int pick_thr(const unsigned *thr, int n, unsigned r) {
    int i = 0;
    while (i < n - 1 && r >= thr[i]) i++;
    return i;
}

// first i in [0, n-1] with r < thr[i] (n-1 if none): same result as the linear scan of pick_thr (thr is non-decreasing)
__device__ __forceinline__ int pick_thr_bsearch(const unsigned *thr, int n, int top_step, unsigned r) {
    int i = 0;
    for (int step = top_step; step > 0; step >>= 1)
        if (i + step <= n - 1 && r >= thr[i + step - 1]) i += step;
    return i;
}

// ---------------------------------------------------------------- the request stream (DESIGN.md section 5)
// _next_service's draws (rmsa_env.py:548-561) from the counter-based generator, in pieces: the persistent and the fast kernels
// draw the times before their tables have landed and the nodes from the tables in shared memory.  The Philox blocks themselves
// stay at the call sites: behind a function boundary the compiler orders the XORs of the rounds differently and the code of
// the persistent and fast kernels changes.

// inter-arrival and holding time from stream 0 (the arrival is now + the inter-arrival time)
__device__ __forceinline__ double request_iat(const Params &p, const uint32_t c[4]) { return __dmul_rn(neg_log_u32(c[0]), p.mean_iat); }
__device__ __forceinline__ double request_holding(const Params &p, const uint32_t c[4]) { return __dmul_rn(neg_log_u32(c[1]), p.mean_holding); }

// source and destination from stream 0: node_thr is the node CDF in global or in shared memory
__device__ __forceinline__ void request_nodes(const Params &p, const unsigned *node_thr, const uint32_t c[4], int &src, int &dst) {
    const int n = p.N;
    src = pick_thr_bsearch(node_thr, n, p.node_top_step, c[2]);        // binary search: up to 255 nodes, every lane its own draw
    const unsigned lo = src ? node_thr[src - 1] : 0u;
    const unsigned long long hi = (src == n - 1) ? 4294967296ULL : (unsigned long long)node_thr[src];
    const unsigned long long mass = hi - lo;
    unsigned long long tt = ((unsigned long long)c[3] * (4294967296ULL - mass)) >> 32;
    if (tt >= lo) tt += mass;
    dst = pick_thr_bsearch(node_thr, n, p.node_top_step, (unsigned)tt);
    if (dst == src) dst = (src + 1) % n;
}

// bit rate from word 0 of stream 1: the discrete CDF when the handle has one (only compiled in with DISCRETE), else uniform
template <bool DISCRETE>
__device__ __forceinline__ int request_bit_rate(const Params &p, uint32_t d0) {
    if (DISCRETE && p.n_bit_rates > 0) return p.bit_rates[pick_thr(p.br_thr, p.n_bit_rates, d0)];
    return p.br_lo + (int)__umulhi(d0, (unsigned)p.br_span);
}

__device__ __forceinline__ void philox_request(const Params &p, const unsigned *node_thr, int env, unsigned ridx, double now,
                                               double &arrival, double &holding, int &src, int &dst, int &br) {
    unsigned long long gid = (unsigned long long)(p.env_id_base + env);
    uint32_t c[4] = {ridx, 0u, (uint32_t)gid, 0u};
    philox4x32_10(c, (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
    arrival = __dadd_rn(now, request_iat(p, c));
    holding = request_holding(p, c);
    request_nodes(p, node_thr, c, src, dst);
    br = 0;
    if (p.kind != ORLG_RWA) {
        uint32_t d[4] = {ridx, 0u, (uint32_t)gid, 1u};
        philox4x32_10(d, (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
        br = request_bit_rate<true>(p, d[0]);
    }
}

// request ridx of env e from the recorded trace, its bit rate clamped to [0, br_cap]; above br_cap it sets
// ORLG_ERR_TRACE_RANGE when flag_range.  Past the end of the trace: ORLG_ERR_TRACE_EXHAUSTED and the request
// (now, holding 0, node 0 -> 1, br_past_end).
__device__ __forceinline__ orlg_request trace_request(const Params &p, int e, unsigned ridx, double now, int br_cap, int br_past_end,
                                                      bool flag_range, unsigned &err) {
    orlg_request r;
    if ((long long)ridx < p.trace_len) {
        r = p.trace[(size_t)e * p.trace_len + ridx];
        if (flag_range && r.bit_rate > br_cap) err |= ORLG_ERR_TRACE_RANGE;
        r.bit_rate = min(max(r.bit_rate, 0), br_cap);
    } else {
        err |= ORLG_ERR_TRACE_EXHAUSTED;
        r.arrival = now; r.holding = 0.0; r.src = 0; r.dst = 1; r.bit_rate = br_past_end;
    }
    return r;
}

// ---------------------------------------------------------------- the counters
// cnt = services_processed, services_accepted, episode_services_processed, episode_services_accepted, bit_rate_requested,
// bit_rate_provisioned, episode_bit_rate_requested, episode_bit_rate_provisioned.  The persistent rollout kernel keeps the
// same updates in its register form (orlg_rollout.cuh).

// the decision on the pending request (rmsa_env.py:163-209, rwa_env.py:135-136, rmcsa_env.py:292-295): RWA and RMCSA count
// the request here, RMCSA its bit rate as well (it is counted again when the request is drawn)
template <int KIND>
__device__ __forceinline__ void count_decision(long long cnt[8], bool accepted, int br) {
    if (accepted) {
        cnt[1] += 1; cnt[3] += 1;                                // services_accepted (+episode)
        if (KIND != ORLG_RWA) { cnt[5] += br; cnt[7] += br; }   // bit_rate_provisioned (+episode)
    }
    if (KIND == ORLG_RWA || KIND == ORLG_RMCSA) {
        cnt[0] += 1; cnt[2] += 1;
        if (KIND == ORLG_RMCSA) { cnt[4] += br; cnt[6] += br; }
    }
}

// a new request (_next_service, rmsa_env.py:570-573, rmcsa_env.py:730-731)
template <int KIND>
__device__ __forceinline__ void count_request(long long cnt[8], int br) {
    if (KIND == ORLG_RMSA || KIND == ORLG_DEEPRMSA) { cnt[0] += 1; cnt[2] += 1; cnt[4] += br; cnt[6] += br; }
    else if (KIND == ORLG_RMCSA) { cnt[4] += br; cnt[6] += br; }
}

// reset(only_episode_counters=True) (rmsa_env.py:285-330, rwa_env.py:164-179, rmcsa_env.py:387-430): the pending request
// (bit rate br) stays counted in the new episode, except on RWA
template <int KIND>
__device__ __forceinline__ void reset_episode_counters(long long cnt[8], int br) {
    cnt[2] = 0; cnt[3] = 0; cnt[6] = 0; cnt[7] = 0;
    if (KIND != ORLG_RWA) { cnt[2] = 1; cnt[6] = br; }
}

// ---------------------------------------------------------------- row f1: float statistics
// Per link, from the packed mask (identities checked against the reference, SURVEY.md section 8f):
// used = ~free; used blocks = popc(used & ~(used << 1)); lambda_min = ffs(used), lambda_max = fls(used) + 1;
// free runs inside [lambda_min, lambda_max) = popc(free & ~(free << 1)) less the free runs at slot 0 and at slot S - 1: with
// two or more used runs those are exactly the free runs outside the window.
struct LinkShape {
    int free_cnt, used_runs, span, free_runs_in;
    int free_runs, longest_free;       // number of free runs and the longest one (external fragmentation)
    bool free_at_both_ends;            // slot 0 and slot S - 1 are free
};
template <int V>
__device__ __forceinline__ LinkShape link_shape(const WBits<V> &fr, int S) {
    const WBits<V> valid = bits_range<V>(0, S), last = bits_range<V>(S - 1, S);
    WBits<V> used;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) used.w[i] = valid.w[i] & ~fr.w[i];
    const WBits<V> ul = bits_shl1(used), fl = bits_shl1(fr);
    LinkShape r;
    int ur = 0, frn = 0;
    uint32_t at_end = 0;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) {
        ur += __popc(used.w[i] & ~ul.w[i]);
        frn += __popc(fr.w[i] & ~fl.w[i]);
        at_end |= fr.w[i] & last.w[i];
    }
    const int f0 = fr.w[0] & 1u, f1 = at_end != 0;
    r.free_cnt = bits_popc(fr);
    r.used_runs = ur;
    r.free_runs = frn;
    r.longest_free = bits_longest_run(fr);
    r.free_at_both_ends = f0 && f1;
    r.span = 0; r.free_runs_in = 0;
    if (ur > 1) {
        r.span = bits_fls(used) + 1 - bits_ffs(used);
        r.free_runs_in = frn - f0 - f1;
    }
    return r;
}

// _get_network_compactness from its integer sums over the links: occupied = sum of spans, unused = free runs inside them
__device__ __forceinline__ double compactness_value(const Params &p, long long occupied, long long unused, long long sum_nh) {
    if (unused > 0) return __dmul_rn(__ddiv_rn((double)occupied, (double)sum_nh), __ddiv_rn((double)p.E, (double)unused));
    return 1.0;
}

// _get_network_compactness (rmsa_env.py:699-744)
// (rmcsa_env.py:825-871: the links of ONE core, number_slots * hops summed over all running services)
__device__ __forceinline__ double network_compactness(const Params &p, int env, long long sum_nh, int core = 0) {
    long long occupied = 0, unused = 0;
    for (int l = 0; l < p.E; l++) {
        const LinkShape s = link_shape(bits_from(p.masks[(size_t)(core * p.E + l) * p.n + env]), p.S);
        occupied += s.span; unused += s.free_runs_in;
    }
    return compactness_value(p, occupied, unused, sum_nh);
}

// _update_link_stats (rmsa_env.py:464-543, rmcsa_env.py:591-688, rwa_env.py:365-383: utilisation only) for link l whose (already
// updated) mask -- of the core being touched -- has the shape `shape()`; the statistics are per LINK (RMCSA's cores share them)
template <typename ShapeFn>
__device__ __forceinline__ void update_link_stats_with(const Params &p, int env, int l, double now, ShapeFn shape) {
    const size_t i = (size_t)l * p.n + env;
    const double last_update = p.link_last[i];
    const double time_diff = __dadd_rn(now, -last_update);
    if (now > 0) {
        const LinkShape s = shape();
        const double cur_util = __ddiv_rn((double)(p.S - s.free_cnt), (double)p.S);
        p.link_util[i] = __ddiv_rn(__dadd_rn(__dmul_rn(p.link_util[i], last_update), __dmul_rn(cur_util, time_diff)), now);
        if (p.kind != ORLG_RWA) {
            double cur_comp = 0.0, cur_frag = 0.0;
            if (s.free_cnt > 0) {
                cur_comp = s.used_runs > 1 ? __dmul_rn(__ddiv_rn((double)s.span, (double)(p.S - s.free_cnt)), __ddiv_rn(1.0, (double)s.used_runs)) : 1.0;
                // max_empty stays 0 for fewer than two free runs and when they are exactly the first and the last block
                const int max_empty = (s.free_runs > 1 && !(s.free_runs == 2 && s.free_at_both_ends)) ? s.longest_free : 0;
                cur_frag = __dadd_rn(1.0, -__ddiv_rn((double)max_empty, (double)s.free_cnt));
            }
            p.link_frag[i] = __ddiv_rn(__dadd_rn(__dmul_rn(p.link_frag[i], last_update), __dmul_rn(cur_frag, time_diff)), now);
            p.link_comp[i] = __ddiv_rn(__dadd_rn(__dmul_rn(p.link_comp[i], last_update), __dmul_rn(cur_comp, time_diff)), now);
        }
    }
    p.link_last[i] = now;
}
__device__ __forceinline__ void update_link_stats(const Params &p, int env, int l, const Bits &fr, double now) {
    update_link_stats_with(p, env, l, now, [&] { return link_shape(fr, p.S); });
}

// _update_network_stats (rmsa_env.py:439-462, rmcsa_env.py:560-589; a no-op for RWA): called by _provision_path only, after the
// new service joined graph["running_services"]; `compactness()` is _get_network_compactness of the core being provisioned
template <typename CompactnessFn>
__device__ __forceinline__ void update_network_stats_with(const Params &p, int env, long long run_br, double now, CompactnessFn compactness) {
    double *g = p.graph_stats + env;
    const double last_update = g[2 * (size_t)p.n];
    const double time_diff = __dadd_rn(now, -last_update);
    if (now > 0) {
        g[0] = __ddiv_rn(__dadd_rn(__dmul_rn(g[0], last_update), __dmul_rn((double)run_br, time_diff)), now);
        g[p.n] = __ddiv_rn(__dadd_rn(__dmul_rn(g[p.n], last_update), __dmul_rn(compactness(), time_diff)), now);
    }
    g[2 * (size_t)p.n] = now;
}
__device__ __forceinline__ void update_network_stats(const Params &p, int env, long long sum_nh, long long run_br, int core, double now) {
    update_network_stats_with(p, env, run_br, now, [&] { return network_compactness(p, env, sum_nh, core); });
}

// numpy's pairwise summation of the n <= 128 links at positions [off, off + n) of topology.edges() order (8 partial sums)
__device__ __forceinline__ double links_block_sum(const Params &p, const double *per_link, int env, int off, int n) {
    const int *order = p.link_order + off;
    double res;
    if (n < 8) {
        res = 0.0;
        for (int i = 0; i < n; i++) res = __dadd_rn(res, per_link[(size_t)order[i] * p.n + env]);
    } else {
        double r[8];
#pragma unroll
        for (int j = 0; j < 8; j++) r[j] = per_link[(size_t)order[j] * p.n + env];
        int i;
        for (i = 8; i < n - (n % 8); i += 8) {
#pragma unroll
            for (int j = 0; j < 8; j++) r[j] = __dadd_rn(r[j], per_link[(size_t)order[i + j] * p.n + env]);
        }
        res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
        for (; i < n; i++) res = __dadd_rn(res, per_link[(size_t)order[i] * p.n + env]);
    }
    return res;
}

// np.mean over the links in topology.edges() order.  Above 128 links numpy's pairwise_sum splits a range of n at
// n2 = n / 2 - (n / 2) % 8 and adds the sums of the two halves; that recursion runs here on an explicit stack (16 frames
// reach far beyond the 65535 links a hop list can name).
__device__ __forceinline__ double mean_over_links(const Params &p, const double *per_link, int env) {
    const int n = p.E;
    double res;
    if (n <= 128) {
        res = links_block_sum(p, per_link, env, 0, n);
    } else {
        int off[16], len[16], phase[16];     // phase 0: left half next, 1: right half next, 2: add the halves
        double left[16];
        int sp = 1;
        off[0] = 0; len[0] = n; phase[0] = 0;
        res = 0.0;
        while (sp > 0) {
            const int i = sp - 1;
            if (len[i] <= 128) { res = links_block_sum(p, per_link, env, off[i], len[i]); sp--; continue; }
            int n2 = len[i] / 2;
            n2 -= n2 % 8;
            if (phase[i] == 0) { phase[i] = 1; off[sp] = off[i]; len[sp] = n2; phase[sp] = 0; sp++; }
            else if (phase[i] == 1) { phase[i] = 2; left[i] = res; off[sp] = off[i] + n2; len[sp] = len[i] - n2; phase[sp] = 0; sp++; }
            else { res = __dadd_rn(left[i], res); sp--; }
        }
    }
    return __ddiv_rn(res, (double)n);
}

// _provision_path / _release_path with the per-link statistics, links in hop order (rmsa_env.py:381-396, 418-436)
__device__ __forceinline__ void path_update_stats(const Params &p, int env, int row, int core, const Bits &rm, bool set, double now) {
    for (int h = p.path_link_ptr[row]; h < p.path_link_ptr[row + 1]; h++) {
        const int l = p.path_links16[h];
        uint4 *m = p.masks + (size_t)(core * p.E + l) * p.n + env;
        Bits b = bits_from(*m);
        b = set ? bits_or(b, rm) : bits_andnot(b, rm);
        *m = bits_to(b);
        update_link_stats(p, env, l, b, now);
    }
}

// Release every service due at `now` on a handle with statistics (rmsa_env.py:591-597).  The reference releases in heap order
// (by time) and every release updates the statistics of its links, so the due services are collected, sorted by release time
// and applied in that order.  Beyond 24 of them in one step the rest are applied as they come (the masks stay exact, the order
// of the statistics does not) and ORLG_ERR_STATS_ORDER is set.  release(payload) provisions the service's slots back with the
// link statistics and returns its number_slots * hops, which leaves sum_nh; its bit rate leaves run_br.
template <typename ReleaseFn>
__device__ __forceinline__ void release_due_in_order(const Params &p, int env, const Events &ev, unsigned &nheap, double &hmin,
                                                     double &tailmin, double now, unsigned &err, ReleaseFn release) {
    constexpr int MAXR = 24;
    double rt[MAXR];
    unsigned long long rp[MAXR];
    int nr = 0;
    long long rel_br = 0;                                // bit rates leaving graph["running_services"]
    events_release(ev, nheap, hmin, tailmin, now, apply_timed([&](unsigned long long pl, double t, unsigned sbr) {
        rel_br += sbr;
        if (nr < MAXR) { rt[nr] = t; rp[nr] = pl; nr++; }
        else { err |= ORLG_ERR_STATS_ORDER; p.sum_nh[env] -= release(pl); }
    }));
    if (rel_br) p.run_br[env] -= rel_br;
    for (int a = 1; a < nr; a++) {                       // insertion sort by release time
        const double t = rt[a];
        const unsigned long long q = rp[a];
        int b = a - 1;
        while (b >= 0 && rt[b] > t) { rt[b + 1] = rt[b]; rp[b + 1] = rp[b]; b--; }
        rt[b + 1] = t; rp[b + 1] = q;
    }
    long long snh = p.sum_nh[env];
    for (int a = 0; a < nr; a++) snh -= release(rp[a]);
    p.sum_nh[env] = snh;
}

// the float statistics at a full reset (optical_network_env.py:181-203, rmsa_env.py:332-359)
__device__ __forceinline__ void clear_stats(const Params &p, int env) {
    for (int l = 0; l < p.E; l++) {
        const size_t i = (size_t)l * p.n + env;
        p.link_util[i] = 0.0; p.link_comp[i] = 0.0; p.link_last[i] = 0.0; p.link_frag[i] = 0.0;
    }
    p.sum_nh[env] = 0; p.run_br[env] = 0;
    for (int q = 0; q < 3; q++) p.graph_stats[(size_t)q * p.n + env] = 0.0;
}

template <typename T>
__device__ __forceinline__ T obs_ratio(int num, int den);
// float32 observations: one correctly rounded division of the exact rational (<= 1 ulp of the
// reference's float64 value, i.e. ~6e-8 relative)
template <>
__device__ __forceinline__ float obs_ratio<float>(int num, int den) { return __fdiv_rn((float)num, (float)den); }

struct PathFeat {            // integer pre-image of one row of deeprmsa_env.py:72-108
    int n, total, runs;
};

// ---------------------------------------------------------------- the step kernel
template <int KIND, int KM>
__global__ void __launch_bounds__(STEP_THREADS) step_kernel(const Params p, const StepIO io, const int mode) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int env = blockIdx.x * STEP_THREADS + threadIdx.x;
    const bool live = env < p.n;
    const int e = live ? env : p.n - 1;       // clamp: out-of-range threads recompute env n-1 but never store

    // ---- load the scalar block
    double now = p.now[e];
    double hold = p.cur_hold[e];
    uint2 rq = p.cur_req[e];
    int src = rq.x & 0xff, dst = (rq.x >> 8) & 0xff, br = (int)(rq.x >> 16), sid = (int)rq.y;
    long long cnt[8];
#pragma unroll
    for (int q = 0; q < 8; q++) cnt[q] = p.counters[(size_t)q * p.n + e];
    unsigned ridx = p.req_index[e];
    unsigned nheap = p.nheap[e];
    double hmin = p.heap_min[e];
    unsigned err = p.errors[e];
    const Events ev = {p.ev_time + (size_t)e * p.heap_cap, p.ev_pay + (size_t)e * p.heap_cap, p.ev_gmin + (size_t)e * p.ev_groups,
                       p.stats ? p.ev_br + (size_t)e * p.heap_cap : nullptr};
    double tailmin = p.ev_tail[e];

    bool accepted = false;
    int d_row = -1, d_start = -1, d_n = -1, d_core = -1, d_mod = -1;
    bool done = false;

  if (live) {      // ---- everything below touches only this thread's environment
    if (mode == MODE_FULL_RESET) {
        // optical_network_env.py:181-203 + rmsa_env.py:332-359: empty network, clock 0, counters 0
        Bits full = bits_range(0, p.S);
        if (live)
            for (int l = 0; l < p.C * p.E; l++) p.masks[(size_t)l * p.n + env] = bits_to(full);
        now = 0.0; nheap = 0; hmin = ORLG_INF; tailmin = ORLG_INF; ridx = 0; err = 0;
#pragma unroll
        for (int q = 0; q < 8; q++) cnt[q] = 0;
        if (KIND == ORLG_RMSA) br_hist_clear(p, env);
        if (KIND == ORLG_RWA) act_hist_clear(p, env);          // rwa_env.py:195-201
    }

    if (mode == MODE_STEP) {
        // ================= Phase A: the action on the pending request ==================
        const int pair = src * p.N + dst;
        const int first = p.pair_first[pair];
        const int npaths = p.pair_count[pair];
        int row = -1, start = 0, n = 0, core = 0, mod = -1;
        unsigned lm = 0;
        if (KIND == ORLG_DEEPRMSA) {
            // deeprmsa_env.py:48-58: block-th first-fit block of route; the block starts of the pending
            // request were computed (from the same masks) when its observation was built.
            int a = io.actions[e];
            if (a >= 0 && a < p.k * p.J) {
                int route = a / p.J;
                if (route < npaths) {
                    unsigned st = p.cand[(size_t)e * p.cand_stride + a];
                    if (st != CAND_NONE) {
                        row = first + route;
                        unsigned meta = p.path_meta[row];
                        n = p.nslots[meta_se(meta) * (p.br_max + 1) + br];
                        start = (int)st;
                        lm = p.path_linkmask[row];
                        accepted = true;
                    }
                } else {
                    err |= ORLG_ERR_NO_SUCH_PATH;
                }
            }
        } else if (KIND == ORLG_RMSA || KIND == ORLG_RWA) {
            // rmsa_env.py:174-200 / rwa_env.py:104-127
            int path = io.actions[2 * e], slot = io.actions[2 * e + 1];
            if (KIND == ORLG_RWA) act_hist_bump(p, env, path, slot, err);
            if (path >= 0 && path < p.k && slot >= 0 && slot < p.S) {
                if (path < npaths) {
                    row = first + path;
                    unsigned meta = p.path_meta[row];
                    n = (KIND == ORLG_RWA) ? 1 : p.nslots[meta_se(meta) * (p.br_max + 1) + br];
                    start = slot;
                    lm = p.path_linkmask[row];
                    if (start + n <= p.S) {                      // is_path_free, rmsa_env.py:623-636
                        Bits A = path_free(p, e, lm, 0);
                        accepted = bits_contains(A, bits_range(start, start + n));
                    }
                } else {
                    err |= ORLG_ERR_NO_SUCH_PATH;
                }
            }
        } else {
            // rmcsa_env.py:209-277: (path, modulation, core, initial_slot)
            int path = io.actions[4 * e], am = io.actions[4 * e + 1], ac = io.actions[4 * e + 2], slot = io.actions[4 * e + 3];
            if (path >= 0 && path < p.k && am >= 0 && am < p.M && ac >= 0 && ac < p.C && slot >= 0 && slot < p.S) {
                if (path < npaths) {
                    row = first + path;
                    n = p.nslots[p.mod_se[am] * (p.br_max + 1) + br];
                    start = slot; core = ac; mod = am;
                    lm = p.path_linkmask[row];
                    if (start + n <= p.S) {
                        Bits A = path_free(p, e, lm, core);
                        accepted = bits_contains(A, bits_range(start, start + n)) &&
                                   (p.path_length[row] < p.reach[am * (p.br_max + 1) + br]);   // _crosstalk_is_acceptable
                    }
                } else {
                    err |= ORLG_ERR_NO_SUCH_PATH;
                }
            }
        }
        if (accepted && nheap + 1 > (unsigned)p.heap_cap) {
            accepted = false;
            err |= ORLG_ERR_HEAP_OVERFLOW;
        }
        const bool do_stats = p.stats != 0;
        const bool info_stats = do_stats && p.stats_out && (KIND == ORLG_RMSA || KIND == ORLG_DEEPRMSA);
        long long snh = do_stats ? p.sum_nh[env] : 0;
        const double prev_compactness = info_stats ? network_compactness(p, env, snh) : 0.0;     // rmsa_env.py:168-170
        if (accepted) {
            if (live) {
                if (do_stats) {
                    path_update_stats(p, env, row, core, bits_range(start, start + n), false, now);
                    snh += (long long)n * meta_hops(p.path_meta[row]);
                    p.sum_nh[env] = snh;
                    if (KIND != ORLG_RWA) {
                        const long long rb = p.run_br[env] + br;
                        p.run_br[env] = rb;
                        update_network_stats(p, env, snh, rb, core, now);
                    }
                } else
                path_update(p, env, lm, core, bits_range(start, start + n), false);
                double rel = __dadd_rn(now, hold);          // arrival_time + holding_time (now == arrival)
                events_push(ev, nheap, hmin, tailmin, rel, pack_service(row, start, n, core, sid), (unsigned)br);
            }
            if (KIND == ORLG_RMSA) br_hist_bump(p, env, 1, br);     // rmsa_env.py:408-415
            d_row = row; d_start = start; d_n = n; d_core = core; d_mod = mod;
        }
        count_decision<KIND>(cnt, accepted, br);
        if (live) {
            if (io.reward) io.reward[env] = accepted ? 1.0f : (KIND == ORLG_DEEPRMSA ? -1.0f : 0.0f);
            if (io.decision) {
                int *d = io.decision + (size_t)env * 6;
                d[0] = accepted; d[1] = d_row; d[2] = d_start; d[3] = d_n;
                d[4] = (KIND == ORLG_RMCSA) ? d_core : (accepted ? 0 : -1);
                d[5] = d_mod;
            }
            if (io.info) {
#pragma unroll
                for (int q = 0; q < 8; q++) io.info[(size_t)env * 8 + q] = cnt[q];
            }
            if (info_stats) {                                   // rmsa_env.py:229-264
                const double cur = network_compactness(p, env, snh);
                double *so = p.stats_out + (size_t)env * 4;
                so[0] = cur;
                so[1] = __dadd_rn(prev_compactness, -cur);
                so[2] = mean_over_links(p, p.link_comp, env);
                so[3] = mean_over_links(p, p.link_util, env);
            }
        }
    }

    if (mode == MODE_FULL_RESET && p.stats) clear_stats(p, env);

    if (mode == MODE_STEP || mode == MODE_FULL_RESET) {
        // ================= Phase B: _next_service (rmsa_env.py:545-597) ==================
        double arrival, holding;
        int nsrc, ndst, nbr;
        if (p.traffic == ORLG_TRAFFIC_PHILOX) {
            philox_request(p, p.node_thr, e, ridx, now, arrival, holding, nsrc, ndst, nbr);
        } else {
            const orlg_request r = trace_request(p, e, ridx, now, p.br_max, p.br_lo, false, err);
            arrival = r.arrival; holding = r.holding; nsrc = r.src; ndst = r.dst; nbr = r.bit_rate;
        }
        ridx++;
        now = arrival; hold = holding; src = nsrc; dst = ndst; br = nbr;
        sid = (int)cnt[2];                                    // Service(self.episode_services_processed, ...)
        count_request<KIND>(cnt, br);
        if (KIND == ORLG_RMSA) br_hist_bump(p, env, 0, br);     // rmsa_env.py:579-581
        // release every service whose time has come (rmsa_env.py:591-597)
        if (p.stats)
            release_due_in_order(p, env, ev, nheap, hmin, tailmin, now, err, [&](unsigned long long pl) {
                const int rs = svc_start(pl);
                path_update_stats(p, env, svc_row(pl), svc_core(pl), bits_range(rs, rs + svc_slots(pl)), true, now);
                return (long long)svc_slots(pl) * meta_hops(p.path_meta[svc_row(pl)]);
            });
        else
        events_release(ev, nheap, hmin, tailmin, now, apply_payload([&](unsigned long long pl) {
            const int rs = svc_start(pl);
            path_update(p, env, p.path_linkmask[svc_row(pl)], svc_core(pl), bits_range(rs, rs + svc_slots(pl)), true);
        }));
        done = (cnt[2] == (long long)p.episode_length);
    }

    if (mode == MODE_EPISODE_RESET || (mode == MODE_STEP && done && p.auto_reset)) reset_episode_counters<KIND>(cnt, br);

    // ================= Phase C: observation of the pending request (deeprmsa_env.py:60-121) =========
    if (KIND == ORLG_DEEPRMSA) {
        const int pair = src * p.N + dst;
        const int first = p.pair_first[pair];
        const int npaths = min((int)p.pair_count[pair], KM);
        unsigned lms[KM];
        int ns[KM];
        Bits A[KM];
#pragma unroll
        for (int q = 0; q < KM; q++) {
            A[q] = bits_ones();
            lms[q] = 0; ns[q] = 1;
            if (q < npaths) {
                lms[q] = p.path_linkmask[first + q];
                ns[q] = p.nslots[meta_se(p.path_meta[first + q]) * (p.br_max + 1) + br];
            }
        }
        {
            // one coalesced sweep over all links; each path keeps the AND of its own links in registers
            const uint4 *mr = p.masks + e;
#pragma unroll 2
            for (int l = 0; l < p.E; l++) {
                uint4 m = mr[(size_t)l * p.n];
#pragma unroll
                for (int q = 0; q < KM; q++) {
                    unsigned keep = ((lms[q] >> l) & 1u) - 1u;      // on the path: 0, else all ones
                    A[q].w[0] &= m.x | keep; A[q].w[1] &= m.y | keep;
                    A[q].w[2] &= m.z | keep; A[q].w[3] &= m.w | keep;
                }
            }
        }
        const int W = 2 * p.J + 3;
        float *so32 = reinterpret_cast<float *>(smem_raw) + (size_t)threadIdx.x * p.obs_dim;
        double *so64 = reinterpret_cast<double *>(smem_raw) + (size_t)threadIdx.x * p.obs_dim;
        const bool want_obs = io.obs != nullptr;
        if (want_obs) {
            if (p.obs_f64) {
                for (int q = 0; q < p.obs_dim; q++) so64[q] = (q > 2 * p.N) ? -1.0 : 0.0;
                so64[0] = __ddiv_rn((double)br, 100.0);
                so64[1 + min(src, dst)] = 1.0;
                so64[1 + p.N + max(src, dst)] = 1.0;
            } else {
                for (int q = 0; q < p.obs_dim; q++) so32[q] = (q > 2 * p.N) ? -1.0f : 0.0f;
                so32[0] = obs_ratio<float>(br, 100);
                so32[1 + min(src, dst)] = 1.0f;
                so32[1 + p.N + max(src, dst)] = 1.0f;
            }
        }
#pragma unroll
        for (int q = 0; q < KM; q++) {
            if (q < npaths) {
                const int n = ns[q];
                Bits B = bits_runs_ge(A[q], n);
                Bits starts = bits_andnot(B, bits_shl1(B));                 // run starts (SURVEY.md 7.6)
                const int total = bits_popc(A[q]);
                const int runs = bits_popc(bits_andnot(A[q], bits_shl1(A[q])));
                const int ob = 1 + 2 * p.N + q * W;
                for (int b = 0; b < p.J; b++) {
                    int st = bits_ffs(starts);
                    if (live) p.cand[(size_t)env * p.cand_stride + q * p.J + b] = (unsigned char)(st < 0 ? CAND_NONE : st);
                    if (st < 0) {
                        if (live && io.obs_int) { io.obs_int[((size_t)env * p.k + q) * W + 2 * b] = -1; io.obs_int[((size_t)env * p.k + q) * W + 2 * b + 1] = -1; }
                        continue;
                    }
                    starts = bits_clear_lowest(starts);
                    int len = bits_run_length(A[q], st);
                    if (want_obs) {
                        if (p.obs_f64) {
                            // 2 * (initial_index - 0.5 * S) / S ; (length - 8) / 8
                            so64[ob + 2 * b] = __ddiv_rn(__dmul_rn(2.0, __dadd_rn((double)st, -__dmul_rn(0.5, (double)p.S))), (double)p.S);
                            so64[ob + 2 * b + 1] = __ddiv_rn(__dadd_rn((double)len, -8.0), 8.0);
                        } else {
                            so32[ob + 2 * b] = obs_ratio<float>(2 * st - p.S, p.S);
                            so32[ob + 2 * b + 1] = obs_ratio<float>(len - 8, 8);
                        }
                    }
                    if (live && io.obs_int) { io.obs_int[((size_t)env * p.k + q) * W + 2 * b] = st; io.obs_int[((size_t)env * p.k + q) * W + 2 * b + 1] = len; }
                }
                if (want_obs) {
                    if (p.obs_f64) {
                        so64[ob + 2 * p.J] = __ddiv_rn(__dadd_rn((double)n, -5.5), 3.5);
                        so64[ob + 2 * p.J + 1] = __ddiv_rn(__dmul_rn(2.0, __dadd_rn((double)total, -__dmul_rn(0.5, (double)p.S))), (double)p.S);
                        if (runs > 0)   // (np.mean(lengths) - 4) / 4
                            so64[ob + 2 * p.J + 2] = __ddiv_rn(__dadd_rn(__ddiv_rn((double)total, (double)runs), -4.0), 4.0);
                    } else {
                        so32[ob + 2 * p.J] = obs_ratio<float>(2 * n - 11, 7);
                        so32[ob + 2 * p.J + 1] = obs_ratio<float>(2 * total - p.S, p.S);
                        if (runs > 0) so32[ob + 2 * p.J + 2] = obs_ratio<float>(total - 4 * runs, 4 * runs);
                    }
                }
                if (live && io.obs_int) {
                    int *oi = io.obs_int + ((size_t)env * p.k + q) * W;
                    oi[2 * p.J] = n; oi[2 * p.J + 1] = total; oi[2 * p.J + 2] = runs;
                }
            }
        }
        if (live) {
            for (int q = npaths * p.J; q < p.k * p.J; q++) p.cand[(size_t)env * p.cand_stride + q] = (unsigned char)CAND_NONE;
            if (io.obs_int)
                for (int q = npaths * W; q < p.k * W; q++) io.obs_int[(size_t)env * p.k * W + q] = -1;
        }
    }
  }                // ---- end of the per-env body

    if (KIND == ORLG_DEEPRMSA) {
        if (io.obs != nullptr) {
            // block-wide coalesced copy of the [STEP_THREADS, obs_dim] tile
            __syncthreads();
            const size_t tile0 = (size_t)blockIdx.x * STEP_THREADS * p.obs_dim;
            const int rows = min(STEP_THREADS, p.n - blockIdx.x * STEP_THREADS);
            const int total_el = rows * p.obs_dim;
            if (p.obs_f64) {
                const double *s = reinterpret_cast<const double *>(smem_raw);
                double *g = reinterpret_cast<double *>(io.obs) + tile0;
                for (int q = threadIdx.x; q < total_el; q += STEP_THREADS) g[q] = s[q];
            } else {
                const float *s = reinterpret_cast<const float *>(smem_raw);
                float *g = reinterpret_cast<float *>(io.obs) + tile0;
                for (int q = threadIdx.x; q < total_el; q += STEP_THREADS) g[q] = s[q];
            }
        }
    }

    // ---- store the scalar block
    if (live && mode != MODE_OBSERVE) {
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

// uniform random policy: Philox stream 2, counter = requests generated so far (DESIGN.md "Traffic")
// Programmatic dependent launch (griddepcontrol): a kernel launched with the programmatic-stream-serialization
// attribute may start while its predecessor in the stream drains; it must not touch the predecessor's outputs before
// pdl_wait().  Both are no-ops for an ordinary launch.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__global__ void random_action_kernel(const Params p, int *actions) {
    pdl_launch_dependents();
    pdl_wait();                      // req_index is written by the preceding step kernel
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    unsigned long long gid = (unsigned long long)(p.env_id_base + env);
    uint32_t c[4] = {p.req_index[env], 0u, (uint32_t)gid, 2u};
    philox4x32_10(c, (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
    const unsigned rej = p.allow_rejection ? 1u : 0u;
    if (p.kind == ORLG_DEEPRMSA) {
        actions[env] = (int)__umulhi(c[0], (unsigned)(p.k * p.J) + rej);
    } else if (p.kind == ORLG_RMCSA) {
        actions[4 * env] = (int)__umulhi(c[0], (unsigned)p.k + rej);
        actions[4 * env + 1] = (int)__umulhi(c[1], (unsigned)p.M);
        actions[4 * env + 2] = (int)__umulhi(c[2], (unsigned)p.C + rej);
        actions[4 * env + 3] = (int)__umulhi(c[3], (unsigned)p.S + rej);
    } else {
        actions[2 * env] = (int)__umulhi(c[0], (unsigned)p.k + rej);
        actions[2 * env + 1] = (int)__umulhi(c[1], (unsigned)p.S + rej);
    }
}

// full reset: empty release-event tables (every time slot and every directory entry = +INF)
__global__ void fill_events_kernel(const Params p) {
    const size_t nt = (size_t)p.n * p.heap_cap, ng = (size_t)p.n * p.ev_groups;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nt; i += stride) p.ev_time[i] = ORLG_INF;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < ng; i += stride) p.ev_gmin[i] = ORLG_INF_F;
}

// ---------------------------------------------------------------- introspection kernels
__global__ void export_kernel(const Params p, unsigned *masks_out, int *alloc_out, double *now_out, int *nheap_out,
                              long long *counters_out, orlg_request *req_out, int *sid_out, unsigned *err_out) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    const int CE = p.C * p.E;
    if (masks_out)
        for (int l = 0; l < CE; l++) {
            uint4 m = p.masks[(size_t)l * p.n + env];
            unsigned *o = masks_out + ((size_t)env * CE + l) * NW;
            o[0] = m.x; o[1] = m.y; o[2] = m.z; o[3] = m.w;
        }
    if (alloc_out) {
        // spectrum_slots_allocation rebuilt from the live services (rmsa_env.py:386-389)
        int *o = alloc_out + (size_t)env * CE * p.S;
        for (int q = 0; q < CE * p.S; q++) o[q] = -1;
        const unsigned long long *h = p.ev_pay + (size_t)env * p.heap_cap;
        const unsigned nh = p.nheap[env];
        for (unsigned s = 0; s < nh; s++) {
            unsigned long long pl = h[s];
            unsigned lm = p.path_linkmask[svc_row(pl)];
            while (lm) {
                int l = __ffs(lm) - 1;
                lm &= lm - 1;
                for (int q = 0; q < svc_slots(pl); q++) o[((size_t)svc_core(pl) * p.E + l) * p.S + svc_start(pl) + q] = svc_id(pl);
            }
        }
    }
    if (now_out) now_out[env] = p.now[env];
    if (nheap_out) nheap_out[env] = (int)p.nheap[env];
    if (counters_out)
        for (int q = 0; q < 8; q++) counters_out[(size_t)env * 8 + q] = p.counters[(size_t)q * p.n + env];
    if (req_out) {
        uint2 rq = p.cur_req[env];
        orlg_request r;
        r.arrival = p.now[env]; r.holding = p.cur_hold[env];
        r.src = rq.x & 0xff; r.dst = (rq.x >> 8) & 0xff; r.bit_rate = (int)(rq.x >> 16); r.reserved = 0;
        req_out[env] = r;
    }
    if (sid_out) sid_out[env] = (int)p.cur_req[env].y;
    if (err_out) err_out[env] = p.errors[env];
}

// row f1 read-out: the statistics the reference keeps on the topology graph.  link_out [n][E][3] = utilization,
// external_fragmentation, compactness per link index; graph_out [n][2] = throughput, compactness
__global__ void link_stats_kernel(const Params p, double *link_out, double *graph_out) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    if (link_out)
        for (int l = 0; l < p.E; l++) {
            const size_t i = (size_t)l * p.n + env;
            double *o = link_out + ((size_t)env * p.E + l) * 3;
            o[0] = p.link_util[i]; o[1] = p.link_frag[i]; o[2] = p.link_comp[i];
        }
    if (graph_out) { graph_out[2 * (size_t)env] = p.graph_stats[env]; graph_out[2 * (size_t)env + 1] = p.graph_stats[(size_t)p.n + env]; }
}

// info["bit_rate_blocking_<rate>"] and info["fairness"] (rmsa_env.py:217-227, 268-273) as the reference sees them when
// it builds `info`: the pending request (drawn after that point) is taken out of the requested histogram again.
__global__ void bit_rate_blocking_kernel(const Params p, double *out) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    const int B = p.n_bit_rates;
    const int pending = br_index(p, (int)(p.cur_req[env].x >> 16));
    double lo = 0.0, hi = 0.0;
    for (int i = 0; i < B; i++) {
        const int req = p.br_hist[(size_t)i * p.n + env] - (i == pending ? 1 : 0);
        const int prov = p.br_hist[((size_t)B + i) * p.n + env];
        const double b = req > 0 ? __ddiv_rn((double)(req - prov), (double)req) : 0.0;
        out[(size_t)env * (B + 1) + i] = b;
        lo = i == 0 ? b : fmin(lo, b);
        hi = i == 0 ? b : fmax(hi, b);
    }
    out[(size_t)env * (B + 1) + B] = __dadd_rn(hi, -lo);
}

// info["path_action_probability"] ++ info["wavelength_action_probability"] (rwa_env.py:148-151): marginals of
// actions_output divided by its total (int / int -> float64, like numpy)
__global__ void action_probability_kernel(const Params p, double *out) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    const int R = p.k + p.allow_rejection, Cn = p.S + p.allow_rejection;
    long long total = 0;
    for (int i = 0; i < R; i++) total += p.act_hist[(size_t)i * p.n + env];
    for (int i = 0; i < R + Cn; i++)
        out[(size_t)env * (R + Cn) + i] = __ddiv_rn((double)p.act_hist[(size_t)i * p.n + env], (double)total);
}

// per-device sums of the 8 counters (+ #envs with an error flag) for the cross-GPU all-reduce
__global__ void reduce_counters_kernel(const Params p, unsigned long long *sums) {
    __shared__ unsigned long long part[9];
    if (threadIdx.x < 9) part[threadIdx.x] = 0;
    __syncthreads();
    unsigned long long loc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int env = blockIdx.x * blockDim.x + threadIdx.x; env < p.n; env += gridDim.x * blockDim.x) {
#pragma unroll
        for (int q = 0; q < 8; q++) loc[q] += (unsigned long long)p.counters[(size_t)q * p.n + env];
        loc[8] += p.errors[env] ? 1 : 0;
    }
#pragma unroll
    for (int q = 0; q < 9; q++) {
        unsigned long long v = loc[q];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) atomicAdd(&part[q], v);
    }
    __syncthreads();
    if (threadIdx.x < 9) atomicAdd(&sums[threadIdx.x], part[threadIdx.x]);
}

}  // namespace orlg
