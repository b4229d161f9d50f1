// orlg_step_wide.cuh -- step / heuristic / export kernels for topologies beyond the NSFNET class:
// any number of links (path -> link lists in CSR form instead of 32-bit link bitmaps), up to 512 slots
// per link (NWV = 1..4 128-bit word groups per (core, link)), up to 31 cores, k <= 16 candidate paths.
// Covers BASELINE.json configs[3] (RMSA-v0, 100 nodes / 300 links, 320 slots, k = 10) and configs[4]
// (RMCSA-v0, 7 cores x 320 slots).  Same semantics, same state arrays and the same release-event table as
// step_kernel (orlg_kernels.cuh); one thread per environment, masks accessed in place:
//     masks[(env * C * E + core * E + link) * wstride + v]   (uint4; env-major: an entry's words share one DRAM burst,
//     an env's entries one page -- every thread walks its OWN path, so the [link][env] layout of the NSFNET-class kernels
//     would put each of its accesses on a different 2 MB page)
#pragma once
#include "orlg_kernels.cuh"

namespace orlg {

template <int NWV>
struct WBits {
    uint32_t w[4 * NWV];
};

template <int NWV>
__device__ __forceinline__ WBits<NWV> wb_fill(uint32_t v) {
    WBits<NWV> b;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) b.w[i] = v;
    return b;
}
// bits [lo, hi) set
template <int NWV>
__device__ __forceinline__ WBits<NWV> wb_range(int lo, int hi) {
    WBits<NWV> r;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) {
        int a = min(max(lo - 32 * i, 0), 32), b = min(max(hi - 32 * i, 0), 32);
        uint32_t ma = a >= 32 ? 0u : (0xFFFFFFFFu << a);
        uint32_t mb = b >= 32 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu << b);
        r.w[i] = ma & mb;
    }
    return r;
}
template <int NWV>
__device__ __forceinline__ bool wb_contains(const WBits<NWV> &a, const WBits<NWV> &m) {
    uint32_t miss = 0;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) miss |= (~a.w[i]) & m.w[i];
    return miss == 0;
}
template <int NWV>
__device__ __forceinline__ int wb_popc(const WBits<NWV> &a) {
    int c = 0;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) c += __popc(a.w[i]);
    return c;
}
template <int NWV>
__device__ __forceinline__ int wb_ffs(const WBits<NWV> &a) {
    int r = -1;
#pragma unroll
    for (int i = 4 * NWV - 1; i >= 0; i--)
        if (a.w[i]) r = 32 * i + __ffs(a.w[i]) - 1;
    return r;
}
template <int NWV>
__device__ __forceinline__ int wb_fls(const WBits<NWV> &a) {
    int r = -1;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++)
        if (a.w[i]) r = 32 * i + 31 - __clz(a.w[i]);
    return r;
}
template <int NWV>
__device__ __forceinline__ WBits<NWV> wb_shr_small(const WBits<NWV> &a, int s) {     // 0 <= s < 32
    WBits<NWV> r;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) r.w[i] = __funnelshift_r(a.w[i], i + 1 < 4 * NWV ? a.w[i + 1] : 0u, s);
    return r;
}
template <int NWV>
__device__ __forceinline__ WBits<NWV> wb_shl1(const WBits<NWV> &a) {
    WBits<NWV> r;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) r.w[i] = __funnelshift_l(i > 0 ? a.w[i - 1] : 0u, a.w[i], 1);
    return r;
}
// B[i] = 1 iff A[i .. i+n-1] are all 1 (shift-AND doubling, shifts kept below 32)
template <int NWV>
__device__ __forceinline__ WBits<NWV> wb_runs_ge(const WBits<NWV> &a, int n) {
    WBits<NWV> b = a;
    int len = 1;
    while (len < n) {
        const int s = min(min(len, n - len), 31);
        const WBits<NWV> sh = wb_shr_small(b, s);
#pragma unroll
        for (int i = 0; i < 4 * NWV; i++) b.w[i] &= sh.w[i];
        len += s;
    }
    return b;
}
template <int NWV>
__device__ __forceinline__ WBits<NWV> wb_clear_lowest(const WBits<NWV> &a) {
    WBits<NWV> r = a;
    bool done = false;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++)
        if (!done && r.w[i]) { r.w[i] &= r.w[i] - 1; done = true; }
    return r;
}
// length of the run of ones starting at bit `start`
template <int NWV>
__device__ __forceinline__ int wb_run_length(const WBits<NWV> &a, int start) {
    const WBits<NWV> from = wb_range<NWV>(start, 128 * NWV);
    WBits<NWV> z;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) z.w[i] = ~a.w[i] & from.w[i];
    const int pos = wb_ffs(z);
    return (pos < 0 ? 128 * NWV : pos) - start;
}

// get_available_slots (rmsa_env.py:638-649): AND of the path's link masks.  Four hops at a time: the four link indices are
// fetched together, then all 4 x NWV mask words are requested before any is used (2 dependent round trips per 4 hops instead
// of 2 per hop: the kernel is latency-bound, every lane walks its own path).
template <int NWV>
__device__ __forceinline__ WBits<NWV> wide_path_free(const Params &p, int env, int row, int core) {
    WBits<NWV> a = wb_fill<NWV>(0xFFFFFFFFu);
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
// longest run of ones: one pass over the words, ctz / clz at every run boundary (no shift-AND pass per slot)
template <int NWV>
__device__ __forceinline__ int wb_longest_run(const WBits<NWV> &a) {
    int best = 0, cur = 0;                             // cur: the run that reaches the top of the words seen so far
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) {
        const uint32_t x = a.w[i];
        if (x == 0xFFFFFFFFu) { cur += 32; continue; }
        best = max(best, cur + __ffs(~x) - 1);         // the run coming from below ends at the lowest 0 of x
        const int top = __clz(~x);                     // ones reaching bit 31 start the next carried run
        uint32_t y = (x & (x + 1u)) & (0xFFFFFFFFu >> top);   // the runs strictly inside x (bit 0 of y is 0)
        while (y) {
            const int s = __ffs(y) - 1, len = __ffs(~(y >> s)) - 1;      // s >= 1, so len <= 31
            best = max(best, len);
            y &= ~(((1u << len) - 1u) << s);
        }
        cur = top;
    }
    return max(best, cur);
}

// link_shape (orlg_kernels.cuh) of a multi-word mask: the same integers.  With two or more used runs the free runs outside
// [ffs(used), fls(used) + 1) are exactly the one at slot 0 and the one at slot S - 1 (when those slots are free).
template <int NWV>
__device__ __forceinline__ LinkShape wb_link_shape(const WBits<NWV> &fr, int S) {
    const WBits<NWV> valid = wb_range<NWV>(0, S), last = wb_range<NWV>(S - 1, S);
    WBits<NWV> used;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) used.w[i] = valid.w[i] & ~fr.w[i];
    const WBits<NWV> ul = wb_shl1(used), fl = wb_shl1(fr);
    LinkShape r;
    int ur = 0, frn = 0;
    uint32_t at_end = 0;
#pragma unroll
    for (int i = 0; i < 4 * NWV; i++) {
        ur += __popc(used.w[i] & ~ul.w[i]);
        frn += __popc(fr.w[i] & ~fl.w[i]);
        at_end |= fr.w[i] & last.w[i];
    }
    const int f0 = fr.w[0] & 1u, f1 = at_end != 0;
    r.free_cnt = wb_popc(fr);
    r.used_runs = ur;
    r.free_runs = frn;
    r.longest_free = wb_longest_run(fr);
    r.free_at_both_ends = f0 && f1;
    r.span = 0; r.free_runs_in = 0;
    if (ur > 1) {
        r.span = wb_fls(used) + 1 - wb_ffs(used);
        r.free_runs_in = frn - f0 - f1;
    }
    return r;
}

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
    const WBits<NWV> rm = wb_range<NWV>(start, start + n);
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
            s.free_cnt = wb_popc(b);                   // rwa_env.py:365-383: utilisation only
        } else {
            s = wb_link_shape(b, p.S);
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

// heuristic action sources (SURVEY a21) for the wide layout: the action of env's pending request (src, dst, br) into a[0..3]
// Returns true when the action is KNOWN to fit (it was derived from the path's free mask just now), so that the fused step
// does not have to read the masks a second time for is_path_free.
template <int KIND, int NWV>
__device__ __forceinline__ bool wide_heuristic(const Params &p, const int env, const int which, const int src, const int dst, const int br, int *a) {
    const int pair = src * p.N + dst;
    const int first = p.pair_first[pair];
    const int npaths = min((int)p.pair_count[pair], p.k);
    if (KIND == ORLG_DEEPRMSA) {
        int act = p.k * p.J;
        if (which == ORLG_HEUR_SP_FF) act = (!p.allow_rejection || p.cand16[(size_t)env * p.cand_stride] != 0xFFFFu) ? 0 : p.k * p.J;
        else
            for (int q = 0; q < npaths; q++)
                if (p.cand16[(size_t)env * p.cand_stride + q * p.J] != 0xFFFFu) { act = q * p.J; break; }
        a[0] = act;
        return false;
    } else if (KIND == ORLG_RMSA) {
        int ap = p.k, as = p.S, max_free = 0;
        const int np_ = (which == ORLG_HEUR_SP_FF) ? min(npaths, 1) : npaths;
        for (int q = 0; q < np_; q++) {
            const int n = wide_nslots(p, meta_se(p.path_meta[first + q]), br);
            const WBits<NWV> A = wide_path_free<NWV>(p, env, first + q, 0);
            WBits<NWV> B = wb_runs_ge(A, n);
            const WBits<NWV> lim = wb_range<NWV>(0, max(p.S - n, 0));          // range(0, S - n): App. B-5
#pragma unroll
            for (int i = 0; i < 4 * NWV; i++) B.w[i] &= lim.w[i];
            const int s = wb_ffs(B);
            if (s >= 0) {
                if (which == ORLG_HEUR_LLP_FF) {
                    const int fr = wb_popc(A);
                    if (fr > max_free) { ap = q; as = s; max_free = fr; }
                } else { ap = q; as = s; break; }
            }
        }
        a[0] = ap; a[1] = as;
        return ap < p.k;
    } else if (KIND == ORLG_RWA) {
        int ap = p.k, as = p.S;
        if (which == ORLG_HEUR_SP_FF) {
            if (npaths > 0) {
                const int s = wb_ffs(wide_path_free<NWV>(p, env, first, 0));
                if (s >= 0) { ap = 0; as = s; }
            }
        } else if (which == ORLG_HEUR_SAP_FF || which == ORLG_HEUR_SAP_LF) {
            int best_hops = 0x7fffffff;
            for (int q = 0; q < npaths; q++) {
                const int hops = p.path_link_ptr[first + q + 1] - p.path_link_ptr[first + q];
                if (hops < best_hops) {
                    WBits<NWV> A = wide_path_free<NWV>(p, env, first + q, 0);
                    int s;
                    if (which == ORLG_HEUR_SAP_FF) s = wb_ffs(A);
                    else { A.w[0] &= ~1u; s = wb_fls(A); }
                    if (s >= 0) { best_hops = hops; ap = q; as = s; }
                }
            }
        } else {
            int best = -1;
            for (int q = 0; q < npaths; q++) {
                const WBits<NWV> A = wide_path_free<NWV>(p, env, first + q, 0);
                const int cap = wb_popc(A);
                if (cap > best) {
                    const int s = wb_ffs(A);
                    if (s >= 0) { best = cap; ap = q; as = s; }
                }
            }
        }
        a[0] = ap; a[1] = as;
        return ap < p.k;
    } else {
        int a0 = p.k, a1 = p.M, a2 = p.C, a3 = p.S;
        bool found = false;
        for (int q = 0; q < npaths && !found; q++) {
            const int mod = meta_mod(p.path_meta[first + q]);
            const int n = wide_nslots(p, p.mod_se[mod], br);
            const WBits<NWV> lim = wb_range<NWV>(0, max(p.S - n, 0));
            for (int c = 0; c < p.C && !found; c++) {
                WBits<NWV> B = wb_runs_ge(wide_path_free<NWV>(p, env, first + q, c), n);
#pragma unroll
                for (int i = 0; i < 4 * NWV; i++) B.w[i] &= lim.w[i];
                const int s = wb_ffs(B);
                if (s >= 0) { a0 = q; a1 = mod; a2 = c; a3 = s; found = true; }
            }
        }
        a[0] = a0; a[1] = a1; a[2] = a2; a[3] = a3;
        return found;
    }
}

template <int KIND, int NWV>
__global__ void heuristic_wide_kernel(const Params p, const int which, int *actions) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    const uint2 rq = p.cur_req[env];
    constexpr int AD = KIND == ORLG_DEEPRMSA ? 1 : (KIND == ORLG_RMCSA ? 4 : 2);
    int a[4];
    wide_heuristic<KIND, NWV>(p, env, which, rq.x & 0xff, (rq.x >> 8) & 0xff, (int)(rq.x >> 16), a);
#pragma unroll
    for (int i = 0; i < AD; i++) actions[AD * env + i] = a[i];
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
        const WBits<NWV> full = wb_range<NWV>(0, p.S);
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
                    else if (start + n <= p.S) accepted = wb_contains(wide_path_free<NWV>(p, env, row, 0), wb_range<NWV>(start, start + n));
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
                        accepted = (known_free || wb_contains(wide_path_free<NWV>(p, env, row, core), wb_range<NWV>(start, start + n))) &&
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
            cnt[1] += 1; cnt[3] += 1;
            if (KIND != ORLG_RWA) { cnt[5] += br; cnt[7] += br; }
            if (KIND == ORLG_RMSA) br_hist_bump(p, env, 1, br);
        }
        if (KIND == ORLG_RWA || KIND == ORLG_RMCSA) {
            cnt[0] += 1; cnt[2] += 1;
            if (KIND == ORLG_RMCSA) { cnt[4] += br; cnt[6] += br; }
        }
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
        for (int l = 0; l < p.E; l++) {
            const size_t i = (size_t)l * p.n + env;
            p.link_util[i] = 0.0; p.link_comp[i] = 0.0; p.link_last[i] = 0.0; p.link_frag[i] = 0.0;
        }
        p.sum_nh[env] = 0; p.run_br[env] = 0;
        for (int q = 0; q < 3; q++) p.graph_stats[(size_t)q * p.n + env] = 0.0;
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
        } else if ((long long)ridx < p.trace_len) {
            const orlg_request r = p.trace[(size_t)env * p.trace_len + ridx];
            arrival = r.arrival; holding = r.holding; nsrc = r.src; ndst = r.dst;
            nbr = min(max(r.bit_rate, 0), p.br_max);
        } else {
            err |= ORLG_ERR_TRACE_EXHAUSTED;
            arrival = now; holding = 0.0; nsrc = 0; ndst = 1; nbr = p.br_lo;
        }
        ridx++;
        now = arrival; hold = holding; src = nsrc; dst = ndst; br = nbr;
        sid = (int)cnt[2];
        if (KIND == ORLG_RMSA || KIND == ORLG_DEEPRMSA) { cnt[0] += 1; cnt[2] += 1; cnt[4] += br; cnt[6] += br; }
        if (KIND == ORLG_RMSA) br_hist_bump(p, env, 0, br);
        else if (KIND == ORLG_RMCSA) { cnt[4] += br; cnt[6] += br; }
        if constexpr (STATS) {
            // the reference releases in heap order (by time) and every release updates the statistics of its links: the due
            // services are collected, sorted by release time and applied in that order (as in step_kernel)
            constexpr int MAXR = 24;
            double rt[MAXR];
            unsigned long long rp[MAXR];
            int nr = 0;
            long long rel_br = 0;                                // bit rates leaving graph["running_services"]
            long long snh = p.sum_nh[env];
            events_release(ev, nheap, hmin, tailmin, now, apply_timed([&](unsigned long long pl, double t, unsigned sbr) {
                rel_br += sbr;
                if (nr < MAXR) { rt[nr] = t; rp[nr] = pl; nr++; }
                else {                                           // overflow: masks stay exact, statistics order is not
                    err |= ORLG_ERR_STATS_ORDER;
                    wide_path_update_stats<KIND, NWV>(p, env, svc_row(pl), svc_core(pl), svc_start(pl), svc_slots(pl), true, now);
                    snh -= (long long)svc_slots(pl) * wide_hops(p, svc_row(pl));
                }
            }));
            if (rel_br) p.run_br[env] -= rel_br;
            for (int a = 1; a < nr; a++) {                       // insertion sort by release time
                const double t = rt[a];
                const unsigned long long q = rp[a];
                int b = a - 1;
                while (b >= 0 && rt[b] > t) { rt[b + 1] = rt[b]; rp[b + 1] = rp[b]; b--; }
                rt[b + 1] = t; rp[b + 1] = q;
            }
            for (int a = 0; a < nr; a++) {
                const unsigned long long pl = rp[a];
                wide_path_update_stats<KIND, NWV>(p, env, svc_row(pl), svc_core(pl), svc_start(pl), svc_slots(pl), true, now);
                snh -= (long long)svc_slots(pl) * wide_hops(p, svc_row(pl));
            }
            p.sum_nh[env] = snh;
        } else
        events_release(ev, nheap, hmin, tailmin, now, apply_payload([&](unsigned long long pl) {
            wide_path_update<NWV>(p, env, svc_row(pl), svc_core(pl), svc_start(pl), svc_slots(pl), true);
        }));
        done = (cnt[2] == (long long)p.episode_length);
    }

    if (mode == MODE_EPISODE_RESET || (mode == MODE_STEP && done && p.auto_reset)) {
        cnt[2] = 0; cnt[3] = 0; cnt[6] = 0; cnt[7] = 0;
        if (KIND != ORLG_RWA) { cnt[2] = 1; cnt[6] = br; }
    }

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
            const WBits<NWV> B = wb_runs_ge(A, n);
            const WBits<NWV> Bl = wb_shl1(B), Al = wb_shl1(A);
            WBits<NWV> starts, arun;
#pragma unroll
            for (int i = 0; i < 4 * NWV; i++) { starts.w[i] = B.w[i] & ~Bl.w[i]; arun.w[i] = A.w[i] & ~Al.w[i]; }
            const int total = wb_popc(A), runs = wb_popc(arun);
            const int ob = head + q * W;
            for (int b = 0; b < p.J; b++) {
                const int st = wb_ffs(starts);
                p.cand16[(size_t)env * p.cand_stride + q * p.J + b] = (unsigned short)(st < 0 ? 0xFFFF : st);
                int len = -1;
                if (st >= 0) {
                    starts = wb_clear_lowest(starts);
                    len = wb_run_length(A, st);
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
