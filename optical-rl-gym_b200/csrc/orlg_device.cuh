// orlg_device.cuh -- device-side building blocks of the batched step path (sm_100a).
//
// Spectrum state is bit-packed: one 128-bit word group per (core, link, env); bit s = slot s
// free (the reference's available_slots[link, s] == 1, rmsa_env.py:337-339); bits >= S are 0.
// Every RLE / np.any / np.sum of the reference collapses to popc / ffs / funnel shifts here
// (identities verified against the reference in SURVEY.md section 7 step 6).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace orlg {

constexpr int NW = 4;              // 32-bit words per (core, link): S <= 128
constexpr int MAX_SLOTS = 32 * NW;
constexpr uint32_t CAND_NONE = 0xFFu;

// ---------------------------------------------------------------- slot masks of V x 128 bits
// V = 1 (Bits) for the NSFNET-class kernels; the wide kernels take V = 1..4 word groups (S <= 512).  Each operation deduces V
// from its argument; bits_ones and bits_range take no mask and default to V = 1.
template <int V>
struct WBits {
    uint32_t w[4 * V];
};
using Bits = WBits<1>;

__device__ __forceinline__ Bits bits_from(uint4 v) {
    Bits b;
    b.w[0] = v.x; b.w[1] = v.y; b.w[2] = v.z; b.w[3] = v.w;
    return b;
}
__device__ __forceinline__ uint4 bits_to(const Bits &b) { return make_uint4(b.w[0], b.w[1], b.w[2], b.w[3]); }
template <int V = 1>
__device__ __forceinline__ WBits<V> bits_ones() {
    WBits<V> b;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) b.w[i] = 0xFFFFFFFFu;
    return b;
}
template <int V>
__device__ __forceinline__ WBits<V> bits_and(const WBits<V> &a, const WBits<V> &b) {
    WBits<V> r;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) r.w[i] = a.w[i] & b.w[i];
    return r;
}
template <int V>
__device__ __forceinline__ WBits<V> bits_or(const WBits<V> &a, const WBits<V> &b) {
    WBits<V> r;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) r.w[i] = a.w[i] | b.w[i];
    return r;
}
template <int V>
__device__ __forceinline__ WBits<V> bits_andnot(const WBits<V> &a, const WBits<V> &b) {   // a & ~b
    WBits<V> r;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) r.w[i] = a.w[i] & ~b.w[i];
    return r;
}
template <int V>
__device__ __forceinline__ bool bits_contains(const WBits<V> &a, const WBits<V> &m) {   // (a & m) == m
    uint32_t miss = 0;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) miss |= (~a.w[i]) & m.w[i];
    return miss == 0;
}
// logical shift right by 0 <= s < 32
template <int V>
__device__ __forceinline__ WBits<V> bits_shr_small(const WBits<V> &a, int s) {
    WBits<V> r;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) r.w[i] = __funnelshift_r(a.w[i], i + 1 < 4 * V ? a.w[i + 1] : 0u, s);
    return r;
}
template <int V>
__device__ __forceinline__ WBits<V> bits_shl1(const WBits<V> &a) {
    WBits<V> r;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) r.w[i] = __funnelshift_l(i > 0 ? a.w[i - 1] : 0u, a.w[i], 1);
    return r;
}
template <int V>
__device__ __forceinline__ int bits_popc(const WBits<V> &a) {
    int c = 0;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) c += __popc(a.w[i]);
    return c;
}
// index of the lowest set bit, or -1
template <int V>
__device__ __forceinline__ int bits_ffs(const WBits<V> &a) {
    int r = -1;
#pragma unroll
    for (int i = 4 * V - 1; i >= 0; i--)
        if (a.w[i]) r = 32 * i + __ffs(a.w[i]) - 1;
    return r;
}
// index of the highest set bit, or -1: the highest non-zero word by selects, then one clz (an empty mask leaves x = 0,
// base = 0, and 31 - clz(0) = -1)
template <int V>
__device__ __forceinline__ int bits_fls(const WBits<V> &a) {
    uint32_t x = 0;
    int base = 0;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) {
        const bool nz = a.w[i] != 0u;
        x = nz ? a.w[i] : x;
        base = nz ? 32 * i : base;
    }
    return base + 31 - __clz(x);
}
template <int V>
__device__ __forceinline__ WBits<V> bits_clear_lowest(const WBits<V> &a) {
    WBits<V> r = a;
    bool done = false;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) {
        if (!done && r.w[i]) { r.w[i] &= r.w[i] - 1; done = true; }
    }
    return r;
}
// bits [lo, hi) set, 0 <= lo <= hi <= 128 * V
template <int V = 1>
__device__ __forceinline__ WBits<V> bits_range(int lo, int hi) {
    WBits<V> r;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) {
        int a = min(max(lo - 32 * i, 0), 32), b = min(max(hi - 32 * i, 0), 32);
        uint32_t ma = a >= 32 ? 0u : (0xFFFFFFFFu << a);     // bits >= a
        uint32_t mb = b >= 32 ? 0xFFFFFFFFu : ~(0xFFFFFFFFu << b);   // bits < b
        r.w[i] = ma & mb;
    }
    return r;
}
// B[i] = 1 iff A[i .. i+n-1] are all 1 (n >= 1): shift-AND doubling, shifts kept below 32
template <int V>
__device__ __forceinline__ WBits<V> bits_runs_ge(const WBits<V> &a, int n) {
    WBits<V> b = a;
    int len = 1;
    while (len < n) {
        const int s = min(min(len, n - len), 31);
        const WBits<V> sh = bits_shr_small(b, s);
#pragma unroll
        for (int i = 0; i < 4 * V; i++) b.w[i] &= sh.w[i];
        len += s;
    }
    return b;
}
// length of the run of ones starting at bit `start` (A[start] must be 1; bit 128 * V counts as 0)
template <int V>
__device__ __forceinline__ int bits_run_length(const WBits<V> &a, int start) {
    const WBits<V> from = bits_range<V>(start, 128 * V);
    WBits<V> z;
#pragma unroll
    for (int i = 0; i < 4 * V; i++) z.w[i] = ~a.w[i] & from.w[i];
    const int pos = bits_ffs(z);
    return (pos < 0 ? 128 * V : pos) - start;
}
// the longest run of ones: one pass over the words, ctz / clz at every run boundary (no shift-AND pass per slot)
template <int V>
__device__ __forceinline__ int bits_longest_run(const WBits<V> &a) {
    int best = 0, cur = 0;                             // cur: the run that reaches the top of the words seen so far
#pragma unroll
    for (int i = 0; i < 4 * V; i++) {
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

// 128-bit variants of the fast DeepRMSA and rollout kernels, each compiling to different code on purpose:
// bits_runs_ge with the four shift amounts of n packed one per byte (table built by the host: orlg_api.cu): no loop control
__device__ __forceinline__ Bits bits_runs_ge_sched(const Bits &a, unsigned sched) {
    Bits b = a;
#pragma unroll
    for (int it = 0; it < 4; it++) {
        b = bits_and(b, bits_shr_small(b, (int)((sched >> (8 * it)) & 0xffu)));
    }
    return b;
}
// bits_runs_ge without any branch; valid for 1 <= n <= 16 (the caller takes bits_runs_ge otherwise)
__device__ __forceinline__ Bits bits_runs_ge_flat(const Bits &a, int n) {
    Bits b = a;
    int len = 1;
#pragma unroll
    for (int it = 0; it < 4; it++) {
        int s = max(min(len, n - len), 0);
        Bits sh = bits_shr_small(b, s);       // s == 0: funnel shift by 0 returns b
        b = bits_and(b, sh);
        len += s;
    }
    return b;
}
// bits [start, start + n) for 1 <= n <= 32, 0 <= start, start + n <= 128: one 64-bit shift placed at word start / 32
__device__ __forceinline__ Bits bits_range_short(int start, int n) {
    const unsigned long long m = ((1ULL << n) - 1ULL) << (start & 31);
    const unsigned lo = (unsigned)m, hi = (unsigned)(m >> 32);
    const int ws = start >> 5;
    Bits r;
#pragma unroll
    for (int i = 0; i < NW; i++) r.w[i] = (i == ws) ? lo : ((i == ws + 1) ? hi : 0u);
    return r;
}
// bits [start, start + n): bits_range_short where it applies (the common case), else bits_range
__device__ __forceinline__ Bits bits_range_auto(int start, int n) {
    return (n <= 32) ? bits_range_short(start, n) : bits_range(start, start + n);
}
// bits_ffs without branches: the lowest non-zero word by selects, then one ffs (an empty mask leaves x = 0, base = 0,
// and ffs(0) - 1 = -1).  One bit scan instead of four: BREV + FLO sit on the dependent chain of every caller.
__device__ __forceinline__ int bits_ffs_flat(const Bits &a) {
    uint32_t x = 0;
    int base = 0;
#pragma unroll
    for (int i = NW - 1; i >= 0; i--) {
        const bool nz = a.w[i] != 0u;
        x = nz ? a.w[i] : x;
        base = nz ? 32 * i : base;
    }
    return base + __ffs(x) - 1;
}

// ---------------------------------------------------------------- Philox4x32-10 (counter-based traffic)
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

// -ln((r + 0.5) / 2^32) with every rounding fixed (DESIGN.md "Traffic"): IEEE add/mul/div/fma only,
// so the CPU oracle reproduces it bit-for-bit.
__device__ __forceinline__ double neg_log_u32(uint32_t r) {
    double x = __dadd_rn((double)r, 0.5);
    long long bits = __double_as_longlong(x);
    int e = (int)((bits >> 52) & 0x7ff) - 1023;
    double m = __longlong_as_double((bits & 0x000fffffffffffffLL) | 0x3ff0000000000000LL);
    if (m > 1.4142135623730951) { m = __dmul_rn(m, 0.5); e += 1; }
    double s = __ddiv_rn(__dadd_rn(m, -1.0), __dadd_rn(m, 1.0));
    double z = __dmul_rn(s, s);
    double p = 1.0 / 23.0;
    p = __fma_rn(p, z, 1.0 / 21.0);
    p = __fma_rn(p, z, 1.0 / 19.0);
    p = __fma_rn(p, z, 1.0 / 17.0);
    p = __fma_rn(p, z, 1.0 / 15.0);
    p = __fma_rn(p, z, 1.0 / 13.0);
    p = __fma_rn(p, z, 1.0 / 11.0);
    p = __fma_rn(p, z, 1.0 / 9.0);
    p = __fma_rn(p, z, 1.0 / 7.0);
    p = __fma_rn(p, z, 1.0 / 5.0);
    p = __fma_rn(p, z, 1.0 / 3.0);
    p = __fma_rn(p, z, 1.0);
    double lnm = __dmul_rn(__dmul_rn(2.0, s), p);
    double lnx = __fma_rn((double)e, 0.6931471805599453, lnm);
    return __dadd_rn(22.180709777918249, -lnx);
}

// ---------------------------------------------------------------- per-env release-event table (HBM)
// Replaces the reference's heapq of (release_time, service) (optical_network_env.py:143-154,
// rmsa_env.py:591-597).  The reference only ever asks "which services have release_time <= now?",
// and the order in which those are released does not change the masks, so no total order is kept:
//   * the n live services occupy slots [0, n) of two parallel arrays (f64 time, u64 payload), UNSORTED;
//   * a directory holds, per group of EV_GROUP consecutive slots, a float LOWER BOUND of the group's
//     earliest release time (the open tail group's bound lives in the scalar block), and the scalar
//     `tmin` is a lower bound over all groups;
//   * push   = two stores at slot n (no load at all);
//   * a step with tmin > now touches nothing;
//   * otherwise: ONE fetch of the directory, ONE fetch of each group whose bound is due (usually one
//     128-byte line), ONE fetch of the due payloads + the tail entry that fills the hole.  Constant
//     number of dependent round trips per step, however many services expire.
// (A binary/d-ary heap costs 3-4 dependent DRAM round trips PER POP and was measured to dominate both
//  the mean and the tail of the step; a plain scan of all n times is latency-bound too: profiles/.)
#define ORLG_INF __longlong_as_double(0x7ff0000000000000LL)
constexpr int EV_GROUP = 16;

// Optional cycle accounting (instrumented builds only: -DORLG_PHASE_TIMING, tools/phase_timing.py)
#ifdef ORLG_PHASE_TIMING
__device__ unsigned long long g_phase_cycles[16];
#define SUBPHASE_BEGIN() long long sub_t_ = clock64()
#define SUBPHASE_MARK(k)                                                                 \
    do {                                                                                 \
        long long sub_n_ = clock64();                                                    \
        if ((threadIdx.x & 31) == 0) atomicAdd(&g_phase_cycles[k], (unsigned long long)(sub_n_ - sub_t_)); \
        sub_t_ = sub_n_;                                                                 \
    } while (0)
#else
#define SUBPHASE_BEGIN() do { } while (0)
#define SUBPHASE_MARK(k) do { } while (0)
#endif

struct Events {
    double *t;                    // [cap] release times of this env; every slot >= n holds +INF
    unsigned long long *p;        // [cap] packed services
    float *gmin;                  // [cap / EV_GROUP] lower bound of each FULL group's earliest time; +INF from the tail group on
    unsigned short *br;           // [cap] bit rate of each service (statistics mode only: graph "throughput"), else null
};

__device__ __forceinline__ void prefetch_l2(const void *ptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr)); }

__device__ __forceinline__ float lower_f32(double x) { return __double2float_rd(x); }
#define ORLG_INF_F __int_as_float(0x7f800000)
// plain minimum of finite values (fmin()'s NaN handling costs several extra instructions)
__device__ __forceinline__ double dmin(double a, double b) { return a < b ? a : b; }

__device__ __forceinline__ void events_push(const Events &ev, unsigned &n, double &tmin, double &tail_min, double t,
                                            unsigned long long payload, unsigned bit_rate = 0) {
    if ((n & (EV_GROUP - 1)) == 0) {             // opening a new tail group: publish the previous group's bound
        if (n > 0) ev.gmin[(n / EV_GROUP) - 1] = lower_f32(tail_min);
        tail_min = ORLG_INF;
    }
    ev.t[n] = t;
    ev.p[n] = payload;
    if (ev.br) ev.br[n] = (unsigned short)bit_rate;
    n++;
    tail_min = dmin(tail_min, t);
    tmin = dmin(tmin, t);
}

// Releases every service with time <= now; `apply(payload)` frees its slots.  Updates n, tmin, tail_min.
// Invariants: gmin[g] <= every time in full group g (g < tail group) and +INF from the tail group on;
// tail_min <= every time in the tail group; tmin <= every time; t[s] = +INF for s >= n.  Due services can
// therefore only sit in groups whose bound is <= now; those are scanned from the highest group down, so the
// tail entry that fills a hole is never itself due.  All bounds are lower bounds (floats rounded down), which
// is all the gate needs; the comparisons that decide a release use the exact float64 times.
// adapter: a plain lambda taking the payload (release order irrelevant: masks only)
template <typename F>
struct ApplyPayload {
    static constexpr bool wants_time = false;
    F f;
    __device__ __forceinline__ void operator()(unsigned long long pl, double, unsigned) const { f(pl); }
};
template <typename F>
__device__ __forceinline__ ApplyPayload<F> apply_payload(F f) { return ApplyPayload<F>{f}; }
// adapter: payload + exact release time (row f1 needs the reference's release order = by time)
template <typename F>
struct ApplyTimed {
    static constexpr bool wants_time = true;
    F f;
    __device__ __forceinline__ void operator()(unsigned long long pl, double t, unsigned br) const { f(pl, t, br); }
};
template <typename F>
__device__ __forceinline__ ApplyTimed<F> apply_timed(F f) { return ApplyTimed<F>{f}; }

template <typename Apply>
__device__ __forceinline__ void events_release(const Events &ev, unsigned &n, double &tmin, double &tail_min,
                                               const double now, Apply apply) {
    SUBPHASE_BEGIN();
    if (n == 0 || tmin > now) return;
    const unsigned tail0 = (n - 1) / EV_GROUP;     // tail group on entry
    const float now_up = __double2float_ru(now);    // f <= now_up whenever (double)f <= now
    float fb = ORLG_INF_F;                          // lower bound over everything that stays
    unsigned tail_pub = tail0;                      // the group that `tail_min` currently describes
    // The directory is walked in blocks of 64 groups, HIGHEST block first and highest group first inside a block, so that
    // the tail entry that fills a hole is never itself due (any number of groups: the capacity is not tied to a 64-bit mask).
    for (int blk = (int)(tail0 / 64); blk >= 0; blk--) {
        const unsigned g0 = (unsigned)blk * 64;
        // ---- directory: which full groups of this block may hold a due service?  (entries >= tail0 are +INF)
        unsigned long long due_groups = 0;
        const unsigned gend = min(g0 + 64u, tail0);
        for (unsigned c = g0; c < gend; c += 16) {
            float4 d[4];
#pragma unroll
            for (int q = 0; q < 4; q++) d[q] = reinterpret_cast<const float4 *>(ev.gmin + c)[q];
            unsigned m16 = 0;
#pragma unroll
            for (int q = 0; q < 16; q++) {
                const float4 v = d[q >> 2];
                const float f = (q & 3) == 0 ? v.x : ((q & 3) == 1 ? v.y : ((q & 3) == 2 ? v.z : v.w));
                const bool due = f <= now_up;
                m16 |= due ? (1u << q) : 0u;
                fb = fminf(fb, due ? ORLG_INF_F : f);
            }
            due_groups |= (unsigned long long)m16 << (c - g0);
        }
        if (tail0 >= g0 && tail0 < g0 + 64u) {      // the open tail group lives in this block
            if (tail_min <= now) due_groups |= 1ULL << (tail0 - g0); else fb = fminf(fb, lower_f32(tail_min));
        }
        SUBPHASE_MARK(13);                         // directory
        {   // start every fetch the scans below will need (times + payloads of the due groups, the tail entry)
            unsigned long long m = due_groups;
            while (m) {
                const unsigned g = g0 + 63 - __clzll(m);
                m &= ~(1ULL << (g - g0));
                prefetch_l2(ev.t + g * EV_GROUP);
                prefetch_l2(ev.p + g * EV_GROUP);
            }
            if (due_groups && n > 0) {
                prefetch_l2(ev.t + (n - 1));
                prefetch_l2(ev.p + (n - 1));
            }
        }
        while (due_groups) {
            const unsigned g = g0 + 63 - __clzll(due_groups);
            due_groups &= ~(1ULL << (g - g0));
            const unsigned s0 = g * EV_GROUP;
            if (s0 >= n) continue;                 // the group vanished while the tail shrank
            unsigned duebits = 0;
            float gm = ORLG_INF_F;                 // lower bound of what stays in this group
#pragma unroll
            for (int q = 0; q < EV_GROUP / 2; q++) {
                const double2 v = reinterpret_cast<const double2 *>(ev.t + s0)[q];
                const bool d0 = v.x <= now, d1 = v.y <= now;        // slots >= n hold +INF: never due
                duebits |= (d0 ? (1u << (2 * q)) : 0u) | (d1 ? (2u << (2 * q)) : 0u);
                gm = fminf(gm, d0 ? ORLG_INF_F : lower_f32(v.x));
                gm = fminf(gm, d1 ? ORLG_INF_F : lower_f32(v.y));
            }
            SUBPHASE_MARK(14);                     // group fetch + classify
            while (duebits) {                      // highest slot first
                const unsigned q = 31 - __clz(duebits);
                duebits &= ~(1u << q);
                const unsigned s = s0 + q;
                const unsigned last = n - 1;
                const unsigned long long pl = ev.p[s];
                const double pt = Apply::wants_time ? ev.t[s] : 0.0;
                const unsigned pb = (Apply::wants_time && ev.br) ? ev.br[s] : 0u;
                if (s != last) {                   // fill the hole with the tail entry (never due, see above)
                    const double lt = ev.t[last];
                    const unsigned long long lp = ev.p[last];
                    ev.t[s] = lt;
                    ev.p[s] = lp;
                    if (ev.br) ev.br[s] = ev.br[last];
                    gm = fminf(gm, lower_f32(lt));
                }
                ev.t[last] = ORLG_INF;             // keep "t[s] = +INF for s >= n"
                n--;
                apply(pl, pt, pb);
            }
            SUBPHASE_MARK(15);                     // payload fetch, hole fill, apply
            if (s0 < n) {                          // publish the bound of what is left of this group
                if (g == (n - 1) / EV_GROUP) { tail_min = (double)gm; tail_pub = g; }
                else ev.gmin[g] = gm;
                fb = fminf(fb, gm);
            }
        }
    }
    if (n == 0) {
        for (unsigned g = 0; g <= tail0; g++) ev.gmin[g] = ORLG_INF_F;
        tmin = ORLG_INF; tail_min = ORLG_INF;
        return;
    }
    const unsigned tail_g = (n - 1) / EV_GROUP;
    if (tail_g != tail_pub) tail_min = (double)ev.gmin[tail_g];    // the tail shrank into an older, published group
    for (unsigned g = tail_g; g < tail0; g++) ev.gmin[g] = ORLG_INF_F;   // directory is +INF from the (new) tail group on
    tmin = (double)fb;
}

// payload: path row (20 bits) | start (9) | slots (8) | core (5) | service id (22)
__device__ __forceinline__ unsigned long long pack_service(int row, int start, int n, int core, int sid) {
    return (unsigned long long)(uint32_t)row | ((unsigned long long)(uint32_t)start << 20) |
           ((unsigned long long)(uint32_t)n << 29) | ((unsigned long long)(uint32_t)core << 37) |
           ((unsigned long long)((uint32_t)sid & 0x3FFFFFu) << 42);
}
__device__ __forceinline__ int svc_row(unsigned long long p) { return (int)(p & 0xFFFFFu); }
__device__ __forceinline__ int svc_start(unsigned long long p) { return (int)((p >> 20) & 0x1FFu); }
__device__ __forceinline__ int svc_slots(unsigned long long p) { return (int)((p >> 29) & 0xFFu); }
__device__ __forceinline__ int svc_core(unsigned long long p) { return (int)((p >> 37) & 0x1Fu); }
__device__ __forceinline__ int svc_id(unsigned long long p) { return (int)((p >> 42) & 0x3FFFFFu); }

}  // namespace orlg
