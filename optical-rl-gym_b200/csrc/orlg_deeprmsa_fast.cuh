// orlg_deeprmsa_fast.cuh -- latency-oriented DeepRMSA step kernel (the headline path).
//
// Same semantics as step_kernel<ORLG_DEEPRMSA> (orlg_kernels.cuh), reorganised so that one thread's
// step is ONE round trip to HBM plus the release-heap chain, with few registers:
//   * the E link masks of the env (E x 16 B, contiguous across the warp) are brought into shared
//     memory with cp.async (no registers, L1 bypass) at kernel entry, overlapping the scalar loads,
//     the traffic draw and the heap work; allocation, releases and the candidate-path AND-reduction
//     then index them dynamically in shared memory ([link][thread] layout: conflict-free LDS.128);
//     only dirty links are written back;
//   * the read-only topology tables (pair -> paths, path -> link bitmap / spectral efficiency,
//     slots-per-bit-rate, node CDF, f32 normalisation tables) are staged once per CTA in shared memory;
//   * the observation tile of the CTA overlays the mask area once the masks are dead and is written
//     to HBM with full-line stores.
#pragma once
#include <cuda.h>          // CUtensorMap (type only: the encoder is fetched with cudaGetDriverEntryPoint)
#include "orlg_kernels.cuh"

namespace orlg {

#ifndef ORLG_FAST_THREADS
#define ORLG_FAST_THREADS 128
#endif
#ifndef ORLG_FAST_MIN_BLOCKS
#define ORLG_FAST_MIN_BLOCKS 4
#endif
constexpr int FAST_THREADS = ORLG_FAST_THREADS;
constexpr int FAST_MIN_BLOCKS = ORLG_FAST_MIN_BLOCKS;     // threads/SM x 148 SMs >= 65536 envs in one wave

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Optional per-phase cycle accounting (build with -DORLG_PHASE_TIMING; read with orlg_debug_phase_cycles):
// sum over warps of the cycles between consecutive marks.  Not part of the product build.
#ifdef ORLG_PHASE_TIMING
#define PHASE_MARK(k)                                                        \
    do {                                                                     \
        long long t_now_ = clock64();                                        \
        if ((threadIdx.x & 31) == 0) atomicAdd(&g_phase_cycles[k], (unsigned long long)(t_now_ - t_prev_)); \
        t_prev_ = t_now_;                                                    \
    } while (0)
#define PHASE_INIT() long long t_prev_ = clock64(); unsigned long long gt0_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt0_))
__device__ unsigned long long g_warp_timeline[2 * 65536];      // per warp: globaltimer at entry / exit (ns), last launch
#define PHASE_END()                                                                          \
    do {                                                                                     \
        unsigned long long gt1_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1_));    \
        const unsigned w_ = (blockIdx.x * FAST_THREADS + threadIdx.x) >> 5;                   \
        if ((threadIdx.x & 31) == 0 && w_ < 65536) { g_warp_timeline[2 * w_] = gt0_; g_warp_timeline[2 * w_ + 1] = gt1_; } \
    } while (0)
#else
#define PHASE_END() do { } while (0)
#define PHASE_MARK(k) do { } while (0)
#define PHASE_INIT() do { } while (0)
#endif

// HOT = the instance for the steady-state rollout step (chosen by the host when it holds): mode == MODE_STEP, Philox
// traffic with continuous bit rates < 128 Gb/s, every request fits the 4-round shift-AND (n <= 16), k == KM, j == 1,
// float32 observation + reward + done requested, no decision / integer-observation outputs.  Same code with those
// conditions as compile-time constants: the reset / trace / generic-feature paths disappear from the instruction stream.
// ---- TMA: the warp's [E links] x [32 envs x 16 B] tile of the mask tensor arrives with ONE cp.async.bulk.tensor.2d,
// completion on a per-warp mbarrier (HOT instance; the general instance keeps per-thread cp.async)
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    unsigned ok = 0, spins = 0;
    while (!ok) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
        if (!ok && ++spins > (1u << 22)) asm volatile("trap;");      // a copy that never lands must fail loudly, not hang
    }
}
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const CUtensorMap *tmap, int x, int y, unsigned long long *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(tmap), "r"(x), "r"(y),
                   "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}

template <int ET, int KM, int JT, bool OBS64, bool HOT = false>
__global__ void __launch_bounds__(FAST_THREADS, FAST_MIN_BLOCKS)
deeprmsa_fast_kernel(const Params p, const StepIO io_rt, const int mode_rt, const __grid_constant__ CUtensorMap mask_map) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int mode = HOT ? (int)MODE_STEP : mode_rt;
    const bool philox = HOT ? true : (p.traffic == ORLG_TRAFFIC_PHILOX);
    const bool cand8 = HOT ? true : (p.cand_stride == 8);
    StepIO io = io_rt;
    if (HOT) { io.decision = nullptr; io.obs_int = nullptr; }
    const int tid = threadIdx.x;
    const int env = blockIdx.x * FAST_THREADS + tid;
    const bool live = env < p.n;
    const int e = live ? env : p.n - 1;
    const int J = JT == 1 ? 1 : p.J;
    const int E = p.E;
    // Work area after the tables: one region per warp, [link][lane] uint4 (conflict-free LDS.128).  Once the
    // warp's masks are dead the same region holds the warp's 32 observation rows, so only __syncwarp() is
    // needed between the two uses: no CTA-wide barrier after the table load.
    const int lane = tid & 31, wid = tid >> 5;
    unsigned char *warp_area = smem + p.tab_vec * 16 + (size_t)wid * p.warp_area_bytes;
    uint4 *sm = reinterpret_cast<uint4 *>(warp_area) + lane;                   // this thread's masks: sm[l * 32]
    unsigned long long *mask_bar = reinterpret_cast<unsigned long long *>(smem + p.tab_vec * 16 + (size_t)(FAST_THREADS / 32) * p.warp_area_bytes) + wid;
    if (HOT) pdl_launch_dependents();      // the next kernel in the stream may be scheduled as soon as SMs drain
    unsigned long long *tab_bar = reinterpret_cast<unsigned long long *>(smem + p.tab_vec * 16 + (size_t)(FAST_THREADS / 32) * p.warp_area_bytes) + FAST_THREADS / 32;
    PHASE_INIT();

    // ---------------- stage 0: asynchronous copies (group 0 = tables, group 1 = this env's link masks)
    {
        uint4 *dst = reinterpret_cast<uint4 *>(smem);
        if (HOT) {                   // one bulk copy for the whole table blob, completion on the CTA's mbarrier
            if (tid == 0) {
                mbar_init(tab_bar, 1);
                mbar_expect_tx(tab_bar, (unsigned)p.tab_vec * 16u);
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(p.tab_blob), "r"((unsigned)p.tab_vec * 16u),
                               "r"((unsigned)__cvta_generic_to_shared(tab_bar)) : "memory");
            }
        } else {
            for (int i = tid; i < p.tab_vec; i += FAST_THREADS) cp_async16(dst + i, p.tab_blob + i);
        }
        cp_async_commit();
        if (HOT) {
            if (lane == 0) mbar_init(mask_bar, 1);      // the tile itself is requested after the dependency wait below
        } else if (mode != MODE_FULL_RESET) {
            const uint4 *mr = p.masks + e;
            unsigned sdst = (unsigned)__cvta_generic_to_shared(sm);
            for (int l = 0; l < E; l++) {
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sdst), "l"(mr) : "memory");
                sdst += 32 * 16;
                mr += p.n;
            }
        }
        cp_async_commit();
    }
    const unsigned short *s_pair_first = reinterpret_cast<const unsigned short *>(smem + p.off_pair_first);
    const unsigned char *s_pair_count = smem + p.off_pair_count;
    const unsigned *s_path_lm = reinterpret_cast<const unsigned *>(smem + p.off_path_lm);
    const unsigned char *s_path_se = smem + p.off_path_se;
    const unsigned long long *s_path_ll = reinterpret_cast<const unsigned long long *>(smem + p.off_path_ll);   // packed hop lists
    const unsigned char *s_nslots = smem + p.off_nslots;              // [se][128]
    const unsigned *s_node_thr = reinterpret_cast<const unsigned *>(smem + p.off_node_thr);
    const float *s_pos = reinterpret_cast<const float *>(smem + p.off_pos);     // (2v - S) / S
    const float *s_nsl = reinterpret_cast<const float *>(smem + p.off_nsl);     // (2n - 11) / 7, n < 32
    const float *s_rcp4 = reinterpret_cast<const float *>(smem + p.off_rcp4);   // 1 / (4 r), r <= (S + 1) / 2 free runs
    const unsigned *s_dbl = reinterpret_cast<const unsigned *>(smem + p.off_dbl);   // shift-AND doubling schedule of n <= 16

    // ---------------- stage 1: the scalar block
    // The traffic draw of _next_service needs only (seed, global env id, request index).  All envs of a
    // handle are reset and stepped together, so the request index is a launch parameter and the Philox
    // rounds + the two logarithms run while the loads above are still in flight.
    uint32_t rc_[4] = {0u, 0u, 0u, 0u}, rd_[4] = {0u, 0u, 0u, 0u};
    double e_iat = 0.0, e_hold = 0.0;
    if (philox && (mode == MODE_STEP || mode == MODE_FULL_RESET)) {
        const unsigned long long gid = (unsigned long long)(p.env_id_base + e);
        const unsigned r0 = mode == MODE_FULL_RESET ? 0u : p.lockstep_ridx;
        rc_[0] = r0; rc_[2] = (uint32_t)gid; rc_[3] = 0u;
        rd_[0] = r0; rd_[2] = (uint32_t)gid; rd_[3] = 1u;
        philox4x32_10(rc_, (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
        philox4x32_10(rd_, (uint32_t)p.seed, (uint32_t)(p.seed >> 32));
        e_iat = request_iat(p, rc_);
        e_hold = request_holding(p, rc_);
    }
    // HOT: the rest of the draw (source, destination, bit rate) and the candidate-path tables of the NEXT request
    // also depend on nothing but the tables and the Philox words: done here, ahead of the dependency wait.
    int p_src = 0, p_dst = 1, p_br = 0, p_first = 0, p_npaths = 0;
    unsigned p_pm[KM];
    int p_ns[KM];
#pragma unroll
    for (int q = 0; q < KM; q++) { p_pm[q] = 0u; p_ns[q] = 1; }
    if (HOT) {
        __syncthreads();             // the table barrier initialised by thread 0 is visible ...
        mbar_wait(tab_bar, 0);       // ... and the tables have landed
        request_nodes(p, s_node_thr, rc_, p_src, p_dst);
        p_br = request_bit_rate<false>(p, rd_[0]);
        const int pair = p_src * p.N + p_dst;
        p_first = s_pair_first[pair];
        p_npaths = min((int)s_pair_count[pair], KM);
#pragma unroll
        for (int q = 0; q < KM; q++) {
            const bool have = q < p_npaths;
            const int row = have ? p_first + q : p_first;
            p_ns[q] = s_nslots[s_path_se[row] * 128 + p_br];
            p_pm[q] = have ? s_path_lm[row] : 0u;
        }
    }
    if (HOT) {
        // Everything above is independent of the previous kernels in the stream (tables, Philox, logarithms, the
        // next request): with a programmatic dependent launch it runs while they drain.  State and actions are only
        // touched from here on.
        pdl_wait();
        if (lane == 0) {
            mbar_expect_tx(mask_bar, (unsigned)(E * 32 * 16));
            tma_load_2d(warp_area, &mask_map, (blockIdx.x * FAST_THREADS + wid * 32) * 4, 0, mask_bar);
        }
    }
    double now = p.now[e];
    double hold = p.cur_hold[e];
    uint2 rq = p.cur_req[e];
    long long cnt[8];
#pragma unroll
    for (int q = 0; q < 8; q++) cnt[q] = p.counters[(size_t)q * p.n + e];
    unsigned ridx = p.req_index[e];
    unsigned nheap = p.nheap[e];
    double hmin = p.heap_min[e];
    unsigned err = p.errors[e];
    const int act = (mode == MODE_STEP) ? io.actions[e] : -1;
    unsigned long long candw = 0;
    if (cand8) candw = *reinterpret_cast<const unsigned long long *>(p.cand + (size_t)e * 8);
    const Events ev = {p.ev_time + (size_t)e * p.heap_cap, p.ev_pay + (size_t)e * p.heap_cap, p.ev_gmin + (size_t)e * p.ev_groups};
    double tailmin = p.ev_tail[e];
    if (mode == MODE_STEP && hmin <= now + 4.0 * p.mean_iat) prefetch_l2(ev.gmin);     // a release is likely: warm the directory

    PHASE_MARK(0);               // issue of the async copies + scalar loads
    if (!HOT) {                  // (HOT waited for its tables in the prologue)
        cp_async_wait<1>();      // tables landed (this thread's part) ...
        __syncthreads();         // ... and everybody else's
    }
    PHASE_MARK(1);               // wait for tables (first round trip)

    int src = rq.x & 0xff, dst = (rq.x >> 8) & 0xff, br = (int)(rq.x >> 16), sid = (int)rq.y;
    bool accepted = false, done = false;
    int d_row = -1, d_start = -1, d_n = -1;
    unsigned dirty = 0;
    int npaths = 0;
    int ns[KM];
    Bits A[KM];

    if (mode == MODE_FULL_RESET) {
        now = 0.0; nheap = 0; hmin = ORLG_INF; tailmin = ORLG_INF; ridx = 0; err = 0;
        dirty = E >= 32 ? 0xFFFFFFFFu : ((1u << E) - 1u);
        const uint4 full = bits_to(bits_range(0, p.S));
        for (int l = 0; l < E; l++) sm[l * 32] = full;
#pragma unroll
        for (int q = 0; q < 8; q++) cnt[q] = 0;
    }

    if (live) {
        // ============ Phase A decision (deeprmsa_env.py:48-58): needs no mask, only the cached block starts
        int a_row = 0, a_start = 0, a_n = 0;
        unsigned a_lm = 0;
        if (mode == MODE_STEP) {
            const int pair = src * p.N + dst;
            const int first = s_pair_first[pair];
            const int np_a = s_pair_count[pair];
            if (act >= 0 && act < p.k * J) {
                const int route = JT == 1 ? act : act / J;
                if (route < np_a) {
                    const unsigned st = cand8 ? (unsigned)((candw >> (8 * act)) & 0xffu)
                                                           : (unsigned)p.cand[(size_t)e * p.cand_stride + act];
                    if (st != CAND_NONE) {
                        if (nheap + 1 > (unsigned)p.heap_cap) {
                            err |= ORLG_ERR_HEAP_OVERFLOW;
                        } else {
                            a_row = first + route;
                            const int se = s_path_se[a_row];
                            a_n = (HOT || br < 128) ? s_nslots[se * 128 + br] : p.nslots[se * (p.br_max + 1) + br];
                            a_lm = s_path_lm[a_row];
                            a_start = (int)st;
                            const double rel = __dadd_rn(now, hold);
                            events_push(ev, nheap, hmin, tailmin, rel, pack_service(a_row, a_start, a_n, 0, sid));
                            count_decision<ORLG_DEEPRMSA>(cnt, true, br);
                            accepted = true;
                            d_row = a_row; d_start = a_start; d_n = a_n;
                        }
                    }
                } else {
                    err |= ORLG_ERR_NO_SUCH_PATH;
                }
            }
            if (HOT || io.reward) io.reward[env] = accepted ? 1.0f : -1.0f;
            if (io.decision) {
                int *d = io.decision + (size_t)env * 6;
                d[0] = accepted; d[1] = d_row; d[2] = d_start; d[3] = d_n; d[4] = accepted ? 0 : -1; d[5] = -1;
            }
            if (io.info) {
#pragma unroll
                for (int q = 0; q < 8; q++) io.info[(size_t)env * 8 + q] = cnt[q];
            }
        }

        PHASE_MARK(2);               // phase A: decision + heap push
        // ============ Phase B draw: _next_service (rmsa_env.py:545-580)
        if (mode == MODE_STEP || mode == MODE_FULL_RESET) {
            double arrival, holding;
            int nsrc, ndst, nbr;
            if (HOT) {
                if (ridx != p.lockstep_ridx) err |= ORLG_ERR_LOCKSTEP;
                arrival = __dadd_rn(now, e_iat);
                holding = e_hold;
                nsrc = p_src; ndst = p_dst; nbr = p_br;
            } else if (philox) {
                if (ridx != (mode == MODE_FULL_RESET ? 0u : p.lockstep_ridx)) err |= ORLG_ERR_LOCKSTEP;
                arrival = __dadd_rn(now, e_iat);
                holding = e_hold;
                request_nodes(p, s_node_thr, rc_, nsrc, ndst);
                nbr = request_bit_rate<!HOT>(p, rd_[0]);
            } else {
                const orlg_request r = trace_request(p, e, ridx, now, p.br_max, p.br_lo, false, err);
                arrival = r.arrival; holding = r.holding; nsrc = r.src; ndst = r.dst; nbr = r.bit_rate;
            }
            ridx++;
            now = arrival; hold = holding; src = nsrc; dst = ndst; br = nbr;
            sid = (int)cnt[2];
            count_request<ORLG_DEEPRMSA>(cnt, br);
        }

        PHASE_MARK(3);               // phase B: traffic draw
        if (HOT) mbar_wait(mask_bar, 0);       // the warp's tile has landed (TMA)
        else cp_async_wait<0>();               // this thread's masks are in shared memory
        PHASE_MARK(4);               // wait for masks

        if (accepted) {              // _provision_path: clear [start, start+n) on the path's links
            const Bits rm = HOT ? bits_range_short(a_start, a_n) : bits_range_auto(a_start, a_n);
            unsigned m = a_lm;
            while (m) {
                const int l = __ffs(m) - 1;
                m &= m - 1;
                uint4 v = sm[l * 32];
                v.x &= ~rm.w[0]; v.y &= ~rm.w[1]; v.z &= ~rm.w[2]; v.w &= ~rm.w[3];
                sm[l * 32] = v;
                if (HOT) p.masks[(size_t)l * p.n + env] = v;       // write-through: no dirty-link pass later
            }
            dirty |= a_lm;
        }
        if (mode == MODE_STEP || mode == MODE_FULL_RESET) {
            events_release(ev, nheap, hmin, tailmin, now, apply_payload([&](unsigned long long pl) {     // rmsa_env.py:591-597
                const unsigned lm = s_path_lm[svc_row(pl)];
                const int rs = svc_start(pl);
                const Bits rm = HOT ? bits_range_short(rs, svc_slots(pl)) : bits_range_auto(rs, svc_slots(pl));
                unsigned m = lm;
                while (m) {
                    const int l = __ffs(m) - 1;
                    m &= m - 1;
                    uint4 v = sm[l * 32];
                    v.x |= rm.w[0]; v.y |= rm.w[1]; v.z |= rm.w[2]; v.w |= rm.w[3];
                    sm[l * 32] = v;
                    if (HOT) p.masks[(size_t)l * p.n + env] = v;
                }
                dirty |= lm;
            }));
            done = (cnt[2] == (long long)p.episode_length);
        }
        if (mode == MODE_EPISODE_RESET || (mode == MODE_STEP && done && p.auto_reset)) reset_episode_counters<ORLG_DEEPRMSA>(cnt, br);
        if (mode != MODE_OBSERVE) {      // ---- store the scalar block (final from here on: frees its registers for phase C)
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
            if (mode == MODE_STEP && (HOT || io.done)) io.done[env] = done ? 1 : 0;
        }
        PHASE_MARK(5);               // allocation + release loop (heap pops)

        // ============ Phase C, part 1: free-slot mask of every candidate path of the pending request
        const int pair = src * p.N + dst;
        const int first = s_pair_first[pair];
        npaths = HOT ? p_npaths : min((int)s_pair_count[pair], KM);
        // get_available_slots (rmsa_env.py:638-649): every candidate path walks its packed hop list
        // (5 bits per link, hop count in the top 4 bits); the KM paths advance in lockstep so that the
        // LDS -> AND chains of different paths overlap.
        unsigned long long ll[KM];
        unsigned pm[KM];
        int hops[KM], mh = 0;
#pragma unroll
        for (int q = 0; q < KM; q++) {
            const bool have = q < npaths;
            const int row = have ? first + q : first;
            if (HOT) {
                ns[q] = p_ns[q];
                pm[q] = p_pm[q];
            } else {
                const int se = s_path_se[row];
                ns[q] = s_nslots[se * 128 + min(br, 127)];
                if (br >= 128) ns[q] = p.nslots[se * (p.br_max + 1) + br];
                pm[q] = have ? s_path_lm[row] : 0u;
            }
            ll[q] = s_path_ll[row];
            hops[q] = have ? (int)(ll[q] >> 60) : 0;
            mh = max(mh, hops[q]);
            A[q] = have ? bits_ones() : Bits{{0u, 0u, 0u, 0u}};
        }
        if (ET > 0) {
            // known link count: one static sweep over the E links, 20 independent accumulator words
            // (more instructions than walking the hop lists, but throughput- instead of latency-bound)
#pragma unroll
            for (int l = 0; l < (ET > 0 ? ET : 1); l++) {
                const uint4 v = sm[l * 32];
#pragma unroll
                for (int q = 0; q < KM; q++) {
                    // predicated AND (LOP3 with a predicate output + 4 predicated LOP3): 5 instructions per (link, path)
                    if (pm[q] & (1u << l)) { A[q].w[0] &= v.x; A[q].w[1] &= v.y; A[q].w[2] &= v.z; A[q].w[3] &= v.w; }
                }
            }
        } else {
            for (int h = 0; h < mh; h++) {
#pragma unroll
                for (int q = 0; q < KM; q++) {
                    if (h < hops[q]) {
                        const int l = (int)(ll[q] & 31u);
                        const uint4 v = sm[l * 32];
                        A[q].w[0] &= v.x; A[q].w[1] &= v.y; A[q].w[2] &= v.z; A[q].w[3] &= v.w;
                    }
                    ll[q] >>= 5;
                }
            }
        }
        PHASE_MARK(6);               // candidate-path AND
        if (!HOT) {   // write back the links this step touched
            uint4 *mw = p.masks + env;
            unsigned m = dirty;
            while (m) {
                const int l = __ffs(m) - 1;
                m &= m - 1;
                mw[(size_t)l * p.n] = sm[l * 32];
            }
        }
    }

    PHASE_MARK(7);          // dirty write-back
    __syncwarp();           // every lane is done with its masks: the warp's area becomes its observation tile
    unsigned char *stage = warp_area;
    PHASE_MARK(8);          // barrier (mask area -> observation tile)

    if (live) {
        // ============ Phase C, part 2: block features (deeprmsa_env.py:60-121)
        const int W = 2 * J + 3;
        const bool want_obs = HOT ? true : (io.obs != nullptr);
        float *so32 = reinterpret_cast<float *>(stage) + (size_t)lane * p.obs_dim;
        double *so64 = reinterpret_cast<double *>(stage) + (size_t)lane * p.obs_dim;
        if (want_obs) {
            const int lo = min(src, dst), hi = max(src, dst);
            if (OBS64) {
                for (int q = 0; q < p.obs_dim; q++) so64[q] = (q > 2 * p.N) ? -1.0 : 0.0;
                so64[0] = __ddiv_rn((double)br, 100.0);
                so64[1 + lo] = 1.0; so64[1 + p.N + hi] = 1.0;
            } else {
                // rows are 8-byte aligned (obs_dim even) or handled element-wise
                const int head = 1 + 2 * p.N;
                if (HOT || (JT == 1 && io.obs_int == nullptr && p.k == KM && (p.obs_dim & 1) == 0)) {
                    // every feature entry is written below: only the head (bit rate + one-hots) needs zeros
                    float2 *r2 = reinterpret_cast<float2 *>(so32);
                    for (int q = 0; q < (head + 1) / 2; q++) r2[q] = make_float2(0.0f, 0.0f);
                } else if ((p.obs_dim & 1) == 0) {
                    float2 *r2 = reinterpret_cast<float2 *>(so32);
                    for (int q = 0; q < p.obs_dim / 2; q++) r2[q] = (2 * q >= head) ? make_float2(-1.0f, -1.0f) : make_float2(0.0f, (2 * q + 1 >= head) ? -1.0f : 0.0f);
                } else {
                    for (int q = 0; q < p.obs_dim; q++) so32[q] = (q >= head) ? -1.0f : 0.0f;
                }
                so32[0] = __fdiv_rn((float)br, 100.0f);
                so32[1 + lo] = 1.0f; so32[1 + p.N + hi] = 1.0f;
            }
        }
        unsigned long long cand_out = 0xFFFFFFFFFFFFFFFFULL;
        int n_max = 0;
#pragma unroll
        for (int q = 0; q < KM; q++) n_max = max(n_max, ns[q]);
        const bool flat = HOT ? true : (JT == 1 && !OBS64 && io.obs_int == nullptr && p.k == KM && n_max <= 16);
        if (flat) {
            // j = 1, float32: straight-line code, the KM paths are independent instruction streams.
            // With B = positions where a free run of >= n slots starts-or-continues (shift-AND doubling):
            //   first block start = lowest set bit of B; its B-run ends at the lowest set bit of B & ~(B >> 1),
            //   so the full free run has length (that end) - start + n            (get_available_blocks, rmsa_env.py:667-697)
#pragma unroll
            for (int q = 0; q < KM; q++) {
                const int n = ns[q];
                const Bits B = bits_runs_ge_sched(A[q], s_dbl[n]);
                const int st = bits_ffs_flat(B);
                const int fe = bits_ffs_flat(bits_andnot(B, bits_shr_small(B, 1)));
                const int len = fe - st + n;
                const int total = bits_popc(A[q]);
                const int runs = bits_popc(bits_andnot(A[q], bits_shl1(A[q])));
                const bool have = q < npaths;
                const bool blk = st >= 0;
                cand_out = blk ? ((cand_out & ~(0xFFULL << (8 * q))) | ((unsigned long long)st << (8 * q))) : cand_out;
                if (want_obs) {
                    const int ob = 1 + 2 * p.N + q * 5;
                    so32[ob] = blk ? s_pos[max(st, 0)] : -1.0f;
                    so32[ob + 1] = blk ? (float)(len - 8) * 0.125f : -1.0f;
                    so32[ob + 2] = have ? s_nsl[n] : -1.0f;                 // n <= 16 here
                    so32[ob + 3] = have ? s_pos[total] : -1.0f;
                    so32[ob + 4] = runs > 0 ? (float)(total - 4 * runs) * s_rcp4[runs] : -1.0f;   // x * fl(1/y): <= 1.5 ulp
                }
            }
        } else {
#pragma unroll
        for (int q = 0; q < KM; q++) {
            if (q < npaths) {
                const int n = ns[q];
                const Bits B = n <= 16 ? bits_runs_ge_flat(A[q], n) : bits_runs_ge(A[q], n);
                Bits starts = bits_andnot(B, bits_shl1(B));
                const int total = bits_popc(A[q]);
                const int runs = bits_popc(bits_andnot(A[q], bits_shl1(A[q])));
                const int ob = 1 + 2 * p.N + q * W;
                if (JT == 1) {
                    const int st = bits_ffs(starts);
                    const int len = bits_run_length(A[q], max(st, 0));
                    if (st >= 0) cand_out = (cand_out & ~(0xFFULL << (8 * q))) | ((unsigned long long)st << (8 * q));
                    if (want_obs && st >= 0) {
                        if (OBS64) {
                            so64[ob] = __ddiv_rn(__dmul_rn(2.0, __dadd_rn((double)st, -__dmul_rn(0.5, (double)p.S))), (double)p.S);
                            so64[ob + 1] = __ddiv_rn(__dadd_rn((double)len, -8.0), 8.0);
                        } else {
                            so32[ob] = s_pos[st];
                            so32[ob + 1] = (float)(len - 8) * 0.125f;
                        }
                    }
                    if (io.obs_int) {
                        int *oi = io.obs_int + ((size_t)env * p.k + q) * W;
                        oi[0] = st; oi[1] = st >= 0 ? len : -1;
                    }
                } else {
                    for (int b = 0; b < J; b++) {
                        const int st = bits_ffs(starts);
                        if (p.cand_stride == 8) {
                            if (st >= 0) cand_out = (cand_out & ~(0xFFULL << (8 * (q * J + b)))) | ((unsigned long long)st << (8 * (q * J + b)));
                        } else {
                            p.cand[(size_t)env * p.cand_stride + q * J + b] = (unsigned char)(st < 0 ? CAND_NONE : st);
                        }
                        int len = -1;
                        if (st >= 0) {
                            starts = bits_clear_lowest(starts);
                            len = bits_run_length(A[q], st);
                            if (want_obs) {
                                if (OBS64) {
                                    so64[ob + 2 * b] = __ddiv_rn(__dmul_rn(2.0, __dadd_rn((double)st, -__dmul_rn(0.5, (double)p.S))), (double)p.S);
                                    so64[ob + 2 * b + 1] = __ddiv_rn(__dadd_rn((double)len, -8.0), 8.0);
                                } else {
                                    so32[ob + 2 * b] = s_pos[st];
                                    so32[ob + 2 * b + 1] = (float)(len - 8) * 0.125f;
                                }
                            }
                        }
                        if (io.obs_int) {
                            int *oi = io.obs_int + ((size_t)env * p.k + q) * W;
                            oi[2 * b] = st; oi[2 * b + 1] = len;
                        }
                    }
                }
                if (want_obs) {
                    if (OBS64) {
                        so64[ob + 2 * J] = __ddiv_rn(__dadd_rn((double)n, -5.5), 3.5);
                        so64[ob + 2 * J + 1] = __ddiv_rn(__dmul_rn(2.0, __dadd_rn((double)total, -__dmul_rn(0.5, (double)p.S))), (double)p.S);
                        if (runs > 0) so64[ob + 2 * J + 2] = __ddiv_rn(__dadd_rn(__ddiv_rn((double)total, (double)runs), -4.0), 4.0);
                    } else {
                        so32[ob + 2 * J] = n < 32 ? s_nsl[n] : __fdiv_rn((float)(2 * n - 11), 7.0f);
                        so32[ob + 2 * J + 1] = s_pos[total];
                        if (runs > 0) so32[ob + 2 * J + 2] = __fdividef((float)(total - 4 * runs), (float)(4 * runs));   // <= 2 ulp
                    }
                }
                if (io.obs_int) {
                    int *oi = io.obs_int + ((size_t)env * p.k + q) * W;
                    oi[2 * J] = n; oi[2 * J + 1] = total; oi[2 * J + 2] = runs;
                }
            }
        }
        }
        if (cand8) {
            *reinterpret_cast<unsigned long long *>(p.cand + (size_t)env * 8) = cand_out;
        } else {
            for (int q = npaths * J; q < p.k * J; q++) p.cand[(size_t)env * p.cand_stride + q] = (unsigned char)CAND_NONE;
        }
        if (io.obs_int)
            for (int q = npaths * W; q < p.k * W; q++) io.obs_int[(size_t)env * p.k * W + q] = -1;

        PHASE_MARK(9);                   // block features + observation row
    }

    PHASE_MARK(10);         // scalar stores
    if (HOT || io.obs != nullptr) {
        // The warp's 32 rows are one contiguous run of the [N, obs_dim] tensor: a single bulk (TMA) store from shared
        // memory, issued by one lane (generic-proxy writes -> fence.proxy.async by every writer -> warp sync -> store).
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        PHASE_MARK(11);     // (warp-level sync before the tile copy)
        const int row0 = blockIdx.x * FAST_THREADS + wid * 32;          // first env of this warp
        const int rows = min(32, p.n - row0);
        if (rows > 0) {
            const size_t esz = OBS64 ? 8 : 4;
            unsigned char *g = reinterpret_cast<unsigned char *>(io.obs) + (size_t)row0 * p.obs_dim * esz;
            const unsigned bytes = (unsigned)(rows * p.obs_dim * esz);
            if ((reinterpret_cast<size_t>(g) & 15) == 0 && (bytes & 15u) == 0) {
                if (lane == 0) {
                    const unsigned ssrc = (unsigned)__cvta_generic_to_shared(stage);
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(g), "r"(ssrc), "r"(bytes) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");      // shared memory must outlive the read
                }
            } else {                 // ragged tail or unaligned view: element loop
                const int total_el = rows * p.obs_dim;
                if (OBS64) {
                    const double *sv = reinterpret_cast<const double *>(stage);
                    double *gv = reinterpret_cast<double *>(g);
                    for (int q = lane; q < total_el; q += 32) gv[q] = sv[q];
                } else {
                    const float *sv = reinterpret_cast<const float *>(stage);
                    float *gv = reinterpret_cast<float *>(g);
                    for (int q = lane; q < total_el; q += 32) gv[q] = sv[q];
                }
            }
        }
    }
    PHASE_MARK(12);         // observation tile copy-out
    PHASE_END();
}

}  // namespace orlg
