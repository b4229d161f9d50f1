// orlg_policy.cuh -- an SB3 MlpPolicy (a tanh trunk of L hidden layers of width H, then action_net / value_net), evaluated
// for a whole batch of observations in ONE fused kernel: model.predict(obs, deterministic=True).  The agent the reference
// trains and ships (examples/stable_baselines3/DeepRMSA.ipynb cell 13: PPO(MlpPolicy, env, policy_kwargs=dict(net_arch=5*[128]));
// bkp/deeprmsa-ppo-trained/best_model.zip) is H = 128, L = 5; SB3's default PPO / A2C trunk is H = 64, L = 2.
//
//   obs f32 [n, 54] -> L x (Linear H + tanh) -> action_net (5 logits) / value_net (1) -> argmax -> int32 action
//
// This IS a contraction (146 kFLOP per env at 5 x 128, 9.6 GFLOP per 65536-env step), so it runs on the 5th-generation
// tensor cores: a persistent CTA per SM keeps all L + 1 weight matrices (bf16, 148 KB at 5 x 128) in shared memory in the
// UMMA K-major core-matrix layout, and walks tiles of 128 environments.  Per tile and layer one elected thread issues
// tcgen05.mma (M = 128, N = H, K = 16 per instruction) with A = the tile's activations (bf16, shared memory),
// B = the layer's weights, D = fp32 accumulators in TMEM; the warps then read their 32 TMEM lanes back with
// tcgen05.ld, add the bias, apply tanh and write the next layer's A operand.  Nothing but the observation rows and
// the actions touches HBM.  A second instance (mlp_policy_kernel<true>) ends in a sampling epilogue: the action drawn from
// softmax(logits) with Philox stream 3, its log-probability and the value (PPO's rollout collection, orlg_policy_sample), and
// its MASKED variant draws under an invalid-action mask (orlg_policy_sample_masked).
#pragma once
#include <cuda_bf16.h>
#include "orlg_deeprmsa_fast.cuh"

namespace orlg {

constexpr int PL_TILE = 128;          // environments per tile = UMMA M
constexpr int PL_HMAX = 128;          // widest hidden layer: the TMEM columns and the A buffer of a tile group
constexpr int PL_K0 = 64;             // observation width padded to a multiple of 16 (54 -> 64)
constexpr int PL_NOUT = 16;           // output layer padded: 5 logits + 1 value
constexpr int PL_SMEM_MAX = 232448;   // dynamic shared memory a block may opt in to on sm_100 (227 KB)

struct PolicyParams {
    const uint4 *w_blob;              // all weights, bf16, already in the shared-memory operand layout (orlg_policy_create)
    int w_bytes;                      // H * 64 * 2 + (L - 1) * H * H * 2 + 16 * H * 2
    const float *bias;                // [L * H + 16]
    int obs_dim, n_actions;           // 54, 5
    int H, L;                         // hidden width (multiple of 16, 16..128) and number of hidden layers (>= 1)
};

// bytes of weights and of dynamic shared memory of a policy with hidden width H and L hidden layers
inline size_t pl_weight_bytes(int H, int L) { return (size_t)H * PL_K0 * 2 + (size_t)(L - 1) * H * H * 2 + (size_t)PL_NOUT * H * 2; }
constexpr int PL_GROUPS = 2;          // tile groups per CTA
inline size_t pl_smem_bytes(int H, int L) {
    return pl_weight_bytes(H, L) + (size_t)PL_GROUPS * PL_TILE * PL_HMAX * 2 + ((size_t)L * H + PL_NOUT) * 4 + 64;
}

// The sampling epilogue (mlp_policy_kernel<true>, orlg_policy_sample): one Philox4x32-10 block per row, key = seed,
// counter = (c0, 0, row_id_base + row, 3) -- stream 3 of DESIGN.md section 5 -- where c0 = counter_dev[row] (the env's
// request index) or `counter`.  Every output may be NULL.
struct PolicyDraw {
    unsigned long long seed;
    const unsigned *counter_dev;
    unsigned counter;
    int deterministic;                // 1: argmax (first maximum); 0: inverse-CDF draw from softmax(logits)
    long long row_id_base;
    float *log_prob;                  // [n] log softmax(logits)[action]
    float *value;                     // [n] the value head
    const unsigned char *mask;        // [n, n_actions] invalid-action mask, 0 = invalid (read by the MASKED instances only)
};

// Shared-memory operand layout (no swizzle): 8 x 8 bf16 core matrices of 128 contiguous bytes (row r of the core matrix at
// r * 16); core matrix (row block i, k block j) of an operand with R rows at j * (R / 8) * 128 + i * 128.  In descriptor terms:
// leading-dimension (K) byte offset = (R / 8) * 128, stride-dimension (M / N) byte offset = 128.
__host__ __device__ inline int pl_operand_offset(int rows, int r, int k) {       // byte offset of element (r, k)
    return (k >> 3) * (rows >> 3) * 128 + (r >> 3) * 128 + (r & 7) * 16 + (k & 7) * 2;
}

__device__ __forceinline__ unsigned long long pl_smem_desc(unsigned smem_addr, unsigned lbo_bytes, unsigned sbo_bytes) {
    // tcgen05 shared-memory matrix descriptor: start address >> 4 [0,14), LBO >> 4 [16,30), SBO >> 4 [32,46), version 1 [46,48),
    // layout type 0 = no swizzle [61,64)
    return (unsigned long long)((smem_addr & 0x3FFFFu) >> 4) | ((unsigned long long)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((unsigned long long)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ULL << 46);
}
__device__ __forceinline__ unsigned pl_instr_desc(int M, int N) {
    // kind::f16 instruction descriptor: D = F32 [4,6), A = BF16 [7,10), B = BF16 [10,13), both K-major, N >> 3 [17,23), M >> 4 [24,29)
    return (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(N >> 3) << 17) | ((unsigned)(M >> 4) << 24);
}
__device__ __forceinline__ void pl_mma(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc, unsigned idesc, unsigned accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void pl_commit(unsigned long long *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ float pl_tanh(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// 32 consecutive accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void pl_tmem_ld32(unsigned taddr, float (&v)[32]) {
    unsigned r[32];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}
// the same without the wait: several loads in flight, one pl_tmem_wait() before the first use
__device__ __forceinline__ void pl_tmem_ld32_nowait(unsigned taddr, unsigned *r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void pl_tmem_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void pl_tmem_ld16(unsigned taddr, float (&v)[16]) {
    unsigned r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}

// Output layer of the sampling instance, one thread = one row, all in registers (static indices over the 15 possible logits):
// l_a = acc_a + bias_a, m = max l, e_a = expf(l_a - m), S = e_0 + ... in index order; the action is the argmax (deterministic)
// or the smallest a with u S < e_0 + ... + e_a for u = (Philox word 0 >> 8) 2^-24 (the last action if rounding leaves none);
// log_prob = l_a - m - logf(S).  expf / logf, not the intrinsics: 15 values per row.
// MASKED (sb3-contrib's MaskableCategorical): l_a = -1e8 where the row's mask byte is 0, before all of the above, and the
// rounding fallback is the last action with e_a > 0, so a masked action is never drawn while any action is valid.  An all-zero
// row gives the uniform distribution (action 0 when deterministic).  The unmasked instances compile as before: every MASKED
// statement is a constant-false branch there.
template <bool MASKED>
__device__ __forceinline__ void pl_sample_epilogue(const PolicyParams &pp, const PolicyDraw &dr, const float (&v)[16], const float *b,
                                                   int env, int *actions) {
    constexpr int NA = PL_NOUT - 1;
    const int na = pp.n_actions;
    unsigned valid = 0;               // bit a = action a is valid
    if (MASKED) {
        const unsigned char *mrow = dr.mask + (size_t)env * na;
#pragma unroll
        for (int a = 0; a < NA; a++)
            if (a < na && mrow[a]) valid |= 1u << a;
    }
    float l[NA], m = v[0] + b[0];
    if (MASKED && !(valid & 1u)) m = -1e8f;
#pragma unroll
    for (int a = 0; a < NA; a++) {
        l[a] = v[a] + b[a];
        if (MASKED && !((valid >> a) & 1u)) l[a] = -1e8f;
        if (a < na && l[a] > m) m = l[a];
    }
    float value = 0.0f;
#pragma unroll
    for (int a = 1; a < PL_NOUT; a++)
        if (a == na) value = v[a] + b[a];
    if (dr.value) dr.value[env] = value;
    if (!actions && !dr.log_prob) return;                           // a critic launch: the value only
    float e[NA], S = 0.0f;
#pragma unroll
    for (int a = 0; a < NA; a++) {
        e[a] = a < na ? expf(l[a] - m) : 0.0f;
        S += e[a];                                                   // (+ 0.0f beyond n_actions: exact)
    }
    int pick = 0;
    if (dr.deterministic) {
        float bv = l[0];
#pragma unroll
        for (int a = 1; a < NA; a++)
            if (a < na && l[a] > bv) { bv = l[a]; pick = a; }
    } else {
        uint32_t c[4] = {dr.counter_dev ? dr.counter_dev[env] : dr.counter, 0u, (uint32_t)(unsigned long long)(dr.row_id_base + env), 3u};
        philox4x32_10(c, (uint32_t)dr.seed, (uint32_t)(dr.seed >> 32));
        const float us = (float)(c[0] >> 8) * 0x1p-24f * S;
        float acc = 0.0f;
        bool found = false;
        pick = na - 1;
        if (MASKED) {
            pick = 0;
#pragma unroll
            for (int a = 0; a < NA; a++)
                if (a < na && e[a] > 0.0f) pick = a;
        }
#pragma unroll
        for (int a = 0; a < NA; a++) {
            if (a < na) {
                acc += e[a];
                if (!found && us < acc) { pick = a; found = true; }
            }
        }
    }
    float lp = l[0];
#pragma unroll
    for (int a = 1; a < NA; a++)
        if (a == pick) lp = l[a];
    if (actions) actions[env] = pick;
    if (dr.log_prob) dr.log_prob[env] = lp - m - logf(S);
}

// Two groups of EIGHT warps per CTA, each walking its own stream of 128-environment tiles with its own A buffer, TMEM accumulator
// and mbarrier (they only share the weights): one group's tensor-core work and TMEM reads overlap the other's epilogue math.
// Inside a group warp w reads TMEM lanes 32 (w % 4) .. + 31 (the hardware's lane quarter of a warp) and takes columns
// (H / 2) (w / 4) .. + H / 2 - 1: thread t owns row t % 128 and one half of its columns, so the epilogue of a layer (128 x H
// tanh, the chain that bounds this kernel) is spread over 8 warps with all of a thread's TMEM loads in flight before the first use.
// smem: [weights w_bytes][2 x A tile 128 x 128 bf16 = 64 KB][bias floats][mbarriers][tmem base]  (pl_smem_bytes)
constexpr int PL_WG = 256;            // threads per group
__device__ __forceinline__ void pl_group_sync(int group) {          // named barrier of one group (ids 1, 2; 0 = __syncthreads)
    asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(PL_WG) : "memory");
}

// SAMPLE = false: orlg_policy_act (argmax, optional logits; `dr` unused).  SAMPLE = true: orlg_policy_sample (the epilogue
// of PolicyDraw; `actions` may be NULL, `logits_out` is unused).  HC, LC: the hidden width and depth fixed at compile time
// (they must equal pp.H, pp.L), or 0: read from pp at run time.  MASKED (with SAMPLE only): the epilogue draws under the
// invalid-action mask dr.mask (orlg_policy_sample_masked); a template flag, so that the unmasked instances keep their code.
template <bool SAMPLE, int HC, int LC, bool MASKED = false>
__global__ void __launch_bounds__(PL_WG * PL_GROUPS, 1)
mlp_policy_kernel(const PolicyParams pp, const float *__restrict__ obs, const int n, int *__restrict__ actions,
                  float *__restrict__ logits_out /* [n, n_actions + 1] = logits + value, or NULL */, const PolicyDraw dr) {
    extern __shared__ __align__(128) unsigned char psm[];
    const int H = HC ? HC : pp.H, L = LC ? LC : pp.L;
    const int group = threadIdx.x / PL_WG, tid = threadIdx.x % PL_WG, warp = (tid >> 5) & 3;     // warp = TMEM lane quarter of this warp
    const int half = tid >> 7;        // which half of the H columns (K elements of the next layer) this thread produces
    unsigned char *s_w = psm;
    unsigned char *s_a = psm + pp.w_bytes + (size_t)group * PL_TILE * PL_HMAX * 2;
    float *s_bias = reinterpret_cast<float *>(psm + pp.w_bytes + (size_t)PL_GROUPS * PL_TILE * PL_HMAX * 2);
    unsigned long long *bars = reinterpret_cast<unsigned long long *>(s_bias + L * H + PL_NOUT);   // [0] weights, [1 + g] mma of group g
    unsigned *s_tmem = reinterpret_cast<unsigned *>(bars + 1 + PL_GROUPS);

    pdl_launch_dependents();
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        for (int g = 0; g < PL_GROUPS; g++) mbar_init(&bars[1 + g], 1);
        mbar_expect_tx(&bars[0], (unsigned)pp.w_bytes);
        // the weights do not depend on the previous kernel of the stream: requested before the dependency wait
        const unsigned chunk = 32768u;
        for (unsigned off = 0; off < (unsigned)pp.w_bytes; off += chunk) {
            const unsigned bytes = min(chunk, (unsigned)pp.w_bytes - off);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"((unsigned)__cvta_generic_to_shared(s_w + off)), "l"(reinterpret_cast<const unsigned char *>(pp.w_blob) + off),
                           "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(&bars[0])) : "memory");
        }
    }
    for (int i = threadIdx.x; i < L * H + PL_NOUT; i += PL_WG * PL_GROUPS) s_bias[i] = pp.bias[i];
    if (threadIdx.x < 32) {     // TMEM: 128 columns (one 128 x 128 fp32 accumulator tile, of which H are used) per tile group
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"((unsigned)__cvta_generic_to_shared(s_tmem)), "r"(128u * PL_GROUPS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem = *s_tmem + (unsigned)group * 128u;           // this warpgroup's accumulator columns
    const unsigned t_lane = tmem + ((unsigned)(warp * 32) << 16);       // this warp's 32 TMEM lanes
    mbar_wait(&bars[0], 0);           // weights have landed
    pdl_wait();                       // the observations come from the previous kernel of the stream

    const unsigned a_addr = (unsigned)__cvta_generic_to_shared(s_a);
    const unsigned w_addr = (unsigned)__cvta_generic_to_shared(s_w);
    unsigned phase = 0;
    const int row = tid & 127;        // thread t owns row t % 128 of the tile: TMEM lane, A-operand row
    unsigned char *a_row = s_a + (row >> 3) * 128 + (row & 7) * 16;        // + (k >> 3) * 2048 + (k & 7) * 2

    unsigned long long *bar = &bars[1 + group];
    for (int tile = blockIdx.x * PL_GROUPS + group; tile * PL_TILE < n; tile += gridDim.x * PL_GROUPS) {
        const int env = tile * PL_TILE + row;
        // ---- layer-0 input: the tile's observation rows as bf16, K padded to 64 with zeros.  The 128 rows are one contiguous
        // 27 KB run of obs: they are fetched with coalesced 16-byte loads, 64 rows at a time, into the upper half of the A
        // buffer (k blocks 8..15: unused by layer 0), and each thread then converts its 32 of a row's 64 elements from there.
        // (A thread reading its own 216-byte row from global memory cost 32 sectors per load instruction: 42 % of the kernel's
        // stall samples were lg_throttle / long scoreboard on those loads.)
        {
            constexpr int KH = PL_K0 / 2;
            unsigned char *stage = s_a + 8 * 2048;                          // 16 KB
            const bool fast = (pp.obs_dim * 4 * 64) % 16 == 0 && (reinterpret_cast<size_t>(obs) & 15) == 0 && pp.obs_dim * 4 * 64 <= 16384;
            for (int hseg = 0; hseg < 2; hseg++) {
                const int r0 = tile * PL_TILE + hseg * 64;                  // first env of this half tile
                const int rows_here = min(64, n - r0);                      // may be <= 0 in the last tile
                float x[KH];
#pragma unroll
                for (int k = 0; k < KH; k++) x[k] = 0.0f;
                if (fast) {
                    const int vec_total = rows_here > 0 ? (rows_here * pp.obs_dim) / 4 : 0;          // whole 16-byte vectors available
                    const int tail = rows_here > 0 ? rows_here * pp.obs_dim - 4 * vec_total : 0;     // (a ragged last tile: 0..3 floats)
                    const uint4 *g = reinterpret_cast<const uint4 *>(obs + (size_t)r0 * pp.obs_dim);
#pragma unroll
                    for (int it = 0; it < 4; it++) {
                        const int v = tid + it * PL_WG;
                        if (v < vec_total) *reinterpret_cast<uint4 *>(stage + v * 16) = g[v];
                    }
                    if (tid < tail) reinterpret_cast<float *>(stage)[4 * vec_total + tid] = obs[(size_t)r0 * pp.obs_dim + 4 * vec_total + tid];
                    pl_group_sync(group);
                    if ((row >> 6) == hseg && env < n) {
                        const float2 *src = reinterpret_cast<const float2 *>(stage + (row & 63) * pp.obs_dim * 4) + half * (KH / 2);
#pragma unroll
                        for (int k = 0; k < KH / 2; k++)
                            if (half * KH + 2 * k < pp.obs_dim) { const float2 v = src[k]; x[2 * k] = v.x; x[2 * k + 1] = v.y; }
                    }
                } else if ((row >> 6) == hseg && env < n) {
                    const float2 *src = reinterpret_cast<const float2 *>(obs + (size_t)env * pp.obs_dim) + half * (KH / 2);     // obs_dim is even: rows are 8-byte aligned
#pragma unroll
                    for (int k = 0; k < KH / 2; k++)
                        if (half * KH + 2 * k < pp.obs_dim) { const float2 v = src[k]; x[2 * k] = v.x; x[2 * k + 1] = v.y; }
                }
                if ((row >> 6) == hseg) {
#pragma unroll
                    for (int j = 0; j < KH / 8; j++) {
                        uint4 pk;
                        __nv_bfloat162 h0 = __floats2bfloat162_rn(x[8 * j], x[8 * j + 1]), h1 = __floats2bfloat162_rn(x[8 * j + 2], x[8 * j + 3]);
                        __nv_bfloat162 h2 = __floats2bfloat162_rn(x[8 * j + 4], x[8 * j + 5]), h3 = __floats2bfloat162_rn(x[8 * j + 6], x[8 * j + 7]);
                        pk.x = *reinterpret_cast<unsigned *>(&h0); pk.y = *reinterpret_cast<unsigned *>(&h1);
                        pk.z = *reinterpret_cast<unsigned *>(&h2); pk.w = *reinterpret_cast<unsigned *>(&h3);
                        *reinterpret_cast<uint4 *>(a_row + (half * (KH / 8) + j) * 2048) = pk;
                    }
                }
                if (fast) pl_group_sync(group);                             // the stage is refilled (or becomes operand space) next
            }
        }
        int w_off = 0;                 // byte offset of the current layer's weights in s_w
        for (int layer = 0; layer <= L; layer++) {
            const int K = layer == 0 ? PL_K0 : H;
            const int N = layer == L ? PL_NOUT : H;
            // activations written by the generic proxy -> visible to the tensor core (async proxy); previous TMEM reads done
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            pl_group_sync(group);
            if (tid == 0) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const unsigned idesc = pl_instr_desc(PL_TILE, N);
                const unsigned a_lbo = (PL_TILE / 8) * 128, b_lbo = (unsigned)(N / 8) * 128;
#pragma unroll 1
                for (int kk = 0; kk < K / 16; kk++) {            // one instruction per 16 elements of K (two core matrices)
                    const unsigned long long ad = pl_smem_desc(a_addr + (unsigned)kk * 2u * a_lbo, a_lbo, 128u);
                    const unsigned long long bd = pl_smem_desc(w_addr + (unsigned)w_off + (unsigned)kk * 2u * b_lbo, b_lbo, 128u);
                    pl_mma(tmem, ad, bd, idesc, kk > 0 ? 1u : 0u);
                }
                pl_commit(bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1u;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const float *b = s_bias + layer * H;
            if (layer < L) {
                // ---- epilogue: bias + tanh, next layer's A operand (bf16) back into shared memory.  This thread's H / 2
                // columns are m chunks of 8 (register r[8 j ..] = column cb + 8 j ..).  Both .x32 loads are issued whatever H
                // is -- columns cb .. cb + 63 lie inside the group's 128 TMEM columns, chunks from m on are not used: loads
                // sized to H (.x16 / .x8, or a second .x32 only when H > 64) give a register two possible definitions, which
                // costs some 17 registers and spills at the 128 that 512 threads leave.
                const int m = H >> 4;
                const int cb = half * (H >> 1);
                unsigned r[64];
                pl_tmem_ld32_nowait(t_lane + (unsigned)cb, r);
                pl_tmem_ld32_nowait(t_lane + (unsigned)cb + 32u, r + 32);
                pl_tmem_wait();
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    if (j < m) {
                        const int c0 = cb + 8 * j;
                        const float4 b0 = *reinterpret_cast<const float4 *>(b + c0), b1 = *reinterpret_cast<const float4 *>(b + c0 + 4);
                        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                        unsigned w4[4];
#pragma unroll
                        for (int q = 0; q < 4; q++) {
                            const float v0 = __uint_as_float(r[8 * j + 2 * q]), v1 = __uint_as_float(r[8 * j + 2 * q + 1]);
                            __nv_bfloat162 h = __floats2bfloat162_rn(pl_tanh(v0 + bb[2 * q]), pl_tanh(v1 + bb[2 * q + 1]));
                            w4[q] = *reinterpret_cast<unsigned *>(&h);
                        }
                        *reinterpret_cast<uint4 *>(a_row + (c0 >> 3) * 2048) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
                    }
                }
            } else {
                // ---- output layer: 5 logits (+ value); deterministic action = argmax (first maximum, like torch.argmax)
                if (half == 0) {                                   // warp-uniform: the four warps of the first half hold the 128 rows
                    float v[16];
                    pl_tmem_ld16(t_lane, v);
                    if (SAMPLE) {
                        if (env < n) pl_sample_epilogue<MASKED>(pp, dr, v, b, env, actions);
                    } else if (env < n) {
                        int best = 0;
                        float bv = v[0] + b[0];
#pragma unroll
                        for (int a = 1; a < PL_NOUT - 1; a++) {          // static indices: the accumulator row stays in registers
                            const float l = v[a] + b[a];
                            if (a < pp.n_actions && l > bv) { bv = l; best = a; }
                        }
                        actions[env] = best;
                        if (logits_out) {
#pragma unroll
                            for (int a = 0; a < PL_NOUT; a++)
                                if (a <= pp.n_actions) logits_out[(size_t)env * (pp.n_actions + 1) + a] = v[a] + b[a];
                        }
                    }
                }
            }
            w_off += N * K * 2;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*s_tmem), "r"(128u * PL_GROUPS) : "memory");
}

}  // namespace orlg
