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
// its MASKED variant draws under an invalid-action mask (orlg_policy_sample_masked).  The WIDE instances
// (orlg_policy_create_wide) take observations up to 256 wide, layer 0 in chunks of 64 inputs.
#pragma once
#include <cuda_bf16.h>
#include "orlg_deeprmsa_fast.cuh"

namespace orlg {

constexpr int PL_TILE = 128;          // environments per tile = UMMA M
constexpr int PL_HMAX = 128;          // widest hidden layer: the TMEM columns and the A buffer of a tile group
constexpr int PL_K0 = 64;             // observation width padded to a multiple of 16 (54 -> 64)
constexpr int PL_K0_WIDE = 256;       // widest observation of the WIDE instances (orlg_policy_create_wide), K0 = obs_dim rounded up to 16
constexpr int PL_NOUT = 16;           // output layer padded: 5 logits + 1 value
constexpr int PL_SMEM_MAX = 232448;   // dynamic shared memory a block may opt in to on sm_100 (227 KB)

struct PolicyParams {
    const uint4 *w_blob;              // all weights, bf16, already in the shared-memory operand layout (orlg_policy_create)
    int w_bytes;                      // H * K0 * 2 + (L - 1) * H * H * 2 + 16 * H * 2 (K0 = 64; WIDE: obs_dim rounded up to 16)
    const float *bias;                // [L * H + 16]
    int obs_dim, n_actions;           // 54, 5
    int H, L;                         // hidden width (multiple of 16, 16..128) and number of hidden layers (>= 1)
};

// MATRIX instances (orlg_policy_create_matrix): the agent reads SimpleMatrixObservation rows packed as bits (orlg_matrix_observation
// _packed): uint32 [n, W], W = 4 + 4 NWV E, word 0 = min(src, dst) | max(src, dst) << 8, then per link NWV groups of 4 words,
// bit b of word w of group v = slot 128 v + 32 w + b.  Layer 0 has K0 = 64 ceil(2 N / 64) + 128 NWV E columns: the one-hot
// header, then link l's slots at 128 NWV l + s.  It does not fit in shared memory (360 KB at NSFNET / S = 100 / H = 64): it
// stays in a device buffer and every tile streams it, 64 columns (H x 128 bytes) at a time, through a ring of `stages` buffers
// per tile group; chunks whose 64 columns are all padding (slots >= S) are skipped.
constexpr int PL_MX_RMAX = 6;         // most ring stages per tile group
struct PolicyMatrix {
    const uint4 *w0;                  // layer 0, bf16, [K0 / 64 chunks][H x 64 operand] (chunk c at c * H * 128 bytes); NULL = not MATRIX
    int nodes, links, slots, nwv;     // N, E, S, 128-bit word groups per link (ceil(S / 128))
    int hdr_chunks, link_chunks;      // ceil(2 N / 64); ceil(S / 64): the chunks of a link that hold slots
    int stages, seg_q;                // ring stages per group (3..PL_MX_RMAX); 16-byte words per row of the row stage (1..8)
};

// bytes of weights and of dynamic shared memory of a policy with hidden width H, L hidden layers, layer 0 padded to K0 inputs
// and G tile groups per CTA (the 2-argument forms: K0 = 64, G = 2, the instances of orlg_policy_create)
inline size_t pl_weight_bytes(int H, int L, int K0) {
    return (size_t)H * K0 * 2 + (size_t)(L - 1) * H * H * 2 + (size_t)PL_NOUT * H * 2;
}
inline size_t pl_weight_bytes(int H, int L) { return pl_weight_bytes(H, L, PL_K0); }
constexpr int PL_GROUPS = 2;          // tile groups per CTA
inline size_t pl_smem_bytes(int H, int L, int K0, int G) {
    return pl_weight_bytes(H, L, K0) + (size_t)G * PL_TILE * PL_HMAX * 2 + ((size_t)L * H + PL_NOUT) * 4 + 64;
}
inline size_t pl_smem_bytes(int H, int L) { return pl_smem_bytes(H, L, PL_K0, PL_GROUPS); }
// a MATRIX handle: the resident weights are layers 1.. and the heads (K0 = 0), and each group adds its ring, its row stage and
// 2 + PL_MX_RMAX mbarriers
inline size_t pl_matrix_smem_bytes(int H, int L, int G, int stages, int seg_q) {
    return pl_smem_bytes(H, L, 0, G) + (size_t)G * ((size_t)stages * H * 128 + (size_t)seg_q * PL_TILE * 16 + (2 + PL_MX_RMAX) * 8);
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
// smem: [weights w_bytes][G x A tile 128 x 128 bf16 = G x 32 KB][bias floats][mbarriers][tmem base]  (pl_smem_bytes; G = 2, or
// 1 on a WIDE handle whose layer-0 weights leave room for one group only)
constexpr int PL_WG = 256;            // threads per group
__device__ __forceinline__ void pl_group_sync(int group) {          // named barrier of one group (ids 1, 2; 0 = __syncthreads)
    asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(PL_WG) : "memory");
}

// SAMPLE = false: orlg_policy_act (argmax, optional logits; `dr` unused).  SAMPLE = true: orlg_policy_sample (the epilogue
// of PolicyDraw; `actions` may be NULL, `logits_out` is unused).  HC, LC: the hidden width and depth fixed at compile time
// (they must equal pp.H, pp.L), or 0: read from pp at run time.  MASKED (with SAMPLE only): the epilogue draws under the
// invalid-action mask dr.mask (orlg_policy_sample_masked); a template flag, so that the unmasked instances keep their code.
// WIDE (run-time H, L only; orlg_policy_create_wide): observations up to 256 wide, any parity.  Layer 0 has K0 = obs_dim
// rounded up to 16 inputs and runs in chunks of 64 columns through the A buffer (see the staging block), and the CTA has
// G = blockDim.x / PL_WG tile groups (1 or 2: what fits in shared memory next to the larger layer-0 weights).
// MATRIX (run-time H, L, act and sample only; orlg_policy_create_matrix): `obs` is packed matrix rows (PolicyMatrix), layer 0
// streamed through a ring (see the MATRIX block); G as for WIDE.  `mx` is read by the MATRIX instances only.
template <bool SAMPLE, int HC, int LC, bool MASKED = false, bool WIDE = false, bool MATRIX = false>
__global__ void __launch_bounds__(PL_WG * PL_GROUPS, 1)
mlp_policy_kernel(const PolicyParams pp, const float *__restrict__ obs, const int n, int *__restrict__ actions,
                  float *__restrict__ logits_out /* [n, n_actions + 1] = logits + value, or NULL */, const PolicyDraw dr,
                  const PolicyMatrix mx) {
    extern __shared__ __align__(128) unsigned char psm[];
    const int H = HC ? HC : pp.H, L = LC ? LC : pp.L;
    const int G = WIDE || MATRIX ? (int)(blockDim.x / PL_WG) : PL_GROUPS;         // tile groups of this CTA
    const int K0 = WIDE ? (pp.obs_dim + 15) & ~15 : PL_K0;                        // layer-0 inputs
    const int nch = WIDE ? (K0 + 63) >> 6 : 1;                                    // layer-0 chunks of 64 columns
    const int group = threadIdx.x / PL_WG, tid = threadIdx.x % PL_WG, warp = (tid >> 5) & 3;     // warp = TMEM lane quarter of this warp
    const int half = tid >> 7;        // which half of the H columns (K elements of the next layer) this thread produces
    unsigned char *s_w = psm;
    unsigned char *s_a = psm + pp.w_bytes + (size_t)group * PL_TILE * PL_HMAX * 2;
    // MATRIX: [G][stages][H x 128 B] ring, then [G][seg_q][128 rows x 16 B] row stage, after the A buffers
    const size_t mx_ring = MATRIX ? (size_t)mx.stages * H * 128 : 0, mx_stage = MATRIX ? (size_t)mx.seg_q * PL_TILE * 16 : 0;
    unsigned char *s_ring = psm + pp.w_bytes + (size_t)G * PL_TILE * PL_HMAX * 2 + (size_t)group * mx_ring;
    unsigned char *s_rows = psm + pp.w_bytes + (size_t)G * (PL_TILE * PL_HMAX * 2 + mx_ring) + (size_t)group * mx_stage;
    float *s_bias = reinterpret_cast<float *>(psm + pp.w_bytes + (size_t)G * PL_TILE * PL_HMAX * 2 + (MATRIX ? (size_t)G * (mx_ring + mx_stage) : 0));
    // [0] weights, [1 + g] mma of group g; MATRIX: [1 + G + (2 + PL_MX_RMAX) g ..] group g's A-half barriers, then its ring stages
    unsigned long long *bars = reinterpret_cast<unsigned long long *>(s_bias + L * H + PL_NOUT);
    const int nbars = 1 + G + (MATRIX ? G * (2 + PL_MX_RMAX) : 0);
    unsigned *s_tmem = reinterpret_cast<unsigned *>(bars + 1 + G + (MATRIX ? G * (2 + PL_MX_RMAX) : 0));

    pdl_launch_dependents();
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        for (int g = 0; g < G; g++) mbar_init(&bars[1 + g], 1);
        if (MATRIX)
            for (int g = 1 + G; g < nbars; g++) mbar_init(&bars[g], 1);
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
    for (int i = threadIdx.x; i < L * H + PL_NOUT; i += PL_WG * G) s_bias[i] = pp.bias[i];
    if (threadIdx.x < 32) {     // TMEM: 128 columns (one 128 x 128 fp32 accumulator tile, of which H are used) per tile group
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"((unsigned)__cvta_generic_to_shared(s_tmem)), "r"(128u * G) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem = *s_tmem + (unsigned)group * 128u;           // this warpgroup's accumulator columns
    const unsigned t_lane = tmem + ((unsigned)(warp * 32) << 16);       // this warp's 32 TMEM lanes
    // MATRIX: layer-0 chunk c of the compact chunk list (header chunks, then each link's chunks that hold slots) -> its first
    // weight column; chunk gq of this group's stream (continuous over its tiles) goes to ring stage gq % stages
    const int mnch = MATRIX ? mx.hdr_chunks + mx.links * mx.link_chunks : 0;
    unsigned long long *abar = bars + 1 + G + (2 + PL_MX_RMAX) * group, *fullb = abar + 2;
    auto mx_col = [&](int c) {
        const int lc = c - mx.hdr_chunks;
        return c < mx.hdr_chunks ? 64 * c : 64 * mx.hdr_chunks + 128 * mx.nwv * (lc / mx.link_chunks) + 64 * (lc % mx.link_chunks);
    };
    auto mx_fetch = [&](long long gq) {                                   // thread 0 of the group: chunk gq into its stage
        const long long t = gq / mnch;
        if ((long long)(blockIdx.x * G + group + t * gridDim.x * G) * PL_TILE >= n) return;  // past this group's last tile: never consumed
        const unsigned bytes = (unsigned)H * 128u;
        unsigned long long *fb = &fullb[gq % mx.stages];
        mbar_expect_tx(fb, bytes);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"((unsigned)__cvta_generic_to_shared(s_ring + (size_t)(gq % mx.stages) * bytes)),
                       "l"(reinterpret_cast<const unsigned char *>(mx.w0) + (size_t)(mx_col((int)(gq % mnch)) >> 6) * bytes),
                       "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(fb)) : "memory");
    };
    if (MATRIX && tid == 0)           // the layer-0 weights do not depend on the previous kernel either
        for (int gq = 0; gq < mx.stages - 2; gq++) mx_fetch(gq);
    long long mx_gq = 0;
    unsigned aph = 0u;                // bit h: phase parity of A-half barrier h
    mbar_wait(&bars[0], 0);           // weights have landed
    pdl_wait();                       // the observations come from the previous kernel of the stream

    const unsigned a_addr = (unsigned)__cvta_generic_to_shared(s_a);
    const unsigned w_addr = (unsigned)__cvta_generic_to_shared(s_w);
    unsigned phase = 0;
    const int row = tid & 127;        // thread t owns row t % 128 of the tile: TMEM lane, A-operand row
    unsigned char *a_row = s_a + (row >> 3) * 128 + (row & 7) * 16;        // + (k >> 3) * 2048 + (k & 7) * 2

    unsigned long long *bar = &bars[1 + group];
    for (int tile = blockIdx.x * G + group; tile * PL_TILE < n; tile += gridDim.x * G) {
        const int env = tile * PL_TILE + row;
        if (MATRIX) {
            // ---- layer 0 of the MATRIX instance, in chunks of 64 columns.  Chunk c goes to half c & 1 of the A buffer as bf16
            // 0.0 / 1.0: header chunks from the one-hot positions of word 0, link chunks from 64 bits of each row.  It waits
            // for chunk c - 2's MMAs (which read that half and whose ring stage the refill below overwrites) on the half's
            // barrier, so the expansion of chunk c overlaps the MMAs of chunk c - 1.  B is the chunk's ring stage.  The last two
            // chunks commit nowhere: layer 0 of the layer loop (no MMA of its own) commits after them.
            // Rows: the tile's 128 packed rows are one contiguous run; 16-byte words seg_q s .. seg_q s + seg_q - 1 of every row
            // are loaded as consecutive uint4 of each row (coalesced) into the row stage, word qq of row r at
            // qq * 2048 + ((r ^ qq) & 127) * 16 (consecutive rows on consecutive 16-byte slots for the reads; the XOR spreads the
            // stores of one row's words over the banks).  A chunk needs one 16-byte word of its row (word 0 for the header).
            const int U = 1 + mx.nwv * mx.links;                            // 16-byte words per packed row
            const uint4 *rows4 = reinterpret_cast<const uint4 *>(obs);
            int seg = -1;
            for (int c = 0; c < mnch; c++, mx_gq++) {
                const int h = c & 1;
                const bool hdr = c < mx.hdr_chunks;
                const int lc = c - mx.hdr_chunks, lj = hdr ? 0 : lc % mx.link_chunks;
                const int q = hdr ? 0 : 1 + mx.nwv * (lc / mx.link_chunks) + (lj >> 1);
                if (q / mx.seg_q != seg) {                                  // (the stage's last readers passed chunk c - 1's sync)
                    seg = q / mx.seg_q;
                    const int cnt = min(mx.seg_q, U - seg * mx.seg_q);
                    uint4 v[4];
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const int e = tid + i * PL_WG, r = e / cnt, qq = e - r * cnt;
                        v[i] = make_uint4(0u, 0u, 0u, 0u);
                        if (e < PL_TILE * cnt && tile * PL_TILE + r < n) v[i] = rows4[(size_t)(tile * PL_TILE + r) * U + seg * mx.seg_q + qq];
                    }
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const int e = tid + i * PL_WG, r = e / cnt, qq = e - r * cnt;
                        if (e < PL_TILE * cnt) *reinterpret_cast<uint4 *>(s_rows + qq * 2048 + (((r ^ qq) & 127) << 4)) = v[i];
                    }
                    pl_group_sync(group);
                }
                if (c >= 2) {                                               // chunk c - 2's MMAs are done
                    mbar_wait(&abar[h], (aph >> h) & 1u);
                    aph ^= 1u << h;
                }
                if (tid == 0) mx_fetch(mx_gq + mx.stages - 2);              // into the stage chunk c - 2 read
                const int qq = q - seg * mx.seg_q;
                const uint4 x = *reinterpret_cast<const uint4 *>(s_rows + qq * 2048 + (((row ^ qq) & 127) << 4));
                unsigned bits;
                if (hdr) {                                                  // this thread's columns 64 c + 32 half .. + 31
                    const int base = 64 * c + 32 * half, lo = (int)(x.x & 0xffu) - base, hi = mx.nodes + (int)((x.x >> 8) & 0xffu) - base;
                    bits = (lo >= 0 && lo < 32 ? 1u << lo : 0u) | (hi >= 0 && hi < 32 ? 1u << hi : 0u);
                } else {
                    const int comp = 2 * (lj & 1) + half;                   // slots 64 lj + 32 half .. + 31 of the link
                    bits = comp == 0 ? x.x : (comp == 1 ? x.y : (comp == 2 ? x.z : x.w));
                }
#pragma unroll
                for (int j = 0; j < 4; j++) {                               // columns 8 j .. + 7 of this thread's 32
                    unsigned w4[4];
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        const unsigned b = bits >> (8 * j + 2 * e);
                        w4[e] = ((b & 1u) ? 0x3F80u : 0u) | ((b & 2u) ? 0x3F800000u : 0u);
                    }
                    *reinterpret_cast<uint4 *>(a_row + (h * 8 + half * 4 + j) * 2048) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                pl_group_sync(group);
                if (tid == 0) {
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    mbar_wait(&fullb[mx_gq % mx.stages], (unsigned)((mx_gq / mx.stages) & 1));
                    const unsigned idesc = pl_instr_desc(PL_TILE, H);
                    const unsigned a_lbo = (PL_TILE / 8) * 128, b_lbo = (unsigned)(H / 8) * 128;
                    const unsigned b_addr = (unsigned)__cvta_generic_to_shared(s_ring + (size_t)(mx_gq % mx.stages) * H * 128);
#pragma unroll 1
                    for (int kk = 0; kk < 4; kk++) {
                        const unsigned long long ad = pl_smem_desc(a_addr + (unsigned)(h * 8 + 2 * kk) * a_lbo, a_lbo, 128u);
                        const unsigned long long bd = pl_smem_desc(b_addr + (unsigned)(2 * kk) * b_lbo, b_lbo, 128u);
                        pl_mma(tmem, ad, bd, idesc, c > 0 || kk > 0 ? 1u : 0u);
                    }
                    if (c + 2 < mnch) pl_commit(&abar[h]);
                }
            }
        } else if (WIDE) {
            // ---- layer-0 input of the WIDE instance, in chunks of 64 columns.  Chunk c (columns 64 c .. + 63) goes to half c & 1
            // of the A buffer (k blocks 8 (c & 1) .. + 7) as bf16; its fp32 rows are staged, 64 at a time, in the other half.  That
            // half is what chunk c - 1's MMAs read, so chunk c waits for them (their commit, on the group's mbarrier) before its
            // first stage store; its global loads are issued before that wait.  Every chunk but the last is multiplied here,
            // accumulating into the tile's TMEM columns from the second chunk on; the last one is layer 0 of the layer loop.  With
            // K0 <= 64 this is the narrow instance's single pass on the same bf16 operands.
            // Loads: thread tid reads elements tid + 256 i (i < 16) of the 64 x 64 block, so a warp reads 32 consecutive floats of
            // one row, coalesced whatever the row's alignment (rows are obs_dim * 4 bytes, only 4-byte aligned when obs_dim is
            // odd); columns >= obs_dim and rows >= n are zeros.  Stage: row r at r * 256, its 16-byte word q at word q ^ (r & 15),
            // so the float4 reads of one word by a warp's 32 rows take 4 wavefronts instead of the 32 of a plain 256-byte stride.
            for (int c = 0; c < nch; c++) {
                const int h = c & 1;
                unsigned char *stage = s_a + (1 - h) * 8 * 2048;              // 16 KB: 64 rows x 64 floats
                for (int hseg = 0; hseg < 2; hseg++) {
                    const int r0 = tile * PL_TILE + hseg * 64;                  // first env of this half tile
                    float v[16];
#pragma unroll
                    for (int i = 0; i < 16; i++) {
                        const int e = tid + i * PL_WG, rr = e >> 6, col = 64 * c + (e & 63);
                        v[i] = col < pp.obs_dim && r0 + rr < n ? obs[(size_t)(r0 + rr) * pp.obs_dim + col] : 0.0f;
                    }
                    if (c > 0 && hseg == 0) {                                   // chunk c - 1's MMAs have read the stage half
                        mbar_wait(bar, phase);
                        phase ^= 1u;
                    }
#pragma unroll
                    for (int i = 0; i < 16; i++) {
                        const int e = tid + i * PL_WG, rr = e >> 6, k = e & 63;
                        *reinterpret_cast<float *>(stage + rr * 256 + (((k >> 2) ^ (rr & 15)) << 4) + (k & 3) * 4) = v[i];
                    }
                    pl_group_sync(group);
                    if ((row >> 6) == hseg) {
                        const int rr = row & 63;
                        const unsigned char *src = stage + rr * 256;
#pragma unroll
                        for (int j = 0; j < 4; j++) {                           // this thread's columns half * 32 + 8 j .. + 7
                            const int q = half * 8 + 2 * j;
                            const float4 x0 = *reinterpret_cast<const float4 *>(src + ((q ^ (rr & 15)) << 4));
                            const float4 x1 = *reinterpret_cast<const float4 *>(src + (((q + 1) ^ (rr & 15)) << 4));
                            uint4 pk;
                            __nv_bfloat162 h0 = __floats2bfloat162_rn(x0.x, x0.y), h1 = __floats2bfloat162_rn(x0.z, x0.w);
                            __nv_bfloat162 h2 = __floats2bfloat162_rn(x1.x, x1.y), h3 = __floats2bfloat162_rn(x1.z, x1.w);
                            pk.x = *reinterpret_cast<unsigned *>(&h0); pk.y = *reinterpret_cast<unsigned *>(&h1);
                            pk.z = *reinterpret_cast<unsigned *>(&h2); pk.w = *reinterpret_cast<unsigned *>(&h3);
                            *reinterpret_cast<uint4 *>(a_row + (h * 8 + half * 4 + j) * 2048) = pk;
                        }
                    }
                    pl_group_sync(group);                                       // the stage is refilled next
                }
                if (c + 1 < nch) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    pl_group_sync(group);
                    if (tid == 0) {
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const unsigned idesc = pl_instr_desc(PL_TILE, H);
                        const unsigned a_lbo = (PL_TILE / 8) * 128, b_lbo = (unsigned)(H / 8) * 128;
#pragma unroll 1
                        for (int kk = 0; kk < 4; kk++) {
                            const unsigned long long ad = pl_smem_desc(a_addr + (unsigned)(h * 8 + 2 * kk) * a_lbo, a_lbo, 128u);
                            const unsigned long long bd = pl_smem_desc(w_addr + (unsigned)(8 * c + 2 * kk) * b_lbo, b_lbo, 128u);
                            pl_mma(tmem, ad, bd, idesc, c > 0 || kk > 0 ? 1u : 0u);
                        }
                        pl_commit(bar);
                    }
                }
            }
        } else {
        // ---- layer-0 input: the tile's observation rows as bf16, K padded to 64 with zeros.  The 128 rows are one contiguous
        // 27 KB run of obs: they are fetched with coalesced 16-byte loads, 64 rows at a time, into the upper half of the A
        // buffer (k blocks 8..15: unused by layer 0), and each thread then converts its 32 of a row's 64 elements from there.
        // (A thread reading its own 216-byte row from global memory cost 32 sectors per load instruction: 42 % of the kernel's
        // stall samples were lg_throttle / long scoreboard on those loads.)
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
            const int K = layer == 0 ? (MATRIX ? 0 : WIDE ? K0 - 64 * (nch - 1) : PL_K0) : H;     // WIDE layer 0: its last chunk; MATRIX: none
            const int N = layer == L ? PL_NOUT : H;
            const bool chunked = WIDE && layer == 0 && nch > 1;
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
                    unsigned a_k = a_addr + (unsigned)kk * 2u * a_lbo, w_k = w_addr + (unsigned)w_off + (unsigned)kk * 2u * b_lbo;
                    if (chunked) {                                // the last chunk: A half (nch - 1) & 1, weight columns 64 (nch - 1) ..
                        a_k += (unsigned)((nch - 1) & 1) * 8u * a_lbo;
                        w_k += (unsigned)(nch - 1) * 8u * b_lbo;
                    }
                    const unsigned long long ad = pl_smem_desc(a_k, a_lbo, 128u);
                    const unsigned long long bd = pl_smem_desc(w_k, b_lbo, 128u);
                    pl_mma(tmem, ad, bd, idesc, kk > 0 || chunked ? 1u : 0u);
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
            w_off += N * (WIDE && layer == 0 ? K0 : K) * 2;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*s_tmem), "r"(128u * G) : "memory");
}

}  // namespace orlg
