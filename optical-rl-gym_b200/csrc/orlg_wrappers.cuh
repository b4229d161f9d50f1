// orlg_wrappers.cuh -- device versions of the reference's gym wrappers (SURVEY.md row f2).
// Both kernels use the generic CSR hop lists and multi-word masks, so they serve every handle
// (any link count, up to 512 slots, any env kind).
#pragma once
#include "orlg_step_wide.cuh"

namespace orlg {

// PathOnlyFirstFitAction.action (rmsa_env.py:840-874, rwa_env.py:505-536): the agent names a path, the
// wrapper picks the first-fit slot / wavelength on it.  RMSA scans range(0, S - n): the last feasible start
// is never tried (SURVEY.md App. B-5); RWA scans range(W).  Anything else becomes the reject action (k, S).
template <int NWV>
__global__ void path_only_first_fit_kernel(const Params p, const int *path_actions, int *actions) {
    const int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= p.n) return;
    const int a = path_actions[env];
    int ap = p.k, as = p.S;
    if (a >= 0 && a < p.k) {
        const uint2 rq = p.cur_req[env];
        const int src = rq.x & 0xff, dst = (rq.x >> 8) & 0xff, br = (int)(rq.x >> 16);
        const int pair = src * p.N + dst;
        if (a < (int)p.pair_count[pair]) {
            const int row = p.pair_first[pair] + a;
            const WBits<NWV> A = wide_path_free<NWV>(p, env, row, 0);
            int s;
            if (p.kind == ORLG_RWA) {
                s = bits_ffs(A);
            } else {
                const int n = wide_nslots(p, meta_se(p.path_meta[row]), br);
                WBits<NWV> B = bits_runs_ge(A, n);
                const WBits<NWV> lim = bits_range<NWV>(0, max(p.S - n, 0));
#pragma unroll
                for (int i = 0; i < 4 * NWV; i++) B.w[i] &= lim.w[i];
                s = bits_ffs(B);
            }
            if (s >= 0) { ap = a; as = s; }
        }
    }
    actions[2 * env] = ap;
    actions[2 * env + 1] = as;
}

// SimpleMatrixObservation.observation (rmsa_env.py:806-837, rmcsa_env.py:914-947):
// [one-hot(min(src_id, dst_id)) | one-hot(max(src_id, dst_id)) | available_slots flattened (core, link, slot)]
// as bytes; consecutive threads write consecutive bytes of one env's row.
__global__ void matrix_observation_kernel(const Params p, unsigned char *out) {
    const int CE = p.C * p.E;
    const long long D = 2LL * p.N + (long long)CE * p.S;
    const long long total = D * p.n;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
        const int env = (int)(idx / D);
        const int pos = (int)(idx - (long long)env * D);
        unsigned char v;
        if (pos < 2 * p.N) {
            const uint2 rq = p.cur_req[env];
            const int src = rq.x & 0xff, dst = (rq.x >> 8) & 0xff;
            v = pos < p.N ? (pos == min(src, dst)) : (pos - p.N == max(src, dst));
        } else {
            const int cell = pos - 2 * p.N;
            const int l = cell / p.S, s = cell - l * p.S;
            const uint4 m = p.masks[mask_index(p, l, s >> 7, env)];
            const int w = (s >> 5) & 3;
            const unsigned word = w == 0 ? m.x : (w == 1 ? m.y : (w == 2 ? m.z : m.w));
            v = (word >> (s & 31)) & 1u;
        }
        out[idx] = v;
    }
}

// The same observation packed as bits (RMSA-v0 / RWA-v0: one core), what the MATRIX policy instances read: uint32 [n, W] with
// W = 4 + 4 nwv E.  Word 0 = min(src, dst) | max(src, dst) << 8 (the two one-hot positions), words 1..3 = 0; then link l's mask
// words in link order, word 4 + 4 nwv l + 4 v + w = word w of its 128-bit group v (bit b = slot 128 v + 32 w + b; bits at and
// above S are 0, as in the masks).  One thread per word, through mask_index: either mask layout.  Launched as a programmatic
// dependent launch whose threads all wait first, so it may sit between a step kernel and a policy kernel that waits on it only.
__global__ void matrix_observation_packed_kernel(const Params p, unsigned *out) {
    pdl_launch_dependents();
    pdl_wait();
    const int W = 4 + 4 * p.nwv * p.E;
    const long long total = (long long)W * p.n;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
        const int env = (int)(idx / W);
        const int w = (int)(idx - (long long)env * W);
        unsigned v = 0u;
        if (w == 0) {
            const uint2 rq = p.cur_req[env];
            const unsigned src = rq.x & 0xffu, dst = (rq.x >> 8) & 0xffu;
            v = min(src, dst) | max(src, dst) << 8;
        } else if (w >= 4) {
            const int q = w - 4, l = q / (4 * p.nwv), r = q - l * 4 * p.nwv;
            const uint4 m = p.masks[mask_index(p, l, r >> 2, env)];
            v = (r & 3) == 0 ? m.x : ((r & 3) == 1 ? m.y : ((r & 3) == 2 ? m.z : m.w));
        }
        out[idx] = v;
    }
}

}  // namespace orlg
