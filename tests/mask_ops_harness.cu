// mask_ops_harness.cu -- test harness of the slot-mask operations (orlg_device.cuh, link_shape in orlg_kernels.cuh).
//
// Built by tests/test_wide_limits.py into a temporary directory and loaded with ctypes; it is not part of the library.  One
// extern "C" launcher per word-group count V = 1..4 runs every operation on a batch of V x 128-bit masks (thread per mask) and
// writes the results to device buffers that the test compares with a numpy restatement on boolean arrays.
#include "orlg_kernels.cuh"

using namespace orlg;

namespace {

// device outputs, all [M][...] row-major
struct MaskOpsOut {
    uint32_t *runs_ge;        // [M][NR][4V]: bits_runs_ge(a, n) for n = 1..NR
    int *run_len;             // [M][128V]: bits_run_length(a, s) where bit s is set, else -1
    int *scalars;             // [M][4]: bits_longest_run, bits_ffs, bits_fls, bits_popc
    uint32_t *clear_lowest;   // [M][4V]
    uint32_t *shr;            // [M][32][4V]: bits_shr_small(a, s) for s = 0..31
    uint32_t *shl1;           // [M][4V]
    int *contains;            // [M][2]: bits_contains(a, a & b), bits_contains(a, b) with b = mask (i + 1) % M
    int *shape;               // [M][7]: link_shape(a, S[i]) free_cnt, used_runs, span, free_runs_in, free_runs, longest_free,
                              //         free_at_both_ends
};

template <int V>
__device__ WBits<V> load(const uint32_t *in, int i) {
    WBits<V> a;
    for (int w = 0; w < 4 * V; w++) a.w[w] = in[(size_t)i * 4 * V + w];
    return a;
}
template <int V>
__device__ void store(uint32_t *out, size_t row, const WBits<V> &a) {
    for (int w = 0; w < 4 * V; w++) out[row * 4 * V + w] = a.w[w];
}

template <int V>
__global__ void mask_ops_kernel(const uint32_t *in, const int *S, int M, int NR, MaskOpsOut o) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const WBits<V> a = load<V>(in, i), b = load<V>(in, (i + 1) % M);
    for (int n = 1; n <= NR; n++) store(o.runs_ge, (size_t)i * NR + n - 1, bits_runs_ge(a, n));
    for (int s = 0; s < 128 * V; s++)
        o.run_len[(size_t)i * 128 * V + s] = (a.w[s >> 5] >> (s & 31)) & 1u ? bits_run_length(a, s) : -1;
    int *sc = o.scalars + (size_t)i * 4;
    sc[0] = bits_longest_run(a); sc[1] = bits_ffs(a); sc[2] = bits_fls(a); sc[3] = bits_popc(a);
    store(o.clear_lowest, i, bits_clear_lowest(a));
    for (int s = 0; s < 32; s++) store(o.shr, (size_t)i * 32 + s, bits_shr_small(a, s));
    store(o.shl1, i, bits_shl1(a));
    o.contains[2 * (size_t)i] = bits_contains(a, bits_and(a, b));
    o.contains[2 * (size_t)i + 1] = bits_contains(a, b);
    const LinkShape r = link_shape(a, S[i]);
    int *sh = o.shape + (size_t)i * 7;
    sh[0] = r.free_cnt; sh[1] = r.used_runs; sh[2] = r.span; sh[3] = r.free_runs_in;
    sh[4] = r.free_runs; sh[5] = r.longest_free; sh[6] = r.free_at_both_ends;
}

// bits_range<V>(lo, hi) for every pair
template <int V>
__global__ void range_kernel(const int *lohi, int P, uint32_t *out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    store(out, i, bits_range<V>(lohi[2 * i], lohi[2 * i + 1]));
}

// the shift schedule of bits_runs_ge_sched for run length nn, by the rule orlg_api.cu builds its table with (n <= 16)
__device__ unsigned doubling_schedule(int nn) {
    unsigned sched = 0;
    int len = 1;
    for (int it = 0; it < 4; it++) {
        int sh = len < nn - len ? len : nn - len;
        if (sh < 0) sh = 0;
        sched |= (unsigned)sh << (8 * it);
        len += sh;
    }
    return sched;
}

// the 128-bit variants: bits_runs_ge_flat / bits_runs_ge_sched for n = 1..16 ([M][16][4] each), bits_ffs_flat ([M])
__global__ void variants_kernel(const uint32_t *in, int M, uint32_t *flat, uint32_t *sched, int *ffs_flat) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const Bits a = load<1>(in, i);
    for (int n = 1; n <= 16; n++) {
        store(flat, (size_t)i * 16 + n - 1, bits_runs_ge_flat(a, n));
        store(sched, (size_t)i * 16 + n - 1, bits_runs_ge_sched(a, doubling_schedule(n)));
    }
    ffs_flat[i] = bits_ffs_flat(a);
}

// bits_range_short (n <= 32) and bits_range_auto for every (start, n) pair; short_out rows with n > 32 are left alone
__global__ void range_variants_kernel(const int *sn, int P, uint32_t *short_out, uint32_t *auto_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const int start = sn[2 * i], n = sn[2 * i + 1];
    if (n <= 32) store(short_out, i, bits_range_short(start, n));
    store(auto_out, i, bits_range_auto(start, n));
}

int finish() {
    const cudaError_t e = cudaDeviceSynchronize();
    return e == cudaSuccess ? (int)cudaGetLastError() : (int)e;
}

int blocks(int n) { return (n + 127) / 128; }

template <int V>
int mask_ops(const uint32_t *in, const int *S, int M, int NR, uint32_t *runs_ge, int *run_len, int *scalars, uint32_t *clear_lowest,
             uint32_t *shr, uint32_t *shl1, int *contains, int *shape) {
    const MaskOpsOut o = {runs_ge, run_len, scalars, clear_lowest, shr, shl1, contains, shape};
    mask_ops_kernel<V><<<blocks(M), 128>>>(in, S, M, NR, o);
    return finish();
}

template <int V>
int mask_range(const int *lohi, int P, uint32_t *out) {
    range_kernel<V><<<blocks(P), 128>>>(lohi, P, out);
    return finish();
}

}  // namespace

#define MASK_OPS_ENTRY(V)                                                                                                       \
    extern "C" int mask_ops_v##V(const uint32_t *in, const int *S, int M, int NR, uint32_t *runs_ge, int *run_len, int *scalars, \
                                 uint32_t *clear_lowest, uint32_t *shr, uint32_t *shl1, int *contains, int *shape) {            \
        return mask_ops<V>(in, S, M, NR, runs_ge, run_len, scalars, clear_lowest, shr, shl1, contains, shape);                 \
    }                                                                                                                           \
    extern "C" int mask_range_v##V(const int *lohi, int P, uint32_t *out) { return mask_range<V>(lohi, P, out); }
MASK_OPS_ENTRY(1)
MASK_OPS_ENTRY(2)
MASK_OPS_ENTRY(3)
MASK_OPS_ENTRY(4)

extern "C" int mask_variants_v1(const uint32_t *in, int M, uint32_t *flat, uint32_t *sched, int *ffs_flat) {
    variants_kernel<<<blocks(M), 128>>>(in, M, flat, sched, ffs_flat);
    return finish();
}

extern "C" int mask_range_variants_v1(const int *sn, int P, uint32_t *short_out, uint32_t *auto_out) {
    range_variants_kernel<<<blocks(P), 128>>>(sn, P, short_out, auto_out);
    return finish();
}
