// Microbenchmark: throughput and latency of the bit-scan instructions (FLO = clz, BREV, POPC, and __ffs = BREV + FLO) against
// LOP3, the full-rate logic op they compete with for issue slots in the rollout kernel's dependent chains.
//   throughput: one CTA of 1024 threads per SM, 8 independent chains per thread; ops per cycle and SM from clock64 inside the
//               CTA (slowest warp of the CTA), so the figure does not depend on the clock the card runs at;
//   latency:    one thread, one dependent chain; cycles per op from clock64.
// nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o bitscan tools/micro/bitscan.cu && ./bitscan
#include <cstdio>
#include <cuda_runtime.h>

enum { OP_LOP3 = 0, OP_POPC = 1, OP_FLO = 2, OP_BREV = 3, OP_FFS = 4, N_OPS = 5 };
static const char *OP_NAME[N_OPS] = {"LOP3", "POPC", "FLO (clz)", "BREV", "ffs (BREV+FLO)"};

// inline PTX so that no op can be folded away or merged with its neighbour
template <int OP>
__device__ __forceinline__ unsigned op(unsigned x, unsigned c) {
    unsigned r;
    if (OP == OP_LOP3) asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(r) : "r"(x), "r"(c), "r"(c ^ 0x5bd1e995u));
    if (OP == OP_POPC) asm("popc.b32 %0, %1;" : "=r"(r) : "r"(x));
    if (OP == OP_FLO) asm("clz.b32 %0, %1;" : "=r"(r) : "r"(x));
    if (OP == OP_BREV) asm("brev.b32 %0, %1;" : "=r"(r) : "r"(x));
    if (OP == OP_FFS) r = (unsigned)__ffs((int)x);
    return r;
}

constexpr int CHAINS = 8;

template <int OP>
__global__ void __launch_bounds__(1024, 1) throughput(unsigned *out, unsigned long long *cycles, int iters, unsigned c) {
    unsigned x[CHAINS];
#pragma unroll
    for (int i = 0; i < CHAINS; i++) x[i] = threadIdx.x * 0x9E3779B9u + (unsigned)i * 0x85EBCA6Bu + c;
    __syncthreads();
    const long long t0 = clock64();
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
#pragma unroll
            for (int i = 0; i < CHAINS; i++) x[i] = op<OP>(x[i], c);
        }
    }
    __syncthreads();
    const long long t1 = clock64();
    unsigned acc = 0;
#pragma unroll
    for (int i = 0; i < CHAINS; i++) acc ^= x[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
    if (threadIdx.x == 0) cycles[blockIdx.x] = (unsigned long long)(t1 - t0);
}

template <int OP>
__global__ void latency(unsigned *out, unsigned long long *cycles, int iters, unsigned c) {
    unsigned x = threadIdx.x + c;
    const long long t0 = clock64();
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 16; u++) x = op<OP>(x, c);
    }
    const long long t1 = clock64();
    out[0] = x;
    cycles[0] = (unsigned long long)(t1 - t0);
}

#define CK(x)                                                                                  \
    do {                                                                                       \
        cudaError_t e_ = (x);                                                                  \
        if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); return 1; } \
    } while (0)

template <int OP>
int run(int sms, unsigned *out, unsigned long long *cyc, unsigned long long *hcyc) {
    const int t_iters = 4096, l_iters = 4096;
    for (int w = 0; w < 2; w++) throughput<OP><<<sms, 1024>>>(out, cyc, t_iters, 7u);        // warm-up, then the timed launch
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(hcyc, cyc, sizeof(unsigned long long) * sms, cudaMemcpyDeviceToHost));
    double mean = 0;
    for (int b = 0; b < sms; b++) mean += (double)hcyc[b] / sms;
    const double ops = 1024.0 * CHAINS * 4 * t_iters;
    for (int w = 0; w < 2; w++) latency<OP><<<1, 1>>>(out, cyc, l_iters, 7u);
    CK(cudaDeviceSynchronize());
    unsigned long long lc = 0;
    CK(cudaMemcpy(&lc, cyc, sizeof(lc), cudaMemcpyDeviceToHost));
    printf("%-16s throughput %6.1f ops/cycle/SM   latency %5.2f cycles (dependent chain, loop overhead included)\n", OP_NAME[OP],
           ops / mean, (double)lc / (16.0 * l_iters));
    return 0;
}

int main() {
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    const int sms = prop.multiProcessorCount;
    printf("%s, %d SMs\n", prop.name, sms);
    unsigned *out;
    unsigned long long *cyc, *hcyc = new unsigned long long[sms];
    CK(cudaMalloc(&out, sizeof(unsigned) * 1024 * sms));
    CK(cudaMalloc(&cyc, sizeof(unsigned long long) * sms));
    int rc = run<OP_LOP3>(sms, out, cyc, hcyc);
    if (!rc) rc = run<OP_POPC>(sms, out, cyc, hcyc);
    if (!rc) rc = run<OP_FLO>(sms, out, cyc, hcyc);
    if (!rc) rc = run<OP_BREV>(sms, out, cyc, hcyc);
    if (!rc) rc = run<OP_FFS>(sms, out, cyc, hcyc);
    cudaFree(out);
    cudaFree(cyc);
    delete[] hcyc;
    return rc;
}
