// orlg_api.cu -- the C ABI (include/orlg.h) on top of the step kernels.  Links cudart only.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <emmintrin.h>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "orlg_deeprmsa_fast.cuh"
#include "orlg_rollout.cuh"
#include "orlg_policy.cuh"
#include "orlg_step_wide.cuh"
#include "orlg_wrappers.cuh"

using namespace orlg;

static thread_local std::string g_err;

static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

#define CUDA_OK(call)                                                                        \
    do {                                                                                     \
        cudaError_t e_ = (call);                                                             \
        if (e_ != cudaSuccess)                                                               \
            return fail(ORLG_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));    \
    } while (0)

constexpr int RO_HOST_BUFFERS = 3;       // orlg_rollout_host: record buffers in flight (device runs two chunks ahead of the decoder)

namespace {
// orlg_rollout_host: packed records on the device and in pinned host memory, the copy stream with its events, and the device
// copies of replayed action chunks.  Allocated by the first call, grown by later calls that need more rows.
struct HostPipeline {
    uint4 *pk_dev[RO_HOST_BUFFERS] = {};
    uint4 *pk_host[RO_HOST_BUFFERS] = {};
    size_t pk_rows = 0;                        // rows (env-steps) each buffer holds
    cudaEvent_t pk_ev[RO_HOST_BUFFERS] = {};   // records of the chunk are in pinned host memory (copy stream)
    cudaEvent_t k_ev[RO_HOST_BUFFERS] = {};    // the chunk's kernel is done (user stream)
    cudaStream_t copy_stream = nullptr;        // D2H of chunk c overlaps the kernel of chunk c + 1
    int32_t *act_dev[RO_HOST_BUFFERS] = {};    // ORLG_POLICY_REPLAY: the host's action chunks on the device
    size_t act_rows = 0;

    int reserve(size_t rows, bool replay, size_t action_dim) {
        if (pk_rows < rows) {                  // (re)allocate the record buffers (device + pinned host)
            for (int i = 0; i < RO_HOST_BUFFERS; i++) {
                if (pk_dev[i]) cudaFree(pk_dev[i]);
                if (pk_host[i]) cudaFreeHost(pk_host[i]);
                pk_dev[i] = nullptr; pk_host[i] = nullptr;
                if (cudaMalloc(&pk_dev[i], rows * 32) != cudaSuccess) return fail(ORLG_E_NOMEM, "cudaMalloc (packed records) failed");
                if (cudaHostAlloc(&pk_host[i], rows * 32, cudaHostAllocDefault) != cudaSuccess) return fail(ORLG_E_NOMEM, "cudaHostAlloc (packed records) failed");
                if (!pk_ev[i]) CUDA_OK(cudaEventCreateWithFlags(&pk_ev[i], cudaEventDisableTiming));
                if (!k_ev[i]) CUDA_OK(cudaEventCreateWithFlags(&k_ev[i], cudaEventDisableTiming));
            }
            pk_rows = rows;
        }
        if (!copy_stream) CUDA_OK(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
        if (replay && act_rows < rows) {       // device copies of the action chunks
            for (int i = 0; i < RO_HOST_BUFFERS; i++) {
                if (act_dev[i]) cudaFree(act_dev[i]);
                act_dev[i] = nullptr;
                if (cudaMalloc(&act_dev[i], rows * action_dim * sizeof(int32_t)) != cudaSuccess) return fail(ORLG_E_NOMEM, "cudaMalloc (action chunks) failed");
            }
            act_rows = rows;
        }
        return ORLG_OK;
    }
    ~HostPipeline() {
        for (int i = 0; i < RO_HOST_BUFFERS; i++) {
            if (pk_dev[i]) cudaFree(pk_dev[i]);
            if (pk_host[i]) cudaFreeHost(pk_host[i]);
            if (pk_ev[i]) cudaEventDestroy(pk_ev[i]);
            if (k_ev[i]) cudaEventDestroy(k_ev[i]);
            if (act_dev[i]) cudaFree(act_dev[i]);
        }
        if (copy_stream) cudaStreamDestroy(copy_stream);
    }
};
}  // namespace

// Owns every device resource of a handle.  Deleted on the handle's device (orlg_destroy).
struct orlg_env {
    Params p;
    orlg_config cfg;
    int device;
    bool fast = false;            // DeepRMSA fast kernel applicable (NSFNET-class: 22 links, k <= 5)
    bool hot = false;             // ... and its steady-state specialisation qualifies (hot_launch)
    bool ro_ok = false;           // the persistent rollout kernel qualifies (rollout_kernel_applies)
    int ro_lpw;                   // envs per warp of the rollout kernel (8 or 32): fixed per handle, the event slabs follow it
    bool ro_last_persistent = false;   // the last orlg_rollout* call ran the persistent kernel (orlg_kernel_info)
    CUtensorMap mask_map;         // TMA view of the mask tensor: [C*E rows][n x 16 bytes], box = E rows x 512 bytes
    bool wide;                    // beyond 32 links / 128 slots / 8 paths: CSR link lists, multi-word masks
    size_t fast_smem;
    int64_t state_bytes = 0;
    std::vector<void *> allocs;
    // the per-environment STATE arrays among them (orlg_state_save / orlg_state_load), in allocation order
    std::vector<std::pair<void *, size_t>> state_allocs;
    bool alloc_is_state = false;
    // T-steps-per-launch rollout path (orlg_rollout.cuh): window / scratch buffers, allocated by the first call
    WinEntry *ro_ev = nullptr;
    unsigned *ro_st_u32 = nullptr;             // [4][n] table size, window head, window end, canonical size
    double *ro_st_f64 = nullptr;               // [2 + RO_SIDE][n] table minimum, horizon, side-buffer times
    unsigned long long *ro_st_u64 = nullptr;   // [RO_SIDE][n] side-buffer payloads
    bool ro_valid = false;                     // the events live in the rollout-private storage (canonical tables are stale)
    HostPipeline host_pipe;
    int *ro_actions = nullptr;    // [n, action_dim] scratch of the generic (kernel-per-step) rollout

    ~orlg_env() { for (void *ptr : allocs) cudaFree(ptr); }
};

namespace {

// every entry point runs on the handle's device whatever the caller's current device is (and puts it back)
struct DeviceGuard {
    int prev = -1;
    bool changed = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (changed) cudaSetDevice(prev); }
};

template <typename T>
int dev_alloc(orlg_env *env, T **out, size_t count, bool zero = true) {
    void *ptr = nullptr;
    size_t bytes = sizeof(T) * (count ? count : 1);
    if (cudaMalloc(&ptr, bytes) != cudaSuccess) return fail(ORLG_E_NOMEM, "cudaMalloc failed for " + std::to_string(bytes) + " bytes");
    env->allocs.push_back(ptr);
    if (zero && cudaMemset(ptr, 0, bytes) != cudaSuccess) return fail(ORLG_E_CUDA, "cudaMemset failed");
    if (env->alloc_is_state) env->state_allocs.emplace_back(ptr, bytes);
    env->state_bytes += (int64_t)bytes;
    *out = reinterpret_cast<T *>(ptr);
    return ORLG_OK;
}

template <typename T>
int dev_upload(orlg_env *env, const T **out, const std::vector<T> &host) {
    T *ptr = nullptr;
    int rc = dev_alloc(env, &ptr, host.size(), false);
    if (rc) return rc;
    if (!host.empty() && cudaMemcpy(ptr, host.data(), sizeof(T) * host.size(), cudaMemcpyHostToDevice) != cudaSuccess)
        return fail(ORLG_E_CUDA, "cudaMemcpy (table upload) failed");
    *out = ptr;
    return ORLG_OK;
}

// integer CDF thresholds of the Philox node / bit-rate draws (DESIGN.md "Traffic")
std::vector<unsigned> thresholds(const double *prob, int n) {
    std::vector<unsigned> thr(n);
    double tot = 0.0, acc = 0.0;
    for (int i = 0; i < n; i++) tot += prob[i];
    for (int i = 0; i < n; i++) {
        acc += prob[i];
        double v = std::floor(acc / tot * 4294967296.0 + 0.5);
        if (v > 4294967295.0) v = 4294967295.0;
        thr[i] = (unsigned)v;
    }
    thr[n - 1] = 4294967295u;
    return thr;
}

// rmcsa_env.py:341-384: longest reach (km) of a modulation at a bit rate = min(lmax_snr, lmax_xt)
double reach_km(double osnr, double inband_xt_raw, int se, int bit_rate, double worst_xt_raw) {
    double average_power = 1, nf_db = 5.5;
    double nf = std::pow(10.0, nf_db / 10.0);
    double amp_spam = 100, amp_gain_db = 20;
    double amp_gain = std::pow(10.0, amp_gain_db / 10.0);
    double lambda_ = 1550, h = 6.626068e-34;
    double f_hz = 2.99e8 / (lambda_ * 1e-9);
    double inband_xt = inband_xt_raw + 4;        // rmcsa_env.py:127-129 (+4 dB margins)
    double worst_xt = worst_xt_raw + 4;
    double snr_min = std::pow(10.0, (osnr + 2) / 10);
    double lmax_snr = (average_power * amp_spam) /
                      (snr_min * h * f_hz * amp_gain * nf * ((double)bit_rate / (double)se) * 1e9);
    lmax_snr = lmax_snr / 1000;
    double lmax_xt = std::pow(10.0, (inband_xt - worst_xt - 4) / 10);
    return lmax_snr < lmax_xt ? lmax_snr : lmax_xt;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no libcuda link dependency)
bool encode_mask_map(orlg_env *env) {
    typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
        qres != cudaDriverEntryPointSuccess)
        return false;
    const Params &p = env->p;
    const cuuint64_t gdim[2] = {(cuuint64_t)p.n * 4, (cuuint64_t)p.C * p.E};        // uint32 elements per row, rows
    const cuuint64_t gstride[1] = {(cuuint64_t)p.n * 16};                           // bytes between rows
    const cuuint32_t box[2] = {128, (cuuint32_t)p.E};                               // 32 envs x 16 B, all links
    const cuuint32_t estr[2] = {1, 1};
    return reinterpret_cast<encode_fn>(fn)(&env->mask_map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, p.masks, gdim, gstride, box, estr,
                                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                           CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

size_t step_obs_smem(const Params &p) { return (size_t)STEP_THREADS * p.obs_dim * (p.obs_f64 ? 8 : 4); }

template <int KIND>
void launch_step_kind(const orlg_env *env, const StepIO &io, int mode, cudaStream_t s) {
    const int blocks = (env->p.n + STEP_THREADS - 1) / STEP_THREADS;
    const size_t smem = (KIND == ORLG_DEEPRMSA && io.obs) ? step_obs_smem(env->p) : 0;
    if (env->p.k <= 5) step_kernel<KIND, 5><<<blocks, STEP_THREADS, smem, s>>>(env->p, io, mode);
    else step_kernel<KIND, KMAX><<<blocks, STEP_THREADS, smem, s>>>(env->p, io, mode);
}

// launch configuration with the programmatic-stream-serialization attribute (griddepcontrol in the kernels)
cudaLaunchConfig_t pdl_config(int blocks, int threads, size_t smem, cudaStream_t s) {
    static thread_local cudaLaunchAttribute g_pdl_attr[1];          // one host thread per handle (orlg.h)
    g_pdl_attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    g_pdl_attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cfg.attrs = g_pdl_attr;
    cfg.numAttrs = 1;
    return cfg;
}

// ---- kernel-instance decisions: each is made here and nowhere else

// f(std::integral_constant<int, KIND>()) for the env kind
template <typename F>
void for_kind(int kind, F &&f) {
    switch (kind) {
    case ORLG_RWA: f(std::integral_constant<int, ORLG_RWA>()); break;
    case ORLG_RMSA: f(std::integral_constant<int, ORLG_RMSA>()); break;
    case ORLG_DEEPRMSA: f(std::integral_constant<int, ORLG_DEEPRMSA>()); break;
    default: f(std::integral_constant<int, ORLG_RMCSA>()); break;
    }
}

// f(std::integral_constant<int, W>()) for the 128-slot mask words per (core, link) of the wide kernels
template <typename F>
void for_words(int nwv, F &&f) {
    switch (nwv) {
    case 1: f(std::integral_constant<int, 1>()); break;
    case 2: f(std::integral_constant<int, 2>()); break;
    case 3: f(std::integral_constant<int, 3>()); break;
    default: f(std::integral_constant<int, 4>()); break;
    }
}

// link-count template of the fast and rollout kernels: 22 (NSFNET) is compiled in, 0 reads the link count at run time
int link_template(const orlg_env *env) { return !env->wide && env->p.E == 22 ? 22 : 0; }

// the steady-state instance (HOT = true) of the fast kernel runs for this launch: the handle qualifies (orlg_create) and the
// launch is a float32 Philox step that writes observation, reward and done and nothing else
bool hot_launch(const orlg_env *env, const StepIO &io, int mode) {
    return env->hot && env->p.J == 1 && !env->p.obs_f64 && mode == MODE_STEP && env->p.traffic == ORLG_TRAFFIC_PHILOX &&
           io.obs && io.reward && io.done && !io.decision && !io.obs_int;
}

// nullptr when the env kind has heuristic `which`, else why it is refused
constexpr const char *heuristic_refusal(int kind, int which) {
    return kind == ORLG_RMSA && which == ORLG_HEUR_SAP_LF         ? "last-fit exists for RWA only"
           : kind == ORLG_DEEPRMSA && which > ORLG_HEUR_SAP_FF ? "DeepRMSA has SP-FF and SAP-FF only"
                                                                : nullptr;
}

// the persistent rollout kernel runs this policy on this handle (given a shared-memory plan, rollout_plan); it writes the
// counters of info but not the RWA action probabilities (about 90 doubles per env-step): a call that wants them steps
bool rollout_kernel_applies(const orlg_env *env, int policy, const orlg_info_out *info) {
    const Params &p = env->p;
    const bool policy_ok = p.traffic == ORLG_TRAFFIC_TRACE ? policy == ORLG_POLICY_REPLAY
                           : policy == ORLG_POLICY_RANDOM || policy == ORLG_POLICY_REPLAY || !heuristic_refusal(p.kind, policy);
    return env->ro_ok && !p.stats && !p.obs_f64 && !p.br_hist && !(info && info->action_probability_dev) && policy_ok;
}

// refusals of the float entries of info, shared by the per-step entry points and the rollouts that keep every step's info
constexpr const char *NO_STATS_INFO = "info has float statistics only after orlg_enable_stats (RMSA-v0 / DeepRMSA-v0)";
constexpr const char *NO_BIT_RATES = "per-bit-rate statistics exist for RMSA-v0 with bit_rate_selection='discrete'";
constexpr const char *NO_ACTION_HIST = "action probabilities are part of info for RWA-v0 only (rwa_env.py:148-151)";

// nullptr when the handle has every output `info` asks for, else why it is refused
const char *info_refusal(const Params &p, const orlg_info_out *info) {
    if (!info) return nullptr;
    if (info->stats_dev && !p.stats_out) return NO_STATS_INFO;
    if (info->bit_rate_blocking_dev && !p.br_hist) return NO_BIT_RATES;
    if (info->action_probability_dev && !p.act_hist) return NO_ACTION_HIST;
    return nullptr;
}

// the fast-kernel instances launch_fast picks from, [j != 1][float64 obs][link template 0] then HOT [link template 0]
using FastKernel = void (*)(Params, StepIO, int, CUtensorMap);
const FastKernel FAST_KERNELS[] = {
    deeprmsa_fast_kernel<22, 5, 1, false>, deeprmsa_fast_kernel<0, 5, 1, false>, deeprmsa_fast_kernel<22, 5, 1, true>, deeprmsa_fast_kernel<0, 5, 1, true>,
    deeprmsa_fast_kernel<22, 5, 0, false>, deeprmsa_fast_kernel<0, 5, 0, false>, deeprmsa_fast_kernel<22, 5, 0, true>, deeprmsa_fast_kernel<0, 5, 0, true>,
    deeprmsa_fast_kernel<22, 5, 1, false, true>, deeprmsa_fast_kernel<0, 5, 1, false, true>};

void launch_fast(const orlg_env *env, const StepIO &io, int mode, cudaStream_t s) {
    const int blocks = (env->p.n + FAST_THREADS - 1) / FAST_THREADS;
    const bool hot = hot_launch(env, io, mode);
    const int et = link_template(env) == 22 ? 0 : 1;
    const FastKernel kernel = FAST_KERNELS[hot ? 8 + et : (env->p.J == 1 ? 0 : 4) + (env->p.obs_f64 ? 2 : 0) + et];
    if (hot) {
        // programmatic dependent launch: the prologue overlaps the tail of the preceding kernel of the stream
        cudaLaunchConfig_t cfg = pdl_config(blocks, FAST_THREADS, env->fast_smem, s);
        cudaLaunchKernelEx(&cfg, kernel, env->p, io, mode, env->mask_map);
        return;
    }
    kernel<<<blocks, FAST_THREADS, env->fast_smem, s>>>(env->p, io, mode, env->mask_map);
}

int launch_step(const orlg_env *env, const StepIO &io, int mode, cudaStream_t s) {
    const Params &p = env->p;
    if (env->wide) {
        const int blocks = (p.n + ORLG_WIDE_THREADS - 1) / ORLG_WIDE_THREADS;
        for_kind(p.kind, [&](auto K) { for_words(p.nwv, [&](auto W) {
            constexpr int KIND = decltype(K)::value, NWV = decltype(W)::value;
            if (p.stats) step_wide_kernel<KIND, NWV, true><<<blocks, ORLG_WIDE_THREADS, 0, s>>>(p, io, mode);
            else step_wide_kernel<KIND, NWV, false><<<blocks, ORLG_WIDE_THREADS, 0, s>>>(p, io, mode); }); });
    } else if (env->fast && !p.stats) launch_fast(env, io, mode, s);
    else for_kind(p.kind, [&](auto K) { launch_step_kind<decltype(K)::value>(env, io, mode, s); });
    CUDA_OK(cudaGetLastError());
    return ORLG_OK;
}

// envs per warp of the rollout kernel: a batch that would leave most SMs with one or two warps is spread over more warps
// with fewer lanes in use (less divergence per warp, more warps to hide latency).  Chosen by orlg_create (ORLG_RO_LPW = 8 or
// 32 overrides it for the handles created while it is set) and fixed per handle: the event slabs follow it.
int choose_rollout_lpw(int n) {
    const char *v = std::getenv("ORLG_RO_LPW");
    const int w = v ? std::atoi(v) : 0;
    if (w == 8 || w == 32) return w;
    return n >= 16384 ? 32 : 8;
}

void rollout_state_args(const orlg_env *env, RolloutArgs *ra) {
    const size_t n = (size_t)env->p.n;
    ra->lpw = env->ro_lpw;
    ra->ev = env->ro_ev;
    ra->st_ntab = env->ro_st_u32; ra->st_wh = env->ro_st_u32 + n; ra->st_wn = env->ro_st_u32 + 2 * n; ra->st_ncanon = env->ro_st_u32 + 3 * n;
    ra->st_tmin = env->ro_st_f64; ra->st_hzn = env->ro_st_f64 + n; ra->st_side_t = env->ro_st_f64 + 2 * n;
    ra->st_side_p = env->ro_st_u64;
}

// Every entry point that reads or writes the release-event tables calls this first: after an orlg_rollout the events live in
// the rollout kernel's private storage until somebody else needs them.
int ensure_canonical(orlg_env *env, cudaStream_t s) {
    if (!env->ro_valid) return ORLG_OK;
    RolloutArgs ra;
    std::memset(&ra, 0, sizeof(ra));
    rollout_state_args(env, &ra);
    ro_canonicalize_kernel<<<(env->p.n + 127) / 128, 128, 0, s>>>(env->p, ra);
    CUDA_OK(cudaGetLastError());
    env->ro_valid = false;
    return ORLG_OK;
}

// shared-memory plan of the rollout kernel: as many warps per CTA as cover the batch in one wave (<= 14), each with
// its mask tile + side buffer, plus a pool of observation tiles
bool rollout_plan(const orlg_env *env, int *wpc_out, RolloutArgs *ra, size_t *smem_out) {
    const Params &p = env->p;
    const int warps = (p.n + env->ro_lpw - 1) / env->ro_lpw;
    int wpc = (warps + 147) / 148;
    if (wpc > RO_MAX_THREADS / 32) wpc = RO_MAX_THREADS / 32;
    if (wpc < 1) wpc = 1;
    if (const char *v = std::getenv("ORLG_RO_WARPS")) { int w = std::atoi(v); if (w >= 1 && w <= RO_MAX_THREADS / 32) wpc = w; }
    const int tile = (32 * p.obs_dim * 4 + 127) / 128 * 128;
    const int warp_bytes = p.E * 512 + RO_SIDE * 512;
    const size_t budget = 227 * 1024;
    for (; wpc >= 1; wpc--) {
        const size_t fixed = (size_t)p.tab_vec * 16 + (size_t)wpc * warp_bytes + 16;
        if (fixed + tile > budget) continue;
        int tiles = tile > 0 ? (int)((budget - fixed) / tile) : 0;       // kinds without a tensor observation need no tile
        if (tiles > wpc) tiles = wpc;
        if (tiles > 32) tiles = 32;
        if (const char *v = std::getenv("ORLG_RO_TILES")) { int w = std::atoi(v); if (w >= 1 && w <= tiles) tiles = w; }
        ra->pool_tiles = tiles; ra->tile_bytes = tile; ra->warp_bytes = warp_bytes;
        *wpc_out = wpc;
        *smem_out = fixed + (size_t)tiles * tile;
        return true;
    }
    return false;
}

template <int ET, int KIND>
cudaError_t launch_rollout_kind(const orlg_env *env, const RolloutArgs &ra, int policy, int wpc, size_t smem, cudaStream_t s) {
    const int warps = (env->p.n + ra.lpw - 1) / ra.lpw;
    const int threads = wpc * 32, blocks = (warps + wpc - 1) / wpc;
    cudaLaunchConfig_t cfg = pdl_config(blocks, threads, smem, s);
    cudaError_t e = cudaErrorInvalidValue;
    const bool trace = env->p.traffic == ORLG_TRAFFIC_TRACE;
#define ORLG_RO_LAUNCH2(POL, TR, LP, INF)                                                                                \
    do {                                                                                                                 \
        e = cudaFuncSetAttribute(deeprmsa_rollout_kernel<ET, POL, TR, KIND, LP, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e == cudaSuccess) e = cudaLaunchKernelEx(&cfg, deeprmsa_rollout_kernel<ET, POL, TR, KIND, LP, INF>, env->p, ra); \
    } while (0)
#define ORLG_RO_LAUNCH1(POL, TR, LP) do { if (ra.info) ORLG_RO_LAUNCH2(POL, TR, LP, true); else ORLG_RO_LAUNCH2(POL, TR, LP, false); } while (0)
#define ORLG_RO_LAUNCH(POL, TR) do { if (ra.lpw == 32) ORLG_RO_LAUNCH1(POL, TR, 32); else ORLG_RO_LAUNCH1(POL, TR, 8); } while (0)
    if (policy == ORLG_POLICY_REPLAY) {
        if (trace) ORLG_RO_LAUNCH(RO_POLICY_REPLAY, true); else ORLG_RO_LAUNCH(RO_POLICY_REPLAY, false);
    } else if (trace) {
        return cudaErrorInvalidValue;                          // (filtered by the caller: trace traffic is replay-only here)
    } else if (policy == ORLG_POLICY_RANDOM) ORLG_RO_LAUNCH(RO_POLICY_RANDOM, false);
    else if (policy == ORLG_HEUR_SP_FF) ORLG_RO_LAUNCH(RO_POLICY_SP_FF, false);
    else if (policy == ORLG_HEUR_SAP_FF) ORLG_RO_LAUNCH(RO_POLICY_SAP_FF, false);
    else if (policy == ORLG_HEUR_LLP_FF) { if (!heuristic_refusal(KIND, ORLG_HEUR_LLP_FF)) ORLG_RO_LAUNCH(RO_POLICY_LLP_FF, false); }
    else if (policy == ORLG_HEUR_SAP_LF) { if (!heuristic_refusal(KIND, ORLG_HEUR_SAP_LF)) ORLG_RO_LAUNCH(RO_POLICY_SAP_LF, false); }
#undef ORLG_RO_LAUNCH
#undef ORLG_RO_LAUNCH1
#undef ORLG_RO_LAUNCH2
    return e;
}

template <int ET>
cudaError_t launch_rollout(const orlg_env *env, const RolloutArgs &ra, int policy, int wpc, size_t smem, cudaStream_t s) {
    switch (env->p.kind) {
    case ORLG_DEEPRMSA: return launch_rollout_kind<ET, ORLG_DEEPRMSA>(env, ra, policy, wpc, smem, s);
    case ORLG_RMSA: return launch_rollout_kind<ET, ORLG_RMSA>(env, ra, policy, wpc, smem, s);
    case ORLG_RWA: return launch_rollout_kind<ET, ORLG_RWA>(env, ra, policy, wpc, smem, s);
    default: return cudaErrorInvalidValue;
    }
}

int slots_needed(int bit_rate, int se, double channel_width) {   // get_number_slots (rmsa_env.py:610-621), same float expression
    return (int)std::ceil((double)bit_rate / ((double)se * channel_width)) + 1;
}

// Step 1.  Every refusal of a configuration, in a fixed order: an input with several faults is always refused for the same
// one.  Nothing is allocated; the device query is the only CUDA call.  Fills the scalar launch parameters, whether the wide
// kernels serve the handle, and the largest spectral efficiency (the extent of the slot-count tables).
int configure(const orlg_config &cfg, const orlg_tables &t, int device, Params &p, bool &wide, int &se_max) {
    if (cfg.kind < ORLG_RWA || cfg.kind > ORLG_RMCSA) return fail(ORLG_E_INVALID, "unknown env kind");
    if (cfg.num_envs <= 0) return fail(ORLG_E_INVALID, "num_envs must be positive");
    if (cfg.num_slots > 512 || cfg.num_slots <= 0) return fail(ORLG_E_UNSUPPORTED, "1..512 slots per link");
    if (t.num_links < 1 || t.num_links > 65535) return fail(ORLG_E_UNSUPPORTED, "1..65535 links");
    if (t.num_nodes > 255 || t.num_nodes < 2) return fail(ORLG_E_UNSUPPORTED, "2..255 nodes");
    if (t.k_paths > 16 || t.k_paths < 1) return fail(ORLG_E_UNSUPPORTED, "k_paths must be 1..16");
    if (t.num_paths >= (1 << 20)) return fail(ORLG_E_UNSUPPORTED, "too many paths");
    const int C = cfg.kind == ORLG_RMCSA ? cfg.num_cores : 1;
    if (C < 1 || C > 31) return fail(ORLG_E_UNSUPPORTED, "1..31 cores");
    const int J = cfg.kind == ORLG_DEEPRMSA ? cfg.j : 1;
    if (J < 1 || J > 16) return fail(ORLG_E_INVALID, "j must be 1..16");
    if (cfg.episode_length < 1 || cfg.episode_length >= (1 << 22)) return fail(ORLG_E_UNSUPPORTED, "episode_length must be < 2^22");
    if (!(cfg.mean_holding > 0) || !(cfg.mean_iat > 0)) return fail(ORLG_E_INVALID, "holding / inter-arrival times must be positive");
    if (cfg.kind != ORLG_RWA && t.num_bit_rates == 0 && cfg.bit_rate_hi < cfg.bit_rate_lo)
        return fail(ORLG_E_INVALID, "bit_rate_higher_bound < bit_rate_lower_bound");
    if (cfg.kind == ORLG_RMCSA && t.num_mods < 1) return fail(ORLG_E_INVALID, "RMCSA needs a modulation table");

    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev) return fail(ORLG_E_CUDA, "no such CUDA device");
    wide = t.num_links > 32 || cfg.num_slots > MAX_SLOTS || t.k_paths > KMAX;
    std::memset(&p, 0, sizeof(p));
    p.kind = cfg.kind; p.n = cfg.num_envs; p.N = t.num_nodes; p.E = t.num_links; p.C = C; p.S = cfg.num_slots;
    p.k = t.k_paths; p.J = J; p.M = t.num_mods;
    p.episode_length = cfg.episode_length; p.allow_rejection = cfg.allow_rejection ? 1 : 0;
    p.auto_reset = cfg.auto_reset ? 1 : 0; p.traffic = cfg.traffic; p.obs_f64 = cfg.obs_dtype == ORLG_OBS_F64;
    p.n_bit_rates = t.num_bit_rates;
    p.br_lo = cfg.bit_rate_lo; p.br_span = cfg.bit_rate_hi - cfg.bit_rate_lo + 1;
    int br_max = cfg.kind == ORLG_RWA ? 0 : (cfg.bit_rate_hi > 1023 ? cfg.bit_rate_hi : 1023);   // traces may carry any rate <= 1023
    for (int i = 0; i < t.num_bit_rates; i++) br_max = t.bit_rates[i] > br_max ? t.bit_rates[i] : br_max;
    if (br_max < 0 || br_max > 65535) return fail(ORLG_E_UNSUPPORTED, "bit rates must be 0..65535");
    p.br_max = br_max;
    p.seed = cfg.seed; p.env_id_base = cfg.env_id_base;
    p.mean_holding = cfg.mean_holding; p.mean_iat = cfg.mean_iat;
    p.obs_dim = cfg.kind == ORLG_DEEPRMSA ? 1 + 2 * p.N + (2 * J + 3) * p.k : 0;
    p.node_top_step = 1;                   // highest power of two <= N - 1: binary search over the node CDF
    while (p.node_top_step * 2 <= p.N - 1) p.node_top_step *= 2;
    p.cand_stride = ((p.k * J + 7) / 8) * 8;
    p.nwv = wide ? (p.S + 127) / 128 : 1;
    p.wstride = wide ? (p.nwv == 3 ? 4 : p.nwv) : 0;      // 3-word entries padded to 64 bytes: one DRAM burst per (env, core, link)
    if (step_obs_smem(p) > 200 * 1024) return fail(ORLG_E_UNSUPPORTED, "observation too large for the staging tile");

    // heap capacity: live services ~ Poisson(load) at most (M/M/inf bound); hard bound E*S*C/2 slots pairs
    int cap = cfg.heap_capacity;
    if (cap <= 0) {
        double load = cfg.mean_holding / cfg.mean_iat;
        double want = load + 8.0 * std::sqrt(load) + 16.0;
        double hard = cfg.kind == ORLG_RWA ? (double)p.E * p.S * C : (double)p.E * p.S * C / 2.0;
        cap = (int)std::ceil(want < hard ? want : hard);
    }
    cap = ((cap + EV_GROUP - 1) / EV_GROUP) * EV_GROUP;
    // up to 4096 live services per env (RWA's physical bound on NSFNET is E * W = 1760).  A derived capacity is capped
    // there (overflow is flagged per env, ORLG_ERR_HEAP_OVERFLOW); an explicit request beyond it is refused.
    if (cfg.heap_capacity > 256 * EV_GROUP) return fail(ORLG_E_UNSUPPORTED, "heap_capacity above 4096 live services per environment");
    if (cap > 256 * EV_GROUP) cap = 256 * EV_GROUP;
    p.ev_groups = ((cap / EV_GROUP + 15) / 16) * 16;
    p.heap_cap = cap;

    se_max = 1;
    for (int r = 0; r < t.num_paths; r++) {
        for (int h = t.path_link_ptr[r]; h < t.path_link_ptr[r + 1]; h++)
            if (t.path_links[h] < 0 || t.path_links[h] >= p.E) return fail(ORLG_E_INVALID, "path link index out of range");
        if (t.path_hops[r] > 255 || t.path_link_ptr[r + 1] - t.path_link_ptr[r] != t.path_hops[r]) return fail(ORLG_E_INVALID, "inconsistent path hop counts");
        se_max = t.path_se[r] > se_max ? t.path_se[r] : se_max;
    }
    for (int m = 0; m < t.num_mods; m++) se_max = t.mod_se[m] > se_max ? t.mod_se[m] : se_max;
    // slot counts are 8-bit table entries / payload fields: harmless above 200 only while 200 slots can never fit
    bool unrepresentable = false;
    auto check = [&](int b) {
        for (int se = 1; se <= se_max; se++) { const int n = slots_needed(b, se, cfg.channel_width); unrepresentable |= n > 200 && n <= p.S; }
    };
    if (cfg.kind != ORLG_RWA && t.num_bit_rates > 0) for (int i = 0; i < t.num_bit_rates; i++) check(t.bit_rates[i]);
    else if (cfg.kind != ORLG_RWA) for (int b = cfg.bit_rate_lo < 0 ? 0 : cfg.bit_rate_lo; b <= cfg.bit_rate_hi; b++) check(b);
    if (unrepresentable)
        return fail(ORLG_E_UNSUPPORTED, "a request of this configuration may need 201.." + std::to_string(p.S) + " slots: at most 200 slots per service are representable");
    return ORLG_OK;
}

// the host copies of the lookup tables that the fast-kernel blob and the instance selection read after the upload
struct HostTables {
    std::vector<int> pair_first;
    std::vector<unsigned char> pair_count, nslots;     // nslots: [se][bit rate]
    std::vector<unsigned> linkmask, meta, node_thr;
};

// Step 2.  The lookup tables (paths, slot counts, reach, traffic CDFs): built on the host, uploaded.
int upload_tables(orlg_env *env, const orlg_config &cfg, const orlg_tables &t, int se_max, HostTables &h) {
    Params &p = env->p;
    const int NN = p.N * p.N, P = t.num_paths, br_max = p.br_max;
    h.pair_first.assign(t.pair_first, t.pair_first + NN);
    h.pair_count.resize(NN);
    for (int i = 0; i < NN; i++) h.pair_count[i] = (unsigned char)(t.pair_count[i] < 0 ? 0 : (t.pair_count[i] > p.k ? p.k : t.pair_count[i]));
    h.linkmask.resize(P); h.meta.resize(P);
    for (int r = 0; r < P; r++) {
        unsigned lm = 0;
        if (!env->wide) for (int h0 = t.path_link_ptr[r]; h0 < t.path_link_ptr[r + 1]; h0++) lm |= 1u << t.path_links[h0];
        h.linkmask[r] = lm;
        int se = t.path_se[r] < 1 ? 1 : t.path_se[r];
        h.meta[r] = (unsigned)(t.path_hops[r] & 0xff) | ((unsigned)(se & 0xff) << 8) | ((unsigned)(t.path_mod[r] & 0xff) << 16);
    }
    std::vector<unsigned char> mod_se(t.num_mods > 0 ? t.num_mods : 1, 1);
    for (int m = 0; m < t.num_mods; m++) mod_se[m] = (unsigned char)t.mod_se[m];
    h.nslots.assign((size_t)(se_max + 1) * (br_max + 1), 1);
    for (int se = 1; se <= se_max; se++)
        for (int b = 0; b <= br_max; b++) {
            const int n = slots_needed(b, se, cfg.channel_width);
            h.nslots[(size_t)se * (br_max + 1) + b] = (unsigned char)(n > 200 ? 200 : n);
        }
    std::vector<double> reach((size_t)(t.num_mods > 0 ? t.num_mods : 1) * (br_max + 1), 0.0);
    if (cfg.kind == ORLG_RMCSA)
        for (int m = 0; m < t.num_mods; m++)
            for (int b = 0; b <= br_max; b++)
                reach[(size_t)m * (br_max + 1) + b] = b == 0 ? 1e300 : reach_km(t.mod_osnr[m], t.mod_xt[m], t.mod_se[m], b, cfg.worst_xt);
    std::vector<double> plen(t.path_length, t.path_length + P);
    h.node_thr = thresholds(t.node_prob, p.N);
    std::vector<unsigned> br_thr = t.num_bit_rates > 0 ? thresholds(t.bit_rate_prob, t.num_bit_rates) : std::vector<unsigned>(1, 0u);
    std::vector<int> link_order(p.E);
    for (int l = 0; l < p.E; l++) link_order[l] = t.link_order ? t.link_order[l] : l;
    std::vector<int> bit_rates(t.num_bit_rates > 0 ? t.num_bit_rates : 1, 0);
    for (int i = 0; i < t.num_bit_rates; i++) bit_rates[i] = t.bit_rates[i];
    std::vector<int> lptr(t.path_link_ptr, t.path_link_ptr + P + 1);
    std::vector<unsigned short> l16(lptr[P] > 0 ? lptr[P] : 1, 0);
    for (int i = 0; i < lptr[P]; i++) l16[i] = (unsigned short)t.path_links[i];

    int rc = dev_upload(env, &p.pair_first, h.pair_first);
    if (!rc) rc = dev_upload(env, &p.pair_count, h.pair_count);
    if (!rc) rc = dev_upload(env, &p.path_linkmask, h.linkmask);
    if (!rc) rc = dev_upload(env, &p.path_meta, h.meta);
    if (!rc) rc = dev_upload(env, &p.path_length, plen);
    if (!rc) rc = dev_upload(env, &p.path_link_ptr, lptr);
    if (!rc) rc = dev_upload(env, &p.path_links16, l16);
    if (!rc) rc = dev_upload(env, &p.nslots, h.nslots);
    if (!rc) rc = dev_upload(env, &p.mod_se, mod_se);
    if (!rc) rc = dev_upload(env, &p.reach, reach);
    if (!rc) rc = dev_upload(env, &p.node_thr, h.node_thr);
    if (!rc) rc = dev_upload(env, &p.br_thr, br_thr);
    if (!rc) rc = dev_upload(env, &p.bit_rates, bit_rates);
    if (!rc) rc = dev_upload(env, &p.link_order, link_order);
    return rc;
}

// Step 3.  The per-environment state arrays (orlg_state_save / orlg_state_load keep them, in this order).
int alloc_state(orlg_env *env, const orlg_tables &t) {
    Params &p = env->p;
    const size_t n = (size_t)p.n;
    env->alloc_is_state = true;
    int rc = dev_alloc(env, &p.masks, (size_t)p.C * p.E * (env->wide ? p.wstride : p.nwv) * n);
    if (!rc) rc = dev_alloc(env, &p.now, n);
    if (!rc) rc = dev_alloc(env, &p.cur_hold, n);
    if (!rc) rc = dev_alloc(env, &p.cur_req, n);
    if (!rc) rc = dev_alloc(env, &p.counters, 8 * n);
    if (!rc) rc = dev_alloc(env, &p.req_index, n);
    if (!rc) rc = dev_alloc(env, &p.nheap, n);
    if (!rc) rc = dev_alloc(env, &p.heap_min, n);
    if (!rc) rc = dev_alloc(env, &p.ev_time, n * (size_t)p.heap_cap, false);
    if (!rc) rc = dev_alloc(env, &p.ev_pay, n * (size_t)p.heap_cap, false);
    if (!rc) rc = dev_alloc(env, &p.ev_gmin, n * (size_t)p.ev_groups);
    if (!rc) rc = dev_alloc(env, &p.ev_tail, n);
    if (!rc) rc = dev_alloc(env, &p.cand, n * (size_t)p.cand_stride);
    if (!rc && env->wide && p.kind == ORLG_DEEPRMSA) rc = dev_alloc(env, &p.cand16, n * (size_t)p.cand_stride);
    if (!rc) rc = dev_alloc(env, &p.errors, n);
    if (!rc && p.kind == ORLG_RMSA && t.num_bit_rates > 0) rc = dev_alloc(env, &p.br_hist, 2 * (size_t)t.num_bit_rates * n);
    if (!rc && p.kind == ORLG_RWA) rc = dev_alloc(env, &p.act_hist, (size_t)(p.k + p.S + 2 * p.allow_rejection) * n);
    env->alloc_is_state = false;
    return rc;
}

// Step 4.  The small tables packed for shared-memory staging by the fast DeepRMSA kernel and the rollout kernel (p.tab_blob),
// and the shared-memory size of the fast kernel.  Nothing is uploaded when the topology does not fit that form.
int upload_fast_blob(orlg_env *env, const orlg_tables &t, const HostTables &h, int se_max) {
    Params &p = env->p;
    const int NN = p.N * p.N, P = t.num_paths, br_max = p.br_max;
    if (env->wide || p.kind == ORLG_RMCSA || p.k > 5 || P > 65535 || se_max > 15) return ORLG_OK;
    std::vector<unsigned char> blob;
    auto put = [&blob](const void *src, size_t bytes) {
        size_t off = (blob.size() + 15) / 16 * 16;
        blob.resize(off + bytes);
        std::memcpy(blob.data() + off, src, bytes);
        return (int)off;
    };
    std::vector<unsigned short> pf16(NN);
    for (int i = 0; i < NN; i++) pf16[i] = (unsigned short)(h.pair_first[i] < 0 ? 0 : h.pair_first[i]);
    std::vector<unsigned char> pse(P);
    for (int r = 0; r < P; r++) pse[r] = (unsigned char)((h.meta[r] >> 8) & 0xff);
    std::vector<unsigned char> ns128((size_t)(se_max + 1) * 128, 1);
    for (int se = 1; se <= se_max; se++)
        for (int b = 0; b < 128 && b <= br_max; b++) ns128[(size_t)se * 128 + b] = h.nslots[(size_t)se * (br_max + 1) + b];
    std::vector<float> pos(p.S + 1), nsl(32);
    for (int v = 0; v <= p.S; v++) pos[v] = (float)(2 * v - p.S) / (float)p.S;      // IEEE f32 division == __fdiv_rn
    for (int v = 0; v < 32; v++) nsl[v] = (float)(2 * v - 11) / 7.0f;
    p.off_pair_first = put(pf16.data(), pf16.size() * 2);
    p.off_pair_count = put(h.pair_count.data(), h.pair_count.size());
    p.off_path_lm = put(h.linkmask.data(), h.linkmask.size() * 4);
    p.off_path_se = put(pse.data(), pse.size());
    std::vector<unsigned long long> pll(P, 0ULL);      // hop list: 5 bits per link index, hop count in bits 60..63
    for (int r = 0; r < P; r++) {
        const int h0 = t.path_link_ptr[r], hn = t.path_link_ptr[r + 1] - h0;
        if (hn > 12) return ORLG_OK;
        unsigned long long v = (unsigned long long)hn << 60;
        for (int i = 0; i < hn; i++) v |= (unsigned long long)(t.path_links[h0 + i] & 31) << (5 * i);
        pll[r] = v;
    }
    p.off_path_ll = put(pll.data(), pll.size() * 8);
    p.off_nslots = put(ns128.data(), ns128.size());
    p.off_node_thr = put(h.node_thr.data(), h.node_thr.size() * 4);
    p.off_pos = put(pos.data(), pos.size() * 4);
    p.off_nsl = put(nsl.data(), nsl.size() * 4);
    std::vector<float> rcp4(p.S / 2 + 2, 0.0f);               // 1 / (4 r): at most (S + 1) / 2 free runs on a path
    for (size_t r = 1; r < rcp4.size(); r++) rcp4[r] = 1.0f / (float)(4 * r);
    p.off_rcp4 = put(rcp4.data(), rcp4.size() * 4);
    std::vector<unsigned> dbl(17, 0u);                          // shift-AND doubling: shifts of the 4 rounds for n <= 16
    for (int nn = 1; nn <= 16; nn++) {
        int len = 1;
        for (int it = 0; it < 4; it++) {
            int sh = len < nn - len ? len : nn - len;
            if (sh < 0) sh = 0;
            dbl[nn] |= (unsigned)sh << (8 * it);
            len += sh;
        }
    }
    p.off_dbl = put(dbl.data(), dbl.size() * 4);
    blob.resize((blob.size() + 127) / 128 * 128);          // the warp areas behind it are TMA destinations (128-byte aligned)
    if (blob.size() > 24 * 1024 || blob.size() + (size_t)FAST_THREADS * 16 * 32 > 100 * 1024) return ORLG_OK;
    std::vector<uint4> blob4(blob.size() / 16);
    std::memcpy(blob4.data(), blob.data(), blob.size());
    int rc = dev_upload(env, &p.tab_blob, blob4);
    if (rc) return rc;
    p.tab_vec = (int)blob4.size();
    size_t per_thread = (size_t)p.obs_dim * (p.obs_f64 ? 8 : 4);      // observation tile overlays the mask area
    if (per_thread < (size_t)p.E * 16) per_thread = (size_t)p.E * 16;
    p.warp_area_bytes = (int)((per_thread * 32 + 127) / 128 * 128);
    env->fast_smem = blob.size() + (size_t)(FAST_THREADS / 32) * p.warp_area_bytes + 8 * (FAST_THREADS / 32 + 1);   // + per-warp mbarriers + the table barrier
    return ORLG_OK;
}

// Step 5.  Which kernel instances the handle may run (the per-launch half is in hot_launch / rollout_kernel_applies), and
// the shared-memory size of each of them.
int select_instances(orlg_env *env, const orlg_config &cfg, const HostTables &h, int se_max) {
    const Params &p = env->p;
    if (p.tab_blob) {
        cudaError_t ea = cudaSuccess;
        if (env->fast_smem > 48 * 1024)
            for (FastKernel k : FAST_KERNELS)
                if (ea == cudaSuccess) ea = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env->fast_smem);
        env->fast = p.kind == ORLG_DEEPRMSA && ea == cudaSuccess;
        // continuous bit rates below 128 Gb/s whose slot counts all fit the 4-round shift-AND
        int n_hi = 0;
        for (int se = 1; se <= se_max; se++)
            for (int b = 0; b <= cfg.bit_rate_hi && b <= p.br_max; b++) n_hi = std::max<int>(n_hi, h.nslots[(size_t)se * (p.br_max + 1) + b]);
        const bool small_n = p.n_bit_rates == 0 && cfg.bit_rate_hi < 128 && cfg.bit_rate_lo >= 0 && n_hi <= 16;
        const bool no_hot = std::getenv("ORLG_NO_HOT") != nullptr;
        // steady-state specialisation: small slot counts, exactly KM candidate paths per pair, j = 1, 8-byte candidate
        // cache, even observation width
        env->hot = env->fast && p.J == 1 && p.k == 5 && p.cand_stride == 8 && small_n && (p.obs_dim & 1) == 0 && p.E <= 256 && !no_hot;
        if (env->hot && !encode_mask_map(env)) env->hot = false;
        // the persistent rollout kernel (orlg_rollout.cuh): DeepRMSA-v0 under the HOT conditions; RMSA-v0 with small slot
        // counts; RWA-v0 (one wavelength per lightpath)
        env->ro_ok = p.kind == ORLG_DEEPRMSA ? env->hot
                     : (ea == cudaSuccess && p.E <= 32 && (p.kind == ORLG_RWA || small_n) && !no_hot);
    }
    if (const size_t obs_smem = step_obs_smem(p); obs_smem > 48 * 1024) {
        cudaError_t e1 = cudaFuncSetAttribute(step_kernel<ORLG_DEEPRMSA, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)obs_smem);
        cudaError_t e2 = cudaFuncSetAttribute(step_kernel<ORLG_DEEPRMSA, KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)obs_smem);
        if (e1 != cudaSuccess || e2 != cudaSuccess) return fail(ORLG_E_CUDA, "cudaFuncSetAttribute(shared memory) failed");
    }
    return ORLG_OK;
}
}  // namespace

extern "C" {

const char *orlg_last_error(void) { return g_err.c_str(); }
int orlg_version(void) { return ORLG_VERSION; }

int orlg_create(const orlg_config *cfg, const orlg_tables *t, int device, orlg_env **out) {
    if (!cfg || !t || !out) return fail(ORLG_E_INVALID, "null argument");
    *out = nullptr;
    Params p; bool wide; int se_max;
    int rc = configure(*cfg, *t, device, p, wide, se_max);
    if (rc) return rc;
    DeviceGuard guard(device);
    std::unique_ptr<orlg_env, int (*)(orlg_env *)> env(new orlg_env(), orlg_destroy);
    env->p = p; env->cfg = *cfg; env->device = device; env->wide = wide;
    env->ro_lpw = choose_rollout_lpw(cfg->num_envs);
    HostTables h;
    rc = upload_tables(env.get(), *cfg, *t, se_max, h);
    if (!rc) rc = alloc_state(env.get(), *t);
    if (!rc) rc = upload_fast_blob(env.get(), *t, h, se_max);
    if (!rc) rc = select_instances(env.get(), *cfg, h, se_max);
    if (rc) return rc;
    *out = env.release();
    return ORLG_OK;
}

int orlg_destroy(orlg_env *env) {
    if (!env) return ORLG_OK;
    DeviceGuard guard(env->device);
    delete env;
    return ORLG_OK;
}

int orlg_action_dim(const orlg_env *env) { return env->p.kind == ORLG_DEEPRMSA ? 1 : (env->p.kind == ORLG_RMCSA ? 4 : 2); }
int orlg_obs_dim(const orlg_env *env) { return env->p.obs_dim; }
int orlg_mask_words(const orlg_env *env) { return NW * env->p.nwv; }
int orlg_heap_capacity(const orlg_env *env) { return env->p.heap_cap; }
int64_t orlg_state_bytes(const orlg_env *env) { return env->state_bytes; }

int orlg_kernel_info(const orlg_env *env, orlg_kernel_info_t *out) {
    if (!env || !out) return fail(ORLG_E_INVALID, "null handle or output");
    out->wide = env->wide;
    out->fast = env->fast;
    out->hot = env->hot;
    out->rollout_kernel = env->ro_ok;
    out->rollout_lanes = env->ro_lpw;
    out->link_template = link_template(env);
    out->last_rollout_persistent = env->ro_last_persistent;
    return ORLG_OK;
}

int orlg_seed(orlg_env *env, uint64_t seed) {
    if (!env) return fail(ORLG_E_INVALID, "null handle");
    env->p.seed = seed;           // a launch parameter: takes effect with the next kernel
    env->cfg.seed = seed;
    return ORLG_OK;
}

int orlg_set_trace(orlg_env *env, const orlg_request *trace_dev, int64_t trace_len) {
    if (!env || (trace_len > 0 && !trace_dev)) return fail(ORLG_E_INVALID, "null trace");
    if (trace_len >= (1LL << 32)) return fail(ORLG_E_UNSUPPORTED, "trace too long");
    env->p.trace = trace_dev;
    env->p.trace_len = trace_len;
    env->p.traffic = ORLG_TRAFFIC_TRACE;
    return ORLG_OK;
}

int orlg_reset(orlg_env *env, int full, void *obs_dev, orlg_stream stream) {
    if (!env) return fail(ORLG_E_INVALID, "null handle");
    DeviceGuard guard(env->device);
    if (env->p.traffic == ORLG_TRAFFIC_TRACE && env->p.trace == nullptr) return fail(ORLG_E_INVALID, "trace traffic selected but orlg_set_trace was not called");
    StepIO io;
    std::memset(&io, 0, sizeof(io));
    io.policy = -1;
    io.obs = env->p.obs_dim ? obs_dev : nullptr;
    if (full) env->ro_valid = false;           // everything is reset below: nothing to convert back
    else if (int rc0 = ensure_canonical(env, (cudaStream_t)stream)) return rc0;
    if (full) {
        fill_events_kernel<<<592, 256, 0, (cudaStream_t)stream>>>(env->p);
        CUDA_OK(cudaGetLastError());
    }
    int rc = launch_step(env, io, full ? MODE_FULL_RESET : MODE_EPISODE_RESET, (cudaStream_t)stream);
    if (rc == ORLG_OK && full) env->p.lockstep_ridx = 1;      // every env has drawn its first request
    return rc;
}

// orlg_step; fused_policy >= 0 (wide kernels only): the heuristic is evaluated inside the step kernel, actions_dev receives it
static int step_impl(orlg_env *env, const int32_t *actions_dev, int fused_policy, int32_t *actions_out, void *obs_dev, float *reward_dev,
                     uint8_t *done_dev, int32_t *decision_dev, int64_t *info_dev, orlg_stream stream) {
    if (int rc0 = ensure_canonical(env, (cudaStream_t)stream)) return rc0;
    StepIO io;
    io.policy = fused_policy;
    io.actions_out = actions_out;
    io.actions = actions_dev;
    io.obs = env->p.obs_dim ? obs_dev : nullptr;
    io.reward = reward_dev;
    io.done = done_dev;
    io.decision = decision_dev;
    io.info = reinterpret_cast<long long *>(info_dev);
    io.obs_int = nullptr;
    int rc = launch_step(env, io, MODE_STEP, (cudaStream_t)stream);
    if (rc == ORLG_OK) env->p.lockstep_ridx++;
    return rc;
}

int orlg_step(orlg_env *env, const int32_t *actions_dev, void *obs_dev, float *reward_dev, uint8_t *done_dev,
              int32_t *decision_dev, int64_t *info_dev, orlg_stream stream) {
    if (!env || !actions_dev) return fail(ORLG_E_INVALID, "null handle or actions");
    DeviceGuard guard(env->device);
    return step_impl(env, actions_dev, -1, nullptr, obs_dev, reward_dev, done_dev, decision_dev, info_dev, stream);
}

int orlg_observation(orlg_env *env, void *obs_dev, orlg_stream stream) {
    if (!env || !obs_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    if (!env->p.obs_dim) return fail(ORLG_E_UNSUPPORTED, "this env kind has a dict observation (no tensor)");
    StepIO io;
    std::memset(&io, 0, sizeof(io));
    io.policy = -1;
    io.obs = obs_dev;
    return launch_step(env, io, MODE_OBSERVE, (cudaStream_t)stream);
}

int orlg_observation_int(orlg_env *env, int32_t *out_dev, orlg_stream stream) {
    if (!env || !out_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    if (!env->p.obs_dim) return fail(ORLG_E_UNSUPPORTED, "this env kind has a dict observation (no tensor)");
    StepIO io;
    std::memset(&io, 0, sizeof(io));
    io.policy = -1;
    io.obs_int = out_dev;
    return launch_step(env, io, MODE_OBSERVE, (cudaStream_t)stream);
}

int orlg_heuristic(orlg_env *env, int which, int32_t *actions_dev, orlg_stream stream) {
    if (!env || !actions_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    if (which < 0 || which > ORLG_HEUR_SAP_LF) return fail(ORLG_E_INVALID, "unknown heuristic");
    const int threads = 128, blocks = (env->p.n + threads - 1) / threads;
    cudaStream_t s = (cudaStream_t)stream;
    if (const char *why = heuristic_refusal(env->p.kind, which)) return fail(ORLG_E_UNSUPPORTED, why);
    for_kind(env->p.kind, [&](auto K) {
        if (env->wide) for_words(env->p.nwv, [&](auto W) {
            heuristic_wide_kernel<decltype(K)::value, decltype(W)::value><<<blocks, threads, 0, s>>>(env->p, which, actions_dev); });
        else heuristic_kernel<decltype(K)::value><<<blocks, threads, 0, s>>>(env->p, which, actions_dev);
    });
    CUDA_OK(cudaGetLastError());
    return ORLG_OK;
}

int orlg_random_actions(orlg_env *env, int32_t *actions_dev, orlg_stream stream) {
    if (!env || !actions_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    const int threads = 256, blocks = (env->p.n + threads - 1) / threads;
    cudaLaunchConfig_t cfg = pdl_config(blocks, threads, 0, (cudaStream_t)stream);
    int *actions = actions_dev;
    CUDA_OK(cudaLaunchKernelEx(&cfg, random_action_kernel, env->p, actions));
    return ORLG_OK;
}

static int run_export(orlg_env *env, uint32_t *masks, int32_t *alloc, double *now, int32_t *nheap, int64_t *counters,
                      orlg_request *req, int32_t *sid, uint32_t *err, orlg_stream stream) {
    if (!env) return fail(ORLG_E_INVALID, "null handle");
    DeviceGuard guard(env->device);
    const int threads = 128, blocks = (env->p.n + threads - 1) / threads;
    if (alloc) {                               // the allocation matrix is rebuilt from the release-event table
        if (int rc0 = ensure_canonical(env, (cudaStream_t)stream)) return rc0;
    }
    if (env->wide && (masks || alloc)) {
        export_wide_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(env->p, masks, alloc);
        CUDA_OK(cudaGetLastError());
        masks = nullptr; alloc = nullptr;
    }
    export_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(env->p, masks, alloc, now, nheap,
                                                                reinterpret_cast<long long *>(counters), req, sid, err);
    CUDA_OK(cudaGetLastError());
    return ORLG_OK;
}

int orlg_get_counters(orlg_env *env, int64_t *counters_dev, orlg_stream stream) {
    return run_export(env, nullptr, nullptr, nullptr, nullptr, counters_dev, nullptr, nullptr, nullptr, stream);
}

int orlg_get_requests(orlg_env *env, orlg_request *requests_dev, int32_t *service_id_dev, orlg_stream stream) {
    return run_export(env, nullptr, nullptr, nullptr, nullptr, nullptr, requests_dev, service_id_dev, nullptr, stream);
}

int orlg_export_state(orlg_env *env, uint32_t *masks_dev, int32_t *alloc_dev, double *now_dev, int32_t *nheap_dev,
                      orlg_stream stream) {
    return run_export(env, masks_dev, alloc_dev, now_dev, nheap_dev, nullptr, nullptr, nullptr, nullptr, stream);
}

int orlg_error_flags(orlg_env *env, uint32_t *flags_dev, orlg_stream stream) {
    return run_export(env, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, flags_dev, stream);
}

// debug (instrumented builds only): cumulative per-phase cycles of the fast kernel, then reset
int orlg_debug_phase_cycles(unsigned long long *out16) {
#ifdef ORLG_PHASE_TIMING
    CUDA_OK(cudaMemcpyFromSymbol(out16, g_phase_cycles, 16 * sizeof(unsigned long long)));
    unsigned long long zero[16] = {0};
    CUDA_OK(cudaMemcpyToSymbol(g_phase_cycles, zero, sizeof(zero)));
    return ORLG_OK;
#else
    (void)out16;
    return fail(ORLG_E_UNSUPPORTED, "built without -DORLG_PHASE_TIMING");
#endif
}

// debug (instrumented builds only): per-warp globaltimer entry/exit of the last fast-kernel launch
int orlg_debug_warp_timeline(unsigned long long *out, int n_warps) {
#ifdef ORLG_PHASE_TIMING
    CUDA_OK(cudaMemcpyFromSymbol(out, g_warp_timeline, (size_t)2 * n_warps * sizeof(unsigned long long)));
    return ORLG_OK;
#else
    (void)out; (void)n_warps;
    return fail(ORLG_E_UNSUPPORTED, "built without -DORLG_PHASE_TIMING");
#endif
}

// debug (instrumented builds only): per-warp timeline of the last orlg_rollout launch (8 words per warp, orlg_rollout.cuh)
int orlg_debug_rollout_timeline(unsigned long long *out, int n_warps) {
#ifdef ORLG_RO_TIMELINE
    CUDA_OK(cudaMemcpyFromSymbol(out, g_ro_timeline, (size_t)8 * (n_warps < 4096 ? n_warps : 4096) * sizeof(unsigned long long)));
    return ORLG_OK;
#else
    (void)out; (void)n_warps;
    return fail(ORLG_E_UNSUPPORTED, "built without -DORLG_RO_TIMELINE");
#endif
}

static int stats_alloc(orlg_env *env) {
    Params &p = env->p;
    if (p.br_max > 65535) return fail(ORLG_E_UNSUPPORTED, "statistics path keeps bit rates in 16 bits");
    if (!p.link_util) {
        const size_t n = (size_t)p.n;
        env->alloc_is_state = true;
        int rc = dev_alloc(env, &p.link_util, (size_t)p.E * n);
        if (!rc) rc = dev_alloc(env, &p.link_comp, (size_t)p.E * n);
        if (!rc) rc = dev_alloc(env, &p.link_last, (size_t)p.E * n);
        if (!rc) rc = dev_alloc(env, &p.link_frag, (size_t)p.E * n);
        if (!rc) rc = dev_alloc(env, &p.graph_stats, 3 * n);
        if (!rc) rc = dev_alloc(env, &p.run_br, n);
        if (!rc) rc = dev_alloc(env, &p.ev_br, n * (size_t)p.heap_cap);
        // wide kernels: the compactness terms follow sum_nh in its allocation (nc_totals / nc_links, orlg_step_wide.cuh), in
        // units of 8 bytes: int2 [n][C], then unsigned [n][C*E]
        const size_t nc = env->wide && p.kind != ORLG_RWA ? (size_t)p.C * n + ((size_t)p.C * p.E * n + 1) / 2 : 0;
        if (!rc) rc = dev_alloc(env, &p.sum_nh, n + nc);
        env->alloc_is_state = false;
        if (rc) return rc;
    }
    return ORLG_OK;
}

int orlg_enable_stats(orlg_env *env, double *stats_dev) {
    if (!env) return fail(ORLG_E_INVALID, "null handle");
    DeviceGuard guard(env->device);
    Params &p = env->p;
    if (!stats_dev) { p.stats = 0; p.stats_out = nullptr; return ORLG_OK; }
    if (p.kind != ORLG_RMSA && p.kind != ORLG_DEEPRMSA) return fail(ORLG_E_UNSUPPORTED, "info has float statistics for RMSA-v0 / DeepRMSA-v0 only (orlg_enable_link_stats covers every kind)");
    int rc = stats_alloc(env);
    if (rc) return rc;
    p.stats = 1;
    p.stats_out = stats_dev;
    return ORLG_OK;
}

int orlg_enable_link_stats(orlg_env *env, int on) {
    if (!env) return fail(ORLG_E_INVALID, "null handle");
    DeviceGuard guard(env->device);
    Params &p = env->p;
    if (!on) { if (!p.stats_out) p.stats = 0; return ORLG_OK; }
    int rc = stats_alloc(env);
    if (rc) return rc;
    p.stats = 1;
    return ORLG_OK;
}

int orlg_link_stats(orlg_env *env, double *link_dev, double *graph_dev, orlg_stream stream) {
    if (!env || (!link_dev && !graph_dev)) return fail(ORLG_E_INVALID, "null handle or buffers");
    if (!env->p.stats) return fail(ORLG_E_INVALID, "statistics are off (orlg_enable_stats / orlg_enable_link_stats before the full reset)");
    DeviceGuard guard(env->device);
    link_stats_kernel<<<(env->p.n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(env->p, link_dev, graph_dev);
    CUDA_OK(cudaGetLastError());
    return ORLG_OK;
}

int orlg_num_bit_rates(const orlg_env *env) { return env->p.br_hist ? env->p.n_bit_rates : 0; }

int orlg_bit_rate_blocking(orlg_env *env, double *out_dev, orlg_stream stream) {
    if (!env || !out_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    if (!env->p.br_hist) return fail(ORLG_E_UNSUPPORTED, NO_BIT_RATES);
    bit_rate_blocking_kernel<<<(env->p.n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(env->p, out_dev);
    CUDA_OK(cudaGetLastError());
    return ORLG_OK;
}

int orlg_action_hist_dim(const orlg_env *env) { return env->p.act_hist ? env->p.k + env->p.S + 2 * env->p.allow_rejection : 0; }

int orlg_action_probability(orlg_env *env, double *out_dev, orlg_stream stream) {
    if (!env || !out_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    if (!env->p.act_hist) return fail(ORLG_E_UNSUPPORTED, NO_ACTION_HIST);
    DeviceGuard guard(env->device);
    action_probability_kernel<<<(env->p.n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(env->p, out_dev);
    CUDA_OK(cudaGetLastError());
    return ORLG_OK;
}

int orlg_matrix_obs_dim(const orlg_env *env) { return 2 * env->p.N + env->p.C * env->p.E * env->p.S; }

int orlg_matrix_observation(orlg_env *env, uint8_t *out_dev, orlg_stream stream) {
    if (!env || !out_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    const long long total = (long long)orlg_matrix_obs_dim(env) * env->p.n;
    long long blocks = (total + 255) / 256;
    if (blocks > 148LL * 32) blocks = 148LL * 32;
    matrix_observation_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(env->p, out_dev);
    CUDA_OK(cudaGetLastError());
    return ORLG_OK;
}

int orlg_path_only_first_fit(orlg_env *env, const int32_t *path_actions_dev, int32_t *actions_dev, orlg_stream stream) {
    if (!env || !path_actions_dev || !actions_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    if (env->p.kind != ORLG_RMSA && env->p.kind != ORLG_RWA)
        return fail(ORLG_E_UNSUPPORTED, "PathOnlyFirstFitAction exists for RMSA-v0 and RWA-v0 (the RMCSA one raises upstream)");
    const int blocks = (env->p.n + 127) / 128;
    cudaStream_t s = (cudaStream_t)stream;
    for_words(env->p.nwv, [&](auto W) { path_only_first_fit_kernel<decltype(W)::value><<<blocks, 128, 0, s>>>(env->p, path_actions_dev, actions_dev); });
    CUDA_OK(cudaGetLastError());
    return ORLG_OK;
}

// row t of the float outputs of info, after step t (the counters come through the step kernel's info_dev)
static int info_row(orlg_env *env, const orlg_info_out *info, int t, orlg_stream stream) {
    const Params &p = env->p;
    const size_t n = (size_t)p.n;
    if (info->stats_dev)
        CUDA_OK(cudaMemcpyAsync(info->stats_dev + (size_t)t * n * 4, p.stats_out, n * 4 * sizeof(double), cudaMemcpyDeviceToDevice,
                                (cudaStream_t)stream));
    int rc = ORLG_OK;
    if (info->bit_rate_blocking_dev)
        rc = orlg_bit_rate_blocking(env, info->bit_rate_blocking_dev + (size_t)t * n * (p.n_bit_rates + 1), stream);
    if (!rc && info->action_probability_dev)
        rc = orlg_action_probability(env, info->action_probability_dev + (size_t)t * n * orlg_action_hist_dim(env), stream);
    return rc;
}

static int rollout_impl(orlg_env *env, int steps, int policy, void *obs_dev, float *reward_dev, uint8_t *done_dev,
                        int32_t *actions_dev, uint32_t *packed_dev, const orlg_info_out *info, orlg_stream stream) {
    if (!env) return fail(ORLG_E_INVALID, "null handle");
    DeviceGuard guard(env->device);
    if (steps < 0) return fail(ORLG_E_INVALID, "steps must be >= 0");
    if (policy != ORLG_POLICY_RANDOM && policy != ORLG_POLICY_REPLAY && (policy < 0 || policy > ORLG_HEUR_SAP_LF)) return fail(ORLG_E_INVALID, "unknown policy");
    if (policy == ORLG_POLICY_REPLAY && !actions_dev) return fail(ORLG_E_INVALID, "ORLG_POLICY_REPLAY needs the action sequence in actions_dev");
    if (env->p.traffic == ORLG_TRAFFIC_TRACE && env->p.trace == nullptr) return fail(ORLG_E_INVALID, "trace traffic selected but orlg_set_trace was not called");
    if (const char *why = info_refusal(env->p, info)) return fail(ORLG_E_UNSUPPORTED, why);
    if (steps == 0) return ORLG_OK;
    Params &p = env->p;
    cudaStream_t s = (cudaStream_t)stream;
    RolloutArgs ra;
    std::memset(&ra, 0, sizeof(ra));
    int wpc = 0;
    size_t smem = 0;
    if (rollout_kernel_applies(env, policy, info) && rollout_plan(env, &wpc, &ra, &smem)) {
        if (!env->ro_ev) {
            const size_t n = (size_t)p.n, warps = (n + env->ro_lpw - 1) / env->ro_lpw;
            int rc = dev_alloc(env, &env->ro_ev, warps * 32 * ((size_t)p.heap_cap + 2 * RO_WCAP), false);
            if (!rc) rc = dev_alloc(env, &env->ro_st_u32, 4 * n, false);
            if (!rc) rc = dev_alloc(env, &env->ro_st_f64, (2 + RO_SIDE) * n, false);
            if (!rc) rc = dev_alloc(env, &env->ro_st_u64, RO_SIDE * n, false);
            if (rc) return rc;
        }
        double span_steps = 40.0;
        if (const char *v = std::getenv("ORLG_RO_SPAN")) { double w = std::atof(v); if (w > 0) span_steps = w; }
        ra.T = steps;
        ra.span = span_steps * p.mean_iat;
        ra.obs = reinterpret_cast<float *>(obs_dev);
        ra.reward = reward_dev; ra.done = done_dev; ra.actions = actions_dev;
        ra.packed = reinterpret_cast<uint4 *>(packed_dev);
        ra.info = info ? reinterpret_cast<long long *>(info->counters_dev) : nullptr;
        if (packed_dev && p.kind != ORLG_DEEPRMSA) return fail(ORLG_E_UNSUPPORTED, "packed records describe the DeepRMSA observation");
        rollout_state_args(env, &ra);
        ra.resume = env->ro_valid ? 1 : 0;
        cudaError_t e = link_template(env) == 22 ? launch_rollout<22>(env, ra, policy, wpc, smem, s) : launch_rollout<0>(env, ra, policy, wpc, smem, s);
        if (e != cudaSuccess) return fail(ORLG_E_CUDA, std::string("rollout launch: ") + cudaGetErrorString(e));
        p.lockstep_ridx += (unsigned)steps;
        env->ro_valid = true;
        env->ro_last_persistent = true;
        return ORLG_OK;
    }
    env->ro_last_persistent = false;
    if (packed_dev) return fail(ORLG_E_UNSUPPORTED, "packed records exist for the persistent DeepRMSA rollout kernel only (k = 5, j = 1, float32)");
    // generic: the same T steps as separate policy + step launches
    int rc = ensure_canonical(env, s);
    if (rc) return rc;
    const int adim = orlg_action_dim(env);
    if (policy != ORLG_POLICY_REPLAY && !actions_dev && !env->ro_actions) {
        rc = dev_alloc(env, &env->ro_actions, (size_t)p.n * adim, false);
        if (rc) return rc;
    }
    const size_t obs_row = (size_t)p.obs_dim * (p.obs_f64 ? 8 : 4);
    // wide kernels: the heuristic runs in the step kernel's prologue (one launch per step; the chosen path's masks are read once)
    const bool fuse = env->wide && policy >= 0 && !heuristic_refusal(p.kind, policy);
    for (int t = 0; t < steps && !rc; t++) {
        int32_t *a = actions_dev ? actions_dev + (size_t)t * p.n * adim : env->ro_actions;
        void *o = (obs_dev && p.obs_dim) ? reinterpret_cast<unsigned char *>(obs_dev) + (size_t)t * p.n * obs_row : nullptr;
        float *r = reward_dev ? reward_dev + (size_t)t * p.n : nullptr;
        uint8_t *d = done_dev ? done_dev + (size_t)t * p.n : nullptr;
        int64_t *c = info && info->counters_dev ? info->counters_dev + (size_t)t * p.n * 8 : nullptr;
        if (fuse) rc = step_impl(env, nullptr, policy, actions_dev ? a : nullptr, o, r, d, nullptr, c, stream);
        else if (policy != ORLG_POLICY_REPLAY)
            rc = policy == ORLG_POLICY_RANDOM ? orlg_random_actions(env, a, stream) : orlg_heuristic(env, policy, a, stream);
        if (!rc && !fuse) rc = orlg_step(env, a, o, r, d, nullptr, c, stream);
        if (!rc && info) rc = info_row(env, info, t, stream);
    }
    return rc;
}


int orlg_rollout(orlg_env *env, int steps, int policy, void *obs_dev, float *reward_dev, uint8_t *done_dev,
                 int32_t *actions_dev, orlg_stream stream) {
    return rollout_impl(env, steps, policy, obs_dev, reward_dev, done_dev, actions_dev, nullptr, nullptr, stream);
}

int orlg_rollout_info(orlg_env *env, int steps, int policy, void *obs_dev, float *reward_dev, uint8_t *done_dev,
                      int32_t *actions_dev, const orlg_info_out *info, orlg_stream stream) {
    return rollout_impl(env, steps, policy, obs_dev, reward_dev, done_dev, actions_dev, nullptr, info, stream);
}

int orlg_rollout_packed(orlg_env *env, int steps, int policy, uint32_t *packed_dev, int32_t *actions_dev, orlg_stream stream) {
    if (!packed_dev) return fail(ORLG_E_INVALID, "null record buffer");
    return rollout_impl(env, steps, policy, nullptr, nullptr, nullptr, actions_dev, packed_dev, nullptr, stream);
}

// ---------------------------------------------------------------- host side of the packed records (no CUDA below this line)
// A persistent pool of host threads: orlg_expand_packed is called once per chunk of a pipelined rollout (every ~0.3 ms),
// so creating threads per call would cost more than the work.  Blocks of rows are handed out through an atomic counter
// (the caller's thread works too), which also balances the load when several ranks share the host's cores.
namespace {
struct HostPool {
    std::mutex mu;
    std::condition_variable cv_work;
    std::vector<std::thread> workers;
    std::function<void(int64_t)> fn;
    int64_t nblocks = 0;
    std::atomic<int64_t> next{0};
    std::atomic<int> active{0};          // workers still inside the current job
    std::atomic<uint64_t> generation{0};
    bool stop = false;
    static constexpr int SPIN = 20000;   // polls of the generation counter (~0.3 ms) before a worker sleeps on the condition variable:
                                         // the chunks of a pipelined rollout follow each other within that time

    void drain() {
        for (;;) {
            const int64_t b = next.fetch_add(1, std::memory_order_relaxed);
            if (b >= nblocks) return;
            fn(b);
        }
    }
    void worker(int id) {
        uint64_t seen = 0;
        for (;;) {
            int spins = 0;
            while (generation.load(std::memory_order_acquire) == seen && spins < SPIN) { _mm_pause(); spins++; }
            if (generation.load(std::memory_order_acquire) == seen) {
                std::unique_lock<std::mutex> lk(mu);
                cv_work.wait(lk, [&] { return stop || generation.load(std::memory_order_acquire) != seen; });
                if (stop) return;
            }
            seen = generation.load(std::memory_order_acquire);
            // the low byte of the generation is the number of workers wanted by THAT job: a worker below it is waited for by
            // run() (so fn / nblocks / next are the job's own); one at or above it touches nothing
            if (id < (int)(seen & 0xffu)) {
                drain();
                active.fetch_sub(1, std::memory_order_acq_rel);
            }
        }
    }
    void run(int threads, int64_t blocks, std::function<void(int64_t)> f) {
        if (threads <= 1 || blocks <= 1) { for (int64_t b = 0; b < blocks; b++) f(b); return; }
        if (threads > 200) threads = 200;
        {
            std::lock_guard<std::mutex> lk(mu);
            while ((int)workers.size() < threads - 1) { const int id = (int)workers.size(); workers.emplace_back(&HostPool::worker, this, id); }
            fn = std::move(f); nblocks = blocks; next.store(0); active.store(threads - 1);
            generation.store((((generation.load(std::memory_order_relaxed) >> 8) + 1) << 8) | (uint64_t)(threads - 1), std::memory_order_release);
        }
        cv_work.notify_all();
        drain();
        while (active.load(std::memory_order_acquire) != 0) _mm_pause();     // the stragglers finish their last block
    }
    ~HostPool() {
        { std::lock_guard<std::mutex> lk(mu); stop = true; }
        cv_work.notify_all();
        for (auto &t : workers) t.join();
    }
};
HostPool g_pool;                         // one job at a time (g_pool_mu); handles on different threads serialise here
std::mutex g_pool_mu;

// Float tables of the observation features, indexed by PAIRS of packed fields so that a candidate path costs three look-ups:
// the same float32 expressions as the device tables built in orlg_create (hence bit-identical rows).  192 KB, L2-resident.
struct F2 { float a, b; };
struct ExpandTables {
    int S = -1;
    std::vector<F2> sl;      // [start | length << 7] -> (start, length) features; (-1, -1) when start == 127 (no block)
    std::vector<F2> tr;      // [free slots | free runs << 7] -> (free-slot feature, average-run feature or -1)
    float need[32], rate[256];
};
const ExpandTables &expand_tables(int S) {
    static std::mutex mu;
    static std::vector<std::unique_ptr<ExpandTables>> cache;
    std::lock_guard<std::mutex> lk(mu);
    for (auto &t : cache) if (t->S == S) return *t;
    std::unique_ptr<ExpandTables> t(new ExpandTables);
    t->S = S; t->sl.resize(1 << 14); t->tr.resize(1 << 13);
    for (int st = 0; st < 128; st++)
        for (int ln = 0; ln < 128; ln++)
            t->sl[st | ln << 7] = st != 127 ? F2{(float)(2 * st - S) / (float)S, (float)(ln - 8) * 0.125f} : F2{-1.0f, -1.0f};
    for (int total = 0; total < 128; total++)
        for (int runs = 0; runs < 64; runs++)
            t->tr[total | runs << 7] = F2{(float)(2 * total - S) / (float)S, runs > 0 ? (float)(total - 4 * runs) * (1.0f / (float)(4 * runs)) : -1.0f};
    for (int n = 0; n < 32; n++) t->need[n] = (float)(2 * n - 11) / 7.0f;
    for (int b = 0; b < 256; b++) t->rate[b] = (float)b / 100.0f;
    cache.push_back(std::move(t));
    return *cache.back();
}

constexpr int EXP_BLOCK = 64;            // rows per staging block: 64 x (4 D) bytes is a multiple of 64 for every D

// rows [r0, r1) of the packed records -> float32 rows.  A block is assembled in a cache-resident staging buffer and leaves
// with non-temporal 16-byte stores when the destination allows it (no read-for-ownership of 14 MB per step).
void expand_rows(const ExpandTables &tb, const uint32_t *pk, int64_t r0, int64_t r1, int N, float *obs, float *reward, uint8_t *done,
                 int32_t *action) {
    const int D = 1 + 2 * N + 25, H = 1 + 2 * N;
    alignas(64) float stage[EXP_BLOCK * (1 + 2 * 255 + 25)];
    const F2 *sl = tb.sl.data(), *tr = tb.tr.data();
    for (int64_t b0 = r0; b0 < r1; b0 += EXP_BLOCK) {
        const int nb = (int)(r1 - b0 < EXP_BLOCK ? r1 - b0 : EXP_BLOCK);
        if (obs) {
            float *dst = obs + b0 * D;
            const bool stream_out = (reinterpret_cast<uintptr_t>(dst) & 15u) == 0 && ((size_t)nb * D) % 4 == 0;
            float *out = stream_out ? stage : dst;
            std::memset(out, 0, sizeof(float) * (size_t)nb * D);
            for (int i = 0; i < nb; i++) {
                const uint32_t *w = pk + (b0 + i) * 8;
                float *o = out + (size_t)i * D;
                const uint32_t q5 = w[5];
                const int src = (int)((q5 >> 8) & 0xffu), dst_n = (int)((q5 >> 16) & 0xffu), npaths = (int)((q5 >> 24) & 0xfu);
                o[0] = tb.rate[q5 & 0xffu];
                o[1 + (src < dst_n ? src : dst_n)] = 1.0f;
                o[1 + N + (src < dst_n ? dst_n : src)] = 1.0f;
                float *v = o + H;
                for (int q = 0; q < 5; q++, v += 5) {
                    const uint32_t f = w[q];
                    const F2 a = sl[f & 0x3fffu], b = tr[(f >> 14) & 0x1fffu];
                    const bool path = q < npaths;
                    v[0] = a.a; v[1] = a.b; v[2] = path ? tb.need[f >> 27] : -1.0f; v[3] = path ? b.a : -1.0f; v[4] = b.b;
                }
            }
            if (stream_out) {
                const __m128i *sv = reinterpret_cast<const __m128i *>(stage);
                __m128i *dv = reinterpret_cast<__m128i *>(dst);
                const size_t nv = (size_t)nb * D / 4;
                for (size_t i = 0; i < nv; i++) _mm_stream_si128(dv + i, _mm_load_si128(sv + i));
            }
        }
        if (reward) for (int i = 0; i < nb; i++) reward[b0 + i] = (pk[(b0 + i) * 8 + 5] >> 28) & 1u ? 1.0f : -1.0f;
        if (done) for (int i = 0; i < nb; i++) done[b0 + i] = (uint8_t)((pk[(b0 + i) * 8 + 5] >> 29) & 1u);
        if (action) for (int i = 0; i < nb; i++) action[b0 + i] = (int32_t)pk[(b0 + i) * 8 + 6];
    }
    _mm_sfence();
}
}  // namespace

int orlg_expand_packed(const uint32_t *packed_host, int64_t rows, int num_nodes, int num_slots, float *obs_host, float *reward_host,
                       uint8_t *done_host, int32_t *action_host, int threads) {
    if (!packed_host || rows < 0 || num_nodes < 2 || num_nodes > 255 || num_slots < 1) return fail(ORLG_E_INVALID, "bad arguments");
    int nt = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
    if (nt < 1) nt = 1;
    const ExpandTables &tb = expand_tables(num_slots);
    constexpr int64_t JOB = 2048;          // rows per hand-out (a multiple of EXP_BLOCK)
    const int64_t blocks = (rows + JOB - 1) / JOB;
    if ((int64_t)nt > blocks) nt = (int)blocks;
    auto job = [&](int64_t b) {
        const int64_t r0 = b * JOB;
        const int64_t r1 = r0 + JOB < rows ? r0 + JOB : rows;
        expand_rows(tb, packed_host, r0, r1, num_nodes, obs_host, reward_host, done_host, action_host);
    };
    if (nt <= 1) { for (int64_t b = 0; b < blocks; b++) job(b); return ORLG_OK; }
    std::lock_guard<std::mutex> lk(g_pool_mu);
    g_pool.run(nt, blocks, job);
    return ORLG_OK;
}

int orlg_rollout_host(orlg_env *env, int steps, int policy, float *obs_host, float *reward_host, uint8_t *done_host,
                      int32_t *actions_host, int chunk_steps, int threads, orlg_stream stream) {
    if (!env) return fail(ORLG_E_INVALID, "null handle");
    if (steps <= 0) return steps == 0 ? ORLG_OK : fail(ORLG_E_INVALID, "steps must be >= 0");
    const bool replay = policy == ORLG_POLICY_REPLAY;       // actions_host is then the INPUT [steps, num_envs, action_dim]
    if (replay && !actions_host) return fail(ORLG_E_INVALID, "ORLG_POLICY_REPLAY needs the actions");
    DeviceGuard guard(env->device);
    Params &p = env->p;
    cudaStream_t s = (cudaStream_t)stream;
    const int chunk = chunk_steps > 0 ? chunk_steps : 4;
    const size_t rows = (size_t)chunk * p.n;
    constexpr int NB = RO_HOST_BUFFERS, AHEAD = RO_HOST_BUFFERS - 1;      // the device runs up to AHEAD chunks ahead of the host decoder
    const size_t adim = (size_t)orlg_action_dim(env);
    HostPipeline &hp = env->host_pipe;
    if (int rc0 = hp.reserve(rows, replay, adim)) return rc0;
    const int nchunks = (steps + chunk - 1) / chunk;
    const size_t D = (size_t)p.obs_dim;
    cudaStream_t sc = hp.copy_stream;
    // chunk c: [user stream] H2D of its actions, the rollout kernel -> [copy stream] D2H of its records.  The kernel
    // of chunk c + 1 overlaps the copy of chunk c; buffer b = c % NB is reused by chunk c + NB, whose kernel waits for the copy
    // of chunk c (event) and which is only enqueued after the host has decoded chunk c (program order below).
    auto enqueue = [&](int c) -> int {
        const int b = c % NB, t0 = c * chunk, tc = steps - t0 < chunk ? steps - t0 : chunk;
        if (replay)
            CUDA_OK(cudaMemcpyAsync(hp.act_dev[b], actions_host + (size_t)t0 * p.n * adim, (size_t)tc * p.n * adim * sizeof(int32_t),
                                    cudaMemcpyHostToDevice, s));
        if (c >= NB) CUDA_OK(cudaStreamWaitEvent(s, hp.pk_ev[b], 0));
        int rc = rollout_impl(env, tc, policy, nullptr, nullptr, nullptr, replay ? hp.act_dev[b] : nullptr,
                              reinterpret_cast<uint32_t *>(hp.pk_dev[b]), nullptr, stream);
        if (rc) return rc;
        CUDA_OK(cudaEventRecord(hp.k_ev[b], s));
        CUDA_OK(cudaStreamWaitEvent(sc, hp.k_ev[b], 0));
        CUDA_OK(cudaMemcpyAsync(hp.pk_host[b], hp.pk_dev[b], (size_t)tc * p.n * 32, cudaMemcpyDeviceToHost, sc));
        CUDA_OK(cudaEventRecord(hp.pk_ev[b], sc));
        return ORLG_OK;
    };
    for (int c = 0; c < AHEAD && c < nchunks; c++) { int rc = enqueue(c); if (rc) return rc; }
    for (int c = 0; c < nchunks; c++) {
        if (c + AHEAD < nchunks) { int rc = enqueue(c + AHEAD); if (rc) return rc; }
        const int b = c % NB, t0 = c * chunk, tc = steps - t0 < chunk ? steps - t0 : chunk;
        CUDA_OK(cudaEventSynchronize(hp.pk_ev[b]));
        const size_t off = (size_t)t0 * p.n;
        int rc = orlg_expand_packed(reinterpret_cast<const uint32_t *>(hp.pk_host[b]), (int64_t)tc * p.n, p.N, p.S,
                                    obs_host ? obs_host + off * D : nullptr, reward_host ? reward_host + off : nullptr,
                                    done_host ? done_host + off : nullptr, (actions_host && !replay) ? actions_host + off : nullptr, threads);
        if (rc) return rc;
    }
    // the user's stream must not run ahead of the copies that still read the record buffers (a later call reuses them)
    CUDA_OK(cudaStreamWaitEvent(s, hp.pk_ev[(nchunks - 1) % NB], 0));
    return ORLG_OK;
}

// ---------------------------------------------------------------- MLP policies on the tensor cores (orlg_policy.cuh)
struct orlg_policy {
    PolicyParams pp;
    int device;
    size_t smem;
    bool general;                     // ORLG_POLICY_GENERAL at orlg_policy_create: the run-time (H, L) instance also for 5 x 128
    void *w_dev = nullptr, *b_dev = nullptr;

    ~orlg_policy() { cudaFree(w_dev); cudaFree(b_dev); }
};

}  // extern "C"

// The one place that picks the kernel instance of a handle: the shipped agent's 5 x 128 has one compiled for it, every other
// architecture runs the instance that reads H and L from PolicyParams.
template <bool SAMPLE>
static decltype(&mlp_policy_kernel<SAMPLE, 0, 0>) policy_kernel(const orlg_policy *pol) {
    if (pol->pp.H == 128 && pol->pp.L == 5 && !pol->general) return mlp_policy_kernel<SAMPLE, 128, 5>;
    return mlp_policy_kernel<SAMPLE, 0, 0>;
}

extern "C" {

static unsigned short f32_to_bf16(float f) {          // round to nearest even
    unsigned u;
    std::memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (unsigned short)((u >> 16) | 0x40u);      // NaN
    return (unsigned short)((u + 0x7fffu + ((u >> 16) & 1u)) >> 16);
}

int orlg_policy_create(int device, int obs_dim, int hidden, int n_hidden_layers, int n_actions, const float *weights,
                       const float *biases, orlg_policy **out) {
    if (!weights || !biases || !out) return fail(ORLG_E_INVALID, "null argument");
    *out = nullptr;
    if (obs_dim < 2 || obs_dim > PL_K0 || (obs_dim & 1) || n_actions < 1 || n_actions + 1 > PL_NOUT)
        return fail(ORLG_E_UNSUPPORTED, "the fused policy kernel is built for obs_dim <= 64 (even), <= 15 actions; got obs_dim " +
                                            std::to_string(obs_dim) + ", " + std::to_string(n_actions) + " actions");
    if (hidden < 16 || hidden > PL_HMAX || hidden % 16)
        return fail(ORLG_E_UNSUPPORTED, "the fused policy kernel needs a hidden width that is a multiple of 16 in 16..128; got " +
                                            std::to_string(hidden));
    if (n_hidden_layers < 1)
        return fail(ORLG_E_UNSUPPORTED, "the fused policy kernel needs at least one hidden layer; got " + std::to_string(n_hidden_layers));
    const int H = hidden, L = n_hidden_layers;
    const size_t smem = pl_smem_bytes(H, L);
    if (smem > (size_t)PL_SMEM_MAX)         // all weights stay resident in shared memory
        return fail(ORLG_E_UNSUPPORTED, "the fused policy kernel needs " + std::to_string(smem) + " bytes of shared memory, " +
                                            std::to_string(PL_SMEM_MAX) + " available, for " + std::to_string(L) +
                                            " hidden layers of " + std::to_string(H));
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev) return fail(ORLG_E_CUDA, "no such CUDA device");
    DeviceGuard guard(device);
    // bf16 weights in the shared-memory operand layout of the kernel: layer l is an [N x K] K-major operand, K = 64 (the
    // padded observation) for layer 0, H after it
    const size_t bytes = pl_weight_bytes(H, L);
    std::vector<unsigned short> blob(bytes / 2, 0);
    std::vector<float> bias((size_t)L * H + PL_NOUT, 0.0f);
    const float *w = weights, *b = biases;
    size_t off = 0;
    for (int l = 0; l < L; l++) {
        const int K = l == 0 ? obs_dim : H, Kp = l == 0 ? PL_K0 : H;
        for (int r = 0; r < H; r++)
            for (int k = 0; k < K; k++) blob[(off + pl_operand_offset(H, r, k)) / 2] = f32_to_bf16(w[(size_t)r * K + k]);
        for (int r = 0; r < H; r++) bias[(size_t)l * H + r] = b[r];
        w += (size_t)H * K; b += H; off += (size_t)H * Kp * 2;
    }
    for (int r = 0; r < n_actions + 1; r++)                     // action_net rows, then value_net
        for (int k = 0; k < H; k++) blob[(off + pl_operand_offset(PL_NOUT, r, k)) / 2] = f32_to_bf16(w[(size_t)r * H + k]);
    for (int r = 0; r < n_actions + 1; r++) bias[(size_t)L * H + r] = b[r];
    std::unique_ptr<orlg_policy, int (*)(orlg_policy *)> pol(new orlg_policy(), orlg_policy_destroy);
    pol->device = device;
    pol->general = std::getenv("ORLG_POLICY_GENERAL") != nullptr;
    if (cudaMalloc(&pol->w_dev, bytes) != cudaSuccess || cudaMalloc(&pol->b_dev, bias.size() * 4) != cudaSuccess ||
        cudaMemcpy(pol->w_dev, blob.data(), bytes, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(pol->b_dev, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess)
        return fail(ORLG_E_NOMEM, "policy weight upload failed");
    pol->pp.w_blob = reinterpret_cast<const uint4 *>(pol->w_dev);
    pol->pp.w_bytes = (int)bytes;
    pol->pp.bias = reinterpret_cast<const float *>(pol->b_dev);
    pol->pp.obs_dim = obs_dim; pol->pp.n_actions = n_actions;
    pol->pp.H = H; pol->pp.L = L;
    pol->smem = smem;
    // the attribute only raises a kernel's limit: a larger policy made earlier on this device keeps its launches valid
    int have_act = 0, have_sample = 0;
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, policy_kernel<false>(pol.get())) == cudaSuccess) have_act = fa.maxDynamicSharedSizeBytes;
    if (cudaFuncGetAttributes(&fa, policy_kernel<true>(pol.get())) == cudaSuccess) have_sample = fa.maxDynamicSharedSizeBytes;
    if ((have_act < (int)smem &&
         cudaFuncSetAttribute(policy_kernel<false>(pol.get()), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) ||
        (have_sample < (int)smem &&
         cudaFuncSetAttribute(policy_kernel<true>(pol.get()), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess))
        return fail(ORLG_E_CUDA, "cudaFuncSetAttribute(policy kernel shared memory) failed");
    *out = pol.release();
    return ORLG_OK;
}

}  // extern "C"

// one launch of the fused policy kernel over n rows: a persistent CTA per SM (each walks PL_GROUPS tile streams)
template <bool SAMPLE>
static int launch_policy(const orlg_policy *pol, const float *obs_dev, int n, int32_t *actions_dev, float *logits_dev,
                         const PolicyDraw &dr, cudaStream_t s) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, pol->device);
    const int pairs = ((n + PL_TILE - 1) / PL_TILE + PL_GROUPS - 1) / PL_GROUPS;
    cudaLaunchConfig_t cfg = pdl_config(pairs < sms ? pairs : sms, PL_WG * PL_GROUPS, pol->smem, s);
    int *actions = actions_dev;
    CUDA_OK(cudaLaunchKernelEx(&cfg, policy_kernel<SAMPLE>(pol), pol->pp, obs_dev, n, actions, logits_dev, dr));
    return ORLG_OK;
}

extern "C" {

int orlg_policy_act(orlg_policy *pol, const float *obs_dev, int n, int32_t *actions_dev, float *logits_dev, orlg_stream stream) {
    if (!pol || !obs_dev || !actions_dev || n < 0) return fail(ORLG_E_INVALID, "null policy or buffer");
    if (n == 0) return ORLG_OK;
    DeviceGuard guard(pol->device);
    PolicyDraw dr;
    std::memset(&dr, 0, sizeof(dr));
    return launch_policy<false>(pol, obs_dev, n, actions_dev, logits_dev, dr, (cudaStream_t)stream);
}

static PolicyDraw policy_draw(const orlg_policy_draw &d, float *log_prob_dev, float *value_dev) {
    PolicyDraw dr;
    std::memset(&dr, 0, sizeof(dr));
    dr.seed = d.seed;
    dr.counter_dev = d.counter_dev;
    dr.counter = d.counter;
    dr.deterministic = d.deterministic ? 1 : 0;
    dr.row_id_base = d.row_id_base;
    dr.log_prob = log_prob_dev;
    dr.value = value_dev;
    return dr;
}

int orlg_policy_sample(orlg_policy *pol, const float *obs_dev, int n, const orlg_policy_draw *draw, int32_t *actions_dev,
                       float *log_prob_dev, float *value_dev, orlg_stream stream) {
    if (!pol || !obs_dev || !draw || n < 0) return fail(ORLG_E_INVALID, "null policy, observation buffer or draw");
    if (n == 0) return ORLG_OK;
    DeviceGuard guard(pol->device);
    return launch_policy<true>(pol, obs_dev, n, actions_dev, nullptr, policy_draw(*draw, log_prob_dev, value_dev), (cudaStream_t)stream);
}

int orlg_rollout_policy(orlg_env *env, int steps, orlg_policy *actor, orlg_policy *critic, uint64_t seed, int deterministic,
                        float *obs_dev, int32_t *actions_dev, float *log_prob_dev, float *value_dev,
                        float *reward_dev, uint8_t *done_dev, orlg_stream stream) {
    return orlg_rollout_policy_info(env, steps, actor, critic, seed, deterministic, obs_dev, actions_dev, log_prob_dev, value_dev,
                                    reward_dev, done_dev, nullptr, stream);
}

int orlg_rollout_policy_info(orlg_env *env, int steps, orlg_policy *actor, orlg_policy *critic, uint64_t seed, int deterministic,
                             float *obs_dev, int32_t *actions_dev, float *log_prob_dev, float *value_dev,
                             float *reward_dev, uint8_t *done_dev, const orlg_info_out *info, orlg_stream stream) {
    if (!env || !actor) return fail(ORLG_E_INVALID, "null env or actor handle");
    const Params &p = env->p;
    if (p.kind != ORLG_DEEPRMSA) return fail(ORLG_E_UNSUPPORTED, "orlg_rollout_policy drives DeepRMSA-v0 (the env kind with a tensor observation)");
    if (p.obs_f64) return fail(ORLG_E_UNSUPPORTED, "orlg_rollout_policy needs float32 observations (the policy kernel reads float32)");
    if (actor->pp.obs_dim != p.obs_dim)
        return fail(ORLG_E_INVALID, "actor obs_dim " + std::to_string(actor->pp.obs_dim) + " != env obs_dim " + std::to_string(p.obs_dim));
    const int n_act = p.k * p.J + p.allow_rejection;
    if (actor->pp.n_actions != n_act)
        return fail(ORLG_E_INVALID, "actor n_actions " + std::to_string(actor->pp.n_actions) + " != k * j + allow_rejection = " + std::to_string(n_act));
    if (critic && critic->pp.obs_dim != p.obs_dim)
        return fail(ORLG_E_INVALID, "critic obs_dim " + std::to_string(critic->pp.obs_dim) + " != env obs_dim " + std::to_string(p.obs_dim));
    if (actor->device != env->device || (critic && critic->device != env->device))
        return fail(ORLG_E_INVALID, "policy and env handles live on different devices");
    if (!obs_dev) return fail(ORLG_E_INVALID, "orlg_rollout_policy needs obs_dev (the policy reads it)");
    if (steps < 0) return fail(ORLG_E_INVALID, "steps must be >= 0");
    if (p.traffic == ORLG_TRAFFIC_TRACE && p.trace == nullptr) return fail(ORLG_E_INVALID, "trace traffic selected but orlg_set_trace was not called");
    if (const char *why = info_refusal(p, info)) return fail(ORLG_E_UNSUPPORTED, why);
    DeviceGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = ensure_canonical(env, s);          // the handle may have been stepped by the persistent rollout kernel
    if (!rc) rc = orlg_observation(env, obs_dev, stream);
    if (rc) return rc;
    if (!actions_dev && steps > 0 && !env->ro_actions) {
        rc = dev_alloc(env, &env->ro_actions, (size_t)p.n, false);
        if (rc) return rc;
    }
    const size_t n = (size_t)p.n, row = n * (size_t)p.obs_dim;
    orlg_policy_draw d;
    d.seed = seed; d.counter_dev = p.req_index; d.counter = 0; d.deterministic = deterministic; d.row_id_base = p.env_id_base;
    for (int t = 0; t < steps; t++) {
        const float *o = obs_dev + (size_t)t * row;
        int32_t *a = actions_dev ? actions_dev + (size_t)t * n : env->ro_actions;
        float *v = value_dev ? value_dev + (size_t)t * n : nullptr;
        rc = launch_policy<true>(actor, o, p.n, a, nullptr, policy_draw(d, log_prob_dev ? log_prob_dev + (size_t)t * n : nullptr,
                                                                       critic ? nullptr : v), s);
        if (!rc && critic && v) rc = launch_policy<true>(critic, o, p.n, nullptr, nullptr, policy_draw(d, nullptr, v), s);
        if (!rc) rc = step_impl(env, a, -1, nullptr, obs_dev + (size_t)(t + 1) * row, reward_dev ? reward_dev + (size_t)t * n : nullptr,
                                done_dev ? done_dev + (size_t)t * n : nullptr, nullptr,
                                info && info->counters_dev ? info->counters_dev + (size_t)t * n * 8 : nullptr, stream);
        if (!rc && info) rc = info_row(env, info, t, stream);
        if (rc) return rc;
    }
    if (value_dev)                              // the bootstrap value of the last observation
        rc = launch_policy<true>(critic ? critic : actor, obs_dev + (size_t)steps * row, p.n, nullptr, nullptr,
                                 policy_draw(d, nullptr, value_dev + (size_t)steps * n), s);
    return rc;
}

int64_t orlg_request_index(const orlg_env *env) { return env ? (int64_t)env->p.lockstep_ridx : -1; }

int orlg_policy_destroy(orlg_policy *pol) {
    if (!pol) return ORLG_OK;
    DeviceGuard guard(pol->device);
    delete pol;
    return ORLG_OK;
}

// ---------------------------------------------------------------- checkpoint / resume (SURVEY.md section 5)
int64_t orlg_state_save_bytes(const orlg_env *env) {
    int64_t b = 16;                                   // header: lockstep request index, number of arrays
    for (const auto &a : env->state_allocs) b += (int64_t)((a.second + 15) / 16 * 16);
    return b;
}

int orlg_state_save(orlg_env *env, void *buf_dev, orlg_stream stream) {
    if (!env || !buf_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    int rc = ensure_canonical(env, s);               // the saved form is the canonical one
    if (rc) return rc;
    const unsigned long long hdr[2] = {env->p.lockstep_ridx, (unsigned long long)env->state_allocs.size()};
    CUDA_OK(cudaMemcpyAsync(buf_dev, hdr, 16, cudaMemcpyHostToDevice, s));
    CUDA_OK(cudaStreamSynchronize(s));               // hdr lives on this stack frame
    size_t off = 16;
    for (const auto &a : env->state_allocs) {
        CUDA_OK(cudaMemcpyAsync(reinterpret_cast<unsigned char *>(buf_dev) + off, a.first, a.second, cudaMemcpyDeviceToDevice, s));
        off += (a.second + 15) / 16 * 16;
    }
    return ORLG_OK;
}

int orlg_state_load(orlg_env *env, const void *buf_dev, orlg_stream stream) {
    if (!env || !buf_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long hdr[2] = {0, 0};
    CUDA_OK(cudaMemcpyAsync(hdr, buf_dev, 16, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
    if (hdr[1] != env->state_allocs.size()) return fail(ORLG_E_INVALID, "checkpoint does not match this handle (different configuration)");
    size_t off = 16;
    for (const auto &a : env->state_allocs) {
        CUDA_OK(cudaMemcpyAsync(a.first, reinterpret_cast<const unsigned char *>(buf_dev) + off, a.second, cudaMemcpyDeviceToDevice, s));
        off += (a.second + 15) / 16 * 16;
    }
    env->p.lockstep_ridx = (unsigned)hdr[0];
    env->ro_valid = false;                           // the loaded tables are canonical
    return ORLG_OK;
}

int orlg_reduce_counters(orlg_env *env, int64_t *sums_dev, orlg_stream stream) {
    if (!env || !sums_dev) return fail(ORLG_E_INVALID, "null handle or buffer");
    DeviceGuard guard(env->device);
    cudaStream_t s = (cudaStream_t)stream;
    CUDA_OK(cudaMemsetAsync(sums_dev, 0, 9 * sizeof(int64_t), s));
    int blocks = (env->p.n + 255) / 256;
    if (blocks > 592) blocks = 592;
    reduce_counters_kernel<<<blocks, 256, 0, s>>>(env->p, reinterpret_cast<unsigned long long *>(sums_dev));
    CUDA_OK(cudaGetLastError());
    return ORLG_OK;
}

}  // extern "C"
