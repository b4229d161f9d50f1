/*
 * orlg.h -- C ABI of the B200-native batched Optical RL-Gym step path (liborlg.so).
 *
 * The reference (carlosnatalino/optical-rl-gym) has no FFI: its "operator API" for this
 * path is the gym.Env method set of RWAEnv / RMSAEnv / DeepRMSAEnv / RMCSAEnv.  Each entry
 * point below names the reference method(s) it replaces for a whole batch of independent
 * environments (file:line relative to the reference tree).  Plain pointers and sizes only;
 * every *_dev pointer is caller-owned DEVICE memory (e.g. a torch tensor's data_ptr()),
 * every call is stream-ordered on the cudaStream_t passed as `stream` (0 = legacy default
 * stream) and never synchronises.  Return value: 0 on success, <0 = ORLG_E_* (see
 * orlg_last_error()).  One host thread per handle.
 */
#ifndef ORLG_H
#define ORLG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORLG_VERSION 1

/* environment kinds = the reference's gym ids (optical_rl_gym/__init__.py:3-26) */
enum { ORLG_RWA = 0, ORLG_RMSA = 1, ORLG_DEEPRMSA = 2, ORLG_RMCSA = 3 };
/* request sources */
enum { ORLG_TRAFFIC_TRACE = 0, ORLG_TRAFFIC_PHILOX = 1 };
/* observation element type (DeepRMSA): f64 reproduces deeprmsa_env.py:60-121 bit-for-bit */
enum { ORLG_OBS_F32 = 0, ORLG_OBS_F64 = 1 };
/* heuristic action sources (rmsa_env.py:747-803, rwa_env.py:425-502, deeprmsa_env.py:135-155,
 * rmcsa_env.py:882-911) */
enum { ORLG_HEUR_SP_FF = 0, ORLG_HEUR_SAP_FF = 1, ORLG_HEUR_LLP_FF = 2, ORLG_HEUR_SAP_LF = 3 };
/* error codes */
enum { ORLG_OK = 0, ORLG_E_INVALID = -1, ORLG_E_UNSUPPORTED = -2, ORLG_E_CUDA = -3, ORLG_E_NOMEM = -4 };
/* per-environment soft error bits (orlg_error_flags) */
enum {
    ORLG_ERR_TRACE_EXHAUSTED = 1,  /* the recorded trace has no request left */
    ORLG_ERR_HEAP_OVERFLOW = 2,    /* more live services than heap_capacity: the request was blocked */
    ORLG_ERR_NO_SUCH_PATH = 4,     /* action chose path >= number of candidate paths (reference: IndexError) */
    ORLG_ERR_LOCKSTEP = 8,         /* internal: an env's request counter left the handle's lockstep count */
    ORLG_ERR_STATS_ORDER = 16,     /* > 24 services released in one step: float statistics updated out of time order */
    ORLG_ERR_TRACE_RANGE = 32      /* orlg_rollout replay: a trace bit rate above 127 Gb/s (clamped) */
};

typedef struct orlg_env orlg_env;     /* opaque handle: owns all per-environment state in HBM */
typedef void *orlg_stream;            /* cudaStream_t */

/* Constructor keyword arguments of the reference envs (optical_network_env.py:14-25,
 * rmsa_env.py:29-46, deeprmsa_env.py:10-21, rwa_env.py:19-31, rmcsa_env.py:29-49). */
typedef struct orlg_config {
    int32_t kind;              /* ORLG_RWA ... */
    int32_t num_envs;          /* environments held by this handle (this GPU's shard) */
    int64_t env_id_base;       /* global id of local env 0: Philox streams are keyed by global id */
    int32_t num_slots;         /* num_spectrum_resources */
    int32_t num_cores;         /* num_spatial_resources (RMCSA), else 1 */
    int32_t j;                 /* DeepRMSA: candidate blocks per path */
    int32_t episode_length;
    int32_t allow_rejection;
    int32_t bit_rate_lo, bit_rate_hi;   /* continuous bit-rate selection: randint bounds */
    int32_t traffic;           /* ORLG_TRAFFIC_* */
    int32_t obs_dtype;         /* ORLG_OBS_* */
    int32_t auto_reset;        /* VecEnv semantics: reset(only_episode_counters=True) right after done */
    int32_t heap_capacity;     /* max live services per env; 0 = derive from the load */
    uint64_t seed;             /* Philox key */
    double channel_width;      /* GHz per slot */
    double mean_holding;       /* mean_service_holding_time */
    double mean_iat;           /* mean_service_inter_arrival_time = holding / load */
    double worst_xt;           /* RMCSA worst aggregate inter-core crosstalk (dB), before the +4 dB margin */
} orlg_config;

/* Host-side topology tables (what topology.graph["ksp"/"modulations"] holds after
 * examples/create_topology.py:96-147).  HOST pointers, copied by orlg_create. */
typedef struct orlg_tables {
    int32_t num_nodes, num_links, k_paths, num_paths, num_mods, num_bit_rates;
    const int32_t *pair_first;     /* [N*N] first path row of (src,dst) */
    const int32_t *pair_count;     /* [N*N] candidate paths of the pair (<= k_paths) */
    const int32_t *path_hops;      /* [P] */
    const int32_t *path_se;        /* [P] spectral efficiency of Path.best_modulation */
    const int32_t *path_mod;       /* [P] index of best_modulation */
    const int32_t *path_link_ptr;  /* [P+1] CSR */
    const int32_t *path_links;     /* link index of every hop */
    const double *path_length;     /* [P] km */
    const int32_t *mod_se;         /* [M] */
    const double *mod_osnr;        /* [M] minimum_osnr */
    const double *mod_xt;          /* [M] inband_xt */
    const double *node_prob;       /* [N] node_request_probabilities */
    const int32_t *bit_rates;      /* [num_bit_rates] discrete bit-rate selection (0 = continuous) */
    const double *bit_rate_prob;   /* [num_bit_rates] */
    const int32_t *link_order;     /* [E] link indices in topology.edges() iteration order (np.mean over links); NULL = 0..E-1 */
} orlg_tables;

/* One recorded request of a trace (ORLG_TRAFFIC_TRACE): what _next_service draws,
 * rmsa_env.py:545-573.  arrival is absolute time. */
typedef struct orlg_request {
    double arrival;
    double holding;
    int32_t src, dst, bit_rate, reserved;
} orlg_request;

/* ---- lifetime ------------------------------------------------------------------------- */
/* gym.make(id, **env_args) for num_envs environments on CUDA device `device`
 * (optical_network_env.py:14-74 + the env constructors).  Does NOT reset: call orlg_reset(full=1). */
int orlg_create(const orlg_config *cfg, const orlg_tables *tables, int device, orlg_env **out);
int orlg_destroy(orlg_env *env);
const char *orlg_last_error(void);
int orlg_version(void);

/* ---- shape queries -------------------------------------------------------------------- */
int orlg_action_dim(const orlg_env *env);   /* 1 DeepRMSA (Discrete), 2 RMSA/RWA, 4 RMCSA (MultiDiscrete) */
int orlg_obs_dim(const orlg_env *env);      /* 1 + 2N + (2j+3)k for DeepRMSA (deeprmsa_env.py:34-40), else 0 */
int orlg_mask_words(const orlg_env *env);   /* 32-bit words per (core, link) in orlg_export_state */
int orlg_heap_capacity(const orlg_env *env);
int64_t orlg_state_bytes(const orlg_env *env);

/* Which compiled kernel instances the handle runs (fixed at orlg_create, except last_rollout_persistent). */
typedef struct orlg_kernel_info {
    int32_t wide;              /* > 32 links, > 128 slots or > 8 paths: CSR link lists, multi-word masks */
    int32_t fast;              /* DeepRMSA: the per-step fast kernel (deeprmsa_fast_kernel) */
    int32_t hot;               /* ... and its steady-state specialisation is allowed */
    int32_t rollout_kernel;    /* the persistent rollout kernel applies to this configuration */
    int32_t rollout_lanes;     /* envs per warp of the rollout kernel: 8 or 32 (environment ORLG_RO_LPW at orlg_create) */
    int32_t link_template;     /* link count the non-wide kernels are compiled for: 22 (NSFNET), 0 = read at run time */
    int32_t last_rollout_persistent;   /* 1: the last orlg_rollout* call ran the persistent kernel, 0: per-step launches or none yet */
} orlg_kernel_info_t;
int orlg_kernel_info(const orlg_env *env, orlg_kernel_info_t *out);

/* ---- traffic -------------------------------------------------------------------------- */
/* env.seed(seed) (optical_network_env.py:205-210): new key of the counter-based request stream from the next
 * request on; the state of the environments is not touched (like the reference, which only replaces its rng). */
int orlg_seed(orlg_env *env, uint64_t seed);
/* Replay mode: trace_dev[e * trace_len + i] is the i-th request of env e since the last full
 * reset.  The buffer must stay valid while the handle steps. */
int orlg_set_trace(orlg_env *env, const orlg_request *trace_dev, int64_t trace_len);

/* ---- the hot path --------------------------------------------------------------------- */
/* env.reset(only_episode_counters = !full) for every env (rmsa_env.py:284-359,
 * rwa_env.py:164-208, rmcsa_env.py:386-483).  obs_dev (may be NULL): [num_envs, obs_dim]. */
int orlg_reset(orlg_env *env, int full, void *obs_dev, orlg_stream stream);

/* obs, reward, done, info = env.step(action) for every env (rmsa_env.py:163-282,
 * deeprmsa_env.py:48-58, rwa_env.py:101-162, rmcsa_env.py:209-339), including _next_service and
 * the release loop (rmsa_env.py:545-597).
 *   actions_dev   int32 [num_envs, action_dim]
 *   obs_dev       f32/f64 [num_envs, obs_dim]           (NULL: skip; ignored for obs_dim == 0)
 *   reward_dev    f32 [num_envs]                         (NULL: skip)
 *   done_dev      u8  [num_envs]                         (NULL: skip)
 *   decision_dev  int32 [num_envs, 6] = accepted, path row, initial slot, slots, core, modulation
 *                 (-1 where not applicable)              (NULL: skip)
 *   info_dev      int64 [num_envs, 8] = the counters at the moment the reference builds `info`:
 *                 processed, accepted, episode processed, episode accepted, bit_rate requested,
 *                 provisioned, episode requested, episode provisioned (NULL: skip)            */
int orlg_step(orlg_env *env, const int32_t *actions_dev, void *obs_dev, float *reward_dev, uint8_t *done_dev,
              int32_t *decision_dev, int64_t *info_dev, orlg_stream stream);

/* T consecutive steps in ONE call: T iterations of { action = policy(env); obs, reward, done, _ = env.step(action) }
 * (the rollout loop of examples/stable_baselines3/DeepRMSA.ipynb / utils.py:103-141 evaluate_heuristic), every step's
 * results kept:
 *   policy        ORLG_POLICY_RANDOM (orlg_random_actions), an ORLG_HEUR_* id (orlg_heuristic), or ORLG_POLICY_REPLAY
 *                 (actions_dev holds the actions to apply: with trace traffic this replays a recorded reference run)
 *   obs_dev       [steps, num_envs, obs_dim]  (NULL: skip)      reward_dev  f32 [steps, num_envs]  (NULL: skip)
 *   done_dev      u8 [steps, num_envs]        (NULL: skip)      actions_dev int32 [steps, num_envs, action_dim] (NULL: skip)
 * Identical results to the step-by-step calls.  For DeepRMSA-v0 on NSFNET-class topologies with Philox traffic and
 * float32 observations the T steps run inside one persistent kernel (state stays on chip); every other configuration
 * issues the per-step kernels. */
enum { ORLG_POLICY_RANDOM = -1, ORLG_POLICY_REPLAY = -2 };   /* REPLAY: actions_dev is the INPUT action sequence [steps, num_envs, action_dim] */
int orlg_rollout(orlg_env *env, int steps, int policy, void *obs_dev, float *reward_dev, uint8_t *done_dev,
                 int32_t *actions_dev, orlg_stream stream);

/* The fourth part of env.step's result, kept for every step of a rollout: row t of each output is what the step-by-step calls
 * give after step t.  Any member may be NULL (not written).  Asking for an output the handle does not have is
 * ORLG_E_UNSUPPORTED, with the message of the per-step entry point. */
typedef struct orlg_info_out {
    int64_t *counters_dev;              /* int64 [steps, num_envs, 8]: at step t exactly what orlg_step's info_dev receives */
    double *stats_dev;                  /* f64 [steps, num_envs, 4]: orlg_enable_stats's values (handles with float statistics) */
    double *bit_rate_blocking_dev;      /* f64 [steps, num_envs, orlg_num_bit_rates + 1]: orlg_bit_rate_blocking (discrete bit rates) */
    double *action_probability_dev;     /* f64 [steps, num_envs, orlg_action_hist_dim]: orlg_action_probability (RWA-v0) */
} orlg_info_out;
/* orlg_rollout (= this call with info NULL) that also keeps every step's info.  The persistent kernel writes the counters
 * itself (64 bytes per env-step); handles with statistics or discrete bit rates already run step by step, and so does an RWA-v0
 * call that asks for action probabilities (about 90 doubles per env-step).  orlg_kernel_info's last_rollout_persistent reports
 * which path ran.  Not offered for orlg_rollout_packed / orlg_rollout_host (a 32-byte record has no room, and int64 counters
 * would triple the bytes that cross PCIe), nor the decision output of orlg_step. */
int orlg_rollout_info(orlg_env *env, int steps, int policy, void *obs_dev, float *reward_dev, uint8_t *done_dev,
                      int32_t *actions_dev, const orlg_info_out *info, orlg_stream stream);

/* The same rollout with ONE 32-byte record per env-step instead of the float observation: uint32 [steps, num_envs, 8]
 *   w0..w4  per candidate path: first-block start (7 bits, 127 = none) | its length (7) | free slots (7) | free runs (6) | slots needed (5)
 *   w5      bit rate (8) | source << 8 | destination << 16 | candidate paths << 24 | accepted << 28 | done << 29  (request = the NEXT one)
 *   w6      the action taken;   w7 reserved
 * i.e. the integer pre-image of deeprmsa_env.py:60-121 (orlg_observation_int) plus reward / done: 6.75x fewer bytes than the
 * float32 row when the result has to cross PCIe.  DeepRMSA-v0 with k = 5, j = 1 (the persistent-kernel configuration) only. */
int orlg_rollout_packed(orlg_env *env, int steps, int policy, uint32_t *packed_dev, int32_t *actions_dev, orlg_stream stream);
/* HOST function: expands `rows` packed records into what env.step returned for them -- float32 observation rows
 * [rows, 1 + 2 * num_nodes + 25] (bit-identical to the rows orlg_rollout writes), reward f32, done u8, action i32 (any output
 * may be NULL) -- using `threads` host threads (<= 0: all cores). */
int orlg_expand_packed(const uint32_t *packed_host, int64_t rows, int num_nodes, int num_slots, float *obs_host, float *reward_host,
                       uint8_t *done_host, int32_t *action_host, int threads);
/* orlg_rollout with HOST buffers (pageable or pinned): the steps run in chunks on the device while the previous chunk's
 * records cross PCIe and are expanded by a persistent pool of `threads` host threads (<= 0: all cores).  obs_host f32
 * [steps, num_envs, obs_dim] etc.; any output may be NULL.  With ORLG_POLICY_REPLAY actions_host is the INPUT: the action of
 * every env at every step, copied to the device chunk by chunk ahead of the kernel that consumes it. */
int orlg_rollout_host(orlg_env *env, int steps, int policy, float *obs_host, float *reward_host, uint8_t *done_host,
                      int32_t *actions_host, int chunk_steps, int threads, orlg_stream stream);

/* ---- SB3 MlpPolicy agents (the PPO agent of the reference's notebook among them), evaluated on the device ---------- */
/* model.predict(obs, deterministic=True) of an SB3 MlpPolicy: obs -> n_hidden_layers x (Linear hidden + tanh) -> action_net /
 * value_net -> argmax.  The agent the reference trains and ships (examples/stable_baselines3/DeepRMSA.ipynb cell 13:
 * PPO(MlpPolicy, env, policy_kwargs=dict(net_arch=5*[128])); bkp/deeprmsa-ppo-trained/best_model.zip) is 5 x 128; SB3's PPO /
 * A2C default trunk is 2 x 64.  One fused kernel on the tensor cores (bf16 operands, fp32 accumulation), all weights resident
 * in shared memory.  Accepted: obs_dim even in 2..64, n_actions 1..15, hidden a multiple of 16 in 16..128, n_hidden_layers
 * >= 1 with hidden * 64 * 2 + (n_hidden_layers - 1) * hidden^2 * 2 + 16 * hidden * 2 (weights) + 65536 (activations) +
 * (n_hidden_layers * hidden + 16) * 4 + 64 <= 232448 bytes of shared memory (5 x 128 and 6 x 112 fit, 6 x 128 does not);
 * anything else is ORLG_E_UNSUPPORTED.  weights: HOST float32, the nn.Linear matrices [out, in] row-major one after the other
 * (the trunk layers, action_net, value_net); biases likewise.  5 x 128 runs a kernel instance compiled for it (environment
 * ORLG_POLICY_GENERAL at create: the run-time instance the other architectures use, the same results bit for bit). */
typedef struct orlg_policy orlg_policy;
int orlg_policy_create(int device, int obs_dim, int hidden, int n_hidden_layers, int n_actions, const float *weights,
                       const float *biases, orlg_policy **out);
/* actions_dev int32 [n]; logits_dev float32 [n, n_actions + 1] = logits then value (NULL: skip) */
int orlg_policy_act(orlg_policy *pol, const float *obs_dev, int n, int32_t *actions_dev, float *logits_dev, orlg_stream stream);
int orlg_policy_destroy(orlg_policy *pol);

/* What PPO's collect_rollouts needs from the same fused kernel: the action, log softmax(logits)[action] and the value head.
 * Deterministic: the argmax (first maximum), as orlg_policy_act.  Sampling: one Philox4x32-10 block per row with key = seed and
 * counter = (c0, 0, row_id_base + row, 3) (stream 3, DESIGN.md section 5); u = (word 0 >> 8) * 2^-24; the action is the
 * smallest a with u * S < e_0 + ... + e_a, e_a = expf(l_a - max l), S = sum of e_a (the last action if rounding leaves none).
 * A draw is therefore a function of (seed, c0, row id, observation) only. */
typedef struct orlg_policy_draw {
    uint64_t seed;               /* Philox key of the action draws */
    const uint32_t *counter_dev; /* per row: counter word 0 (the env's request index); NULL = `counter` for every row */
    uint32_t counter;
    int32_t deterministic;       /* 1: argmax, as model.predict(deterministic=True); 0: sample from softmax(logits) */
    int64_t row_id_base;         /* counter word 2 of row r = row_id_base + r (the global env id) */
} orlg_policy_draw;
/* actions_dev int32 [n], log_prob_dev f32 [n], value_dev f32 [n]: any may be NULL */
int orlg_policy_sample(orlg_policy *pol, const float *obs_dev, int n, const orlg_policy_draw *draw, int32_t *actions_dev,
                       float *log_prob_dev, float *value_dev, orlg_stream stream);

/* A PPO rollout buffer in one call: steps x { a, log p(a), V(obs) = policy(obs); obs, r, done = env.step(a) } for DeepRMSA-v0
 * with float32 observations (per step the sampling kernel, an optional critic launch and the step kernel, chained by
 * programmatic dependent launch).
 *   obs_dev      f32 [steps + 1, N, obs_dim]  required: obs[0] = observation of the pending request, obs[t+1] = what step t returned
 *   actions_dev  i32 [steps, N]      log_prob_dev f32 [steps, N]      value_dev f32 [steps + 1, N] (value[steps] = bootstrap value)
 *   reward_dev   f32 [steps, N]      done_dev     u8  [steps, N]      (all but obs may be NULL)
 *   critic       NULL = the actor's value head; else a handle whose value head is the critic's (separate SB3 >= 1.8 trunk,
 *                which may have its own width and depth: n_actions = 1, value_net as both head rows)
 * The draws are keyed by (seed, global env id, the env's request index): results do not depend on sharding, on how a rollout is
 * split into calls, or on a checkpoint taken between calls.  deterministic = 1: argmax actions. */
int orlg_rollout_policy(orlg_env *env, int steps, orlg_policy *actor, orlg_policy *critic, uint64_t seed, int deterministic,
                        float *obs_dev, int32_t *actions_dev, float *log_prob_dev, float *value_dev,
                        float *reward_dev, uint8_t *done_dev, orlg_stream stream);
/* orlg_rollout_policy (= this call with info NULL) that also keeps every step's info: counters_dev and stats_dev as in
 * orlg_rollout_info (DeepRMSA-v0 has neither discrete bit rates nor action probabilities). */
int orlg_rollout_policy_info(orlg_env *env, int steps, orlg_policy *actor, orlg_policy *critic, uint64_t seed, int deterministic,
                             float *obs_dev, int32_t *actions_dev, float *log_prob_dev, float *value_dev,
                             float *reward_dev, uint8_t *done_dev, const orlg_info_out *info, orlg_stream stream);
/* requests drawn so far by every env of the handle (all step together): counter word 0 of the draws orlg_rollout_policy
 * makes at its next step.  Host state, no device access. */
int64_t orlg_request_index(const orlg_env *env);

/* Float statistics of `info` (rmsa_env.py:229-264, 439-543, 699-744; RMSA-v0 / DeepRMSA-v0, any topology the handle
 * takes: any link count, up to 512 slots): after this call every orlg_step also writes, per env, float64
 *   stats_dev[env][0..3] = network_compactness, network_compactness_difference,
 *                          avg_link_compactness, avg_link_utilization
 * bit-identical to the reference (same float64 operation order, releases applied in time order, numpy's
 * pairwise mean, recursive above 128 links).  Call before orlg_reset(full = 1).  stats_dev = NULL disables it again.  Bit
 * rates must fit 16 bits (<= 65535).  NSFNET-class handles (<= 32 links, <= 128 slots) run the statistics on the generic
 * kernel instead of the fast one; wide handles on the statistics instance of the wide step kernel, which updates each link
 * with a load / store instead of fire-and-forget reductions.  Both are slower than the default path.  orlg_rollout on a
 * handle with statistics on (fused heuristic, random or replay) runs the same kernels step by step. */
int orlg_enable_stats(orlg_env *env, double *stats_dev);
/* The time-averaged statistics the reference keeps ON the topology graph while it provisions and releases (never returned by
 * step, read by users through env.topology): per link `utilization`, `external_fragmentation`, `compactness`
 * (_update_link_stats: rmsa_env.py:464-543, rmcsa_env.py:591-688 -- one set per link, fed by the core being touched --,
 * rwa_env.py:365-383 -- utilization only) and the graph's `throughput` / `compactness` (_update_network_stats:
 * rmsa_env.py:439-462, rmcsa_env.py:560-589; a no-op in rwa_env.py:351-363).  orlg_enable_link_stats(on = 1) before
 * orlg_reset(full = 1) turns them on for ANY env kind (orlg_enable_stats implies it); orlg_link_stats reads them as of the last
 * step: link_dev f64 [num_envs, links, 3] by link index, graph_dev f64 [num_envs, 2] (either may be NULL).  Bit-identical to
 * the reference (same float64 operation order, releases applied in time order; more than 24 releases in one step set
 * ORLG_ERR_STATS_ORDER).  Any link count, up to 512 slots and 31 cores; same kernels and cost as orlg_enable_stats. */
int orlg_enable_link_stats(orlg_env *env, int on);
int orlg_link_stats(orlg_env *env, double *link_dev, double *graph_dev, orlg_stream stream);

/* env.observation() of the pending request (deeprmsa_env.py:60-121) */
int orlg_observation(orlg_env *env, void *obs_dev, orlg_stream stream);
/* integer pre-image of the observation: int32 [num_envs, k, 2j+3] = (start_b, len_b)*j, n_slots,
 * total free slots, number of free runs; -1 = absent */
int orlg_observation_int(orlg_env *env, int32_t *out_dev, orlg_stream stream);

/* heuristic(env) -> action for every env; `which` = ORLG_HEUR_* */
int orlg_heuristic(orlg_env *env, int which, int32_t *actions_dev, orlg_stream stream);
/* uniform random policy (action_space.sample() equivalent, Philox stream 2, see DESIGN.md) */
int orlg_random_actions(orlg_env *env, int32_t *actions_dev, orlg_stream stream);

/* Discrete bit-rate selection (RMSA-v0, rmsa_env.py:88-110): the per-bit-rate blocking rates and `fairness` of
 * `info` (rmsa_env.py:217-227, 268-273) as of the last orlg_step: float64 [num_envs, orlg_num_bit_rates + 1] =
 * bit_rate_blocking_<rate> in the order of `bit_rates`, then fairness = max - min. */
int orlg_num_bit_rates(const orlg_env *env);    /* 0 unless RMSA-v0 with discrete bit rates */
int orlg_bit_rate_blocking(orlg_env *env, double *out_dev, orlg_stream stream);

/* RWA-v0: info["path_action_probability"] and info["wavelength_action_probability"] (rwa_env.py:148-151), the normalised
 * marginals of the actions_output histogram (rwa_env.py:52-58, 103) as of the last orlg_step: float64
 * [num_envs, orlg_action_hist_dim] = (k + rej) path entries, then (W + rej) wavelength entries (rej = allow_rejection).
 * An action outside the histogram (IndexError in the reference) is not counted and sets ORLG_ERR_NO_SUCH_PATH. */
int orlg_action_hist_dim(const orlg_env *env);  /* 0 unless RWA-v0 */
int orlg_action_probability(orlg_env *env, double *out_dev, orlg_stream stream);

/* ---- gym wrappers of the reference, batched (SURVEY.md row f2) ---------------------------- */
/* SimpleMatrixObservation.observation (rmsa_env.py:806-837, rmcsa_env.py:914-947) of every env:
 * uint8 [num_envs, orlg_matrix_obs_dim] = one-hot(min(src_id, dst_id)) [nodes], one-hot(max(src_id, dst_id))
 * [nodes], available_slots flattened as (core, link, slot), 1 = free */
int orlg_matrix_obs_dim(const orlg_env *env);   /* 2*nodes + cores*links*slots */
int orlg_matrix_observation(orlg_env *env, uint8_t *out_dev, orlg_stream stream);
/* PathOnlyFirstFitAction.action (rmsa_env.py:840-874, rwa_env.py:505-536): path_actions_dev int32 [num_envs]
 * (path index, anything else = reject) -> actions_dev int32 [num_envs, 2] = (path, first-fit slot) or (k, S).
 * RMSA-v0 scans range(0, S - n) like the reference (never the last feasible start), RWA-v0 range(W). */
int orlg_path_only_first_fit(orlg_env *env, const int32_t *path_actions_dev, int32_t *actions_dev, orlg_stream stream);

/* ---- checkpoint / resume ------------------------------------------------------------------ */
/* Every per-environment state array of the handle (masks, clocks, pending requests, counters, release-event tables, ...) as one
 * opaque device buffer of orlg_state_save_bytes(env) bytes; orlg_state_load restores it into a handle created with the same
 * configuration (seed and trace are configuration, not state).  Stream-ordered except for one 16-byte header copy. */
int64_t orlg_state_save_bytes(const orlg_env *env);
int orlg_state_save(orlg_env *env, void *buf_dev, orlg_stream stream);
int orlg_state_load(orlg_env *env, const void *buf_dev, orlg_stream stream);

/* ---- introspection (what heuristics / tests read from the reference env object) -------- */
/* counters after the last step: int64 [num_envs, 8], same order as info_dev */
int orlg_get_counters(orlg_env *env, int64_t *counters_dev, orlg_stream stream);
/* env.current_service: requests_dev [num_envs], service_id_dev int32 [num_envs] (either may be NULL) */
int orlg_get_requests(orlg_env *env, orlg_request *requests_dev, int32_t *service_id_dev, orlg_stream stream);
/* topology.graph["available_slots"] bit-packed: uint32 [num_envs, cores*links, mask_words] (bit s of
 * word s/32 = slot s free); spectrum_slots_allocation: int32 [num_envs, cores, links, slots];
 * current_time f64 [num_envs]; len(_events) int32 [num_envs].  Any pointer may be NULL. */
int orlg_export_state(orlg_env *env, uint32_t *masks_dev, int32_t *alloc_dev, double *now_dev, int32_t *nheap_dev,
                      orlg_stream stream);
int orlg_error_flags(orlg_env *env, uint32_t *flags_dev, orlg_stream stream);
/* per-device sums over envs of the 8 counters + number of envs with error flags: int64 [9]
 * (input of the cross-GPU all-reduce of episode statistics) */
int orlg_reduce_counters(orlg_env *env, int64_t *sums_dev, orlg_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* ORLG_H */
