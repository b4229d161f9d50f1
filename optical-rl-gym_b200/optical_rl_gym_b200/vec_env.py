"""Batched drop-in for the reference's gym envs: N independent environments stepped by one
CUDA kernel launch, with observations / rewards / dones returned as device tensors.

API shape: Stable-Baselines3 ``VecEnv`` protocol (``num_envs``, ``reset``, ``step_async`` /
``step_wait`` / ``step``, ``seed``, ``close``, ``get_attr`` ...) over the reference's
constructor keywords (``optical_network_env.py:14-25``, ``rmsa_env.py:29-46``,
``deeprmsa_env.py:10-21``, ``rwa_env.py:19-31``, ``rmcsa_env.py:29-49``) and gym ids
(``optical_rl_gym/__init__.py:3-26``).  Differences by design (DESIGN.md): ``info`` is a
mapping of ``[N]`` tensors instead of a list of dicts; auto-reset on ``done`` performs the
reference's ``reset(only_episode_counters=True)`` (``rmsa_env.py:284-330``).
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple, Optional

import numpy as np
import torch

from . import _native as nat
from . import spaces
from .topology import TopologyTables

_DEFAULTS = {
    "RMSA-v0": dict(episode_length=1000, load=10.0, mean_service_holding_time=10800.0, num_spectrum_resources=100,
                    bit_rate_selection="continuous", bit_rates=(10, 40, 100), bit_rate_probabilities=None,
                    node_request_probabilities=None, bit_rate_lower_bound=25.0, bit_rate_higher_bound=100.0,
                    seed=None, allow_rejection=False, reset=True, channel_width=12.5),
    "DeepRMSA-v0": dict(j=1, episode_length=1000, mean_service_holding_time=25.0, mean_service_inter_arrival_time=0.1,
                        num_spectrum_resources=100, node_request_probabilities=None, seed=None, allow_rejection=False),
    "RWA-v0": dict(episode_length=1000, load=10.0, mean_service_holding_time=10800.0, num_spectrum_resources=80,
                   node_request_probabilities=None, allow_rejection=True, seed=None, reset=True, channel_width=50.0),
    "RMCSA-v0": dict(episode_length=1000, load=10.0, mean_service_holding_time=10800.0, num_spectrum_resources=100,
                     num_spatial_resources=7, modulation_formats=None, worst_xt=None, node_request_probabilities=None,
                     bit_rate_selection="continuous", bit_rates=(10, 40, 100), bit_rate_probabilities=None,
                     bit_rate_lower_bound=25, bit_rate_higher_bound=100, seed=None, allow_rejection=False, reset=True,
                     channel_width=12.5),
}
_WORST_XT_BY_CORE = {7: -84.7, 12: -61.9, 19: -54.8}     # rmcsa_env.py:63-67

METRICS = {   # metadata["metrics"], rmsa_env.py:20-27 / rwa_env.py:17
    "RMSA-v0": ["service_blocking_rate", "episode_service_blocking_rate", "bit_rate_blocking_rate",
                "episode_bit_rate_blocking_rate"],
    "RWA-v0": ["service_blocking_rate", "episode_service_blocking_rate"],
}
STAT_KEYS = ["network_compactness", "network_compactness_difference", "avg_link_compactness", "avg_link_utilization"]
METRICS["DeepRMSA-v0"] = METRICS["RMSA-v0"]
METRICS["RMCSA-v0"] = METRICS["RMSA-v0"]

COUNTER_NAMES = ("services_processed", "services_accepted", "episode_services_processed",
                 "episode_services_accepted", "bit_rate_requested", "bit_rate_provisioned",
                 "episode_bit_rate_requested", "episode_bit_rate_provisioned")


class StepInfo:
    """``info`` of a batched step: blocking rates as float64 ``[N]`` tensors, computed on demand from
    the integer counters the kernel snapshots where the reference builds its dict (rmsa_env.py:234-248).
    The info of a rollout has a leading step axis: every array is ``[T, N, ...]`` and every value ``[T, N]``."""

    _COL = {"service_blocking_rate": (0, 1), "episode_service_blocking_rate": (2, 3),
            "bit_rate_blocking_rate": (4, 5), "episode_bit_rate_blocking_rate": (6, 7)}

    def __init__(self, counters: torch.Tensor, keys, stats: Optional[torch.Tensor] = None,
                 bit_rate_blocking: Optional[torch.Tensor] = None, bit_rates=(),
                 action_probability: Optional[torch.Tensor] = None, n_path_actions: int = 0):
        self.counters = counters       # int64 [N, 8] ([T, N, 8] for a rollout, likewise below)
        self.stats = stats             # float64 [N, 4] (rmsa_env.py:249-263) when link_stats=True
        self.bit_rate_blocking = bit_rate_blocking     # float64 [N, B + 1] (rmsa_env.py:217-227, 268-273), discrete mode
        self._br_keys = ["bit_rate_blocking_%d" % int(b) for b in bit_rates] + ["fairness"] if bit_rate_blocking is not None else []
        # RWA-v0: float64 [N, (k + rej) + (W + rej)] (rwa_env.py:148-151)
        self.action_probability, self._n_path_actions = action_probability, n_path_actions
        self._ap_keys = ["path_action_probability", "wavelength_action_probability"] if action_probability is not None else []
        self._keys = list(keys) + (STAT_KEYS if stats is not None else []) + self._br_keys + self._ap_keys

    def keys(self):
        return list(self._keys)

    def __contains__(self, key):
        return key in self._keys

    def __iter__(self):
        return iter(self._keys)

    def __getitem__(self, key):
        if key not in self._keys:
            raise KeyError(key)
        if key in STAT_KEYS:
            return self.stats[..., STAT_KEYS.index(key)]
        if key in self._br_keys:
            return self.bit_rate_blocking[..., self._br_keys.index(key)]
        if key == "path_action_probability":
            return self.action_probability[..., :self._n_path_actions]
        if key == "wavelength_action_probability":
            return self.action_probability[..., self._n_path_actions:]
        a, b = self._COL[key]
        c = self.counters
        return (c[..., a] - c[..., b]).to(torch.float64) / c[..., a].to(torch.float64)

    def items(self):
        return [(k, self[k]) for k in self._keys]


class PolicyRollout(NamedTuple):
    """A PPO rollout buffer filled on the device by :meth:`OpticalVecEnv.rollout_policy` (T steps of N envs)."""
    obs: torch.Tensor          # float32 [T + 1, N, obs_dim]: obs[0] = the pending request's observation, obs[t + 1] = step t's
    actions: torch.Tensor      # int32 [T, N]
    log_prob: torch.Tensor     # float32 [T, N]: log softmax(logits)[action]
    value: torch.Tensor        # float32 [T + 1, N]: V(obs[t]); value[T] = the bootstrap value of the last observation
    reward: torch.Tensor       # float32 [T, N]
    done: torch.Tensor         # uint8 [T, N]


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class OpticalVecEnv:
    """N batched environments of one kind on one GPU.

    Parameters mirror ``gym.make(env_id, **env_args)`` plus the batching ones:
    ``num_envs``; ``device``; ``env_id_base`` (global id of local env 0 when the batch is one shard of a
    multi-GPU job: Philox traffic is keyed by global id so results do not depend on the GPU count);
    ``traffic`` = "philox" (synthetic, counter-based) or "trace" (replay of recorded requests, see
    :meth:`set_trace`); ``obs_dtype`` float32 (default) or float64 (bit-exact reference arithmetic);
    ``auto_reset``; ``collect_info`` (write the info counters every step).
    """

    metadata = {"metrics": []}

    def __init__(self, env_id: str, num_envs: int, topology, *, device=None, env_id_base: int = 0,
                 traffic: str = "philox", obs_dtype=torch.float32, auto_reset: bool = True, collect_info: bool = True,
                 record_decisions: bool = False, heap_capacity: int = 0, link_stats: bool = False, **env_args):
        if env_id not in nat.KIND:
            raise ValueError("unknown env id %r (have %s)" % (env_id, sorted(nat.KIND)))
        if not torch.cuda.is_available():
            raise nat.NativeError("optical_rl_gym_b200 needs a CUDA device: there is no CPU fallback")
        unknown = set(env_args) - set(_DEFAULTS[env_id])
        if unknown:
            raise TypeError("%s got unexpected keyword arguments %s" % (env_id, sorted(unknown)))
        self.env_id = env_id
        self.kind = nat.KIND[env_id]
        self.args = dict(_DEFAULTS[env_id])
        self.args.update(env_args)
        a = self.args
        self.tables = topology if isinstance(topology, TopologyTables) else TopologyTables.from_graph(topology)
        t = self.tables
        self.num_envs = int(num_envs)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", self._dev_index)       # always an indexed device: buffers, stream and handle agree
        self.metadata = {"metrics": METRICS[env_id]}
        self.k_paths = t.k_paths
        self.num_spectrum_resources = int(a["num_spectrum_resources"])
        self.episode_length = int(a["episode_length"])
        self.allow_rejection = bool(a["allow_rejection"])
        self.reject_action = 1 if self.allow_rejection else 0
        self.j = int(a.get("j", 1))
        self.num_spatial_resources = int(a.get("num_spatial_resources", 1))
        self.channel_width = float(a.get("channel_width", 12.5))
        # set_load (optical_network_env.py:76-94)
        self.mean_service_holding_time = float(a["mean_service_holding_time"])
        if env_id == "DeepRMSA-v0":
            self.load = self.mean_service_holding_time / float(a["mean_service_inter_arrival_time"])
        else:
            self.load = float(a["load"])
        self.mean_service_inter_arrival_time = 1 / float(self.load / float(self.mean_service_holding_time))
        self.rand_seed = 41 if a["seed"] is None else int(a["seed"])       # optical_network_env.py:205-210
        probs = a["node_request_probabilities"]
        self.node_request_probabilities = (np.full(t.num_nodes, 1.0 / t.num_nodes) if probs is None
                                           else np.asarray(probs, np.float64))
        assert len(self.node_request_probabilities) == t.num_nodes
        assert a.get("bit_rate_selection", "continuous") in ("continuous", "discrete")
        discrete = a.get("bit_rate_selection", "continuous") == "discrete"
        if discrete and env_id == "RMCSA-v0":
            raise NotImplementedError("RMCSA discrete bit rates raise TypeError in the reference (SURVEY App. B-7)")
        self.bit_rates = np.asarray(a.get("bit_rates", ()), np.int32) if discrete else np.zeros(0, np.int32)
        bp = a.get("bit_rate_probabilities")
        self.bit_rate_probabilities = (np.full(len(self.bit_rates), 1.0 / max(len(self.bit_rates), 1)) if bp is None
                                       else np.asarray(bp, np.float64))
        worst_xt = a.get("worst_xt")
        if env_id == "RMCSA-v0" and worst_xt is None:
            worst_xt = _WORST_XT_BY_CORE.get(self.num_spatial_resources)
            if worst_xt is None:
                raise ValueError("worst_xt must be given for %d cores" % self.num_spatial_resources)
        assert obs_dtype in (torch.float32, torch.float64)
        self.obs_dtype = obs_dtype
        assert traffic in ("philox", "trace")
        self.traffic = traffic

        # ---- native handle
        self._keep = {}

        def arr(name, x, dt):
            self._keep[name] = np.ascontiguousarray(x, dtype=dt)
            return self._keep[name].ctypes.data_as(C.c_void_p)

        cfg = nat.Config(kind=self.kind, num_envs=self.num_envs, env_id_base=int(env_id_base),
                         num_slots=self.num_spectrum_resources, num_cores=self.num_spatial_resources, j=self.j,
                         episode_length=self.episode_length, allow_rejection=int(self.allow_rejection),
                         # DeepRMSAEnv cannot change the bounds: it always runs RMSAEnv's defaults (SURVEY App. B-14)
                         bit_rate_lo=int(a.get("bit_rate_lower_bound", 25.0)), bit_rate_hi=int(a.get("bit_rate_higher_bound", 100.0)),
                         traffic=nat.TRAFFIC_PHILOX if traffic == "philox" else nat.TRAFFIC_TRACE,
                         obs_dtype=nat.OBS_F64 if obs_dtype == torch.float64 else nat.OBS_F32,
                         auto_reset=int(auto_reset), heap_capacity=int(heap_capacity), seed=self.rand_seed,
                         channel_width=self.channel_width, mean_holding=self.mean_service_holding_time,
                         mean_iat=self.mean_service_inter_arrival_time, worst_xt=float(worst_xt or 0.0))
        tab = nat.Tables(num_nodes=t.num_nodes, num_links=t.num_links, k_paths=t.k_paths, num_paths=t.num_paths,
                         num_mods=len(t.mod_se), num_bit_rates=len(self.bit_rates),
                         pair_first=arr("pf", t.pair_first, np.int32), pair_count=arr("pc", t.pair_count, np.int32),
                         path_hops=arr("ph", t.path_hops, np.int32), path_se=arr("ps", t.path_se, np.int32),
                         path_mod=arr("pm", t.path_mod, np.int32), path_link_ptr=arr("pp", t.path_link_ptr, np.int32),
                         path_links=arr("pl", t.path_links, np.int32), path_length=arr("plen", t.path_length, np.float64),
                         mod_se=arr("ms", t.mod_se, np.int32), mod_osnr=arr("mo", t.mod_osnr, np.float64),
                         mod_xt=arr("mx", t.mod_xt, np.float64),
                         node_prob=arr("np", self.node_request_probabilities, np.float64),
                         bit_rates=arr("br", self.bit_rates if len(self.bit_rates) else [0], np.int32),
                         bit_rate_prob=arr("bp", self.bit_rate_probabilities if len(self.bit_rates) else [1.0], np.float64),
                         link_order=arr("lo", t.link_order, np.int32))
        self._lib = nat.lib()
        self._h = C.c_void_p()
        self._closed = False
        with torch.cuda.device(self.device):
            nat.check(self._lib.orlg_create(C.byref(cfg), C.byref(tab), self._dev_index, C.byref(self._h)))
        self.action_dim = self._lib.orlg_action_dim(self._h)
        self.obs_dim = self._lib.orlg_obs_dim(self._h)
        self.mask_words = self._lib.orlg_mask_words(self._h)
        self.heap_capacity = self._lib.orlg_heap_capacity(self._h)
        self.state_bytes = int(self._lib.orlg_state_bytes(self._h))

        # ---- spaces (rmsa_env.py:138-149, deeprmsa_env.py:34-45, rwa_env.py:70-82, rmcsa_env.py:181-188)
        k, S, rej = self.k_paths, self.num_spectrum_resources, self.reject_action
        if env_id == "DeepRMSA-v0":
            self.action_space = spaces.Discrete(k * self.j + rej)
            self.observation_space = spaces.Box(-2 ** 30, 2 ** 30, (self.obs_dim,),
                                                np.float64 if obs_dtype == torch.float64 else np.float32)
        elif env_id == "RMCSA-v0":
            self.action_space = spaces.MultiDiscrete((k + rej, len(t.mod_se), self.num_spatial_resources + rej, S + rej))
            self.observation_space = spaces.Dict({"topology": spaces.Discrete(10), "current_service": spaces.Discrete(10)})
        else:
            self.action_space = spaces.MultiDiscrete((k + rej, S + rej))
            self.observation_space = spaces.Dict({"topology": spaces.Discrete(10), "current_service": spaces.Discrete(10)})

        # ---- persistent output buffers (overwritten by every step)
        n, dev = self.num_envs, self.device
        self._obs = torch.zeros((n, self.obs_dim), dtype=obs_dtype, device=dev) if self.obs_dim else None
        self._reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self._done = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._info = torch.zeros((n, 8), dtype=torch.int64, device=dev) if collect_info else None
        self._decision = torch.zeros((n, 6), dtype=torch.int32, device=dev) if record_decisions else None
        self._out_ptrs = (_ptr(self._obs), _ptr(self._reward), _ptr(self._done), _ptr(self._decision), _ptr(self._info))
        self._actions = None
        self._trace = None
        # float statistics of info (network / link compactness, utilisation): opt-in; the NSFNET class runs them on the generic
        # kernel, wider topologies on the statistics instance of the wide kernel (any link count, up to 512 slots and 31 cores)
        self._stats = None
        self._link_stats = bool(link_stats)
        if link_stats and env_id in ("RMSA-v0", "DeepRMSA-v0"):
            self._stats = torch.zeros((n, 4), dtype=torch.float64, device=dev)
            nat.check(self._lib.orlg_enable_stats(self._h, _ptr(self._stats)))
        elif link_stats:        # RWA / RMCSA: no float statistics in info, but the graph attributes are kept (graph_statistics())
            nat.check(self._lib.orlg_enable_link_stats(self._h, 1))
        # discrete bit-rate selection: per-bit-rate blocking + fairness of `info` (rmsa_env.py:217-227, 268-273)
        self._brb = None
        nb = self._lib.orlg_num_bit_rates(self._h)
        if nb and collect_info:
            self._brb = torch.zeros((n, nb + 1), dtype=torch.float64, device=dev)
        # RWA-v0: the action-probability entries of `info` (rwa_env.py:148-151)
        self._ap = None
        nh = self._lib.orlg_action_hist_dim(self._h)
        if nh and collect_info:
            self._ap = torch.zeros((n, nh), dtype=torch.float64, device=dev)
        if traffic == "philox" and a.get("reset", True):
            self.reset(full=True)

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        # raw handle of torch's current stream on this device (the private accessor is several times cheaper than
        # building a Stream object per call; the rollout loop issues two launches per ~20 us)
        try:
            return C.c_void_p(torch._C._cuda_getCurrentRawStream(self._dev_index))
        except AttributeError:      # pragma: no cover - older / newer torch without the accessor
            return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if not getattr(self, "_closed", True) and self._h:
            self._lib.orlg_destroy(self._h)
            self._closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def seed(self, seed=None):
        """``env.seed(seed)`` for every env (optical_network_env.py:205-210; VecEnv.seed): the counter-based request
        stream continues under the new key from the next request on (env i keeps its own sub-stream: the key is
        shared, the global env id is part of the counter); state is untouched.  Returns the seed per env."""
        self.rand_seed = 41 if seed is None else int(seed)
        nat.check(self._lib.orlg_seed(self._h, self.rand_seed))
        return [self.rand_seed] * self.num_envs

    def get_attr(self, name, indices=None):
        value = getattr(self, name)
        return [value] * (self.num_envs if indices is None else len(indices))

    def set_attr(self, name, value, indices=None):
        raise NotImplementedError("environment parameters are fixed at construction")

    def env_method(self, name, *args, indices=None, **kwargs):
        return getattr(self, name)(*args, **kwargs)

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False] * self.num_envs

    # ------------------------------------------------------------------ traffic
    def set_trace(self, arrival, holding, src, dst, bit_rate=None):
        """Replay recorded requests: arrays ``[num_envs, T]`` (request i of env e is the i-th request drawn
        by ``_next_service`` since the full reset, rmsa_env.py:545-573)."""
        arrival = np.asarray(arrival, np.float64)
        n, T = arrival.shape
        assert n == self.num_envs
        rec = np.zeros((n, T), nat.REQUEST_DTYPE)
        rec["arrival"], rec["holding"] = arrival, np.asarray(holding, np.float64)
        rec["src"], rec["dst"] = np.asarray(src, np.int32), np.asarray(dst, np.int32)
        rec["bit_rate"] = 0 if bit_rate is None else np.asarray(bit_rate, np.int32)
        if rec["bit_rate"].min() < 0 or rec["bit_rate"].max() > nat.MAX_BIT_RATE:
            raise ValueError("trace bit rates must lie in 0..%d" % nat.MAX_BIT_RATE)
        if rec["src"].min() < 0 or max(rec["src"].max(), rec["dst"].max()) >= self.tables.num_nodes or (rec["src"] == rec["dst"]).any():
            raise ValueError("trace node ids out of range (or src == dst)")
        self._trace = torch.from_numpy(rec.view(np.uint8).reshape(n, T * nat.REQUEST_DTYPE.itemsize)).to(self.device)
        nat.check(self._lib.orlg_set_trace(self._h, _ptr(self._trace), T))
        self.traffic = "trace"

    # ------------------------------------------------------------------ gym / VecEnv API
    def reset(self, full: bool = False):
        """``env.reset(only_episode_counters=not full)`` for every env; returns the observation batch."""
        nat.check(self._lib.orlg_reset(self._h, int(full), _ptr(self._obs), self._stream()))
        return self._obs

    def step_async(self, actions):
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions), device=self.device)
        self._actions = actions.to(device=self.device, dtype=torch.int32).reshape(self.num_envs, self.action_dim).contiguous()

    def step_wait(self):
        nat.check(self._lib.orlg_step(self._h, _ptr(self._actions), _ptr(self._obs), _ptr(self._reward), _ptr(self._done),
                                      _ptr(self._decision), _ptr(self._info), self._stream()))
        info = None
        if self._info is not None:
            if self._brb is not None:
                nat.check(self._lib.orlg_bit_rate_blocking(self._h, _ptr(self._brb), self._stream()))
            if self._ap is not None:
                nat.check(self._lib.orlg_action_probability(self._h, _ptr(self._ap), self._stream()))
            info = StepInfo(self._info, self.metadata["metrics"], self._stats, self._brb, self.bit_rates,
                            self._ap, self.k_paths + self.reject_action)
        return self._obs, self._reward, self._done, info

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    @property
    def info_keys(self):
        """The keys ``info`` carries for this env and configuration (empty with ``collect_info=False``)."""
        if self._info is None:
            return []
        return StepInfo(self._info, self.metadata["metrics"], self._stats, self._brb, self.bit_rates, self._ap,
                        self.k_paths + self.reject_action).keys()

    def _rollout_info(self, steps: int):
        """Device buffers for every step's info of a ``steps``-step rollout: ``(StepInfo, orlg_info_out)``."""
        if self._info is None:
            raise ValueError("want_info=True needs the env's info: construct it with collect_info=True")
        bufs = [None if b is None else torch.empty((steps,) + tuple(b.shape), dtype=b.dtype, device=self.device)
                for b in (self._info, self._stats, self._brb, self._ap)]
        info = StepInfo(bufs[0], self.metadata["metrics"], bufs[1], bufs[2], self.bit_rates, bufs[3],
                        self.k_paths + self.reject_action)
        return info, nat.InfoOut(*(None if b is None else b.data_ptr() for b in bufs))

    def step_raw(self, actions_i32: torch.Tensor):
        """Hot-loop variant: ``actions_i32`` must already be a contiguous int32 CUDA tensor ``[N, action_dim]``."""
        rc = self._lib.orlg_step(self._h, C.c_void_p(actions_i32.data_ptr()), *self._out_ptrs, self._stream())
        if rc:
            nat.check(rc)
        return self._obs, self._reward, self._done

    def rollout(self, steps: int, policy="random", *, obs=None, reward=None, done=None, actions=None,
                want_obs: bool = True, want_actions: bool = True, want_info: bool = False):
        """``steps`` iterations of ``a = policy(env); env.step(a)`` in ONE native call (``orlg_rollout``), every step's
        results kept: returns ``(obs [T, N, obs_dim] | None, reward [T, N], done [T, N], actions [T, N, action_dim] | None)``.
        ``policy``: "random" (:meth:`sample_actions`) or a heuristic name (:meth:`heuristic`).  Identical to the
        step-by-step loop; DeepRMSA-v0 with Philox traffic and float32 observations runs as one persistent kernel.
        ``want_info=True`` (needs ``collect_info=True``) appends every step's ``info``: a :class:`StepInfo` with the keys of
        :attr:`info_keys` and ``[T, N]`` values (``orlg_rollout_info``; RWA-v0's action probabilities make it step by step)."""
        T, n, dev = int(steps), self.num_envs, self.device
        info, info_out = self._rollout_info(T) if want_info else (None, None)
        if policy == "replay":          # the given `actions` [T, N, action_dim] are applied (with trace traffic: a recorded run)
            assert actions is not None, "policy='replay' needs the action sequence"
            actions = torch.as_tensor(actions, device=dev).to(torch.int32).reshape(T, n, self.action_dim).contiguous()
            pol = -2
        else:
            pol = -1 if policy in ("random", None) else (nat.HEURISTICS[policy] if isinstance(policy, str) else int(policy))
        if obs is None and want_obs and self.obs_dim:
            obs = torch.empty((T, n, self.obs_dim), dtype=self.obs_dtype, device=dev)
        if reward is None:
            reward = torch.empty((T, n), dtype=torch.float32, device=dev)
        if done is None:
            done = torch.empty((T, n), dtype=torch.uint8, device=dev)
        if actions is None and want_actions:
            actions = torch.empty((T, n, self.action_dim), dtype=torch.int32, device=dev)
        for tns, shape in ((obs, (T, n, self.obs_dim)), (reward, (T, n)), (done, (T, n)), (actions, (T, n, self.action_dim))):
            if tns is not None:
                assert tuple(tns.shape) == shape and tns.is_contiguous() and tns.device == dev, (tuple(tns.shape), shape)
        with torch.cuda.device(self._dev_index):
            if want_info:
                nat.check(self._lib.orlg_rollout_info(self._h, T, pol, _ptr(obs), _ptr(reward), _ptr(done), _ptr(actions),
                                                      C.byref(info_out), self._stream()))
                return obs, reward, done, actions, info
            nat.check(self._lib.orlg_rollout(self._h, T, pol, _ptr(obs), _ptr(reward), _ptr(done), _ptr(actions), self._stream()))
        return obs, reward, done, actions

    def rollout_policy(self, policy, steps: int, *, deterministic: bool = False, seed: Optional[int] = None,
                       out: Optional[PolicyRollout] = None, want_info: bool = False):
        """``steps`` iterations of ``a, log p(a), V(obs) = policy(obs); obs, r, done = env.step(a)`` in ONE native call
        (``orlg_rollout_policy``): a :class:`PolicyRollout` of device tensors, what SB3's ``collect_rollouts`` gathers.
        ``policy`` is an :class:`~optical_rl_gym_b200.policy.MlpPolicy` on this device (its current weights; the value comes
        from its critic trunk when it has one).  Actions are drawn from softmax(logits) (``deterministic=True``: argmax) with
        Philox stream 3 keyed by ``seed`` (default: the env's seed), the global env id and the env's request index, so the
        result does not depend on the number of GPUs, on how the rollout is split into calls or on a checkpoint in between.
        ``out`` reuses the buffers of an earlier call.  DeepRMSA-v0 with float32 observations.  ``want_info=True`` (needs
        ``collect_info=True``) returns ``(PolicyRollout, StepInfo)``, the latter every step's ``info`` with ``[T, N]`` values."""
        T, n, dev = int(steps), self.num_envs, self.device
        if T < 0:
            raise ValueError("steps must be >= 0")
        info, info_out = self._rollout_info(T) if want_info else (None, None)
        if out is None:
            out = PolicyRollout(torch.empty((T + 1, n, self.obs_dim), dtype=torch.float32, device=dev),
                                torch.empty((T, n), dtype=torch.int32, device=dev),
                                torch.empty((T, n), dtype=torch.float32, device=dev),
                                torch.empty((T + 1, n), dtype=torch.float32, device=dev),
                                torch.empty((T, n), dtype=torch.float32, device=dev),
                                torch.empty((T, n), dtype=torch.uint8, device=dev))
        want = (((T + 1, n, self.obs_dim), torch.float32), ((T, n), torch.int32), ((T, n), torch.float32),
                ((T + 1, n), torch.float32), ((T, n), torch.float32), ((T, n), torch.uint8))
        for name, tns, (shape, dt) in zip(PolicyRollout._fields, out, want):
            if tuple(tns.shape) != shape or tns.dtype != dt or tns.device != dev or not tns.is_contiguous():
                raise ValueError("out.%s must be a contiguous %s tensor %s on %s, got %s %s %s" % (
                    name, dt, shape, dev, tuple(tns.shape), tns.dtype, tns.device))
        actor, critic = policy._native_handles(self._dev_index)
        key = self.rand_seed if seed is None else int(seed)
        with torch.cuda.device(self._dev_index):
            if want_info:
                nat.check(self._lib.orlg_rollout_policy_info(self._h, T, actor, critic, key & (2 ** 64 - 1), int(bool(deterministic)),
                                                             *[_ptr(t) for t in out], C.byref(info_out), self._stream()))
                return out, info
            nat.check(self._lib.orlg_rollout_policy(self._h, T, actor, critic, key & (2 ** 64 - 1), int(bool(deterministic)),
                                                    *[_ptr(t) for t in out], self._stream()))
        return out

    @property
    def request_index(self) -> int:
        """Requests drawn so far by every env (they step together): counter word 0 of the action draws of the next
        :meth:`rollout_policy` step, for a Python loop that wants the same keying (``MlpPolicy.sample_native(counter=...)``)."""
        return int(self._lib.orlg_request_index(self._h))

    def rollout_packed(self, steps: int, policy="random", out=None):
        """Like :meth:`rollout`, but ONE 32-byte record per env-step (int32 ``[T, N, 8]`` on the device): the integer
        pre-image of the observation + request + action / accepted / done (``orlg_rollout_packed``, include/orlg.h).
        :meth:`expand_packed` turns records (on the host) into float32 rows identical to :meth:`rollout`'s."""
        T, n = int(steps), self.num_envs
        pol = -1 if policy in ("random", None) else (nat.HEURISTICS[policy] if isinstance(policy, str) else int(policy))
        if out is None:
            out = torch.empty((T, n, 8), dtype=torch.int32, device=self.device)
        assert tuple(out.shape) == (T, n, 8) and out.is_contiguous() and out.dtype == torch.int32
        with torch.cuda.device(self._dev_index):
            nat.check(self._lib.orlg_rollout_packed(self._h, T, pol, _ptr(out), None, self._stream()))
        return out

    def expand_packed(self, packed, threads: int = 0):
        """Host-side decoder of packed records (numpy / CPU tensor ``[..., 8]`` int32) -> ``(obs f32 [..., obs_dim], reward f32,
        done u8, action i32)`` numpy arrays (``orlg_expand_packed``: all host cores by default)."""
        pk = np.ascontiguousarray(packed.cpu().numpy() if torch.is_tensor(packed) else packed).view(np.uint32)
        lead = pk.shape[:-1]
        rows = int(np.prod(lead))
        obs = np.empty(lead + (self.obs_dim,), np.float32)
        rew, done, act = np.empty(lead, np.float32), np.empty(lead, np.uint8), np.empty(lead, np.int32)
        nat.check(self._lib.orlg_expand_packed(pk.ctypes.data_as(C.c_void_p), rows, self.tables.num_nodes, self.num_spectrum_resources,
                                               obs.ctypes.data_as(C.c_void_p), rew.ctypes.data_as(C.c_void_p),
                                               done.ctypes.data_as(C.c_void_p), act.ctypes.data_as(C.c_void_p), int(threads)))
        return obs, rew, done, act

    def rollout_host(self, steps: int, policy="random", *, obs=None, reward=None, done=None, actions=None, chunk: int = 8,
                     threads: int = 0):
        """:meth:`rollout` with the results delivered in HOST memory (numpy arrays, pageable is fine): the device runs chunk
        c + 1 while chunk c's packed records cross PCIe and the host threads expand them (``orlg_rollout_host``).
        ``policy="replay"``: ``actions`` (int32 ``[steps, num_envs]``, host) is the input action sequence."""
        T, n = int(steps), self.num_envs
        if policy == "replay":
            assert actions is not None, "policy='replay' needs the actions"
            pol = -2
        else:
            pol = -1 if policy in ("random", None) else (nat.HEURISTICS[policy] if isinstance(policy, str) else int(policy))
        obs = np.empty((T, n, self.obs_dim), np.float32) if obs is None else obs
        reward = np.empty((T, n), np.float32) if reward is None else reward
        done = np.empty((T, n), np.uint8) if done is None else done
        actions = np.empty((T, n), np.int32) if actions is None else actions
        for a, shape, dt in ((obs, (T, n, self.obs_dim), np.float32), (reward, (T, n), np.float32), (done, (T, n), np.uint8),
                             (actions, (T, n), np.int32)):
            assert a.shape == shape and a.dtype == dt and a.flags["C_CONTIGUOUS"], (a.shape, shape, a.dtype)
        with torch.cuda.device(self._dev_index):
            nat.check(self._lib.orlg_rollout_host(self._h, T, pol, obs.ctypes.data_as(C.c_void_p), reward.ctypes.data_as(C.c_void_p),
                                                  done.ctypes.data_as(C.c_void_p), actions.ctypes.data_as(C.c_void_p),
                                                  int(chunk), int(threads), self._stream()))
        return obs, reward, done, actions

    def observation(self):
        if not self.obs_dim:
            return None
        nat.check(self._lib.orlg_observation(self._h, _ptr(self._obs), self._stream()))
        return self._obs

    def observation_int(self):
        out = torch.zeros((self.num_envs, self.k_paths, 2 * self.j + 3), dtype=torch.int32, device=self.device)
        nat.check(self._lib.orlg_observation_int(self._h, _ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ action sources
    def heuristic(self, name, out: Optional[torch.Tensor] = None):
        """Device version of the reference's heuristic functions (same names), one action per env."""
        which = nat.HEURISTICS[name] if isinstance(name, str) else int(name)
        if out is None:
            out = torch.empty((self.num_envs, self.action_dim), dtype=torch.int32, device=self.device)
        nat.check(self._lib.orlg_heuristic(self._h, which, _ptr(out), self._stream()))
        return out

    def matrix_observation(self, out: Optional[torch.Tensor] = None):
        """``SimpleMatrixObservation.observation`` of every env (rmsa_env.py:806-837, rmcsa_env.py:914-947):
        uint8 [N, 2*nodes + cores*links*slots]."""
        d = self._lib.orlg_matrix_obs_dim(self._h)
        if out is None:
            out = torch.empty((self.num_envs, d), dtype=torch.uint8, device=self.device)
        nat.check(self._lib.orlg_matrix_observation(self._h, _ptr(out), self._stream()))
        return out

    def path_only_first_fit(self, path_actions, out: Optional[torch.Tensor] = None):
        """``PathOnlyFirstFitAction.action`` for every env (rmsa_env.py:840-874, rwa_env.py:505-536)."""
        pa = torch.as_tensor(path_actions, device=self.device).to(torch.int32).reshape(self.num_envs).contiguous()
        if out is None:
            out = torch.empty((self.num_envs, 2), dtype=torch.int32, device=self.device)
        nat.check(self._lib.orlg_path_only_first_fit(self._h, _ptr(pa), _ptr(out), self._stream()))
        return out

    def sample_actions(self, out: Optional[torch.Tensor] = None):
        """Uniform random policy (``action_space.sample()`` per env) from Philox stream 2."""
        if out is None:
            out = torch.empty((self.num_envs, self.action_dim), dtype=torch.int32, device=self.device)
        rc = self._lib.orlg_random_actions(self._h, C.c_void_p(out.data_ptr()), self._stream())
        if rc:
            nat.check(rc)
        return out

    # ------------------------------------------------------------------ checkpoint / resume
    def state_dict(self):
        """Everything needed to continue this batch later: the native state (one opaque uint8 CUDA tensor) + the request-stream
        key.  ``load_state_dict`` restores it into an env constructed with the same arguments."""
        nbytes = int(self._lib.orlg_state_save_bytes(self._h))
        blob = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self._dev_index):
            nat.check(self._lib.orlg_state_save(self._h, _ptr(blob), self._stream()))
        return {"native": blob, "seed": self.rand_seed, "env_id": self.env_id, "num_envs": self.num_envs}

    def load_state_dict(self, sd):
        if sd["env_id"] != self.env_id or sd["num_envs"] != self.num_envs:
            raise ValueError("checkpoint of %s x %d does not fit %s x %d" % (sd["env_id"], sd["num_envs"], self.env_id, self.num_envs))
        blob = sd["native"].to(self.device).contiguous()
        if blob.numel() != int(self._lib.orlg_state_save_bytes(self._h)):
            raise ValueError("checkpoint was written by a differently configured env")
        with torch.cuda.device(self._dev_index):
            nat.check(self._lib.orlg_state_load(self._h, _ptr(blob), self._stream()))
        self.seed(sd["seed"])

    # ------------------------------------------------------------------ introspection
    def kernel_info(self) -> dict:
        """Which compiled kernel instances this batch runs (``orlg_kernel_info``): ``wide``, ``fast``, ``hot``,
        ``rollout_kernel`` (bools), ``rollout_lanes`` (envs per warp of the rollout kernel, 8 or 32), ``link_template``
        (22: the NSFNET instance, 0: link count read at run time) and ``last_rollout_persistent`` (whether the last
        :meth:`rollout` / :meth:`rollout_packed` / :meth:`rollout_host` ran the persistent kernel)."""
        info = nat.KernelInfo()
        nat.check(self._lib.orlg_kernel_info(self._h, C.byref(info)))
        out = {name: int(getattr(info, name)) for name, _ in nat.KernelInfo._fields_}
        for name in ("wide", "fast", "hot", "rollout_kernel", "last_rollout_persistent"):
            out[name] = bool(out[name])
        return out

    @property
    def decisions(self):
        return self._decision

    def counters(self):
        out = torch.empty((self.num_envs, 8), dtype=torch.int64, device=self.device)
        nat.check(self._lib.orlg_get_counters(self._h, _ptr(out), self._stream()))
        return out

    def current_requests(self):
        """The pending request of every env (``env.current_service``) as a numpy record array + service ids."""
        raw = torch.empty((self.num_envs, nat.REQUEST_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        sid = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        nat.check(self._lib.orlg_get_requests(self._h, _ptr(raw), _ptr(sid), self._stream()))
        return raw.cpu().numpy().view(nat.REQUEST_DTYPE).reshape(self.num_envs), sid.cpu().numpy()

    def export_state(self, masks=True, allocation=False):
        """(bit-packed masks int32 [N, C*E, words], allocation int32 [N, C, E, S] | None, now f64 [N], nheap i32 [N])."""
        n, dev, E = self.num_envs, self.device, self.tables.num_links
        cores = self.num_spatial_resources if self.kind == nat.KIND["RMCSA-v0"] else 1
        m = torch.empty((n, cores * E, self.mask_words), dtype=torch.int32, device=dev) if masks else None
        al = (torch.empty((n, cores, E, self.num_spectrum_resources), dtype=torch.int32, device=dev)
              if allocation else None)
        now = torch.empty(n, dtype=torch.float64, device=dev)
        nh = torch.empty(n, dtype=torch.int32, device=dev)
        nat.check(self._lib.orlg_export_state(self._h, _ptr(m), _ptr(al), _ptr(now), _ptr(nh), self._stream()))
        return m, al, now, nh

    def graph_statistics(self):
        """The time-averaged statistics the reference keeps on ``env.topology`` (needs ``link_stats=True``): ``(link, graph)`` with
        ``link`` float64 [N, E, 3] = each link's ``utilization``, ``external_fragmentation``, ``compactness`` by link index
        (``topology[n1][n2][...]``; rmsa_env.py:464-543, rmcsa_env.py:591-688, RWA: utilization only, rwa_env.py:365-383) and
        ``graph`` float64 [N, 2] = ``topology.graph["throughput"]``, ``["compactness"]`` (rmsa_env.py:439-462)."""
        assert self._link_stats, "construct the env with link_stats=True"
        link = torch.empty((self.num_envs, self.tables.num_links, 3), dtype=torch.float64, device=self.device)
        graph = torch.empty((self.num_envs, 2), dtype=torch.float64, device=self.device)
        nat.check(self._lib.orlg_link_stats(self._h, _ptr(link), _ptr(graph), self._stream()))
        return link, graph

    def available_slots(self):
        """``topology.graph['available_slots']`` of every env: uint8 [N, C*E, S] (1 = free)."""
        m = self.export_state()[0]
        bits = (m.unsqueeze(-1) >> torch.arange(32, device=self.device, dtype=torch.int32)) & 1
        return bits.reshape(self.num_envs, m.shape[1], -1)[:, :, :self.num_spectrum_resources].to(torch.uint8)

    def error_flags(self):
        out = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        nat.check(self._lib.orlg_error_flags(self._h, _ptr(out), self._stream()))
        return out

    def reduce_counters(self):
        """Per-GPU sums of the 8 counters + number of envs with an error flag (int64 [9]) -- the operand of
        the cross-GPU all-reduce of episode statistics."""
        out = torch.empty(9, dtype=torch.int64, device=self.device)
        nat.check(self._lib.orlg_reduce_counters(self._h, _ptr(out), self._stream()))
        return out


def make(env_id: str, num_envs: int = 1, **kwargs) -> OpticalVecEnv:
    """``gym.make(env_id, **env_args)`` for a batch: ``make('DeepRMSA-v0', num_envs=65536, topology=..., seed=10)``."""
    topology = kwargs.pop("topology")
    return OpticalVecEnv(env_id, num_envs, topology, **kwargs)
