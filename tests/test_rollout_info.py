"""Every step's `info` out of the multi-step paths: orlg_rollout_info / orlg_rollout_policy_info, OpticalVecEnv.rollout and
rollout_policy with want_info=True, and the VecMonitor rows they feed.  Row t must be exactly what the step-by-step calls
give after step t: against the reference's goldens, against a twin handle stepped by orlg_step, on the persistent kernel
(which writes the counters itself) and on every per-step path."""
import ctypes as C

import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

from test_gpu_parity import make_env  # noqa: E402
from test_policy_rollout import BASE, SEED, _env, _env_policy, _sb3_state_dict  # noqa: E402


# ------------------------------------------------------------------ CPU: StepInfo with a step axis, VecMonitor bookkeeping
def test_step_info_with_a_step_axis_equals_its_rows():
    from optical_rl_gym_b200.vec_env import METRICS, STAT_KEYS, StepInfo

    g = torch.Generator().manual_seed(0)
    T, n = 5, 7
    c = torch.randint(1, 50, (T, n, 8), generator=g, dtype=torch.int64)
    st = torch.rand((T, n, 4), generator=g, dtype=torch.float64)
    brb = torch.rand((T, n, 4), generator=g, dtype=torch.float64)
    ap = torch.rand((T, n, 9), generator=g, dtype=torch.float64)
    whole = StepInfo(c, METRICS["RMSA-v0"], st, brb, (10, 40, 100), ap, 4)
    assert set(STAT_KEYS) <= set(whole.keys()) and "fairness" in whole and "path_action_probability" in whole
    for t in range(T):
        row = StepInfo(c[t], METRICS["RMSA-v0"], st[t], brb[t], (10, 40, 100), ap[t], 4)
        assert row.keys() == whole.keys()
        for k in whole.keys():
            assert torch.equal(whole[k][t], row[k]), k
    assert whole["service_blocking_rate"].shape == (T, n) and whole["wavelength_action_probability"].shape == (T, n, 5)


class _FakeVenv:
    """What VecMonitor needs of a venv, stepping through preset rewards / dones / info."""

    def __init__(self, reward, done, info):
        self.reward, self.done, self.info = reward, done, info
        self.num_envs, self.device, self.env_id = reward.shape[1], torch.device("cpu"), "DeepRMSA-v0"
        self.action_space = self.observation_space = None
        self._info, self.info_keys, self.t = True, list(info), 0

    def step_async(self, actions):
        pass

    def close(self):
        pass

    def step_wait(self):
        t, self.t = self.t, self.t + 1
        return None, self.reward[t], self.done[t], {k: v[t] for k, v in self.info.items()}


@pytest.mark.parametrize("chunks", [(40,), (1, 13, 26), (0, 17, 1, 1, 21)])
def test_monitor_rollout_rows_equal_the_step_loop_rows(tmp_path, chunks):
    from optical_rl_gym_b200.monitor import VecMonitor

    g = torch.Generator().manual_seed(sum(chunks) + len(chunks))
    T, n = 40, 6
    reward = (torch.randint(0, 3, (T, n), generator=g) - 1).to(torch.float32)
    done = (torch.rand((T, n), generator=g) < 0.15).to(torch.uint8)
    done[:, 0] = 0                                    # an env that never finishes
    done[T - 1, 1] = 1                                # one that finishes on the last step
    info = {"episode_service_blocking_rate": torch.rand((T, n), generator=g, dtype=torch.float64)}
    keys = tuple(info)
    ref = VecMonitor(_FakeVenv(reward, done, info), str(tmp_path / "loop"), info_keywords=keys)
    got = VecMonitor(_FakeVenv(reward, done, info), str(tmp_path / "ro"), info_keywords=keys)
    for _ in range(T):
        ref.step(None)
    t0 = 0
    for ch in chunks:
        sl = slice(t0, t0 + ch)
        got._record_rollout(reward[sl], done[sl], {k: v[sl] for k, v in info.items()})
        t0 += ch
    assert ref.episode_returns == got.episode_returns and ref.episode_lengths == got.episode_lengths
    assert ref.episode_infos == got.episode_infos and ref.total_steps == got.total_steps
    assert torch.equal(ref._ret, got._ret) and torch.equal(ref._len, got._len)
    ref.close(); got.close()
    assert _csv_rows(tmp_path / "loop.monitor.csv") == _csv_rows(tmp_path / "ro.monitor.csv")


def _csv_rows(path):
    """The monitor file without the `t` column (wall-clock seconds)."""
    lines = open(str(path)).read().splitlines()
    return [",".join(x for i, x in enumerate(ln.split(",")) if i != 2) for ln in lines[1:]]


# ------------------------------------------------------------------ GPU helpers
def _info_out(counters=None, stats=None, brb=None, ap=None):
    from optical_rl_gym_b200 import _native as nat

    return nat.InfoOut(*(None if x is None else x.data_ptr() for x in (counters, stats, brb, ap)))


def _rollout_counters(env, T, policy, actions=None):
    """orlg_rollout_info with the counters only (what the persistent kernel writes): (reward, done, actions, counters)."""
    from optical_rl_gym_b200 import _native as nat

    n, dev = env.num_envs, env.device
    pol = -2 if policy == "replay" else (-1 if policy == "random" else nat.HEURISTICS[policy])
    if actions is None:
        actions = torch.empty((T, n, env.action_dim), dtype=torch.int32, device=dev)
    reward = torch.empty((T, n), dtype=torch.float32, device=dev)
    done = torch.empty((T, n), dtype=torch.uint8, device=dev)
    counters = torch.empty((T, n, 8), dtype=torch.int64, device=dev)
    out = _info_out(counters)
    nat.check(env._lib.orlg_rollout_info(env._h, T, pol, None, C.c_void_p(reward.data_ptr()), C.c_void_p(done.data_ptr()),
                                         C.c_void_p(actions.data_ptr()), C.byref(out), env._stream()))
    return reward, done, actions, counters


def _info_arrays(info):
    return [x for x in (info.counters, info.stats, info.bit_rate_blocking, info.action_probability) if x is not None]


def _step_loop(env, T, policy):
    """The same T steps one orlg_step at a time: (reward, done, actions, [every info array stacked over the steps])."""
    rew, dones, acts, infos = [], [], [], []
    for _ in range(T):
        a = env.sample_actions() if policy == "random" else env.heuristic(policy)
        _, r, d, info = env.step(a)
        rew.append(r.clone()); dones.append(d.clone()); acts.append(a.clone())
        infos.append([x.clone() for x in _info_arrays(info)])
    return torch.stack(rew), torch.stack(dones), torch.stack(acts), [torch.stack(x) for x in zip(*infos)]


def _final_state_equal(a, b):
    ma, _, nowa, nha = a.export_state()
    mb, _, nowb, nhb = b.export_state()
    assert torch.equal(ma, mb) and torch.equal(nowa, nowb) and torch.equal(nha, nhb)
    assert torch.equal(a.counters(), b.counters())
    assert int(a.error_flags().abs().sum()) == 0 and int(b.error_flags().abs().sum()) == 0


# ------------------------------------------------------------------ GPU: the reference's goldens
def _golden_info_counters(g, t):
    """The counters of the reference's `info` at step t.  The golden records them after _next_service, which counts the next
    request in RMSA-v0 / DeepRMSA-v0 (rmsa_env.py:545-597) and its bit rate in RMCSA-v0 (the double count of
    rmcsa_env.py:294-295); RWA-v0 counts in step only (rwa_env.py:135-136)."""
    want = g["counters"][:, t].copy()
    kind = g["meta"]["kind"]
    if kind != "RWA-v0":
        br = g["req_bit_rate"][:, t + 1]
        want[:, 4] -= br; want[:, 6] -= br
    if kind in ("RMSA-v0", "DeepRMSA-v0"):
        want[:, 0] -= 1; want[:, 2] -= 1
    return want


def _golden_env(g, **kw):
    meta = g["meta"]
    env = make_env(meta, meta["n_envs"], record_decisions=False, **kw)
    env.set_trace(g["req_arrival"], g["req_holding"], g["req_src"], g["req_dst"], g["req_bit_rate"])
    env.reset(full=True)
    env.reset(full=False)
    return env


def _golden_chunks(T):
    return (1, 7, T - 8)


@pytest.mark.gpu
@pytest.mark.parametrize("name", helpers.golden_names())
def test_goldens_through_rollout_info(name):
    g = helpers.load_golden(name)
    meta = g["meta"]
    kind, args = meta["kind"], meta["env_args"]
    persistent_kind = ((kind == "DeepRMSA-v0" and args.get("j", 1) == 1) or kind == "RWA-v0" or
                       (kind == "RMSA-v0" and args.get("bit_rate_selection") != "discrete"))
    for link_stats in ((False, True) if kind in ("RMSA-v0", "DeepRMSA-v0") else (False,)):
        env = _golden_env(g, link_stats=link_stats)
        if link_stats:
            assert set(["network_compactness", "avg_link_utilization"]) <= set(env.info_keys)
        t0 = 0
        for T in _golden_chunks(meta["T"]):
            acts = torch.as_tensor(np.ascontiguousarray(g["actions"][:, t0:t0 + T].swapaxes(0, 1)), device="cuda")
            _, reward, done, _, info = env.rollout(T, "replay", actions=acts, want_obs=False, want_info=True)
            # RWA-v0's info holds the action probabilities, which the persistent kernel does not write
            assert env.kernel_info()["last_rollout_persistent"] == (persistent_kind and not link_stats and kind != "RWA-v0"), T
            assert info.keys() == env.info_keys
            for tt in range(T):
                t = t0 + tt
                assert np.array_equal(info.counters[tt].cpu().numpy(), _golden_info_counters(g, t)), ("counters", t)
                assert np.array_equal(reward[tt].cpu().numpy().astype(np.float64), g["reward"][:, t]), ("reward", t)
                assert np.array_equal(done[tt].cpu().numpy(), g["done"][:, t]), ("done", t)
            for key in info.keys():
                want = g["info_" + key][:, t0:t0 + T].swapaxes(0, 1)
                assert np.array_equal(info[key].cpu().numpy(), want), (key, t0)
            t0 += T
        assert int(env.error_flags().abs().sum()) == 0
        env.close()
    if kind == "RWA-v0":        # the counters alone: the persistent kernel itself against the reference
        env = _golden_env(g)
        t0 = 0
        for T in _golden_chunks(meta["T"]):
            acts = torch.as_tensor(np.ascontiguousarray(g["actions"][:, t0:t0 + T].swapaxes(0, 1)), device="cuda")
            _, done, _, counters = _rollout_counters(env, T, "replay", actions=acts)
            assert env.kernel_info()["last_rollout_persistent"]
            for tt in range(T):
                assert np.array_equal(counters[tt].cpu().numpy(), _golden_info_counters(g, t0 + tt)), ("counters", t0 + tt)
            t0 += T
        assert int(env.error_flags().abs().sum()) == 0
        env.close()


# ------------------------------------------------------------------ GPU: Philox traffic, persistent kernel against stepping
_RMSA = dict(load=250, mean_service_holding_time=25, allow_rejection=True)
PERSISTENT_CASES = [
    ("DeepRMSA-v0", dict(), "random", True),
    ("DeepRMSA-v0", dict(allow_rejection=True), "sap", True),
    ("DeepRMSA-v0", dict(), "random", False),          # auto_reset=False
    ("RMSA-v0", _RMSA, "sp_ff", True),
    ("RMSA-v0", _RMSA, "sap_ff", True),
    ("RMSA-v0", _RMSA, "llp_ff", True),
    ("RWA-v0", dict(load=450, mean_service_holding_time=25), "sap_lf", True),
]


def _schedule(first_done, period):
    """("ro" | "st", steps): launches of 1 / 3 / 7 / 150 / 8 steps between plain steps, placed so that the 150-step launch
    starts on a terminal step and the 8-step launch ends on one (with auto-reset)."""
    t = first_done + 150
    last = first_done + period * -(-(t + 8 - first_done) // period)      # a terminal step at least 8 steps after t
    return [("ro", 1), ("st", 3), ("ro", 3), ("st", 3), ("ro", 7), ("st", first_done - 17), ("ro", 150),
            ("st", last - 7 - t), ("ro", 8), ("st", 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", ["8", "32"])
@pytest.mark.parametrize("kind,args,policy,auto_reset", PERSISTENT_CASES)
def test_persistent_kernel_counters_equal_stepping(monkeypatch, lanes, kind, args, policy, auto_reset):
    from optical_rl_gym_b200 import OpticalVecEnv

    monkeypatch.setenv("ORLG_RO_LPW", lanes)
    n = 203                                              # ragged: neither lane count divides it
    kw = dict(traffic="philox", seed=5, episode_length=40, auto_reset=auto_reset, **args)
    ro, st = OpticalVecEnv(kind, n, helpers.golden_tables(), **kw), OpticalVecEnv(kind, n, helpers.golden_tables(), **kw)
    assert ro.kernel_info()["rollout_lanes"] == int(lanes)
    # RWA counts a request in step and its reset zeroes the episode; the others count it in _next_service and their reset
    # re-counts the pending request (rmsa_env.py:310-330)
    first_done, period = (39, 40) if kind == "RWA-v0" else (38, 39)
    terminal_seen = 0
    for what, T in _schedule(first_done, period):
        if what == "ro":
            r1, d1, a1, c1 = _rollout_counters(ro, T, policy)
            assert ro.kernel_info()["last_rollout_persistent"]
            r2, d2, a2, (c2, *_) = _step_loop(st, T, policy)
            assert torch.equal(a1, a2) and torch.equal(r1, r2) and torch.equal(d1, d2), (what, T)
            assert torch.equal(c1, c2), ("counters", T)
            terminal_seen += int(d1[0].any()) + int(d1[-1].any())
        else:
            for _ in range(T):
                a = ro.sample_actions() if policy == "random" else ro.heuristic(policy)
                x, y = ro.step(a), st.step(a)
                assert torch.equal(x[1], y[1]) and torch.equal(x[2], y[2])
                assert torch.equal(x[3].counters, y[3].counters)
    assert terminal_seen >= (2 if auto_reset else 1)
    _final_state_equal(ro, st)
    ro.close(); st.close()


# ------------------------------------------------------------------ GPU: the per-step paths
def _wide_tables(name):
    from test_wide_statistics import tables

    return tables(name)


_RMSA320 = dict(episode_length=40, mean_service_holding_time=25, num_spectrum_resources=320, allow_rejection=True)
PER_STEP_CASES = {
    "deeprmsa_j2": ("DeepRMSA-v0", "nsfnet", dict(j=2, episode_length=40), "random", False),
    "rmcsa_7x320": ("RMCSA-v0", "nsfnet", dict(episode_length=40, load=3000, mean_service_holding_time=25, num_spectrum_resources=320,
                                               num_spatial_resources=7, worst_xt=-84.7, allow_rejection=True), "random", False),
    "wide_rmsa_fused": ("RMSA-v0", "ring30", dict(_RMSA320, load=900), "sap_ff", False),
    "nsfnet_link_stats": ("RMSA-v0", "nsfnet", dict(_RMSA, episode_length=40), "sap_ff", True),
    "deeprmsa_link_stats": ("DeepRMSA-v0", "nsfnet", dict(episode_length=40), "random", True),
    "wide_link_stats": ("RMSA-v0", "ring30", dict(_RMSA320, load=700), "random", True),
    "discrete_bit_rates": ("RMSA-v0", "nsfnet", dict(episode_length=40, load=100, mean_service_holding_time=25, allow_rejection=True,
                                                     bit_rate_selection="discrete", num_spectrum_resources=64), "llp_ff", False),
    "rwa_action_probability": ("RWA-v0", "nsfnet", dict(episode_length=40, load=450, mean_service_holding_time=25), "sap_ff", False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PER_STEP_CASES))
def test_per_step_paths_keep_every_info_array(case):
    from optical_rl_gym_b200 import OpticalVecEnv

    kind, topo, args, policy, link_stats = PER_STEP_CASES[case]
    tabs = helpers.golden_tables() if topo == "nsfnet" else _wide_tables(topo)
    kw = dict(traffic="philox", seed=9, link_stats=link_stats, **args)
    ro, st = OpticalVecEnv(kind, 75, tabs, **kw), OpticalVecEnv(kind, 75, tabs, **kw)
    n_arrays = 1 + (ro._stats is not None) + (ro._brb is not None) + (ro._ap is not None)
    assert n_arrays >= (2 if link_stats or case in ("discrete_bit_rates", "rwa_action_probability") else 1)
    for T in (1, 7, 45):
        _, r1, d1, a1, info = ro.rollout(T, policy, want_obs=False, want_info=True)
        assert not ro.kernel_info()["last_rollout_persistent"]
        r2, d2, a2, arrays = _step_loop(st, T, policy)
        assert torch.equal(a1, a2) and torch.equal(r1, r2) and torch.equal(d1, d2), T
        got = _info_arrays(info)
        assert len(got) == len(arrays) == n_arrays
        for g_, w_ in zip(got, arrays):
            assert torch.equal(g_, w_), (case, T)
        x, y = ro.step(a2[0]), st.step(a2[0])           # a plain step in between
        assert torch.equal(x[3].counters, y[3].counters)
    _final_state_equal(ro, st)
    ro.close(); st.close()


# ------------------------------------------------------------------ GPU: full size on the persistent kernel
@pytest.mark.gpu
def test_full_size_persistent_rollout_info():
    from optical_rl_gym_b200 import OpticalVecEnv

    n, T = 65536, 300
    tables = helpers.golden_tables()
    kw = dict(seed=21, episode_length=50)
    env = OpticalVecEnv("DeepRMSA-v0", n, tables, **kw)
    _, _, done, _, info = env.rollout(T, want_obs=False, want_actions=False, want_info=True)
    assert env.kernel_info()["last_rollout_persistent"]
    c = info.counters
    assert bool((c[1:, :, 0] - c[:-1, :, 0] == 1).all()) and bool((c[0, :, 0] == 1).all())
    # the last row + what _next_service and the auto-reset did after it (test_gpu_parity.replay_golden) = the counters now
    want = c[-1].clone()
    br = torch.as_tensor(env.current_requests()[0]["bit_rate"].astype(np.int64), device="cuda")
    want[:, 0] += 1; want[:, 2] += 1; want[:, 4] += br; want[:, 6] += br
    dn = done[-1].bool()
    want[dn, 2] = 1; want[dn, 3] = 0; want[dn, 6] = br[dn]; want[dn, 7] = 0
    assert torch.equal(env.counters(), want)
    # ~100 sampled envs against a stepped twin
    twin = OpticalVecEnv("DeepRMSA-v0", n, tables, **kw)
    idx = torch.as_tensor(np.random.default_rng(0).choice(n, 100, replace=False), device="cuda")
    for t in range(T):
        _, _, _, tinfo = twin.step(twin.sample_actions())
        assert torch.equal(tinfo.counters[idx], c[t, idx]), t
    assert int(env.error_flags().abs().sum()) == 0
    env.close(); twin.close()


# ------------------------------------------------------------------ GPU: rollout_policy
@pytest.mark.gpu
@pytest.mark.parametrize("critic", [False, True])
@pytest.mark.parametrize("link_stats", [False, True])
def test_rollout_policy_info_equals_the_python_loop(critic, link_stats):
    from optical_rl_gym_b200.policy import MlpPolicy

    n, T = 129, 25
    env, twin = _env("nsfnet_j1", n, link_stats=link_stats), _env("nsfnet_j1", n, link_stats=link_stats)
    pol = MlpPolicy.from_state_dict(_sb3_state_dict(separate=True, seed=3)).cuda() if critic else _env_policy(env, seed=2)
    ro, info = env.rollout_policy(pol, T, want_info=True)
    assert info.keys() == env.info_keys
    want = [[] for _ in _info_arrays(info)]
    for t in range(T):
        a, lp, v = pol.sample_native(twin.observation(), seed=SEED, counter=twin.request_index, row_id_base=BASE)
        assert torch.equal(a[:, 0], ro.actions[t]) and torch.equal(lp, ro.log_prob[t]) and torch.equal(v, ro.value[t]), t
        _, r, d, tinfo = twin.step(a)
        assert torch.equal(r, ro.reward[t]) and torch.equal(d, ro.done[t]), t
        for w, x in zip(want, _info_arrays(tinfo)):
            w.append(x.clone())
    for g_, w in zip(_info_arrays(info), want):
        assert torch.equal(g_, torch.stack(w))
    assert int(ro.done.sum()) > 0
    plain = _env("nsfnet_j1", n, link_stats=link_stats).rollout_policy(pol, T)     # the default return is unchanged
    assert isinstance(plain, type(ro)) and torch.equal(plain.obs, ro.obs)
    env.close(); twin.close()


# ------------------------------------------------------------------ GPU: VecMonitor over rollouts
def _monitor_env(link_stats):
    return _env("nsfnet_j1", 96, link_stats=link_stats, episode_length=12)


@pytest.mark.gpu
@pytest.mark.parametrize("link_stats", [False, True])
def test_vec_monitor_rows_are_the_same_for_every_driver(tmp_path, link_stats):
    from optical_rl_gym_b200.monitor import VecMonitor

    keys = ("episode_service_blocking_rate", "episode_bit_rate_blocking_rate") + (("network_compactness",) if link_stats else ())
    T = 60
    mons = {}

    def monitor(name):
        mons[name] = VecMonitor(_monitor_env(link_stats), str(tmp_path / name), info_keywords=keys)
        return mons[name]

    m = monitor("step")
    for _ in range(T):
        m.step(m.unwrapped.sample_actions())
    m = monitor("rollout")
    for ch in (5, 1, 33, 21):
        res = m.rollout(ch)
        assert len(res) == 4
    m = monitor("mix")
    m.rollout(10)
    for _ in range(13):
        m.step(m.unwrapped.sample_actions())
    obs, reward, done, act, info = m.rollout(T - 23, want_info=True)
    assert info.counters.shape == (T - 23, 96, 8)
    # rollout_policy against the step loop it equals
    pol = _env_policy(mons["step"].unwrapped, seed=4)
    m = monitor("policy")
    for ch in (17, 43):
        assert len(m.rollout_policy(pol, ch).obs) == ch + 1
    m = monitor("policy_loop")
    for _ in range(T):
        base = m.unwrapped
        a, _, _ = pol.sample_native(base.observation(), seed=SEED, counter=base.request_index, row_id_base=BASE)
        m.step(a)
    for m in mons.values():
        m.close()
    ref = mons["step"]
    assert len(ref.episode_returns) > 96
    for name in ("rollout", "mix"):
        got = mons[name]
        assert got.episode_returns == ref.episode_returns and got.episode_lengths == ref.episode_lengths, name
        assert got.episode_infos == ref.episode_infos and got.total_steps == ref.total_steps, name
        assert _csv_rows(tmp_path / (name + ".monitor.csv")) == _csv_rows(tmp_path / "step.monitor.csv"), name
    a, b = mons["policy"], mons["policy_loop"]
    assert len(a.episode_returns) > 96
    assert a.episode_returns == b.episode_returns and a.episode_lengths == b.episode_lengths and a.episode_infos == b.episode_infos
    assert _csv_rows(tmp_path / "policy.monitor.csv") == _csv_rows(tmp_path / "policy_loop.monitor.csv")


@pytest.mark.gpu
def test_vec_monitor_rollouts_need_the_env_itself():
    from optical_rl_gym_b200.monitor import VecMonitor
    from optical_rl_gym_b200.wrappers import UseInfoReward

    env = _env("nsfnet_j1", 8)
    mon = VecMonitor(UseInfoReward(env, "episode_service_blocking_rate"))
    with pytest.raises(TypeError, match="UseInfoReward"):
        mon.rollout(3)
    with pytest.raises(TypeError, match="UseInfoReward"):
        mon.rollout_policy(_env_policy(env), 3)
    assert env.request_index == 1                     # nothing ran
    quiet = _env("nsfnet_j1", 8, collect_info=False)
    with pytest.raises(ValueError, match="collect_info"):
        quiet.rollout(3, want_info=True)
    with pytest.raises(ValueError, match="collect_info"):
        quiet.rollout_policy(_env_policy(env), 3, want_info=True)
    assert len(VecMonitor(quiet).rollout(3)) == 4      # no keywords: no info needed


# ------------------------------------------------------------------ GPU: refusals through the C ABI
@pytest.mark.gpu
def test_unsupported_info_outputs_are_refused():
    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200 import _native as nat

    L = nat.lib()
    buf = torch.empty(1 << 16, dtype=torch.float64, device="cuda")
    rmsa = OpticalVecEnv("RMSA-v0", 8, helpers.golden_tables(), seed=1, **_RMSA)
    deep = _env("nsfnet_j1", 8)
    pol = _env_policy(deep)                           # keeps the native handle alive
    actor, _ = pol._native_handles(deep._dev_index)
    obs = torch.empty((3, 8, deep.obs_dim), dtype=torch.float32, device="cuda")

    def rollout(env, out):
        return env._lib.orlg_rollout_info(env._h, 2, -1, None, None, None, None, C.byref(out), env._stream())

    def rollout_policy(out):
        return L.orlg_rollout_policy_info(deep._h, 2, actor, None, 1, 0, C.c_void_p(obs.data_ptr()), None, None, None, None, None,
                                          C.byref(out), deep._stream())

    def message(rc):
        assert rc == -2, (rc, L.orlg_last_error().decode())           # ORLG_E_UNSUPPORTED
        return L.orlg_last_error().decode()

    for call in (lambda o: rollout(rmsa, o), lambda o: rollout(deep, o), rollout_policy):
        assert "orlg_enable_stats" in message(call(_info_out(stats=buf)))
    per_step_br = message(L.orlg_bit_rate_blocking(rmsa._h, C.c_void_p(buf.data_ptr()), rmsa._stream()))
    per_step_ap = message(L.orlg_action_probability(rmsa._h, C.c_void_p(buf.data_ptr()), rmsa._stream()))
    assert message(rollout(rmsa, _info_out(brb=buf))) == per_step_br
    assert message(rollout(rmsa, _info_out(ap=buf))) == per_step_ap
    assert message(rollout_policy(_info_out(brb=buf))) == per_step_br
    assert message(rollout_policy(_info_out(ap=buf))) == per_step_ap
    assert rmsa.request_index == 1 and deep.request_index == 1           # nothing was stepped
    rmsa.close(); deep.close()
