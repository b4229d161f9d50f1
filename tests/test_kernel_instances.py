"""Every compiled instance of the persistent rollout kernel (deeprmsa_rollout_kernel<ET, POLICY, TRACE, KIND, LPW>) against
the CPU oracle.  The launcher picks the instance from the handle: ET = 22 on NSFNET, ET = 0 (link count read at run time) on
any other topology within the non-wide limits; 8 envs per warp below 16384 envs, 32 above (ORLG_RO_LPW forces either at
handle creation).  The ET = 0 cases run on seeded synthetic graphs of 20 and 32 links (32: every bit of the 32-bit path link
mask and the largest hop-list link index in use); batches of 93 envs leave the last warp partly filled at both lane counts.
Each case asserts through kernel_info() that it ran the instance it names and never fell back to per-step launches."""
import os
import re

import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

OBS_RTOL = 1e-6      # float32 observations against the oracle's float64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# loads and spectra at which the heuristics block 10-50 % of the requests on all three topologies within the run
_DEEP = dict(episode_length=45, mean_service_holding_time=40.0, num_spectrum_resources=64)
_RMSA = dict(episode_length=50, load=900, mean_service_holding_time=25, num_spectrum_resources=64, allow_rejection=True)
_RWA = dict(episode_length=64, load=900, mean_service_holding_time=25, num_spectrum_resources=16)
ENV_ARGS = {"DeepRMSA-v0": _DEEP, "RMSA-v0": _RMSA, "RWA-v0": _RWA}

# the policies launch_rollout_kind instantiates per kind; "replay" = given actions on trace traffic, "replay_philox" = given
# actions on Philox traffic (two instances: TRACE = true / false)
POLICIES = {
    "DeepRMSA-v0": ("random", "sp", "sap", "replay", "replay_philox"),
    "RMSA-v0": ("random", "sp_ff", "sap_ff", "llp_ff", "replay", "replay_philox"),
    "RWA-v0": ("random", "sp_ff", "sap_ff", "llp_ff", "sap_lf", "replay", "replay_philox"),
}
RO_POLICY = {"random": "RANDOM", "sp": "SP_FF", "sp_ff": "SP_FF", "sap": "SAP_FF", "sap_ff": "SAP_FF", "llp_ff": "LLP_FF",
             "sap_lf": "SAP_LF", "replay": "REPLAY", "replay_philox": "REPLAY"}
LINK_TEMPLATE = {"nsfnet": 22, "E20": 0, "E32": 0}

CASES = [(kind, policy, topo, lanes) for kind, pols in POLICIES.items() for policy in pols
         for topo in ("E20", "E32", "nsfnet") for lanes in (8, 32)]
N_ENVS = 93
CHUNKS = (1, 7, 64, 150)
STEPS_BETWEEN = 3
T_TOTAL = sum(CHUNKS) + STEPS_BETWEEN * (len(CHUNKS) - 1)


def _instance(kind, policy, topo, lanes):
    return (kind, RO_POLICY[policy], policy == "replay", LINK_TEMPLATE[topo], lanes)


def test_cases_cover_every_rollout_kernel_instance():
    """The case list above covers (kind, policy, trace, link template, lanes) for every instance orlg_api.cu can launch: a
    policy, kind or link template added to the launcher without a case here fails this check."""
    src = open(os.path.join(ROOT, "optical-rl-gym_b200", "csrc", "orlg_api.cu")).read()
    body = src[src.index("cudaError_t launch_rollout_kind("):]
    body = body[:body.index("\n}\n")]
    launched = set(re.findall(r"ORLG_RO_LAUNCH\(RO_POLICY_(\w+), (true|false)\)", body))
    assert launched == {(RO_POLICY[p], str(p == "replay").lower()) for pols in POLICIES.values() for p in pols}
    kinds = set(re.findall(r"launch_rollout_kind<ET, ORLG_(\w+)>", src))
    assert kinds == {"DEEPRMSA", "RMSA", "RWA"}
    assert set(re.findall(r"launch_rollout<(\d+)>\(env", src)) == {"22", "0"}
    assert sorted(set(LINK_TEMPLATE.values())) == [0, 22]
    covered = {_instance(*c) for c in CASES}
    want = {(k, RO_POLICY[p], p == "replay", et, lp) for k, pols in POLICIES.items() for p in pols
            for et in (22, 0) for lp in (8, 32)}
    assert covered == want
    # the topologies are what the cases claim (the GPU cases assert the handle's choice through kernel_info)
    for topo, et in LINK_TEMPLATE.items():
        t = helpers.tables(topo)
        assert (t.num_links == 22) == (et == 22) and t.num_links <= 32 and t.k_paths == 5
        assert np.all(t.pair_count[t.pair_first >= 0] == 5)
    assert helpers.tables("E20").num_links == 20 and helpers.tables("E32").num_links == 32
    assert helpers.tables("E32").path_links.max() == 31


def _trace(kind, tables, n, length, seed):
    """Seeded requests [n, length]: exponential inter-arrival and holding times of the kind's load."""
    rng = np.random.default_rng(seed)
    args = ENV_ARGS[kind]
    hold = args.get("mean_service_holding_time", 25.0)
    iat = 0.1 if kind == "DeepRMSA-v0" else hold / args["load"]
    arrival = np.cumsum(rng.exponential(iat, size=(n, length)), axis=1)
    holding = rng.exponential(hold, size=(n, length))
    src = rng.integers(0, tables.num_nodes, size=(n, length)).astype(np.int32)
    dst = ((src + rng.integers(1, tables.num_nodes, size=(n, length))) % tables.num_nodes).astype(np.int32)
    br = rng.integers(25, 101, size=(n, length)).astype(np.int32) if kind != "RWA-v0" else np.zeros((n, length), np.int32)
    return arrival, holding, src, dst, br


def _replay_actions(kind, tables, env, T, n, seed):
    """Seeded actions [T, n, action_dim] inside the action space (paths, and slots for RMSA / RWA)."""
    rng = np.random.default_rng(seed)
    if kind == "DeepRMSA-v0":
        return rng.integers(0, tables.k_paths, size=(T, n, 1)).astype(np.int32)
    return np.stack([rng.integers(0, tables.k_paths, size=(T, n)),
                     rng.integers(0, env.num_spectrum_resources, size=(T, n))], -1).astype(np.int32)


def _oracle_runs(kind, tables, n, seed, okw, trace=None, actions=None, pol_id=None, T=T_TOTAL, envs=None):
    """One oracle per env (Philox streams of (seed, env) or the env's trace row), T steps of the policy; returns the
    oracles and the stacked results: actions [T, n, A], rewards [T, n], dones [T, n], observations [T, n, D] | None."""
    from oracle import oracle

    orcs, runs = [], []
    for i in (range(n) if envs is None else envs):
        o = oracle.OracleEnv(kind, tables, **okw)
        if trace is not None:
            o.set_trace(*(a[i] for a in trace))
        else:
            o.set_philox(seed, i)
        o.reset(full=True)
        if actions is not None:
            runs.append(o.rollout(T, policy=0, actions=actions[:, i], want_obs=(kind == "DeepRMSA-v0")))
        else:
            runs.append(o.rollout(T, policy=pol_id, want_obs=(kind == "DeepRMSA-v0")))
        orcs.append(o)
    ref = dict(actions=np.stack([r["actions"] for r in runs], 1), rewards=np.stack([r["rewards"] for r in runs], 1),
               dones=np.stack([r["dones"] for r in runs], 1),
               obs=np.stack([r["obs"] for r in runs], 1) if kind == "DeepRMSA-v0" else None)
    return orcs, ref


def _state_matches_oracles(env, orcs, envs=None):
    """Masks, allocation, clock, live services, counters and the pending request of every (listed) env."""
    _, alloc, now, nheap = env.export_state(allocation=True)
    avail = env.available_slots().cpu().numpy()
    alloc, now, nheap = alloc.cpu().numpy(), now.cpu().numpy(), nheap.cpu().numpy()
    cnt = env.counters().cpu().numpy()
    req, sid = env.current_requests()
    for j, o in enumerate(orcs):
        i = j if envs is None else envs[j]
        oa, oal, onow, onh = o.state()
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("masks", i)
        assert np.array_equal(alloc[i], oal), ("allocation", i)
        assert now[i] == onow and nheap[i] == onh, ("clock / live services", i)
        assert np.array_equal(cnt[i], o.counters()), ("counters", i)
        r = o.request()
        assert (req["arrival"][i], req["holding"][i], req["src"][i], req["dst"][i], req["bit_rate"][i], sid[i]) == \
               (r["arrival"], r["holding"], r["src"], r["dst"], r["bit_rate"], r["service_id"]), ("pending request", i)
    assert int(env.error_flags().abs().sum()) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind,policy,topo,lanes", CASES)
def test_rollout_kernel_instance_matches_oracle(monkeypatch, kind, policy, topo, lanes):
    from optical_rl_gym_b200 import OpticalVecEnv

    tables = helpers.tables(topo)
    n, seed = N_ENVS, 29
    args = dict(ENV_ARGS[kind])
    if kind == "DeepRMSA-v0":
        args["allow_rejection"] = policy != "random"
    monkeypatch.setenv("ORLG_RO_LPW", str(lanes))
    trace = _trace(kind, tables, n, T_TOTAL + 8, seed) if policy == "replay" else None
    env = OpticalVecEnv(kind, n, tables, traffic="trace" if trace else "philox", seed=seed, **args)
    monkeypatch.delenv("ORLG_RO_LPW")
    if trace:
        env.set_trace(*trace)
        env.reset(full=True)
    info = env.kernel_info()
    assert info["rollout_kernel"] and not info["wide"], info
    assert info["link_template"] == LINK_TEMPLATE[topo] and info["rollout_lanes"] == lanes, info
    if kind == "DeepRMSA-v0":
        assert info["hot"], info              # the persistent DeepRMSA kernel runs under the steady-state conditions only
    okw = helpers.sim_kwargs(dict(kind=kind, env_args=args))
    actions = _replay_actions(kind, tables, env, T_TOTAL, n, seed + 1) if policy.startswith("replay") else None
    pol_id = 1 if policy == "random" else (10 + helpers.HEURISTIC_ID[policy] if actions is None else None)
    orcs, ref = _oracle_runs(kind, tables, n, seed, okw, trace=trace, actions=actions, pol_id=pol_id)
    act_dev = None if actions is None else torch.as_tensor(actions, device="cuda")

    t0 = 0
    for c, T in enumerate(CHUNKS):
        if c:                             # ordinary steps between the launches: the rollout left canonical state behind
            for t in range(t0, t0 + STEPS_BETWEEN):
                if act_dev is not None:
                    a = act_dev[t]
                else:
                    a = env.sample_actions() if policy == "random" else env.heuristic(policy)
                assert np.array_equal(a.cpu().numpy(), ref["actions"][t]), ("step actions", t)
                o, r, d, _ = env.step(a)
                assert np.array_equal(r.cpu().numpy().astype(np.float64), ref["rewards"][t]), ("step reward", t)
                assert np.array_equal(d.cpu().numpy(), ref["dones"][t]), ("step done", t)
            t0 += STEPS_BETWEEN
        sl = slice(t0, t0 + T)
        if act_dev is not None:
            o, r, d, a = env.rollout(T, "replay", actions=act_dev[sl])
        else:
            o, r, d, a = env.rollout(T, policy)
        assert env.kernel_info()["last_rollout_persistent"], "the rollout fell back to per-step launches"
        assert np.array_equal(a.cpu().numpy(), ref["actions"][sl]), ("actions", t0)
        assert np.array_equal(r.cpu().numpy().astype(np.float64), ref["rewards"][sl]), ("rewards", t0)
        assert np.array_equal(d.cpu().numpy(), ref["dones"][sl]), ("dones", t0)
        if o is not None:
            np.testing.assert_allclose(o.cpu().numpy(), ref["obs"][sl], rtol=OBS_RTOL, atol=0, err_msg="obs at %d" % t0)
        t0 += T
    assert t0 == T_TOTAL
    _state_matches_oracles(env, orcs)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,policy", [("DeepRMSA-v0", "random"), ("RMSA-v0", "sap_ff"), ("RWA-v0", "llp_ff")])
def test_natural_32_lane_rollout_with_partial_last_warp(monkeypatch, kind, policy):
    """16384 + 37 envs select 32 envs per warp by themselves (the last warp holds 5): conservation invariants over every env,
    ~64 sampled envs (the first and last of warps, the last env) bit for bit against the oracle."""
    from optical_rl_gym_b200 import OpticalVecEnv

    monkeypatch.delenv("ORLG_RO_LPW", raising=False)
    tables = helpers.tables("E32")
    n, seed = 16384 + 37, 13
    args = dict(ENV_ARGS[kind])
    env = OpticalVecEnv(kind, n, tables, seed=seed, **args)
    rng = np.random.default_rng(2)
    envs = sorted(set([0, 1, 31, 32, 16383, 16384, n - 2, n - 1] + rng.integers(0, n, 56).tolist()))
    idx = torch.as_tensor(envs, device="cuda")
    acc = torch.zeros(n, dtype=torch.int64, device="cuda")
    ndone = torch.zeros(n, dtype=torch.int64, device="cuda")
    got = dict(actions=[], rewards=[], dones=[], obs=[])
    for T in (100, 37, 163):
        o, r, d, a = env.rollout(T, policy)
        info = env.kernel_info()
        assert info["last_rollout_persistent"] and info["rollout_lanes"] == 32 and info["link_template"] == 0, info
        acc += (r > 0.5).sum(0)
        ndone += d.sum(0)
        got["actions"].append(a[:, idx].cpu().numpy()); got["rewards"].append(r[:, idx].cpu().numpy())
        got["dones"].append(d[:, idx].cpu().numpy())
        if o is not None:
            got["obs"].append(o[:, idx].cpu().numpy())
            last_obs = o[-1]
    T = 300
    assert int(env.error_flags().abs().sum()) == 0
    cnt = env.counters()
    assert torch.all(cnt[:, 0] == cnt[0, 0]) and torch.all(cnt[:, 1] == acc)       # lock step; accepted == rewarded steps
    assert torch.all(ndone == ndone[0]) and int(ndone[0]) > 0
    _, alloc, _, _ = env.export_state(allocation=True)
    avail = env.available_slots()
    assert torch.equal(avail == 0, alloc.reshape(avail.shape) >= 0)              # busy slots == slots of live services
    if kind == "DeepRMSA-v0":
        assert torch.equal(last_obs, env.observation())
    okw = helpers.sim_kwargs(dict(kind=kind, env_args=args))
    pol_id = 1 if policy == "random" else 10 + helpers.HEURISTIC_ID[policy]
    orcs, ref = _oracle_runs(kind, tables, n, seed, okw, pol_id=pol_id, T=T, envs=envs)
    assert np.array_equal(np.concatenate(got["actions"]), ref["actions"])
    assert np.array_equal(np.concatenate(got["rewards"]).astype(np.float64), ref["rewards"])
    assert np.array_equal(np.concatenate(got["dones"]), ref["dones"])
    if kind == "DeepRMSA-v0":
        np.testing.assert_allclose(np.concatenate(got["obs"]), ref["obs"], rtol=OBS_RTOL, atol=0)
    _state_matches_oracles(env, orcs, envs)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,policy", [("DeepRMSA-v0", "random"), ("RMSA-v0", "sap_ff"), ("RWA-v0", "sap_lf")])
def test_checkpoint_moves_between_lane_counts(monkeypatch, kind, policy):
    """state_dict() of an 8-lane handle taken mid-rollout, loaded into a 32-lane handle of the same size: the canonical event
    layout does not depend on the lane mapping, so both continue bit for bit."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tables = helpers.tables("E32")
    kw = dict(traffic="philox", seed=5, **ENV_ARGS[kind])
    monkeypatch.setenv("ORLG_RO_LPW", "8")
    a = OpticalVecEnv(kind, N_ENVS, tables, **kw)
    monkeypatch.setenv("ORLG_RO_LPW", "32")
    b = OpticalVecEnv(kind, N_ENVS, tables, **dict(kw, seed=999))
    monkeypatch.delenv("ORLG_RO_LPW")
    assert a.kernel_info()["rollout_lanes"] == 8 and b.kernel_info()["rollout_lanes"] == 32
    a.rollout(70, policy)
    for _ in range(3):
        a.step(a.sample_actions())
    a.rollout(11, policy)                       # the checkpoint is taken while the events sit in the 8-lane slabs
    sd = a.state_dict()
    b.rollout(5, policy)
    b.load_state_dict(sd)
    for T in (90, 1, 40):
        ra, rb = a.rollout(T, policy), b.rollout(T, policy)
        assert a.kernel_info()["last_rollout_persistent"] and b.kernel_info()["last_rollout_persistent"]
        for x, y in zip(ra, rb):
            assert (x is None and y is None) or torch.equal(x, y), T
    ma, ala, nowa, nha = a.export_state(allocation=True)
    mb, alb, nowb, nhb = b.export_state(allocation=True)
    assert torch.equal(ma, mb) and torch.equal(ala, alb) and torch.equal(nowa, nowb) and torch.equal(nha, nhb)
    assert torch.equal(a.counters(), b.counters())
    assert int(a.error_flags().abs().sum()) == 0 and int(b.error_flags().abs().sum()) == 0
    a.close(); b.close()
