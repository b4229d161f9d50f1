"""GPU parity of the T-steps-per-launch rollout path (orlg_rollout / OpticalVecEnv.rollout):
bit-for-bit against the step-by-step path on a twin handle, and against the CPU oracle replaying the
same Philox streams.  The persistent kernel keeps masks / scalars on chip and consults the release-event
table through a sorted window, so the cases below force every window regime: frequent rebuilds (tiny
horizon), side-buffer and window-capacity overflow (huge horizon), tile-pool contention, ragged batches,
and launch boundaries interleaved with ordinary per-step calls (the state must be canonical there)."""
import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

OBS_RTOL = 1e-6      # north_star tolerance for float32 observations


def _oracles(kind, tables, n, seed, base=0, **okw):
    from oracle import oracle

    out = []
    for i in range(n):
        o = oracle.OracleEnv(kind, tables, **okw)
        o.set_philox(seed, base + i)
        o.reset(full=True)
        out.append(o)
    return out


def _final_state_equal(a, b):
    ma, ala, nowa, nha = a.export_state(allocation=True)
    mb, alb, nowb, nhb = b.export_state(allocation=True)
    assert torch.equal(ma, mb), "masks"
    assert torch.equal(ala, alb), "allocation"
    assert torch.equal(nowa, nowb) and torch.equal(nha, nhb), "clock / live services"
    assert torch.equal(a.counters(), b.counters()), "counters"
    ra, sa = a.current_requests()
    rb, sb = b.current_requests()
    assert np.array_equal(ra, rb) and np.array_equal(sa, sb), "pending request"
    assert int(a.error_flags().abs().sum()) == 0 and int(b.error_flags().abs().sum()) == 0


@pytest.mark.parametrize("policy,span,warps,tiles", [
    ("random", None, None, None),          # defaults
    ("random", "2", None, None),           # horizon of 2 steps: a rebuild almost every step
    ("random", "100000", None, None),      # horizon beyond every release: window capacity + side buffer overflow paths
    ("sap", "7", "14", "1"),               # 14 warps share ONE observation tile
    ("sp", None, "3", "2"),
])
def test_rollout_matches_step_path_and_oracle(monkeypatch, policy, span, warps, tiles):
    from optical_rl_gym_b200 import OpticalVecEnv

    for k, v in (("ORLG_RO_SPAN", span), ("ORLG_RO_WARPS", warps), ("ORLG_RO_TILES", tiles)):
        if v is not None:
            monkeypatch.setenv(k, v)
    tables = helpers.golden_tables()
    n, seed = 1000 if warps == "14" else 200, 17
    kw = dict(traffic="philox", seed=seed, episode_length=45, allow_rejection=(policy != "random"))
    ro = OpticalVecEnv("DeepRMSA-v0", n, tables, **kw)
    st = OpticalVecEnv("DeepRMSA-v0", n, tables, **kw)
    pol_id = {"random": 1, "sp": 10, "sap": 11}[policy]
    n_or = 64
    orc = _oracles("DeepRMSA-v0", tables, n_or, seed, num_slots=100, episode_length=45, allow_rejection=(policy != "random"))

    def step_path(T):
        obs, rew, done, act = [], [], [], []
        for _ in range(T):
            a = st.sample_actions() if policy == "random" else st.heuristic(policy)
            o, r, d, _ = st.step(a)
            obs.append(o.clone()); rew.append(r.clone()); done.append(d.clone()); act.append(a.clone())
        return torch.stack(obs), torch.stack(rew), torch.stack(done), torch.stack(act)

    for T in (1, 7, 64, 3, 150):
        o1, r1, d1, a1 = ro.rollout(T, policy)
        o2, r2, d2, a2 = step_path(T)
        assert torch.equal(a1, a2), ("actions", T)
        assert torch.equal(r1, r2) and torch.equal(d1, d2), ("reward / done", T)
        assert torch.equal(o1, o2), ("observations", T)
        refs = [o.rollout(T, policy=pol_id, want_obs=True) for o in orc]
        assert np.array_equal(a1[:, :n_or].cpu().numpy(), np.stack([r["actions"] for r in refs], 1)), ("oracle actions", T)
        assert np.array_equal(r1[:, :n_or].cpu().numpy().astype(np.float64), np.stack([r["rewards"] for r in refs], 1)), T
        assert np.array_equal(d1[:, :n_or].cpu().numpy(), np.stack([r["dones"] for r in refs], 1)), T
        np.testing.assert_allclose(o1[:, :n_or].cpu().numpy(), np.stack([r["obs"] for r in refs], 1), rtol=OBS_RTOL, atol=0)
        _final_state_equal(ro, st)
        # a few ordinary steps on both handles between the launches: the rollout left canonical state behind
        for _ in range(5):
            a = ro.sample_actions()
            assert torch.equal(a, st.sample_actions())
            x, y = ro.step(a), st.step(a)
            assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1]) and torch.equal(x[2], y[2])
        for o in orc:
            o.rollout(5, policy=1)
    avail = ro.available_slots().cpu().numpy()
    for i, o in enumerate(orc):
        oa, oal, onow, onh = o.state()
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("oracle masks", i)
        assert np.array_equal(ro.counters()[i].cpu().numpy(), o.counters()), ("oracle counters", i)
    ro.close(); st.close()


def test_rollout_without_outputs_and_partial_outputs():
    from optical_rl_gym_b200 import OpticalVecEnv

    tables = helpers.golden_tables()
    kw = dict(traffic="philox", seed=3, episode_length=30)
    a = OpticalVecEnv("DeepRMSA-v0", 97, tables, **kw)
    b = OpticalVecEnv("DeepRMSA-v0", 97, tables, **kw)
    o, r, d, act = a.rollout(80)
    o2, r2, d2, act2 = b.rollout(80, want_obs=False, want_actions=False)
    assert o2 is None and act2 is None
    assert torch.equal(r, r2) and torch.equal(d, d2)
    _final_state_equal(a, b)
    assert torch.equal(a.observation(), b.observation())
    a.close(); b.close()


_RMSA = dict(episode_length=50, load=250, mean_service_holding_time=25, allow_rejection=True)
_RWA = dict(episode_length=64, load=450, mean_service_holding_time=25)


@pytest.mark.parametrize("kind,env_args,policy", [
    # RMSA-v0 / RWA-v0 on NSFNET: the persistent kernel with the reference's heuristics evaluated in-kernel
    ("RMSA-v0", _RMSA, "sap_ff"), ("RMSA-v0", _RMSA, "sp_ff"), ("RMSA-v0", _RMSA, "llp_ff"), ("RMSA-v0", _RMSA, "random"),
    ("RMSA-v0", dict(_RMSA, load=600, num_spectrum_resources=64), "sap_ff"),
    ("RWA-v0", _RWA, "random"), ("RWA-v0", _RWA, "sap_ff"), ("RWA-v0", _RWA, "sap_lf"), ("RWA-v0", _RWA, "llp_ff"),
    ("RWA-v0", dict(_RWA, load=900), "sp_ff"),
    # outside the persistent kernel's limits: the same entry point on the per-step kernels
    ("DeepRMSA-v0", dict(episode_length=40, j=2), "sap"),
    ("RMSA-v0", dict(_RMSA, bit_rate_selection="discrete"), "sap_ff"),
    ("RMCSA-v0", dict(episode_length=50, load=400, mean_service_holding_time=25, num_spectrum_resources=100,
                      num_spatial_resources=3, worst_xt=-84.7, allow_rejection=True), "sap_ff"),
])
def test_generic_rollout_equals_step_loop(kind, env_args, policy):
    from optical_rl_gym_b200 import OpticalVecEnv

    tables = helpers.golden_tables()
    kw = dict(traffic="philox", seed=9, **env_args)
    ro = OpticalVecEnv(kind, 80, tables, **kw)
    st = OpticalVecEnv(kind, 80, tables, **kw)
    for T in (60, 1, 130):
        o1, r1, d1, a1 = ro.rollout(T, policy)
        for t in range(T):
            a = st.sample_actions() if policy == "random" else st.heuristic(policy)
            o, r, d, _ = st.step(a)
            assert torch.equal(a1[t], a), ("actions", t, a1[t][:8], a[:8])
            assert torch.equal(r1[t], r) and torch.equal(d1[t], d), t
            if o is not None:
                assert torch.equal(o1[t], o), t
        _final_state_equal(ro, st)
    if kind == "RWA-v0":          # the action histogram behind info["path_action_probability"] (rwa_env.py:103, 148-151)
        a = ro.sample_actions()
        ia, ib = ro.step(a)[3], st.step(a)[3]
        assert torch.equal(ia["path_action_probability"], ib["path_action_probability"])
        assert torch.equal(ia["wavelength_action_probability"], ib["wavelength_action_probability"])
    ro.close(); st.close()


def test_rollout_full_size_65536_envs_invariants_and_sampled_oracle():
    """BASELINE configs[2] size through the persistent kernel: conservation invariants over all envs, ~100 sampled
    envs bit-for-bit against the oracle (masks, allocation, clock, live services, counters), observations within 1e-6."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tables = helpers.golden_tables()
    n, seed, T = 65536, 21, 1200
    env = OpticalVecEnv("DeepRMSA-v0", n, tables, seed=seed, episode_length=333)
    acc = torch.zeros(n, dtype=torch.int64, device="cuda")
    ndone = torch.zeros(n, dtype=torch.int64, device="cuda")
    last_obs = None
    for chunk in (100, 500, 37, 563):
        o, r, d, a = env.rollout(chunk)
        acc += (r > 0).sum(0)
        ndone += d.sum(0)
        last_obs = o[-1]
    assert int(env.error_flags().abs().sum()) == 0
    cnt = env.counters()
    assert torch.all(cnt[:, 0] == T + 1) and torch.all(cnt[:, 1] == acc)
    assert torch.all(ndone == T // 332)
    m, alloc, now, nheap = env.export_state(allocation=True)
    avail = env.available_slots()
    assert torch.equal((avail == 0), (alloc.reshape(avail.shape) >= 0))          # busy slots == slots of live services
    assert torch.equal(last_obs, env.observation())
    rate = float(acc.sum()) / (n * T)
    assert 0.3 < rate < 0.4, rate
    avail = avail.cpu().numpy()
    cnt = cnt.cpu().numpy()
    rng = np.random.default_rng(1)
    for i in sorted(set([0, 1, 31, 32, 447, 448, n - 1] + rng.integers(0, n, 96).tolist())):
        o = oracle.OracleEnv("DeepRMSA-v0", tables, num_slots=100, episode_length=333)
        o.set_philox(seed, i)
        o.reset(full=True)
        o.rollout(T, policy=1)
        oa, oal, onow, onh = o.state()
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("masks", i)
        assert np.array_equal(alloc[i].cpu().numpy(), oal), ("allocation", i)
        assert now[i].item() == onow and nheap[i].item() == onh, ("clock / live services", i)
        assert np.array_equal(cnt[i], o.counters()), ("counters", i)
        np.testing.assert_allclose(last_obs[i].cpu().numpy(), o.observation(), rtol=OBS_RTOL, atol=0)
    env.close()


@pytest.mark.parametrize("name", helpers.golden_names())
def test_rollout_replays_reference_trace(name):
    """The requests AND actions recorded from the live reference, replayed through orlg_rollout in chunks: for the
    DeepRMSA j = 1 goldens this is the persistent kernel (the one bench.py times) consuming reference traces
    directly; every other golden goes through the same entry point on the per-step kernels."""
    from optical_rl_gym_b200 import OpticalVecEnv

    g = helpers.load_golden(name)
    meta = g["meta"]
    n, T, kind = meta["n_envs"], meta["T"], meta["kind"]
    env = OpticalVecEnv(kind, n, helpers.golden_tables(), traffic="trace", **meta["env_args"])
    env.set_trace(g["req_arrival"], g["req_holding"], g["req_src"], g["req_dst"], g["req_bit_rate"])
    env.reset(full=True)
    obs0 = env.reset(full=False)           # evaluate_heuristic's reset() before the first episode (utils.py:113)
    if kind == "DeepRMSA-v0":
        np.testing.assert_allclose(obs0.cpu().numpy(), g["obs"][:, 0], rtol=OBS_RTOL, atol=0)
    actions = torch.as_tensor(np.ascontiguousarray(np.swapaxes(g["actions"], 0, 1)), device="cuda")     # [T, n, A]
    t0 = 0
    for chunk in (1, 13, 200, T):
        t1 = min(T, t0 + chunk)
        if t1 <= t0:
            break
        obs, rew, done, _ = env.rollout(t1 - t0, "replay", actions=actions[t0:t1])
        acc = (rew > 0).cpu().numpy() if kind == "DeepRMSA-v0" else (rew > 0.5).cpu().numpy()
        assert np.array_equal(acc, np.swapaxes(g["accepted"], 0, 1)[t0:t1].astype(bool)), ("accepted", t0)
        assert np.array_equal(rew.cpu().numpy().astype(np.float64), np.swapaxes(g["reward"], 0, 1)[t0:t1]), ("reward", t0)
        assert np.array_equal(done.cpu().numpy(), np.swapaxes(g["done"], 0, 1)[t0:t1]), ("done", t0)
        if kind == "DeepRMSA-v0":
            np.testing.assert_allclose(obs.cpu().numpy(), np.swapaxes(g["obs"], 0, 1)[t0 + 1:t1 + 1], rtol=OBS_RTOL, atol=0)
        t0 = t1
    m, alloc, now, nheap = env.export_state(allocation=True)
    avail = env.available_slots().cpu().numpy().reshape(g["final_avail"].shape)
    assert np.array_equal(avail, g["final_avail"])
    assert np.array_equal(alloc.cpu().numpy(), g["final_alloc"])
    assert np.array_equal(now.cpu().numpy(), g["final_now"]) and np.array_equal(nheap.cpu().numpy(), g["final_nheap"])
    want = g["counters"][:, T - 1].copy()
    dn = g["done"][:, T - 1].astype(bool)
    if kind == "RWA-v0":
        want[dn, 2] = 0; want[dn, 3] = 0
    else:
        want[dn, 2] = 1; want[dn, 3] = 0; want[dn, 6] = g["req_bit_rate"][dn, T]; want[dn, 7] = 0
    assert np.array_equal(env.counters().cpu().numpy(), want)
    assert int(env.error_flags().abs().sum()) == 0
    env.close()


def test_packed_records_and_host_rollout_equal_the_device_rollout():
    """orlg_rollout_packed + orlg_expand_packed (host decoder) and orlg_rollout_host (chunked, pipelined) against orlg_rollout:
    bit-identical float32 rows, rewards, dones, actions; the three handles end in the same state."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tables = helpers.golden_tables()
    kw = dict(traffic="philox", seed=12, episode_length=33)
    a = OpticalVecEnv("DeepRMSA-v0", 1000, tables, **kw)
    b = OpticalVecEnv("DeepRMSA-v0", 1000, tables, **kw)
    c = OpticalVecEnv("DeepRMSA-v0", 1000, tables, **kw)
    for T, pol in ((1, "random"), (37, "random"), (90, "sap")):
        o, r, d, act = a.rollout(T, pol)
        pk = b.rollout_packed(T, pol)
        o2, r2, d2, a2 = b.expand_packed(pk)
        assert np.array_equal(o.cpu().numpy(), o2), ("obs", T)
        assert np.array_equal(r.cpu().numpy(), r2) and np.array_equal(d.cpu().numpy(), d2), T
        assert np.array_equal(act.cpu().numpy()[..., 0], a2), T
        o3, r3, d3, a3 = c.rollout_host(T, pol, chunk=8, threads=3)
        assert np.array_equal(o2, o3) and np.array_equal(r2, r3) and np.array_equal(d2, d3) and np.array_equal(a2, a3), T
    _final_state_equal(a, b)
    _final_state_equal(a, c)
    # host-provided actions (ORLG_POLICY_REPLAY): the same trajectory as stepping with them one call at a time
    T = 29
    acts = np.random.default_rng(3).integers(0, 6, size=(T, 1000)).astype(np.int32)
    o3, r3, d3, _ = c.rollout_host(T, "replay", actions=acts.copy(), chunk=4, threads=2)
    for t in range(T):
        o, r, d, _ = a.step(torch.from_numpy(acts[t]).cuda())
        assert np.array_equal(o.cpu().numpy(), o3[t]) and np.array_equal(r.cpu().numpy(), r3[t]), t
        assert np.array_equal(d.cpu().numpy().astype(np.uint8), d3[t]), t
    _final_state_equal(a, c)
    a.close(); b.close(); c.close()


@pytest.mark.parametrize("kind,env_args,heuristic,pol_id", [
    ("DeepRMSA-v0", dict(episode_length=50), "shortest_available_path_first_fit", 11),
    ("RMSA-v0", dict(episode_length=60, load=250, mean_service_holding_time=25, allow_rejection=True), "least_loaded_path_first_fit", 12),
    ("RWA-v0", dict(episode_length=40, load=450, mean_service_holding_time=25), "shortest_available_path_first_fit", 11),
])
def test_evaluate_heuristic_matches_the_reference_loop(kind, env_args, heuristic, pol_id):
    """utils.evaluate_heuristic (utils.py:103-141) batched: per-episode rewards / lengths of every env equal the oracle's
    (which restates the reference loop: reset(), then heuristic + step until done)."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200.utils import evaluate_heuristic

    tables = helpers.golden_tables()
    n, episodes, seed = 40, 4, 6
    env = OpticalVecEnv(kind, n, tables, traffic="philox", seed=seed, **env_args)
    rewards, lengths = evaluate_heuristic(env, heuristic, n_eval_episodes=episodes, return_episode_rewards=True, chunk=37)
    okw = helpers.sim_kwargs(dict(kind=kind, env_args=env_args))
    L = env_args["episode_length"] if kind == "RWA-v0" else env_args["episode_length"] - 1
    for i, o in enumerate(_oracles(kind, tables, n, seed, **okw)):
        o.reset(full=False)
        r = o.rollout(episodes * L, policy=pol_id)
        ends = np.nonzero(r["dones"])[0]
        assert list(ends) == [L * (e + 1) - 1 for e in range(episodes)]
        want = [r["rewards"][e * L:(e + 1) * L].sum() for e in range(episodes)]
        assert np.array_equal(rewards[:, i].cpu().numpy(), np.array(want)), i
        assert (lengths[:, i] == L).all()
    mean, std = evaluate_heuristic(OpticalVecEnv(kind, n, tables, traffic="philox", seed=seed, **env_args), heuristic, n_eval_episodes=episodes)
    assert abs(mean - rewards.mean().item()) < 1e-9 and abs(std - rewards.std(unbiased=False).item()) < 1e-9
    env.close()


@pytest.mark.parametrize("kind,env_args,policy", [("DeepRMSA-v0", dict(episode_length=40), "random"),
                                                  ("RMSA-v0", _RMSA, "sap_ff"), ("RWA-v0", _RWA, "sap_ff")])
def test_state_dict_round_trip_continues_bit_for_bit(kind, env_args, policy):
    """state_dict() after a mix of rollouts and steps, load_state_dict() into a FRESH env (also through a CPU copy): both then
    produce identical trajectories and end in the same state."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tables = helpers.golden_tables()
    kw = dict(traffic="philox", seed=5, **env_args)
    a = OpticalVecEnv(kind, 300, tables, **kw)
    a.rollout(70, policy)
    for _ in range(3):
        a.step(a.sample_actions())
    a.rollout(11, policy)                       # the checkpoint is taken while the events sit in the rollout-private storage
    sd = {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in a.state_dict().items()}
    b = OpticalVecEnv(kind, 300, tables, **dict(kw, seed=999))
    b.rollout(5, policy)
    b.load_state_dict(sd)
    _final_state_equal(a, b)
    ra, rb = a.rollout(90, policy), b.rollout(90, policy)
    for x, y in zip(ra, rb):
        assert (x is None and y is None) or torch.equal(x, y)
    _final_state_equal(a, b)
    a.close(); b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("quantum,iat,lifetime", [(4.0, 0.5, 20.0), (1.0, 0.125, 3.0), (16.0, 0.5, 24.0)])
def test_rollout_equal_release_times(quantum, iat, lifetime):
    """Services that expire at EXACTLY the same time (the reference's heapq orders them by insertion, App. B-9: the order
    does not change the masks, but every one of them must leave in the right step).  Release times are multiples of
    `quantum`, so groups of quantum / iat consecutive arrivals tie; the window rebuild's warp-cooperative rank sort has to
    keep tied entries apart (one window row each) on its short-list, single-list and > 32-entry paths."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tables = helpers.golden_tables()
    n, T = 96, 400
    rng = np.random.default_rng(int(quantum * 8))
    arrival = np.tile(iat * np.arange(1, T + 3, dtype=np.float64), (n, 1))
    arrival += iat * rng.integers(0, 3, size=(n, 1))                      # env clocks are not aligned
    holding = quantum * np.ceil((arrival + lifetime) / quantum) - arrival   # exact: everything is a multiple of 2^-3
    assert np.all(arrival + holding == quantum * np.ceil((arrival + lifetime) / quantum))
    src = rng.integers(0, tables.num_nodes, size=arrival.shape).astype(np.int32)
    dst = (src + rng.integers(1, tables.num_nodes, size=arrival.shape).astype(np.int32)) % tables.num_nodes
    br = rng.integers(25, 101, size=arrival.shape).astype(np.int32)
    actions = rng.integers(0, tables.k_paths, size=(T, n, 1)).astype(np.int32)
    kw = dict(episode_length=150, mean_service_holding_time=lifetime, mean_service_inter_arrival_time=iat)
    env = OpticalVecEnv("DeepRMSA-v0", n, tables, traffic="trace", **kw)
    env.set_trace(arrival, holding, src, dst, br)
    env.reset(full=True)
    refs = []
    for i in range(n):
        o = oracle.OracleEnv("DeepRMSA-v0", tables, num_slots=100, episode_length=150, mean_holding=lifetime, mean_iat=iat)
        o.set_trace(arrival[i], holding[i], src[i], dst[i], br[i])
        o.reset(full=True)
        refs.append((o, o.rollout(T, policy=0, actions=actions[:, i], want_obs=True)))
    act_dev = torch.as_tensor(actions, device="cuda")
    t0 = 0
    for chunk in (3, 37, 160, T):
        t1 = min(T, t0 + chunk)
        if t1 <= t0:
            break
        obs, rew, done, _ = env.rollout(t1 - t0, "replay", actions=act_dev[t0:t1])
        assert np.array_equal(rew.cpu().numpy().astype(np.float64), np.stack([r["rewards"][t0:t1] for _, r in refs], 1)), t0
        assert np.array_equal(done.cpu().numpy(), np.stack([r["dones"][t0:t1] for _, r in refs], 1)), t0
        np.testing.assert_allclose(obs.cpu().numpy(), np.stack([r["obs"][t0:t1] for _, r in refs], 1), rtol=OBS_RTOL, atol=0)
        t0 = t1
    avail = env.available_slots().cpu().numpy()
    _, _, now, nheap = env.export_state(allocation=True)
    for i, (o, _) in enumerate(refs):
        oa, _, onow, onh = o.state()
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("masks", i)
        assert now[i].item() == onow and nheap[i].item() == onh, ("clock / live services", i)
    assert int(env.error_flags().abs().sum()) == 0
    env.close()


@pytest.mark.gpu
def test_host_rollout_with_pinned_result_buffer():
    """orlg_rollout_host with a page-locked observation buffer and a ragged env count: the rows expanded from the packed
    records by the host threads must be the device rollout's, bit for bit, across chunk boundaries / a ragged last chunk."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tables = helpers.golden_tables()
    n, T = 8192 + 4096 + 37, 50
    kw = dict(seed=11, episode_length=30, collect_info=False)
    a = OpticalVecEnv("DeepRMSA-v0", n, tables, **kw)
    b = OpticalVecEnv("DeepRMSA-v0", n, tables, **kw)
    o1, r1, d1, a1 = a.rollout(T, "random")
    obs = torch.full((T, n, a.obs_dim), 7.0, dtype=torch.float32).pin_memory()
    o2, r2, d2, a2 = b.rollout_host(T, "random", obs=obs.numpy(), chunk=8, threads=3)
    assert np.array_equal(o1.cpu().numpy(), o2)
    assert np.array_equal(r1.cpu().numpy(), r2) and np.array_equal(d1.cpu().numpy(), d2)
    assert np.array_equal(a1.cpu().numpy()[..., 0], a2)
    # a second call continues from the same state
    o1, r1, d1, _ = a.rollout(T, "random")
    o2, r2, d2, _ = b.rollout_host(T, "random", obs=obs.numpy(), chunk=3, threads=2)
    assert np.array_equal(o1.cpu().numpy(), o2) and np.array_equal(r1.cpu().numpy(), r2) and np.array_equal(d1.cpu().numpy(), d2)
    _final_state_equal(a, b)
    a.close(); b.close()
