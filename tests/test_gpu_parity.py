"""GPU parity tests: the CUDA step path (through the C ABI / VecEnv) against
(a) golden vectors recorded from the live reference and (b) the CPU oracle on Philox traffic.

Bars (BASELINE.json north_star): bit-exact accept/block decisions, slot allocations, link
states, counters and integer observation fields; float64 observations bit-exact (same
operation order); float32 observations within 1e-6 relative of the reference's float64.
"""
import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

OBS_RTOL = 1e-6      # north_star: "Within 1e-6 relative: normalised float observations and rewards"


def make_env(meta, n_envs, **over):
    from optical_rl_gym_b200 import OpticalVecEnv

    args = dict(meta["env_args"])
    kw = dict(traffic="trace", record_decisions=True, collect_info=True, auto_reset=True)
    kw.update(over)
    return OpticalVecEnv(meta["kind"], n_envs, helpers.golden_tables(), **kw, **args)


def unpack_masks(m, S):
    """int32 [N, CE, words] -> uint8 bits [N, CE, ceil(S/8)] in np.packbits(little) layout."""
    b = m.cpu().numpy().view(np.uint8)          # little-endian words -> little bit order bytes
    return b.reshape(m.shape[0], m.shape[1], -1)[:, :, :(S + 7) // 8]


def replay_golden(g, obs_dtype, use_heuristic=False):
    meta = g["meta"]
    n, T, kind = meta["n_envs"], meta["T"], meta["kind"]
    env = make_env(meta, n, obs_dtype=obs_dtype)
    env.set_trace(g["req_arrival"], g["req_holding"], g["req_src"], g["req_dst"], g["req_bit_rate"])
    env.reset(full=True)
    obs = env.reset(full=False)        # evaluate_heuristic's reset() before the first episode (utils.py:113)
    S = env.num_spectrum_resources
    hid = helpers.HEURISTIC_ID[meta["policy"]] if use_heuristic else None
    nm = g["avail_bits"].shape[0]

    def check_obs(o, t):
        if kind != "DeepRMSA-v0":
            assert o is None
            return
        got = o.cpu().numpy()
        if obs_dtype == torch.float64:
            assert np.array_equal(got, g["obs"][:, t]), ("obs f64", t)
        else:
            np.testing.assert_allclose(got, g["obs"][:, t], rtol=OBS_RTOL, atol=0, err_msg="obs f32 step %d" % t)

    check_obs(obs, 0)
    for t in range(T):
        req, sid = env.current_requests()
        assert np.array_equal(req["arrival"], g["req_arrival"][:, t]) and np.array_equal(sid, g["req_id"][:, t]), t
        if hid is not None:
            a = env.heuristic(hid)
            assert np.array_equal(a.cpu().numpy(), g["actions"][:, t]), ("heuristic", t, a.cpu().numpy(), g["actions"][:, t])
        else:
            a = torch.as_tensor(g["actions"][:, t], device="cuda")
        obs, reward, done, info = env.step(a)
        d = env.decisions.cpu().numpy()
        assert np.array_equal(d[:, 0], g["accepted"][:, t]), ("accepted", t)
        assert np.array_equal(d[:, 1], g["path_row"][:, t]), ("path", t)
        assert np.array_equal(d[:, 2], g["initial_slot"][:, t]), ("slot", t)
        assert np.array_equal(d[:, 3], g["number_slots"][:, t]), ("n", t)
        if "core" in g:
            assert np.array_equal(d[:, 4], g["core"][:, t]) and np.array_equal(d[:, 5], g["mod"][:, t]), ("core/mod", t)
        assert np.array_equal(reward.cpu().numpy().astype(np.float64), g["reward"][:, t]), ("reward", t)
        assert np.array_equal(done.cpu().numpy(), g["done"][:, t]), ("done", t)
        for key in info.keys():
            assert np.array_equal(info[key].cpu().numpy(), g["info_" + key][:, t]), (key, t)
        want = g["counters"][:, t].copy()      # recorded before the driver's reset(); the VecEnv auto-resets in-step
        dn = g["done"][:, t].astype(bool)
        if kind == "RWA-v0":                   # rwa_env.py:164-179
            want[dn, 2] = 0; want[dn, 3] = 0
        else:                                  # rmsa_env.py:310-330: the pending request is re-counted
            want[dn, 2] = 1; want[dn, 3] = 0; want[dn, 6] = g["req_bit_rate"][dn, t + 1]; want[dn, 7] = 0
        assert np.array_equal(env.counters().cpu().numpy(), want), ("counters", t)
        check_obs(obs, t + 1)
        if t % 5 == 0 or t == T - 1:
            m = unpack_masks(env.export_state()[0], S)
            assert np.array_equal(m[:nm], g["avail_bits"][:, t]), ("masks", t)
    m, alloc, now, nheap = env.export_state(allocation=True)
    avail = env.available_slots().cpu().numpy().reshape(g["final_avail"].shape)
    assert np.array_equal(avail, g["final_avail"])
    assert np.array_equal(alloc.cpu().numpy(), g["final_alloc"])
    assert np.array_equal(now.cpu().numpy(), g["final_now"]) and np.array_equal(nheap.cpu().numpy(), g["final_nheap"])
    assert int(env.error_flags().abs().sum()) == 0
    env.close()


@pytest.mark.parametrize("name", helpers.golden_names())
def test_cuda_replays_reference_trace_bit_exact(name):
    replay_golden(helpers.load_golden(name), torch.float64)


@pytest.mark.parametrize("name", [n for n in helpers.golden_names() if n.startswith("deeprmsa")])
def test_cuda_float32_observations_within_tolerance(name):
    replay_golden(helpers.load_golden(name), torch.float32)


@pytest.mark.parametrize("name", [n for n in helpers.golden_names()
                                  if helpers.load_golden(n)["meta"]["policy"] in helpers.HEURISTIC_ID])
def test_cuda_heuristics_match_reference(name):
    replay_golden(helpers.load_golden(name), torch.float64, use_heuristic=True)


# ------------------------------------------------------------------ Philox traffic: CUDA vs oracle
PHILOX_CASES = [
    ("DeepRMSA-v0", dict(episode_length=37), "random", 96, 400),
    ("DeepRMSA-v0", dict(episode_length=50, j=3, allow_rejection=True, mean_service_holding_time=10.0,
                         node_request_probabilities=None), "sap", 64, 300),
    ("RMSA-v0", dict(episode_length=50, load=250, mean_service_holding_time=25, allow_rejection=True), "random", 64, 300),
    ("RMSA-v0", dict(episode_length=50, load=300, mean_service_holding_time=25, allow_rejection=True), "sap_ff", 64, 400),
    ("RMSA-v0", dict(episode_length=50, load=100, mean_service_holding_time=25, allow_rejection=True,
                     bit_rate_selection="discrete", num_spectrum_resources=64), "llp_ff", 48, 300),
    ("RWA-v0", dict(episode_length=64, load=450, mean_service_holding_time=25), "sap_ff", 64, 600),
    ("RWA-v0", dict(episode_length=64, load=450, mean_service_holding_time=25), "random", 64, 300),
    ("RMCSA-v0", dict(episode_length=50, load=1200, mean_service_holding_time=25, num_spectrum_resources=64,
                      num_spatial_resources=7, worst_xt=-84.7, allow_rejection=True), "heuristic", 48, 400),
    ("RMCSA-v0", dict(episode_length=50, load=400, mean_service_holding_time=25, num_spectrum_resources=100,
                      num_spatial_resources=3, worst_xt=-84.7, allow_rejection=True), "random", 48, 300),
]
# The DeepRMSA fast kernel with its link count read at run time (link template 0): synthetic graphs of 20 and 32 links
# (helpers.tables) and the 15-link, 3-path topo_small_xml.  env_args["topology"] names the tables (default NSFNET);
# env_args["variant"] the instance: "f64" (default) float64 observations with the decision output, "hot" the steady-state
# instance (float32 observations, no decision output), "general" the float32 instance (ORLG_NO_HOT) with decisions.
_DEEP_BLOCKING = dict(episode_length=37, mean_service_holding_time=40.0, num_spectrum_resources=64)
PHILOX_CASES += [
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="E20", variant="hot"), "random", 93, 300),
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="E32", variant="hot", allow_rejection=True), "sap", 93, 300),
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="E20", variant="general", allow_rejection=True), "sap", 93, 300),
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="E32", variant="general"), "random", 93, 300),
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="E20"), "random", 93, 300),
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="E32", allow_rejection=True), "sap", 93, 300),
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="E20", j=2, allow_rejection=True), "sap", 93, 300),
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="E32", j=2), "random", 93, 300),
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="small_xml"), "random", 93, 300),
    ("DeepRMSA-v0", dict(_DEEP_BLOCKING, topology="small_xml", variant="general", allow_rejection=True), "sap", 93, 300),
]


@pytest.mark.parametrize("kind,env_args,policy,n_envs,T", PHILOX_CASES)
def test_cuda_matches_oracle_on_philox_traffic(monkeypatch, kind, env_args, policy, n_envs, T):
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    env_args = dict(env_args)
    topo, variant = env_args.pop("topology", "nsfnet"), env_args.pop("variant", "f64")
    tables = helpers.tables(topo)
    seed, base = 77, 1000
    meta = dict(kind=kind, env_args=env_args)
    if variant == "general":
        monkeypatch.setenv("ORLG_NO_HOT", "1")
    f64, decisions = variant == "f64", variant != "hot"
    env = OpticalVecEnv(kind, n_envs, tables, traffic="philox", record_decisions=decisions,
                        obs_dtype=torch.float64 if f64 else torch.float32, env_id_base=base, seed=seed, **env_args)
    monkeypatch.delenv("ORLG_NO_HOT", raising=False)
    info = env.kernel_info()
    assert info["link_template"] == (22 if topo == "nsfnet" else 0), info
    if topo != "nsfnet":
        assert info["fast"], info
    if variant != "f64":
        assert info["hot"] == (variant == "hot"), info
    okw = helpers.sim_kwargs(meta)
    if env_args.get("bit_rate_selection") == "discrete":
        okw["bit_rates"] = [10, 40, 100]
    oracles = []
    for i in range(n_envs):
        o = oracle.OracleEnv(kind, tables, **okw)
        o.set_philox(seed, base + i)
        o.reset(full=True)
        oracles.append(o)
    pol = {"random": 1}.get(policy)
    hid = helpers.HEURISTIC_ID.get(policy)
    ref = [o.rollout(T, policy=pol if pol is not None else 10 + hid, want_obs=(kind == "DeepRMSA-v0")) for o in oracles]
    for t in range(T):
        a = env.sample_actions() if pol is not None else env.heuristic(hid)
        want_a = np.stack([r["actions"][t] for r in ref])
        assert np.array_equal(a.cpu().numpy(), want_a), ("actions", t)
        obs, reward, done, _ = env.step(a)
        if decisions:
            d = env.decisions.cpu().numpy()
            want_d = np.stack([r["decisions"][t] for r in ref])
            assert np.array_equal(d[:, :4], want_d), ("decision", t, d[:4], want_d[:4])
        assert np.array_equal(reward.cpu().numpy().astype(np.float64), np.array([r["rewards"][t] for r in ref])), t
        assert np.array_equal(done.cpu().numpy(), np.array([r["dones"][t] for r in ref])), ("done", t)
        if kind == "DeepRMSA-v0" and f64:
            assert np.array_equal(obs.cpu().numpy(), np.stack([r["obs"][t] for r in ref])), ("obs", t)
        elif kind == "DeepRMSA-v0":
            np.testing.assert_allclose(obs.cpu().numpy(), np.stack([r["obs"][t] for r in ref]), rtol=OBS_RTOL, atol=0,
                                       err_msg="obs f32 step %d" % t)
    # final state
    m, alloc, now, nheap = env.export_state(allocation=True)
    avail = env.available_slots().cpu().numpy()
    cnt = env.counters().cpu().numpy()
    req, sid = env.current_requests()
    for i, o in enumerate(oracles):
        oa, oal, onow, onh = o.state()
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("avail", i)
        assert np.array_equal(alloc[i].cpu().numpy(), oal), ("alloc", i)
        assert now[i].item() == onow and nheap[i].item() == onh
        assert np.array_equal(cnt[i], o.counters())
        r = o.request()
        assert (req["arrival"][i], req["holding"][i], req["src"][i], req["dst"][i], req["bit_rate"][i], sid[i]) == \
               (r["arrival"], r["holding"], r["src"], r["dst"], r["bit_rate"], r["service_id"])
    assert int(env.error_flags().abs().sum()) == 0
    env.close()


def test_results_do_not_depend_on_sharding():
    """Envs are keyed by global id: one batch of 128 == two shards of 64 (SURVEY.md 8e)."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tables = helpers.golden_tables()
    kw = dict(traffic="philox", seed=5, episode_length=40, record_decisions=True)
    whole = OpticalVecEnv("DeepRMSA-v0", 128, tables, env_id_base=0, **kw)
    parts = [OpticalVecEnv("DeepRMSA-v0", 64, tables, env_id_base=b, **kw) for b in (0, 64)]
    for t in range(200):
        ow, rw, dw, _ = whole.step(whole.sample_actions())
        outs = [p.step(p.sample_actions()) for p in parts]
        assert torch.equal(ow, torch.cat([o[0] for o in outs])) and torch.equal(rw, torch.cat([o[1] for o in outs]))
        assert torch.equal(dw, torch.cat([o[2] for o in outs]))
    assert torch.equal(whole.reduce_counters(), parts[0].reduce_counters() + parts[1].reduce_counters())
    assert torch.equal(whole.reduce_counters()[:8], whole.counters().sum(0))


def test_full_size_invariants_65536_envs():
    """BASELINE.json config[2] size: properties that hold at any scale + a sampled oracle cross-check."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tables = helpers.golden_tables()
    N, T, seed = 65536, 300, 3
    env = OpticalVecEnv("DeepRMSA-v0", N, tables, traffic="philox", seed=seed, record_decisions=True)
    acc = torch.zeros(N, dtype=torch.int64, device="cuda")
    ndone = torch.zeros(N, dtype=torch.int64, device="cuda")
    for t in range(T):
        obs, reward, done, info = env.step(env.sample_actions())
        acc += (reward > 0)
        ndone += done
    cnt = env.counters()
    assert int(env.error_flags().abs().sum()) == 0
    assert torch.all(cnt[:, 0] == T + 1) and torch.all(cnt[:, 1] == acc)          # processed / accepted
    assert torch.all(ndone == T // 999) or env.episode_length != 1000
    m, alloc, now, nheap = env.export_state(allocation=True)
    # every busy slot belongs to exactly one live service: popcount(busy) == #cells with an id
    avail = env.available_slots()
    assert torch.equal((avail == 0), (alloc.reshape(avail.shape) >= 0))
    assert torch.all(nheap >= 0) and torch.all(nheap <= acc)
    assert torch.isfinite(obs).all() and obs.min() >= -1.0001 and obs.max() <= 24.0   # (mean free run - 4) / 4 on an empty path
    rate = float(acc.sum()) / (N * T)
    assert 0.25 < rate < 0.6, rate                # random policy at 250 Erlang: ~0.34 in steady state, higher while filling
    # sampled envs against the oracle (same Philox streams)
    for i in (0, 1, 4097, 65535):
        o = oracle.OracleEnv("DeepRMSA-v0", tables, num_slots=100)
        o.set_philox(seed, i)
        o.reset(full=True)
        o.rollout(T, policy=1)
        oa = o.state()[0]
        assert np.array_equal(avail[i].cpu().numpy().reshape(oa.shape), oa), i
        assert np.array_equal(cnt[i].cpu().numpy(), o.counters()), i
        assert np.array_equal(obs[i].cpu().numpy(), o.observation().astype(np.float32)) or \
            np.allclose(obs[i].cpu().numpy(), o.observation(), rtol=OBS_RTOL, atol=0), i
    env.close()


def test_rejects_unsupported_and_missing_trace():
    from optical_rl_gym_b200 import OpticalVecEnv, _native

    tables = helpers.golden_tables()
    with pytest.raises(_native.NativeError):
        OpticalVecEnv("RMSA-v0", 4, tables, num_spectrum_resources=1000)       # > 512 slots per link
    env = OpticalVecEnv("RMSA-v0", 4, tables, traffic="trace")
    with pytest.raises(_native.NativeError):
        env.reset(full=True)                                                    # no trace set
    with pytest.raises(TypeError):
        OpticalVecEnv("RWA-v0", 4, tables, j=3)


# ------------------------------------------------------------------ beyond the NSFNET class (BASELINE configs[3], [4])
_WIDE_TABLES = {}


def wide_tables(name):
    """Seeded synthetic 2-edge-connected graphs (ring + chords), k-shortest paths by NetworkX (host, once)."""
    from optical_rl_gym_b200.topology import synthetic_ring_chords

    if name not in _WIDE_TABLES:
        if name == "ring30":
            _WIDE_TABLES[name] = synthetic_ring_chords(num_nodes=30, num_chords=45, k_paths=10, seed=7)     # 75 links
        else:
            _WIDE_TABLES[name] = synthetic_ring_chords(num_nodes=20, num_chords=22, k_paths=6, seed=11)    # 42 links
    return _WIDE_TABLES[name]


WIDE_CASES = [
    # configs[3] shape: RMSA-v0 on a synthetic >32-link graph, 320 slots, k = 10, SAP-FF actions
    ("RMSA-v0", "ring30", dict(episode_length=60, load=900, mean_service_holding_time=25, num_spectrum_resources=320,
                               allow_rejection=True), "sap_ff", 48, 300),
    ("RMSA-v0", "ring30", dict(episode_length=60, load=600, mean_service_holding_time=25, num_spectrum_resources=320,
                               allow_rejection=True), "random", 32, 200),
    ("RMSA-v0", "ring20", dict(episode_length=40, load=300, mean_service_holding_time=25, num_spectrum_resources=200,
                               allow_rejection=True), "llp_ff", 32, 300),
    # configs[4] shape: RMCSA-v0 on NSFNET, 7 cores x 320 slots, first-core first-fit heuristic
    ("RMCSA-v0", "nsfnet", dict(episode_length=80, load=3000, mean_service_holding_time=25, num_spectrum_resources=320,
                                num_spatial_resources=7, worst_xt=-84.7, allow_rejection=True), "heuristic", 32, 400),
    ("RMCSA-v0", "nsfnet", dict(episode_length=80, load=800, mean_service_holding_time=25, num_spectrum_resources=320,
                                num_spatial_resources=3, worst_xt=-84.7, allow_rejection=True), "random", 32, 200),
    ("DeepRMSA-v0", "ring20", dict(episode_length=45, j=2, num_spectrum_resources=160, mean_service_holding_time=25.0,
                                   mean_service_inter_arrival_time=0.05), "sap", 32, 300),
    ("DeepRMSA-v0", "ring30", dict(episode_length=45, j=1, num_spectrum_resources=320, mean_service_holding_time=25.0,
                                   mean_service_inter_arrival_time=0.04, allow_rejection=True), "random", 32, 250),
    ("RWA-v0", "ring20", dict(episode_length=64, load=400, mean_service_holding_time=25, num_spectrum_resources=160), "sap_lf", 32, 300),
]


@pytest.mark.parametrize("kind,topo,env_args,policy,n_envs,T", WIDE_CASES)
def test_wide_layout_matches_oracle(kind, topo, env_args, policy, n_envs, T):
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tables = helpers.golden_tables() if topo == "nsfnet" else wide_tables(topo)
    seed, base = 21, 500
    env = OpticalVecEnv(kind, n_envs, tables, traffic="philox", record_decisions=True, obs_dtype=torch.float64,
                        env_id_base=base, seed=seed, **env_args)
    okw = helpers.sim_kwargs(dict(kind=kind, env_args=env_args))
    oracles = []
    for i in range(n_envs):
        o = oracle.OracleEnv(kind, tables, **okw)
        o.set_philox(seed, base + i)
        o.reset(full=True)
        oracles.append(o)
    pol = {"random": 1}.get(policy)
    hid = helpers.HEURISTIC_ID.get(policy)
    ref = [o.rollout(T, policy=pol if pol is not None else 10 + hid, want_obs=(kind == "DeepRMSA-v0")) for o in oracles]
    n_acc = 0
    for t in range(T):
        a = env.sample_actions() if pol is not None else env.heuristic(hid)
        assert np.array_equal(a.cpu().numpy(), np.stack([r["actions"][t] for r in ref])), ("actions", t)
        obs, reward, done, info = env.step(a)
        d = env.decisions.cpu().numpy()
        assert np.array_equal(d[:, :4], np.stack([r["decisions"][t] for r in ref])), ("decision", t)
        assert np.array_equal(done.cpu().numpy(), np.array([r["dones"][t] for r in ref])), ("done", t)
        if kind == "DeepRMSA-v0":
            assert np.array_equal(obs.cpu().numpy(), np.stack([r["obs"][t] for r in ref])), ("obs", t)
        n_acc += int(d[:, 0].sum())
    assert n_acc > 0.05 * n_envs * T, "case exercises too few accepts (%d)" % n_acc
    m, alloc, now, nheap = env.export_state(allocation=True)
    avail = env.available_slots().cpu().numpy()
    cnt = env.counters().cpu().numpy()
    for i, o in enumerate(oracles):
        oa, oal, onow, onh = o.state()
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("avail", i)
        assert np.array_equal(alloc[i].cpu().numpy(), oal), ("alloc", i)
        assert now[i].item() == onow and nheap[i].item() == onh
        assert np.array_equal(cnt[i], o.counters())
    assert int(env.error_flags().abs().sum()) == 0
    # the same T steps as ONE orlg_rollout call on a fresh handle: for heuristic policies the wide kernels evaluate the heuristic
    # inside the step kernel (fused); actions, rewards, dones and the final state must not change
    twin = OpticalVecEnv(kind, n_envs, tables, traffic="philox", obs_dtype=torch.float64, env_id_base=base, seed=seed, **env_args)
    pname = {"heuristic": "sap_ff"}.get(policy, policy)
    _, r_ro, d_ro, a_ro = twin.rollout(T, pname)
    assert np.array_equal(a_ro.cpu().numpy(), np.stack([np.stack([np.atleast_1d(r["actions"][t]) for r in ref]) for t in range(T)]))
    assert np.array_equal(d_ro.cpu().numpy().astype(bool), np.stack([[bool(r["dones"][t]) for r in ref] for t in range(T)]))
    assert torch.equal(twin.export_state(allocation=True)[0], m) and torch.equal(twin.counters(), env.counters())
    assert torch.equal(twin.export_state(allocation=True)[1], alloc)
    assert int(twin.error_flags().abs().sum()) == 0
    twin.close()
    env.close()


# ------------------------------------------------------------------ row f1: float statistics of info
@pytest.mark.parametrize("name", [n for n in helpers.golden_names() if n.startswith(("rmsa", "deeprmsa"))])
def test_info_float_statistics_bit_exact(name):
    """network_compactness, its difference, avg_link_compactness, avg_link_utilization (rmsa_env.py:229-264):
    float64, bit-identical to the reference on the recorded traces."""
    g = helpers.load_golden(name)
    meta = g["meta"]
    n, T = meta["n_envs"], meta["T"]
    env = make_env(meta, n, obs_dtype=torch.float64, link_stats=True)
    env.set_trace(g["req_arrival"], g["req_holding"], g["req_src"], g["req_dst"], g["req_bit_rate"])
    env.reset(full=True)
    env.reset(full=False)
    for t in range(T):
        obs, reward, done, info = env.step(torch.as_tensor(g["actions"][:, t], device="cuda"))
        assert np.array_equal(env.decisions.cpu().numpy()[:, 0], g["accepted"][:, t]), ("accepted", t)
        for key in ("network_compactness", "network_compactness_difference", "avg_link_compactness", "avg_link_utilization"):
            got = info[key].cpu().numpy()
            assert np.array_equal(got, g["info_" + key][:, t]), (key, t, got, g["info_" + key][:, t])
    assert np.array_equal(env.available_slots().cpu().numpy().reshape(g["final_avail"].shape), g["final_avail"])
    assert int(env.error_flags().abs().sum()) == 0
    env.close()


@pytest.mark.parametrize("name", helpers.golden_names())
def test_graph_statistics_bit_exact(name):
    """Row f1, all four env kinds: the time-averaged statistics the reference keeps on the topology graph -- per link utilization /
    external_fragmentation / compactness (rmsa_env.py:464-543, rmcsa_env.py:591-688, rwa_env.py:365-383) and the graph's
    throughput / compactness (rmsa_env.py:439-462, rmcsa_env.py:560-589) -- float64, bit-identical to the values recorded from
    the live reference at ~140 snapshot steps of env 0."""
    g = helpers.load_golden(name)
    meta = g["meta"]
    n, T = meta["n_envs"], meta["T"]
    env = make_env(meta, n, link_stats=True)
    env.set_trace(g["req_arrival"], g["req_holding"], g["req_src"], g["req_dst"], g["req_bit_rate"])
    env.reset(full=True)
    env.reset(full=False)
    snap = {int(t): k for k, t in enumerate(g["graph_stats_step"][0])}
    for t in range(T):
        env.step(torch.as_tensor(g["actions"][:, t], device="cuda"))
        if t in snap:
            link, graph = env.graph_statistics()
            assert np.array_equal(link[0].cpu().numpy(), g["graph_link_stats"][0, snap[t]]), ("link statistics", t)
            assert np.array_equal(graph[0].cpu().numpy(), g["graph_stats"][0, snap[t]]), ("graph statistics", t)
    assert np.array_equal(env.available_slots().cpu().numpy().reshape(g["final_avail"].shape), g["final_avail"])
    assert int(env.error_flags().abs().sum()) == 0
    env.close()


# ------------------------------------------------------------------ ragged batches and boundary sizes
@pytest.mark.parametrize("kind,n_envs,env_args", [
    ("DeepRMSA-v0", 1, dict(episode_length=20)),                                   # a single env
    ("DeepRMSA-v0", 33, dict(episode_length=20)),                                  # one lane past a warp
    ("DeepRMSA-v0", 129, dict(episode_length=25, num_spectrum_resources=128)),     # one env past a CTA; S = word boundary
    ("DeepRMSA-v0", 31, dict(episode_length=2, j=2, num_spectrum_resources=33)),   # 1-step episodes, S just past a word
    ("RMSA-v0", 127, dict(episode_length=30, load=400, mean_service_holding_time=25, num_spectrum_resources=128,
                          allow_rejection=True)),
    ("RWA-v0", 5, dict(episode_length=10, load=600, mean_service_holding_time=25, num_spectrum_resources=32)),
    ("RMCSA-v0", 3, dict(episode_length=15, load=500, mean_service_holding_time=25, num_spectrum_resources=40,
                         num_spatial_resources=2, worst_xt=-84.7, allow_rejection=True)),
])
def test_ragged_batches_and_boundary_sizes_match_oracle(kind, n_envs, env_args):
    """Batch sizes that are not a multiple of the warp / CTA size, slot counts on and next to a 32-bit word
    boundary, very short episodes: CUDA == oracle on Philox traffic (decisions, dones, observations, final state)."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tables = helpers.golden_tables()
    seed, base, T = 13, 70, 120
    env = OpticalVecEnv(kind, n_envs, tables, traffic="philox", record_decisions=True, obs_dtype=torch.float64,
                        env_id_base=base, seed=seed, **env_args)
    okw = helpers.sim_kwargs(dict(kind=kind, env_args=env_args))
    refs, oracles = [], []
    for i in range(n_envs):
        o = oracle.OracleEnv(kind, tables, **okw)
        o.set_philox(seed, base + i)
        o.reset(full=True)
        refs.append(o.rollout(T, policy=1, want_obs=(kind == "DeepRMSA-v0")))
        oracles.append(o)
    for t in range(T):
        a = env.sample_actions()
        assert np.array_equal(a.cpu().numpy(), np.stack([r["actions"][t] for r in refs])), ("actions", t)
        obs, reward, done, info = env.step(a)
        assert np.array_equal(env.decisions.cpu().numpy()[:, :4], np.stack([r["decisions"][t] for r in refs])), ("decision", t)
        assert np.array_equal(done.cpu().numpy(), np.array([r["dones"][t] for r in refs])), ("done", t)
        if kind == "DeepRMSA-v0":
            assert np.array_equal(obs.cpu().numpy(), np.stack([r["obs"][t] for r in refs])), ("obs", t)
    avail = env.available_slots().cpu().numpy()
    cnt = env.counters().cpu().numpy()
    for i, o in enumerate(oracles):
        oa = o.state()[0]
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("avail", i)
        assert np.array_equal(cnt[i], o.counters()), ("counters", i)
    assert int(env.error_flags().abs().sum()) == 0
    env.close()


def test_heap_overflow_is_flagged_not_silent():
    """More live services than heap_capacity: the request is blocked and the env carries ORLG_ERR_HEAP_OVERFLOW."""
    from optical_rl_gym_b200 import OpticalVecEnv, _native

    env = OpticalVecEnv("RWA-v0", 8, helpers.golden_tables(), seed=2, heap_capacity=16, load=2000,
                        mean_service_holding_time=25, episode_length=1000)
    for _ in range(200):
        env.step(env.heuristic("sap_ff"))
    flags = env.error_flags().cpu().numpy()
    assert (flags & _native.ERR_HEAP_OVERFLOW).all()
    m, alloc, now, nheap = env.export_state(allocation=True)
    assert int(nheap.max()) <= env.heap_capacity
    avail = env.available_slots()
    assert torch.equal((avail == 0), (alloc.reshape(avail.shape) >= 0))      # state stays consistent
    env.close()


def test_steady_state_specialisation_matches_oracle_and_generic_instance(monkeypatch):
    """The HOT instance of the fast kernel (what bench.py and a plain rollout run: Philox traffic, float32
    observation, no decision output) against the oracle, and bit-for-bit against the general instance."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tables = helpers.golden_tables()
    n, T, seed = 200, 300, 31
    kw = dict(traffic="philox", seed=seed, episode_length=45)
    hot = OpticalVecEnv("DeepRMSA-v0", n, tables, **kw)                      # collect_info on: info counters too
    monkeypatch.setenv("ORLG_NO_HOT", "1")
    gen = OpticalVecEnv("DeepRMSA-v0", n, tables, **kw)
    monkeypatch.delenv("ORLG_NO_HOT")
    refs = []
    for i in range(n):
        o = oracle.OracleEnv("DeepRMSA-v0", tables, num_slots=100, episode_length=45)
        o.set_philox(seed, i)
        o.reset(full=True)
        refs.append((o, o.rollout(T, policy=1, want_obs=True)))
    assert torch.equal(hot.reset(), gen.reset())
    for t in range(T):
        a = hot.sample_actions()
        assert torch.equal(a, gen.sample_actions())
        oh, rh_, dh, ih = hot.step(a)
        og, rg, dg, ig = gen.step(a)
        assert torch.equal(oh, og) and torch.equal(rh_, rg) and torch.equal(dh, dg), t
        assert torch.equal(ih.counters, ig.counters), t
        want_r = np.array([r["rewards"][t] for _, r in refs])
        assert np.array_equal(rh_.cpu().numpy().astype(np.float64), want_r), ("reward", t)
        assert np.array_equal(dh.cpu().numpy(), np.array([r["dones"][t] for _, r in refs])), ("done", t)
        np.testing.assert_allclose(oh.cpu().numpy(), np.stack([r["obs"][t] for _, r in refs]), rtol=OBS_RTOL, atol=0)
    avail = hot.available_slots().cpu().numpy()
    cnt = hot.counters().cpu().numpy()
    for i, (o, _) in enumerate(refs):
        oa = o.state()[0]
        assert np.array_equal(avail[i].reshape(oa.shape), oa) and np.array_equal(cnt[i], o.counters()), i
    assert int(hot.error_flags().abs().sum()) == 0
    hot.close(); gen.close()


def test_interleaved_handles_and_side_streams_keep_stream_order():
    """The rollout kernels are launched with the programmatic-stream-serialization attribute (their prologue may run
    under the previous kernel's tail).  Whatever precedes them in the stream -- another handle's kernels, torch
    kernels -- and whichever stream is current, results must equal a plain one-handle-at-a-time run."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tables = helpers.golden_tables()
    kw = dict(traffic="philox", episode_length=30)
    T = 120

    def snap(out):
        return tuple(x.clone() for x in out[:3])

    # reference: each handle alone, synchronised after every step; handle 0 takes one extra step whenever t % 7 == 0
    want = [[], []]
    for i, seed in enumerate((1, 2)):
        e = OpticalVecEnv("DeepRMSA-v0", 96, tables, seed=seed, **kw)
        for t in range(T):
            want[i].append(snap(e.step(e.sample_actions())))
            torch.cuda.synchronize()
            if i == 0 and t % 7 == 0:
                want[i].append(snap(e.step(e.sample_actions())))
                torch.cuda.synchronize()
        assert int(e.error_flags().abs().sum()) == 0
        e.close()
    a, b = [OpticalVecEnv("DeepRMSA-v0", 96, tables, seed=s, **kw) for s in (1, 2)]
    side = torch.cuda.Stream()
    junk = torch.zeros(1 << 20, device="cuda")
    got = [[], []]
    for t in range(T):
        aa = a.sample_actions()
        ab = b.sample_actions()                     # b's action kernel directly behind a's
        got[0].append(snap(a.step(aa)))
        junk.add_(1.0)                              # a torch kernel between the two step kernels
        got[1].append(snap(b.step(ab)))
        if t % 7 == 0:                              # another current stream: order is per stream, hand over with events
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                got[0].append(snap(a.step(a.sample_actions())))
            torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for i in range(2):
        assert len(got[i]) == len(want[i])
        for t, (g, w) in enumerate(zip(got[i], want[i])):
            for x, y in zip(g, w):
                assert torch.equal(x, y), (i, t)
    for e in (a, b):
        assert int(e.error_flags().abs().sum()) == 0
        e.close()


def test_config1_full_size_rmsa_4096_envs_sap_ff_matches_oracle():
    """BASELINE.json configs[1] at its full size: RMSA-v0 on NSFNET (100 slots, 250 Erlang, k = 5), 4096 batched envs,
    device shortest-available-path first-fit actions, 1000 steps: every env's counters, link masks, allocation, clock and
    number of live services equal the oracle's (all host threads), bit for bit."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tables = helpers.golden_tables()
    n, T, seed = 4096, 1000, 17
    args = dict(episode_length=200, load=250, mean_service_holding_time=25, allow_rejection=True)
    env = OpticalVecEnv("RMSA-v0", n, tables, traffic="philox", seed=seed, **args)
    vec = oracle.OracleVec("RMSA-v0", tables, n, seed=seed, **helpers.sim_kwargs(dict(kind="RMSA-v0", env_args=args)))
    accepted_ref = vec.run(T, policy=10 + helpers.HEURISTIC_ID["sap_ff"], with_obs=False)
    acc = torch.zeros((), dtype=torch.int64, device="cuda")
    for t in range(T):
        obs, reward, done, info = env.step(env.heuristic("sap_ff"))
        acc += (reward > 0).sum()
    assert int(acc) == accepted_ref
    cnt = env.counters().cpu().numpy()
    m, alloc, now, nheap = env.export_state(allocation=True)
    avail = env.available_slots().cpu().numpy()
    alloc, now, nheap = alloc.cpu().numpy(), now.cpu().numpy(), nheap.cpu().numpy()
    for i in range(n):
        assert np.array_equal(cnt[i], vec.counters(i)), ("counters", i)
        oa, oal, onow, onh = vec.state(i)
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("masks", i)
        assert np.array_equal(alloc[i], oal), ("allocation", i)
        assert now[i] == onow and nheap[i] == onh, ("clock / live services", i)
    assert int(env.error_flags().abs().sum()) == 0
    env.close(); vec.close()


def test_long_run_at_baseline_size_matches_oracle():
    """65536 envs x 2000 steps through the rollout path (HOT kernel instance, dependent launches), then invariants over
    all envs and a bit-for-bit comparison of ~100 sampled envs with the oracle replaying the same Philox streams."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tables = helpers.golden_tables()
    n, T, seed = 65536, 2000, 99
    env = OpticalVecEnv("DeepRMSA-v0", n, tables, seed=seed, episode_length=777)
    a = torch.empty((n, 1), dtype=torch.int32, device="cuda")
    for t in range(T):
        env.sample_actions(out=a)
        env.step_raw(a)
    assert int(env.error_flags().abs().sum()) == 0
    cnt = env.counters().cpu().numpy()
    assert (cnt[:, 0] == T + 1).all()
    m, alloc, now, nheap = env.export_state(allocation=True)
    avail = env.available_slots()
    assert torch.equal((avail == 0), (alloc.reshape(avail.shape) >= 0))       # busy slots == slots of live services
    avail = avail.cpu().numpy()
    obs = env.observation().cpu().numpy()
    rng = np.random.default_rng(0)
    for i in sorted(set([0, 1, 31, 32, 127, 128, n - 1] + rng.integers(0, n, 96).tolist())):
        o = oracle.OracleEnv("DeepRMSA-v0", tables, num_slots=100, episode_length=777)
        o.set_philox(seed, i)
        o.reset(full=True)
        o.rollout(T, policy=1)
        oa, oal, onow, onh = o.state()
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("masks", i)
        assert np.array_equal(alloc[i].cpu().numpy(), oal), ("allocation", i)
        assert now[i].item() == onow and nheap[i].item() == onh, ("clock / live services", i)
        assert np.array_equal(cnt[i], o.counters()), ("counters", i)
        np.testing.assert_allclose(obs[i], o.observation(), rtol=OBS_RTOL, atol=0)
    env.close()


def test_reseeding_mid_run_matches_oracle():
    """VecEnv.seed(s): the Philox key changes from the next request on, state untouched (the reference's env.seed only
    replaces the rng, optical_network_env.py:205-210)."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tables = helpers.golden_tables()
    n, T = 48, 150
    env = OpticalVecEnv("DeepRMSA-v0", n, tables, seed=5, episode_length=40, obs_dtype=torch.float64)
    orc = []
    for i in range(n):
        o = oracle.OracleEnv("DeepRMSA-v0", tables, num_slots=100, episode_length=40)
        o.set_philox(5, i)
        o.reset(full=True)
        orc.append(o)
    for phase, seed in enumerate((None, 1234, 7)):
        if seed is not None:
            assert env.seed(seed) == [seed] * n
            for i, o in enumerate(orc):
                o.set_philox(seed, i)
        refs = [o.rollout(T, policy=1, want_obs=True) for o in orc]
        for t in range(T):
            a = env.sample_actions()
            assert np.array_equal(a.cpu().numpy(), np.stack([r["actions"][t] for r in refs])), (phase, t)
            obs, reward, done, info = env.step(a)
            assert np.array_equal(obs.cpu().numpy(), np.stack([r["obs"][t] for r in refs])), (phase, t)
            assert np.array_equal(done.cpu().numpy(), np.array([r["dones"][t] for r in refs])), (phase, t)
    assert int(env.error_flags().abs().sum()) == 0
    env.close()
