"""Row f1 on the wide kernels (more than 32 links or 128 slots): the float entries of RMSA / DeepRMSA `info` and the
time-averaged statistics kept on the topology graph, float64 and bit-identical to the C oracle on the same Philox streams,
for every env at every step.  The CPU test pins the oracle's numpy pairwise mean above 128 links to numpy itself."""
import os

import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

STAT_KEYS = ("network_compactness", "network_compactness_difference", "avg_link_compactness", "avg_link_utilization")
ERR_STATS_ORDER = 16


def _topology(name):
    from optical_rl_gym_b200.topology import TopologyTables, synthetic_ring_chords

    if name == "nsfnet":
        return helpers.golden_tables()
    if name == "c3":
        return TopologyTables.load(os.path.join(helpers.GOLDEN_DIR, "topo_c3_ring100_chords200_k10.npz"))
    if name == "germany50":
        return TopologyTables.load(os.path.join(helpers.GOLDEN_DIR, "topo_germany50_tables.npz"))
    if name == "ring30":
        return synthetic_ring_chords(num_nodes=30, num_chords=45, k_paths=10, seed=7)      # 75 links
    return synthetic_ring_chords(num_nodes=20, num_chords=22, k_paths=6, seed=11)           # ring20: 42 links


_TABLES = {}


def tables(name):
    if name not in _TABLES:
        _TABLES[name] = _topology(name)
    return _TABLES[name]


def make_oracles(kind, tabs, env_args, seed, base, n):
    from oracle import oracle

    okw = helpers.sim_kwargs(dict(kind=kind, env_args=env_args))
    out = []
    for i in range(n):
        o = oracle.OracleEnv(kind, tabs, **okw)
        o.set_philox(seed, base + i)
        o.reset(full=True)
        out.append(o)
    return out


def oracle_action(o, policy):
    return o.random_action() if policy == "random" else o.heuristic(helpers.HEURISTIC_ID[policy])


def oracle_step(o, a):
    """One step of an oracle env as the VecEnv takes it (auto-reset of the episode counters at the end of an episode)."""
    out, rc = o.step(a)
    assert rc == 0
    if out.done:
        o.reset(full=False)
    return out


# ------------------------------------------------------------------ CPU: the oracle's mean above 128 links is numpy's
@pytest.mark.parametrize("topo", ["c3", "germany50"])
def test_oracle_link_means_equal_numpy(topo):
    """avg_link_utilization / avg_link_compactness of the oracle == np.mean over its own link statistics in topology.edges()
    order, bit for bit: 300 links (numpy's recursive pairwise sum above 128) and 88.  Compared at every step that releases
    nothing, where the statistics read after the step are the ones `info` averaged."""
    tabs = tables(topo)
    env_args = dict(episode_length=150, load=600, mean_service_holding_time=25, num_spectrum_resources=320, allow_rejection=True)
    o = make_oracles("RMSA-v0", tabs, env_args, seed=3, base=17, n=1)[0]
    order = np.asarray(tabs.link_order)
    compared = 0
    for t in range(300):
        nheap = o.state()[3]
        out = oracle_step(o, o.heuristic(helpers.HEURISTIC_ID["sap_ff"]))
        if o.state()[3] != nheap + out.accepted:
            continue                                  # a release changed the link statistics after `info` was taken
        link, _ = o.link_stats()
        assert out.stats[3] == np.mean(link[order, 0]), ("avg_link_utilization", t)
        assert out.stats[2] == np.mean(link[order, 2]), ("avg_link_compactness", t)
        compared += 1
    assert compared >= 100, compared
    o.close()


# ------------------------------------------------------------------ GPU: every env, every step, against the oracle
_RMSA320 = dict(episode_length=60, mean_service_holding_time=25, num_spectrum_resources=320, allow_rejection=True)
WIDE_STATS_CASES = [
    ("RMSA-v0", "ring30", dict(_RMSA320, load=900), "sap_ff", 48, 400),
    ("RMSA-v0", "ring30", dict(_RMSA320, load=700), "random", 32, 300),
    ("RMSA-v0", "germany50", dict(_RMSA320, load=900), "sap_ff", 48, 400),
    ("DeepRMSA-v0", "ring20", dict(episode_length=45, j=2, num_spectrum_resources=160, mean_service_holding_time=25.0,
                                   mean_service_inter_arrival_time=0.04, allow_rejection=True), "sap", 48, 400),
    ("RWA-v0", "ring20", dict(episode_length=64, load=500, mean_service_holding_time=25, num_spectrum_resources=160), "sap_ff", 32, 400),
    ("RMCSA-v0", "nsfnet", dict(episode_length=80, load=3000, mean_service_holding_time=25, num_spectrum_resources=320,
                                num_spatial_resources=7, worst_xt=-84.7, allow_rejection=True), "heuristic", 32, 500),
    ("RMCSA-v0", "nsfnet", dict(episode_length=80, load=1200, mean_service_holding_time=25, num_spectrum_resources=320,
                                num_spatial_resources=3, worst_xt=-84.7, allow_rejection=True), "random", 32, 400),
]


def _final_state_matches(env, oracles):
    m, alloc, now, nheap = env.export_state(allocation=True)
    avail = env.available_slots().cpu().numpy()
    cnt = env.counters().cpu().numpy()
    for i, o in enumerate(oracles):
        oa, oal, onow, onh = o.state()
        assert np.array_equal(avail[i].reshape(oa.shape), oa), ("avail", i)
        assert np.array_equal(alloc[i].cpu().numpy(), oal), ("alloc", i)
        assert now[i].item() == onow and nheap[i].item() == onh, ("clock / live services", i)
        assert np.array_equal(cnt[i], o.counters()), ("counters", i)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,topo,env_args,policy,n_envs,T", WIDE_STATS_CASES)
def test_wide_statistics_match_oracle(kind, topo, env_args, policy, n_envs, T):
    from optical_rl_gym_b200 import OpticalVecEnv

    tabs = tables(topo)
    seed, base = 29, 300
    env = OpticalVecEnv(kind, n_envs, tabs, traffic="philox", record_decisions=True, env_id_base=base, seed=seed,
                        link_stats=True, **env_args)
    assert env.kernel_info()["wide"]
    oracles = make_oracles(kind, tabs, env_args, seed, base, n_envs)
    info_floats = kind in ("RMSA-v0", "DeepRMSA-v0")
    n_acc = n_rel_multi = 0
    for t in range(T):
        a = env.sample_actions() if policy == "random" else env.heuristic(helpers.HEURISTIC_ID[policy])
        want_a = np.stack([oracle_action(o, policy) for o in oracles])
        assert np.array_equal(a.cpu().numpy(), want_a), ("actions", t)
        nheap0 = np.array([o.state()[3] for o in oracles])
        outs = [oracle_step(o, want_a[i]) for i, o in enumerate(oracles)]
        _, reward, done, info = env.step(a)
        d = env.decisions.cpu().numpy()
        assert np.array_equal(d[:, 0], [x.accepted for x in outs]), ("accepted", t)
        assert np.array_equal(done.cpu().numpy(), [x.done for x in outs]), ("done", t)
        if info_floats:
            for q, key in enumerate(STAT_KEYS):
                assert np.array_equal(info[key].cpu().numpy(), np.array([x.stats[q] for x in outs])), (key, t)
        else:
            assert "network_compactness" not in info.keys()
        link, graph = env.graph_statistics()
        link, graph = link.cpu().numpy(), graph.cpu().numpy()
        for i, o in enumerate(oracles):
            ol, og = o.link_stats()
            assert np.array_equal(link[i], ol), ("link statistics", t, i)
            assert np.array_equal(graph[i], og), ("graph statistics", t, i)
        n_acc += int(d[:, 0].sum())
        released = nheap0 + d[:, 0] - np.array([o.state()[3] for o in oracles])
        n_rel_multi += int((released >= 2).sum())
    assert n_acc > 0.05 * n_envs * T, "case exercises too few accepts (%d)" % n_acc
    assert n_rel_multi > 0, "no step released two or more services"
    _final_state_matches(env, oracles)
    assert int(env.error_flags().abs().sum()) == 0
    env.close()


def _sum_nh(env, sd):
    """sum over the live services of number_slots * hops, per env, from a state_dict: it is the first [N] int64 of the last
    state array (the statistics block allocated by orlg_enable_stats; 16-byte padded in the blob)."""
    n, C, E = env.num_envs, 1, env.tables.num_links
    if env.env_id == "RMCSA-v0":
        C = env.num_spatial_resources
    words = n + (C * n + (C * E * n + 1) // 2 if env.env_id != "RWA-v0" else 0)
    blob = sd["native"].cpu().numpy()
    start = blob.size - (8 * words + 15) // 16 * 16
    return blob[start:start + 8 * n].view(np.int64)


@pytest.mark.gpu
def test_c3_statistics_at_real_shape():
    """BASELINE configs[3] shape (300 links, 320 slots, k = 10) with statistics: 4096 envs x 300 steps of device SAP-FF.
    Sampled envs: every `info` float and the graph statistics at the end against the oracle.  All envs: sum_nh equals
    the busy cells of the allocation (number_slots * hops summed over the live services), no error flag."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tabs = tables("c3")
    n, T, seed = 4096, 300, 5
    env_args = dict(episode_length=120, load=600, mean_service_holding_time=25, num_spectrum_resources=320, allow_rejection=True)
    env = OpticalVecEnv("RMSA-v0", n, tabs, traffic="philox", seed=seed, link_stats=True, **env_args)
    rng = np.random.default_rng(3)
    sample = sorted(set([0, 1, 31, 32, 63, 64, n - 1] + rng.integers(0, n, 57).tolist()))
    idx = torch.as_tensor(sample, device="cuda")
    got = np.zeros((T, len(sample), 4))
    a = torch.empty((n, 2), dtype=torch.int32, device="cuda")
    for t in range(T):
        env.heuristic("sap_ff", out=a)
        _, _, _, info = env.step(a)
        got[t] = torch.stack([info[k][idx] for k in STAT_KEYS], 1).cpu().numpy()
    assert int(env.error_flags().abs().sum()) == 0
    link, graph = env.graph_statistics()
    for j, i in enumerate(sample):
        o = make_oracles("RMSA-v0", tabs, env_args, seed, i, 1)[0]
        for t in range(T):
            out = oracle_step(o, o.heuristic(helpers.HEURISTIC_ID["sap_ff"]))
            assert np.array_equal(got[t, j], np.array(out.stats[:4])), ("info floats", i, t)
        ol, og = o.link_stats()
        assert np.array_equal(link[i].cpu().numpy(), ol) and np.array_equal(graph[i].cpu().numpy(), og), ("graph statistics", i)
        o.close()
    _, alloc, _, _ = env.export_state(allocation=True)
    busy = (alloc >= 0).reshape(n, -1).sum(1).cpu().numpy()
    assert np.array_equal(_sum_nh(env, env.state_dict()), busy)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,topo,env_args,policy", [
    ("RMSA-v0", "ring30", dict(_RMSA320, load=900), "sap_ff"),
    ("RMCSA-v0", "nsfnet", dict(episode_length=80, load=3000, mean_service_holding_time=25, num_spectrum_resources=320,
                                num_spatial_resources=7, worst_xt=-84.7, allow_rejection=True), "random"),
])
def test_rollout_with_statistics_equals_stepping(kind, topo, env_args, policy):
    """orlg_rollout on a wide handle with statistics on (fused heuristic / random) == the same steps one call at a time."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tabs = tables(topo)
    n, T = 64, 250
    kw = dict(traffic="philox", seed=11, link_stats=True, **env_args)
    one = OpticalVecEnv(kind, n, tabs, **kw)
    _, r_ro, d_ro, a_ro = one.rollout(T, policy, want_obs=False)
    two = OpticalVecEnv(kind, n, tabs, **kw)
    for t in range(T):
        a = two.sample_actions() if policy == "random" else two.heuristic(policy)
        assert torch.equal(a, a_ro[t]), t
        _, r, d, info = two.step(a)
        assert torch.equal(r, r_ro[t]) and torch.equal(d, d_ro[t]), t
    for x, y in zip(one.graph_statistics(), two.graph_statistics()):
        assert torch.equal(x, y)
    if one._stats is not None:
        assert torch.equal(one._stats, two._stats)
    assert torch.equal(one.export_state(allocation=True)[1], two.export_state(allocation=True)[1])
    assert torch.equal(one.counters(), two.counters())
    assert int(one.error_flags().abs().sum()) == 0 and int(two.error_flags().abs().sum()) == 0
    one.close(); two.close()


@pytest.mark.gpu
def test_checkpoint_resumes_wide_statistics():
    """state_dict / load_state_dict halfway through a wide statistics run: the restored batch continues with identical
    `info` floats and graph statistics."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tabs = tables("ring30")
    kw = dict(traffic="philox", seed=13, link_stats=True, **dict(_RMSA320, load=900))
    a = OpticalVecEnv("RMSA-v0", 64, tabs, **kw)
    for _ in range(150):
        a.step(a.heuristic("sap_ff"))
    sd = a.state_dict()
    b = OpticalVecEnv("RMSA-v0", 64, tabs, **kw)
    b.load_state_dict(sd)
    for t in range(150):
        _, _, _, ia = a.step(a.heuristic("sap_ff"))
        _, _, _, ib = b.step(b.heuristic("sap_ff"))
        for key in STAT_KEYS:
            assert torch.equal(ia[key], ib[key]), (key, t)
    for x, y in zip(a.graph_statistics(), b.graph_statistics()):
        assert torch.equal(x, y)
    assert int(a.error_flags().abs().sum()) == 0 and int(b.error_flags().abs().sum()) == 0
    a.close(); b.close()


@pytest.mark.gpu
def test_more_than_24_releases_in_one_step_set_the_order_flag():
    """One arrival that releases 30 services at once: ORLG_ERR_STATS_ORDER is set, the masks stay equal to the oracle's.
    Once per slot count: 160 slots on a 42-link ring run the wide kernel, 100 slots on NSFNET the generic step_kernel."""
    for slots in (160, 100):
        _more_than_24_releases(slots)


def _more_than_24_releases(slots):
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tabs = tables("ring20" if slots == 160 else "nsfnet")
    n, R, T = 2, 30, 34
    env_args = dict(episode_length=1000, load=100, mean_service_holding_time=25, num_spectrum_resources=slots)
    arrival = np.concatenate([0.01 * np.arange(1, R + 1), 5.0 + 0.01 * np.arange(T + 2 - R)])
    holding = np.concatenate([np.full(R, 1.0), np.full(T + 2 - R, 100.0)])
    src, dst = np.zeros(T + 2, np.int32), np.ones(T + 2, np.int32)
    env = OpticalVecEnv("RWA-v0", n, tabs, traffic="trace", record_decisions=True, link_stats=True, **env_args)
    env.set_trace(*[np.tile(x, (n, 1)) for x in (arrival, holding, src, dst)])
    env.reset(full=True)
    assert env.kernel_info()["wide"] == (slots == 160), slots
    o = oracle.OracleEnv("RWA-v0", tabs, **helpers.sim_kwargs(dict(kind="RWA-v0", env_args=env_args)))
    o.set_trace(arrival, holding, src, dst)
    o.reset(full=True)
    for t in range(T):
        act = np.array([0, t % slots], np.int32)
        _, _, _, _ = env.step(torch.as_tensor(np.tile(act, (n, 1)), device="cuda"))
        out = oracle_step(o, act)
        assert np.array_equal(env.decisions.cpu().numpy()[:, 0], [out.accepted] * n), (slots, t)
    flags = env.error_flags().cpu().numpy()
    assert np.all(flags == ERR_STATS_ORDER), (slots, flags)
    oa = o.state()[0]
    avail = env.available_slots().cpu().numpy()
    for i in range(n):
        assert np.array_equal(avail[i].reshape(oa.shape), oa), (slots, i)
    assert np.array_equal(env.export_state()[3].cpu().numpy(), [o.state()[3]] * n), slots
    env.close()


@pytest.mark.gpu
def test_vec_monitor_writes_wide_statistics(tmp_path):
    """VecMonitor(info_keywords=("avg_link_utilization", "network_compactness")) on a wide env: one row per episode with the
    oracle's values at the episode's last step."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200.monitor import VecMonitor

    tabs = tables("ring30")
    n, T, seed, base = 8, 130, 31, 0
    env_args = dict(_RMSA320, load=900)
    env = OpticalVecEnv("RMSA-v0", n, tabs, traffic="philox", seed=seed, env_id_base=base, link_stats=True, **env_args)
    keys = ("avg_link_utilization", "network_compactness")
    mon = VecMonitor(env, str(tmp_path / "wide"), info_keywords=keys)
    oracles = make_oracles("RMSA-v0", tabs, env_args, seed, base, n)
    want = []
    for t in range(T):
        mon.step(env.heuristic("sap_ff"))
        for i, o in enumerate(oracles):
            out = oracle_step(o, o.heuristic(helpers.HEURISTIC_ID["sap_ff"]))
            if out.done:
                want.append((t, i, out.stats[3], out.stats[0]))
    assert len(want) == 2 * n                       # episodes of 60 steps: two ends per env in 130 steps
    lines = open(str(tmp_path / "wide.monitor.csv")).read().splitlines()
    assert lines[1] == "r,l,t," + ",".join(keys)
    rows = [ln.split(",") for ln in lines[2:]]
    assert len(rows) == len(want)
    want.sort(key=lambda w: (w[0], w[1]))            # rows are written per step, envs in index order
    for row, (_, _, util, comp) in zip(rows, want):
        assert float(row[3]) == util and float(row[4]) == comp, (row, util, comp)
    assert mon.episode_infos["avg_link_utilization"] == [w[2] for w in want]
    assert mon.episode_infos["network_compactness"] == [w[3] for w in want]
    env.close()
