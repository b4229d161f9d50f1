"""The wide kernels at the limits orlg_create accepts: up to 512 slots (four 128-bit word groups per core and link), 31 cores and
k = 16 candidate paths, against the C oracle.

launch_step picks step_wide_kernel<KIND, NWV, STATS> from 4 kinds x NWV = 1..4 x statistics on / off, and orlg_heuristic /
orlg_path_only_first_fit pick heuristic_kernel<KIND, NWV> / path_only_first_fit_kernel<NWV> by NWV the same way.  The CPU test
reads the launcher and checks that the cases of test_gpu_parity.WIDE_CASES, test_wide_statistics.WIDE_STATS_CASES and LIMIT_CASES
below run every instance it can launch.  The GPU tests run:

* every instance those lists miss, on Philox traffic, step by step against one oracle per env (decisions, rewards, dones, the
  DeepRMSA observations in float64 and float32 and its action masks, every heuristic on every state, the float statistics), then
  as one rollout on a twin handle; each case asserts the instance it ran and that its services reached the top word group and
  crossed every 128-slot boundary;
* replayed actions placed at and around every 32- and 128-bit boundary, with mass releases, on trace traffic;
* every mask operation of orlg_device.cuh (and link_shape) through tests/mask_ops_harness.cu against a numpy restatement on
  boolean arrays;
* PathOnlyFirstFitAction / SimpleMatrixObservation at every NWV and a checkpoint of a 31-core, 512-slot handle with statistics.
"""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

from test_gpu_parity import OBS_RTOL, WIDE_CASES, wide_tables  # noqa: E402
from test_wide_statistics import STAT_KEYS, WIDE_STATS_CASES, make_oracles, oracle_step  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "optical-rl-gym_b200", "csrc")
KIND_NAME = {"RWA": "RWA-v0", "RMSA": "RMSA-v0", "DEEPRMSA": "DeepRMSA-v0", "RMCSA": "RMCSA-v0"}
# the heuristics of each kind (orlg_heuristic refuses the others), all run on every state of a case
HEURISTICS = {"RMSA-v0": ("sp_ff", "sap_ff", "llp_ff"), "RWA-v0": ("sp_ff", "sap_ff", "llp_ff", "sap_lf"),
              "DeepRMSA-v0": ("sp", "sap"), "RMCSA-v0": ("sap_ff",)}

_TABLES = {}


def limit_tables(name):
    """"nsfnet" (22 links, k = 5), "ring20" (42 links, k = 6), "ring30" (75 links, k = 10) as in test_gpu_parity, and
    "ring30k16": the ring30 graph with k = 16 paths per pair (the largest k orlg_create accepts)."""
    if name == "nsfnet":
        return helpers.golden_tables()
    if name in ("ring20", "ring30"):
        return wide_tables(name)
    if name not in _TABLES:
        from optical_rl_gym_b200.topology import synthetic_ring_chords

        _TABLES[name] = synthetic_ring_chords(num_nodes=30, num_chords=45, k_paths=16, seed=7)
    return _TABLES[name]


def _rmsa(S, load, **kw):
    return dict(episode_length=60, load=load, mean_service_holding_time=25, num_spectrum_resources=S, allow_rejection=True, **kw)


def _rmcsa(S, cores, load, **kw):
    return dict(episode_length=80, load=load, mean_service_holding_time=25, num_spectrum_resources=S, num_spatial_resources=cores,
                worst_xt=-84.7, allow_rejection=True, **kw)


def _deep(S, j, iat, hold=25.0, rej=True):
    return dict(episode_length=45, j=j, num_spectrum_resources=S, mean_service_holding_time=hold,
                mean_service_inter_arrival_time=iat, allow_rejection=rej)


def _rwa(S, load):
    return dict(episode_length=64, load=load, mean_service_holding_time=25, num_spectrum_resources=S)


# (kind, topology, env_args, policy, statistics, envs, steps): the instances WIDE_CASES and WIDE_STATS_CASES leave out.  Small
# channel widths make RMSA / RMCSA services of up to ~170 slots; DeepRMSA's long holding times fill 512 slots within the run.
LIMIT_CASES = [
    ("RMSA-v0", "ring30", _rmsa(128, 700), "sap_ff", False, 32, 300),
    ("RMSA-v0", "ring30k16", _rmsa(512, 900, channel_width=0.6), "sap_ff", False, 24, 300),
    ("RMSA-v0", "ring30k16", _rmsa(385, 900, channel_width=0.8), "random", False, 32, 300),     # one slot into group 4
    ("RMCSA-v0", "ring20", _rmcsa(100, 31, 1200), "random", False, 32, 300),
    ("RMCSA-v0", "ring20", _rmcsa(256, 4, 3000, channel_width=2.0), "sap_ff", False, 32, 300),
    ("RMCSA-v0", "nsfnet", _rmcsa(512, 31, 3000, channel_width=2.0), "random", False, 32, 300),
    ("DeepRMSA-v0", "ring30k16", _deep(128, 2, 0.04), "random", False, 32, 300),
    ("DeepRMSA-v0", "nsfnet", _deep(512, 3, 0.02, hold=1000.0), "sap", False, 32, 400),
    ("RWA-v0", "ring30", _rwa(64, 900), "llp_ff", False, 32, 300),
    ("RWA-v0", "ring20", _rwa(320, 4000), "random", False, 32, 300),
    ("RWA-v0", "nsfnet", _rwa(512, 4000), "sap_lf", False, 32, 300),
    ("RMSA-v0", "ring20", _rmsa(100, 300), "random", True, 32, 300),
    ("RMSA-v0", "ring30", _rmsa(256, 900, channel_width=2.0), "llp_ff", True, 32, 300),
    ("RMSA-v0", "ring30k16", _rmsa(512, 900, channel_width=1.0), "random", True, 24, 300),
    ("RMCSA-v0", "ring20", _rmcsa(64, 31, 1200), "random", True, 32, 300),
    ("RMCSA-v0", "ring20", _rmcsa(200, 3, 3000, channel_width=2.0), "sap_ff", True, 32, 300),
    ("RMCSA-v0", "nsfnet", _rmcsa(512, 31, 3000, channel_width=2.0), "random", True, 32, 300),
    ("DeepRMSA-v0", "ring20", _deep(128, 1, 0.04), "sap", True, 32, 300),
    ("DeepRMSA-v0", "ring30k16", _deep(320, 2, 0.02, hold=1000.0), "random", True, 32, 400),
    ("DeepRMSA-v0", "nsfnet", _deep(512, 3, 0.02, hold=1000.0, rej=False), "random", True, 32, 400),
    ("RWA-v0", "ring20", _rwa(64, 900), "sap_lf", True, 32, 300),
    ("RWA-v0", "ring30", _rwa(300, 4000), "sap_lf", True, 32, 300),
    ("RWA-v0", "nsfnet", _rwa(512, 4000), "random", True, 32, 300),
]


def _nwv(env_args):
    return (env_args["num_spectrum_resources"] + 127) // 128


def _case_id(c):
    kind, topo, args, policy, stats, _, _ = c
    return "%s-%s-S%d-%s%s" % (kind, topo, args["num_spectrum_resources"], policy, "-stats" if stats else "")


def _function_body(src, signature):
    body = src[src.index(signature):]
    return body[:body.index("\n}\n")]


# ------------------------------------------------------------------ CPU: the cases cover every instance the launcher has
def test_cases_cover_every_wide_kernel_instance():
    """(kind, NWV, STATS) of WIDE_CASES, WIDE_STATS_CASES and LIMIT_CASES == every step_wide_kernel instance launch_step can
    launch; each case of LIMIT_CASES runs one that the other two lists miss; every (kind, NWV) of heuristic_kernel and every
    NWV of path_only_first_fit_kernel is run as well.  A kind or a word count added to the launcher without a case fails here."""
    src = open(os.path.join(CSRC, "orlg_api.cu")).read()
    kinds = set(re.findall(r"std::integral_constant<int, ORLG_(\w+)>\(\)", _function_body(src, "void for_kind(")))
    words = {int(w) for w in re.findall(r"std::integral_constant<int, (\d+)>\(\)", _function_body(src, "void for_words("))}
    assert kinds == set(KIND_NAME) and words == {1, 2, 3, 4}
    launch = _function_body(src, "int launch_step(")
    assert "for_kind(p.kind, [&](auto K) { for_words(p.nwv, [&](auto W) {" in launch
    assert "step_wide_kernel<KIND, NWV, true><<<" in launch and "step_wide_kernel<KIND, NWV, false><<<" in launch
    assert re.search(r"for_words\(env->p\.nwv, \[&\]\(auto W\) \{\s*heuristic_kernel<decltype\(K\)::value, decltype\(W\)::value>", src)
    assert re.search(r"for_words\(env->p\.nwv, \[&\]\(auto W\) \{ path_only_first_fit_kernel<decltype\(W\)::value>", src)
    want = {(KIND_NAME[k], w, s) for k in kinds for w in words for s in (False, True)}

    existing = {(c[0], _nwv(c[2]), False) for c in WIDE_CASES} | {(c[0], _nwv(c[2]), True) for c in WIDE_STATS_CASES}
    new = {(c[0], _nwv(c[2]), c[4]) for c in LIMIT_CASES}
    for c in LIMIT_CASES:
        assert (c[0], _nwv(c[2]), c[4]) not in existing, ("duplicates an existing case", _case_id(c))
    assert existing | new == want, sorted(want - existing - new)
    # heuristic_kernel<KIND, NWV>: every LIMIT case runs every heuristic of its kind on every state, the other cases their policy
    heur = {(c[0], _nwv(c[2])) for c in LIMIT_CASES} | {(c[0], _nwv(c[2])) for c in WIDE_CASES + WIDE_STATS_CASES if c[3] != "random"}
    assert heur == {(k, w) for k, w, _ in want}
    assert {(c[2] + 127) // 128 for c in PATH_ONLY_CASES} == words
    # the GPU cases assert kernel_info()["wide"]; here: every shape is wide (> 32 links, > 128 slots or k > 8)
    for c in LIMIT_CASES:
        t = limit_tables(c[1])
        assert t.num_links > 32 or c[2]["num_spectrum_resources"] > 128 or t.k_paths > 8, _case_id(c)
    assert limit_tables("ring30k16").k_paths == 16 and limit_tables("ring30k16").num_links == 75
    assert max(c[2].get("num_spatial_resources", 1) for c in LIMIT_CASES) == 31


# ------------------------------------------------------------------ what a case must reach
def reached(kind, S, cores, accepted):
    """Problems of a case's accepted services (rows start, n, core) against what it exists for: services in the top word group
    [128 (NWV - 1), S) (at S = 385, where no RMSA-class service fits in the one slot of group 4, a service ending at S), every
    128-slot boundary below S crossed (not for RWA: a one-slot service cannot cross one), RMCSA's last core in use.  Empty when
    all is reached."""
    a = np.asarray(accepted, np.int64).reshape(-1, 3)
    start, end, core = a[:, 0], a[:, 0] + a[:, 1], a[:, 2]
    lo = 128 * ((S + 127) // 128 - 1)
    bad = []
    if kind == "RWA-v0" or S - lo > 1:
        if not (start >= lo).any():
            bad.append("no service starts in [%d, %d)" % (lo, S))
    elif not (end == S).any():
        bad.append("no service ends at S = %d" % S)
    for b in range(128, S, 128):
        if kind != "RWA-v0" and not ((start < b) & (b < end)).any():
            bad.append("no service crosses slot %d" % b)
    if core.max(initial=-1) != cores - 1:
        bad.append("core %d is never used" % (cores - 1))
    return bad


# ------------------------------------------------------------------ GPU: every missing instance against the oracle
def _packed(avail, words):
    """Oracle available_slots [C, E, S] -> uint32 [C * E, words] with every bit >= S zero (the kernel's mask words)."""
    ce = avail.shape[0] * avail.shape[1]
    bits = np.zeros((ce, 32 * words), np.uint8)
    bits[:, :avail.shape[2]] = avail.reshape(ce, -1)
    return np.packbits(bits, axis=1, bitorder="little").view("<u4")


def _state_matches(env, oracles):
    m, alloc, now, nheap = env.export_state(allocation=True)
    m = m.cpu().numpy().view(np.uint32)
    alloc, now, nheap, cnt = alloc.cpu().numpy(), now.cpu().numpy(), nheap.cpu().numpy(), env.counters().cpu().numpy()
    for i, o in enumerate(oracles):
        oa, oal, onow, onh = o.state()
        assert np.array_equal(m[i], _packed(oa, env.mask_words)), ("masks", i)
        assert np.array_equal(alloc[i], oal), ("allocation", i)
        assert now[i] == onow and nheap[i] == onh, ("clock / live services", i)
        assert np.array_equal(cnt[i], o.counters()), ("counters", i)
    assert int(env.error_flags().abs().sum()) == 0


def _check_heuristics(env, oracles, t):
    for h in HEURISTICS[env.env_id]:
        got = env.heuristic(h).cpu().numpy()
        want = np.stack([o.heuristic(helpers.HEURISTIC_ID[h]) for o in oracles])
        assert np.array_equal(got, want), ("heuristic", h, t)


def _check_deeprmsa(env, f32, oracles, obs, t):
    want = np.stack([o.observation() for o in oracles])
    assert np.array_equal(obs.cpu().numpy(), want), ("obs f64", t)
    np.testing.assert_allclose(f32.observation().cpu().numpy(), want, rtol=OBS_RTOL, atol=0, err_msg="obs f32 step %d" % t)
    oi = np.stack([o.observation_int() for o in oracles])
    assert np.array_equal(env.observation_int().cpu().numpy(), oi), ("integer observation", t)
    k, J = env.k_paths, env.j
    want_m = (oi[:, :, 0:2 * J:2] >= 0).reshape(len(oracles), k * J)
    if env.allow_rejection:
        want_m = np.concatenate([want_m, np.ones((len(oracles), 1), bool)], 1)
    assert np.array_equal(env.action_masks().cpu().numpy(), want_m), ("action masks", t)


def _check_statistics(env, oracles, info, outs, t):
    if env.env_id in ("RMSA-v0", "DeepRMSA-v0"):
        for q, key in enumerate(STAT_KEYS):
            assert np.array_equal(info[key].cpu().numpy(), np.array([x.stats[q] for x in outs])), (key, t)
    link, graph = env.graph_statistics()
    link, graph = link.cpu().numpy(), graph.cpu().numpy()
    for i, o in enumerate(oracles):
        ol, og = o.link_stats()
        assert np.array_equal(link[i], ol) and np.array_equal(graph[i], og), ("graph statistics", t, i)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,topo,env_args,policy,stats,n_envs,T", LIMIT_CASES, ids=[_case_id(c) for c in LIMIT_CASES])
def test_wide_instance_matches_oracle(kind, topo, env_args, policy, stats, n_envs, T):
    from optical_rl_gym_b200 import OpticalVecEnv

    tabs = limit_tables(topo)
    S, V = env_args["num_spectrum_resources"], _nwv(env_args)
    seed, base = 37, 900
    kw = dict(traffic="philox", env_id_base=base, seed=seed, link_stats=stats, **env_args)
    env = OpticalVecEnv(kind, n_envs, tabs, record_decisions=True, obs_dtype=torch.float64, **kw)
    assert env.kernel_info()["wide"] and env.mask_words == 4 * V, (env.kernel_info(), env.mask_words)
    assert ("network_compactness" in env.info_keys) == (stats and kind in ("RMSA-v0", "DeepRMSA-v0"))
    if stats:
        env.graph_statistics()                         # refused (assertion) on a handle without statistics
    deep = kind == "DeepRMSA-v0"
    f32 = OpticalVecEnv(kind, n_envs, tabs, **kw) if deep else None
    oracles = make_oracles(kind, tabs, env_args, seed, base, n_envs)
    acts, dones, accepted = [], [], []
    for t in range(T):
        _check_heuristics(env, oracles, t)
        a = env.sample_actions() if policy == "random" else env.heuristic(policy)
        want_a = np.stack([o.random_action() if policy == "random" else o.heuristic(helpers.HEURISTIC_ID[policy]) for o in oracles])
        assert np.array_equal(a.cpu().numpy(), want_a), ("actions", t)
        acts.append(want_a)
        outs = [oracle_step(o, want_a[i]) for i, o in enumerate(oracles)]
        obs, reward, done, info = env.step(a)
        if deep:
            f32.step(a)
        d = env.decisions.cpu().numpy()
        acc = np.array([x.accepted for x in outs], bool)
        assert np.array_equal(d[:, 0], acc), ("accepted", t)
        want_d = np.array([(x.path_row, x.initial_slot, x.number_slots, x.core) for x in outs])
        assert np.array_equal(d[acc, 1:5], want_d[acc]) and np.all(d[~acc, 1:5] == -1), ("decision", t)
        assert np.array_equal(reward.cpu().numpy().astype(np.float64), [x.reward for x in outs]), ("reward", t)
        assert np.array_equal(done.cpu().numpy(), [x.done for x in outs]), ("done", t)
        dones.append([x.done for x in outs])
        if deep:
            _check_deeprmsa(env, f32, oracles, obs, t)
        if stats:
            _check_statistics(env, oracles, info, outs, t)
        accepted += [(x.initial_slot, x.number_slots, x.core) for x in outs if x.accepted]
    assert len(accepted) > 0.05 * n_envs * T, "case exercises too few accepts (%d)" % len(accepted)
    cores = env_args.get("num_spatial_resources", 1) if kind == "RMCSA-v0" else 1
    assert not reached(kind, S, cores, accepted), reached(kind, S, cores, accepted)
    _state_matches(env, oracles)
    if deep:
        assert int(f32.error_flags().abs().sum()) == 0
        f32.close()
    # the same T steps as ONE rollout call (heuristics: evaluated inside the step kernel, io.policy >= 0)
    twin = OpticalVecEnv(kind, n_envs, tabs, obs_dtype=torch.float64, **kw)
    _, _, d_ro, a_ro = twin.rollout(T, policy)
    assert np.array_equal(a_ro.cpu().numpy(), np.stack(acts).reshape(a_ro.shape))
    assert np.array_equal(d_ro.cpu().numpy(), np.array(dones, np.uint8))
    for x, y in zip(twin.export_state(allocation=True)[:2], env.export_state(allocation=True)[:2]):
        assert torch.equal(x, y)
    assert torch.equal(twin.counters(), env.counters())
    if stats:
        for x, y in zip(twin.graph_statistics(), env.graph_statistics()):
            assert torch.equal(x, y)
    assert int(twin.error_flags().abs().sum()) == 0
    twin.close()
    env.close()


# ------------------------------------------------------------------ GPU: replayed actions at the word and group boundaries
def _boundary_starts(S, n):
    """The start slots a replayed action tries for a service of n slots: b - n, b - n + 1, b - 1 and b at every 32-bit boundary
    b below S, then S - n (legal for step, never tried by the first-fit heuristics) and S - n + 1 (must be blocked)."""
    out = []
    for b in range(32, S, 32):
        out += [b - n, b - n + 1, b - 1, b]
    return [s for s in out if s >= 0] + [S - n, S - n + 1]


def _replay_run(kind, S, stats, n_envs=6, T=260):
    """Trace traffic whose services live long (and whose groups of up to 20 leave at one arrival), actions that put every
    service at a boundary start; device and oracle compared at every step (accept / block, masks, allocation, heuristics on the
    same state, the statistics).  Returns the accepted (start, n) of every env."""
    from optical_rl_gym_b200 import OpticalVecEnv
    from oracle import oracle

    tabs = limit_tables("ring30") if kind == "RMSA-v0" else limit_tables("ring20")
    cw = 2.0                                               # 15..51 slots at the highest spectral efficiency
    env_args = dict(episode_length=100, load=100, mean_service_holding_time=25, num_spectrum_resources=S, channel_width=cw,
                    allow_rejection=True)
    if kind == "RMCSA-v0":
        env_args.update(num_spatial_resources=2, worst_xt=-84.7)
    L = T + 2
    rng = np.random.default_rng(S + 7 * stats)
    i = np.arange(L)
    arrival = np.tile(1.0 + i, (n_envs, 1))
    # the first 20 requests of every 40 leave together just before request 40 g + 30 arrives (at distinct times: the statistics
    # depend on the order of the releases), the others stay 60 time units
    release = np.where(i % 40 < 20, 40.0 * (i // 40) + 30.5 + 0.01 * (i % 40), 1.0 + i + 60.0)
    holding = release - arrival
    src = rng.integers(0, tabs.num_nodes, (n_envs, L))
    dst = (src + rng.integers(1, tabs.num_nodes, (n_envs, L))) % tabs.num_nodes
    br = rng.integers(25, 101, (n_envs, L))
    env = OpticalVecEnv(kind, n_envs, tabs, traffic="trace", record_decisions=True, link_stats=stats, **env_args)
    env.set_trace(arrival, holding, src, dst, br)
    env.reset(full=True)
    assert env.kernel_info()["wide"] and env.mask_words == 4 * ((S + 127) // 128)
    okw = helpers.sim_kwargs(dict(kind=kind, env_args=env_args))
    oracles = []
    for e in range(n_envs):
        o = oracle.OracleEnv(kind, tabs, **okw)
        o.set_trace(arrival[e], holding[e], src[e], dst[e], br[e])
        o.reset(full=True)
        oracles.append(o)
    accepted = [[] for _ in range(n_envs)]
    for t in range(T):
        _check_heuristics(env, oracles, t)
        acts = []
        for e, o in enumerate(oracles):
            r = o.request()
            path = t % min(2, int(tabs.pair_count[r["src"] * tabs.num_nodes + r["dst"]]))
            row = int(tabs.pair_first[r["src"] * tabs.num_nodes + r["dst"]]) + path
            if kind == "RMCSA-v0":
                mod = int(tabs.path_mod[row])
                n = math.ceil(r["bit_rate"] / (int(tabs.mod_se[mod]) * cw)) + 1
            else:
                n = math.ceil(r["bit_rate"] / (int(tabs.path_se[row]) * cw)) + 1
            starts = _boundary_starts(S, n)
            s = starts[(t * 5 + e) % len(starts)]
            acts.append([path, s] if kind == "RMSA-v0" else [path, mod, (t // 3) % 2, s])
        acts = np.array(acts, np.int32)
        outs = [oracle_step(o, acts[e]) for e, o in enumerate(oracles)]
        _, _, _, info = env.step(torch.as_tensor(acts, device="cuda"))
        d = env.decisions.cpu().numpy()
        assert np.array_equal(d[:, 0], [x.accepted for x in outs]), ("accepted", t)
        for e, x in enumerate(outs):
            if acts[e][-1] + x.number_slots > S and x.number_slots > 0:
                assert not x.accepted, ("start past S - n accepted", t, e)
            if x.accepted:
                assert d[e, 3] == x.number_slots
                accepted[e].append((x.initial_slot, x.number_slots))
        _state_matches(env, oracles)
        if stats:
            _check_statistics(env, oracles, info, outs, t)
    env.close()
    return [a for acc in accepted for a in acc]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,S,stats", [("RMSA-v0", 512, False), ("RMSA-v0", 385, False), ("RMCSA-v0", 512, False),
                                          ("RMCSA-v0", 385, False), ("RMSA-v0", 512, True)])
def test_boundary_starts_match_oracle(kind, S, stats):
    acc = np.array(_replay_run(kind, S, stats))
    start, end = acc[:, 0], acc[:, 0] + acc[:, 1]
    for b in range(128, S, 128):                # services end at, start at (room for 2 slots) and cross every group boundary
        assert (end == b).any() and ((start == b).any() or b + 2 > S) and ((start < b) & (b < end)).any(), b
    assert (end == S).any(), "no service at S - n"


# ------------------------------------------------------------------ GPU: the mask operations against boolean arrays
EDGES32 = (32, 64, 96, 128, 160, 192, 224, 256, 288, 320, 352, 384, 416, 448, 480)
TRUNCATE_S = (1, 31, 32, 33, 127, 128, 129, 255, 256, 257, 383, 384, 385, 511, 512)


def ref_run_from(a):
    """R[..., i] = length of the run of ones starting at bit i (0 where bit i is 0), bits past the end counting 0."""
    R = np.zeros(a.shape, np.int64)
    run = np.zeros(a.shape[:-1], np.int64)
    for i in range(a.shape[-1] - 1, -1, -1):
        run = np.where(a[..., i], run + 1, 0)
        R[..., i] = run
    return R


def ref_link_shape(fr, S):
    """link_shape's seven fields from a run-length encoding of the first S slots, as rmsa_env.py's _update_link_stats takes
    them: (free slots, used blocks, lambda_max - lambda_min, free blocks inside [lambda_min, lambda_max), free blocks, longest
    free block, slots 0 and S - 1 both free); span and inner blocks are 0 with fewer than two used blocks."""
    runs, s = [], 0
    while s < S:
        e = s
        while e < S and fr[e] == fr[s]:
            e += 1
        runs.append((int(fr[s]), s, e - s))
        s = e
    used = [r for r in runs if r[0] == 0]
    free = [r for r in runs if r[0] == 1]
    span = inner = 0
    if len(used) > 1:
        lo, hi = used[0][1], used[-1][1] + used[-1][2]
        span = hi - lo
        inner = sum(1 for r in free if lo <= r[1] and r[1] + r[2] <= hi)
    return (int(np.sum(fr[:S])), len(used), span, inner, len(free), max([r[2] for r in free], default=0), int(fr[0] and fr[S - 1]))


def _pack(bits):
    return np.packbits(bits.astype(np.uint8), axis=-1, bitorder="little").view("<u4")


def mask_inputs(V):
    """Boolean masks of 128 V slots and the S of each (link_shape's slot count): all zeros / ones, each single bit, runs of
    many lengths starting or ending on every 32- and 128-bit edge, seeded random masks at densities 0.1 / 0.5 / 0.9, and random
    and full masks with every bit >= S cleared."""
    L = 128 * V
    masks = [np.zeros(L, bool), np.ones(L, bool)]
    for i in range(L):
        m = np.zeros(L, bool)
        m[i] = True
        masks.append(m)
    lengths = sorted(set(range(1, 34)) | {63, 64, 65, 95, 96, 97, 127, 128, 129, 191, 200, 255, 256, 257, 383, 384, 385, 511, 512})
    for e in (0,) + EDGES32 + (512,):
        if e > L:
            continue
        for n in lengths:
            for lo, hi in ((e, e + n), (e - n, e)):
                if 0 <= lo and hi <= L:
                    m = np.zeros(L, bool)
                    m[lo:hi] = True
                    masks.append(m)
    rng = np.random.default_rng(V)
    for p in (0.1, 0.5, 0.9):
        masks += list(rng.random((48, L)) < p)
    S = [L] * len(masks)
    for s in TRUNCATE_S:
        if s <= L:
            for m in [np.ones(L, bool)] + list(rng.random((6, L)) < 0.6):
                m = m.copy()
                m[s:] = False
                masks.append(m)
                S.append(s)
    return np.array(masks), np.array(S, np.int32)


def test_mask_reference_on_hand_worked_masks():
    """The numpy restatement itself, on masks worked out by hand."""
    a = np.zeros(128, bool)
    a[[3, 4, 5, 6, 40, 41, 126, 127]] = True
    R = ref_run_from(a)
    assert R[3] == 4 and R[5] == 2 and R[40] == 2 and R[126] == 2 and R[127] == 1 and R[7] == 0 and R.max() == 4
    assert list(np.flatnonzero(R >= 3)) == [3, 4] and list(np.flatnonzero(R >= 2)) == [3, 4, 5, 40, 126]
    # 8 slots, free = 1: 1 1 0 0 1 0 1 1 -> used blocks [2, 4) and [5, 6): span 4, one free block inside, 3 free blocks
    fr = np.array([1, 1, 0, 0, 1, 0, 1, 1], bool)
    assert ref_link_shape(fr, 8) == (5, 2, 4, 1, 3, 2, 1)
    assert ref_link_shape(fr, 5) == (3, 1, 0, 0, 2, 2, 1)                 # one used block: no span
    assert ref_link_shape(np.ones(8, bool), 8) == (8, 0, 0, 0, 1, 8, 1)
    assert ref_link_shape(np.zeros(8, bool), 8) == (0, 1, 0, 0, 0, 0, 0)
    assert ref_link_shape(np.array([0, 1, 0, 1, 1, 0, 1, 0], bool), 8) == (4, 4, 8, 3, 3, 2, 0)
    w = _pack(np.arange(64) % 33 == 0)
    assert w.tolist() == [1, 2]                                           # bits 0 and 33


_HARNESS = {}


def _harness(tmp_path_factory):
    if "lib" not in _HARNESS:
        from optical_rl_gym_b200 import build

        out = str(tmp_path_factory.mktemp("mask_ops") / "libmask_ops.so")
        cmd = [build.nvcc_path()] + build.NVCC_FLAGS + ["-I", CSRC, "-I", os.path.join(ROOT, "include"), "-o", out,
                                                        os.path.join(ROOT, "tests", "mask_ops_harness.cu")]
        res = subprocess.run(cmd, capture_output=True, text=True)
        assert res.returncode == 0, res.stderr
        _HARNESS["lib"] = C.CDLL(out)
    return _HARNESS["lib"]


def _call(fn, *args):
    conv = [C.c_void_p(a.data_ptr()) if torch.is_tensor(a) else C.c_int(a) for a in args]
    assert fn(*conv) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("V", [1, 2, 3, 4])
def test_mask_operations_match_boolean_reference(tmp_path_factory, V):
    lib = _harness(tmp_path_factory)
    L = 128 * V
    A, S = mask_inputs(V)
    M, NR = len(A), min(200, L)
    dev = lambda *shape, dt=torch.int32: torch.zeros(shape, dtype=dt, device="cuda")   # noqa: E731
    words = torch.as_tensor(_pack(A).view(np.int32), device="cuda")
    out = dict(runs_ge=dev(M, NR, 4 * V), run_len=dev(M, L), scalars=dev(M, 4), clear_lowest=dev(M, 4 * V), shr=dev(M, 32, 4 * V),
               shl1=dev(M, 4 * V), contains=dev(M, 2), shape=dev(M, 7))
    _call(getattr(lib, "mask_ops_v%d" % V), words, torch.as_tensor(S, device="cuda"), M, NR, *out.values())
    got = {k: v.cpu().numpy() for k, v in out.items()}
    u32 = lambda x: x.view(np.uint32)                      # noqa: E731
    R = ref_run_from(A)
    for n in range(1, NR + 1):
        assert np.array_equal(u32(got["runs_ge"][:, n - 1]), _pack(R >= n)), ("bits_runs_ge", n)
    assert np.array_equal(got["run_len"], np.where(A, R, -1)), "bits_run_length"
    idx = np.arange(L)
    ffs = np.where(A.any(1), np.argmax(A, 1), -1)
    fls = np.where(A.any(1), L - 1 - np.argmax(A[:, ::-1], 1), -1)
    assert np.array_equal(got["scalars"], np.stack([R.max(1), ffs, fls, A.sum(1)], 1)), "longest run / ffs / fls / popc"
    cl = A.copy()
    cl[np.flatnonzero(ffs >= 0), ffs[ffs >= 0]] = False
    assert np.array_equal(u32(got["clear_lowest"]), _pack(cl)), "bits_clear_lowest"
    for s in range(32):
        sh = np.zeros_like(A)
        sh[:, :L - s] = A[:, s:]
        assert np.array_equal(u32(got["shr"][:, s]), _pack(sh)), ("bits_shr_small", s)
    sh = np.zeros_like(A)
    sh[:, 1:] = A[:, :-1]
    assert np.array_equal(u32(got["shl1"]), _pack(sh)), "bits_shl1"
    B = np.roll(A, -1, 0)
    assert np.all(got["contains"][:, 0] == 1), "bits_contains(a, a & b)"
    assert np.array_equal(got["contains"][:, 1], np.all(A | ~B, 1).astype(np.int32)), "bits_contains(a, b)"
    for i in range(M):
        assert tuple(got["shape"][i]) == ref_link_shape(A[i], S[i]), ("link_shape", i, S[i])
    # bits_range on a grid of (lo, hi) holding every 32-bit edge, its neighbours and a stride through the rest
    grid = sorted({g for e in range(0, L + 1, 32) for g in (e - 1, e, e + 1) if 0 <= g <= L} | set(range(0, L + 1, 7)))
    pairs = np.array([(lo, hi) for lo in grid for hi in grid if lo <= hi], np.int32)
    rng_out = dev(len(pairs), 4 * V)
    _call(getattr(lib, "mask_range_v%d" % V), torch.as_tensor(pairs, device="cuda"), len(pairs), rng_out)
    want = (idx[None, :] >= pairs[:, :1]) & (idx[None, :] < pairs[:, 1:])
    assert np.array_equal(u32(rng_out.cpu().numpy()), _pack(want)), "bits_range"
    if V == 1:                                 # the 128-bit variants equal their generic ops on their whole domain
        flat, sched, ffs_flat = dev(M, 16, 4), dev(M, 16, 4), dev(M)
        _call(lib.mask_variants_v1, words, M, flat, sched, ffs_flat)
        for n in range(1, 17):
            assert np.array_equal(u32(flat.cpu().numpy()[:, n - 1]), _pack(R >= n)), ("bits_runs_ge_flat", n)
            assert np.array_equal(u32(sched.cpu().numpy()[:, n - 1]), _pack(R >= n)), ("bits_runs_ge_sched", n)
        assert np.array_equal(ffs_flat.cpu().numpy(), ffs), "bits_ffs_flat"
        sn = np.array([(s, n) for n in range(1, 129) for s in range(0, 129 - n)], np.int32)
        short, auto = dev(len(sn), 4), dev(len(sn), 4)
        _call(lib.mask_range_variants_v1, torch.as_tensor(sn, device="cuda"), len(sn), short, auto)
        want = (idx[None, :] >= sn[:, :1]) & (idx[None, :] < sn[:, :1] + sn[:, 1:])
        sel = sn[:, 1] <= 32
        assert np.array_equal(u32(short.cpu().numpy()[sel]), _pack(want[sel])), "bits_range_short"
        assert np.array_equal(u32(auto.cpu().numpy()), _pack(want)), "bits_range_auto"


# ------------------------------------------------------------------ GPU: wrappers at every NWV, a checkpoint at the limits
# (kind, topology, slots): path_only_first_fit_kernel<NWV> for NWV = 1..4 on the wide layout
PATH_ONLY_CASES = [("RMSA-v0", "ring20", 100), ("RMSA-v0", "ring20", 200), ("RMSA-v0", "ring30k16", 320),
                   ("RMSA-v0", "ring30k16", 512)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,topo,S", PATH_ONLY_CASES)
def test_path_only_first_fit_and_matrix_observation_at_every_nwv(kind, topo, S):
    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200.wrappers import PathOnlyFirstFitAction, SimpleMatrixObservation
    from oracle import oracle

    tabs = limit_tables(topo)
    args = _rwa(S, 3000) if kind == "RWA-v0" else _rmsa(S, 900, channel_width=1.0)
    n, T, seed = 16, 200, 9
    base = OpticalVecEnv(kind, n, tabs, traffic="philox", seed=seed, record_decisions=True, **args)
    assert base.kernel_info()["wide"] and base.mask_words == 4 * ((S + 127) // 128)
    env = PathOnlyFirstFitAction(SimpleMatrixObservation(base))
    orc = make_oracles(kind, tabs, args, seed, 0, n)
    rng = np.random.default_rng(S)
    obs = env.reset()
    starts = []
    for t in range(T):
        want_obs = np.stack([oracle.simple_matrix_observation(o, tabs.num_nodes) for o in orc])
        assert np.array_equal(obs.cpu().numpy(), want_obs.astype(np.uint8)), ("matrix", t)
        pa = rng.integers(0, tabs.k_paths + 1, n)
        want = np.array([oracle.path_only_first_fit(o, tabs, int(a)) for o, a in zip(orc, pa)])
        obs, _, _, _ = env.step(torch.as_tensor(pa, device="cuda"))
        assert np.array_equal(env._mapped.cpu().numpy(), want), ("mapped", t)
        for i, o in enumerate(orc):
            so = oracle_step(o, want[i])
            assert so.accepted == int(base.decisions[i, 0]), ("accepted", t, i)
            if so.accepted:
                starts.append(so.initial_slot)
    assert len(starts) > 0.1 * n * T and max(starts) >= 128 * ((S + 127) // 128 - 1), (len(starts), max(starts))
    _state_matches(base, orc)
    base.close()


@pytest.mark.gpu
def test_checkpoint_resumes_31_cores_512_slots_with_statistics():
    """state_dict / load_state_dict halfway through an RMCSA-v0 run of 31 cores x 512 slots (mask entries of 4 word groups)
    with statistics: the restored handle continues bit for bit (decisions, masks, allocation, statistics) and equals the oracle."""
    from optical_rl_gym_b200 import OpticalVecEnv

    tabs = limit_tables("nsfnet")
    args = _rmcsa(512, 31, 3000, channel_width=2.0)
    n, seed = 32, 19
    kw = dict(traffic="philox", seed=seed, link_stats=True, record_decisions=True, **args)
    a = OpticalVecEnv("RMCSA-v0", n, tabs, **kw)
    assert a.kernel_info()["wide"] and a.mask_words == 16
    orc = make_oracles("RMCSA-v0", tabs, args, seed, 0, n)
    for _ in range(150):
        act = a.sample_actions()
        a.step(act)
        for o, x in zip(orc, act.cpu().numpy()):
            oracle_step(o, x)
    sd = a.state_dict()
    b = OpticalVecEnv("RMCSA-v0", n, tabs, **dict(kw, seed=seed + 1))
    b.load_state_dict(sd)
    for t in range(150):
        act = a.sample_actions()
        assert torch.equal(act, b.sample_actions()), t
        _, ra, da, _ = a.step(act)
        ra, da, deca = ra.clone(), da.clone(), a.decisions.clone()
        _, rb, db, _ = b.step(act)
        assert torch.equal(ra, rb) and torch.equal(da, db) and torch.equal(deca, b.decisions), t
        for o, x in zip(orc, act.cpu().numpy()):
            oracle_step(o, x)
    for x, y in zip(a.export_state(allocation=True), b.export_state(allocation=True)):
        assert torch.equal(x, y)
    for x, y in zip(a.graph_statistics(), b.graph_statistics()):
        assert torch.equal(x, y)
    assert torch.equal(a.counters(), b.counters())
    _state_matches(b, orc)
    link, graph = b.graph_statistics()
    for i, o in enumerate(orc):
        ol, og = o.link_stats()
        assert np.array_equal(link[i].cpu().numpy(), ol) and np.array_equal(graph[i].cpu().numpy(), og), i
    a.close(); b.close()
