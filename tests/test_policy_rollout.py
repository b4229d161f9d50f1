"""PPO rollout collection on the device: the sampling epilogue of the fused policy kernel (orlg_policy_sample /
MlpPolicy.sample_native) and the closed loop obs -> policy -> env.step (orlg_rollout_policy / OpticalVecEnv.rollout_policy).

References: a numpy Philox4x32-10 (pinned to the C oracle's), an inverse-CDF sampler on the float64 softmax of
test_policy_kernel.bf16_reference, a Python loop of sample_native + step_raw on a twin env (bit for bit) and the C oracle
replaying the sampled actions."""
import ctypes as C
import os
import subprocess
import tempfile
import types

import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

from test_policy_kernel import BF16_LOGIT_ATOL, _policy, bf16_reference  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M32 = np.uint64(0xFFFFFFFF)
STREAM_POLICY = 3             # Philox counter word 3 of the action draws (DESIGN.md section 5)
# The worst-case shift of a CDF boundary for logits within BF16_LOGIT_ATOL of the reference: e^(2 * 0.02) - 1.
CDF_DELTA = 0.041
OBS_RTOL = 1e-6
# Measured on an NVIDIA B200 (1000 W power limit): over 65536 real NSFNET observations with random seeds and counters, the
# sampled action equalled the reference sampler's on 0.999939 (j = 1) and 0.999908 (j = 2) of the rows; 67 % of the rows
# lie more than CDF_DELTA from every CDF boundary, and there they all agree.
AGREEMENT_MIN = 0.99


# ------------------------------------------------------------------ references (no GPU)
def philox_np(c, key):
    """Philox4x32-10 over numpy arrays: c = 4 uint32 arrays (counter words), key = uint64 seed -> 4 uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(x, np.uint64) & M32 for x in c)
    key = np.asarray(key, np.uint64)
    k0, k1 = key & M32, key >> np.uint64(32)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return [x.astype(np.uint32) for x in (c0, c1, c2, c3)]


def draw_u(seed, counter, row_ids):
    """u of the action draw of each row: (word 0 >> 8) * 2^-24 of the block (counter, 0, row id, 3) under key `seed`."""
    row_ids = np.asarray(row_ids, np.uint64)
    counter = np.broadcast_to(np.asarray(counter, np.uint64), row_ids.shape)
    w = philox_np((counter, np.zeros_like(row_ids), row_ids, np.full_like(row_ids, STREAM_POLICY)), np.uint64(seed))[0]
    return (w >> 8).astype(np.float64) * 2.0 ** -24


def reference_sample(logits, u):
    """Inverse CDF of the float64 softmax: the smallest a with u < p_0 + ... + p_a (the last action if none)."""
    logits = np.asarray(logits, np.float64)
    p = np.exp(logits - logits.max(-1, keepdims=True))
    cdf = np.cumsum(p / p.sum(-1, keepdims=True), -1)
    a = (u[:, None] >= cdf).sum(-1)
    return np.minimum(a, logits.shape[-1] - 1), cdf


def _oracle_philox_shim():
    """The C oracle's philox4x32_10 (static in oracle/orlg_oracle.c), compiled into a small shared object for this test."""
    d = tempfile.mkdtemp(prefix="orlg_philox_")
    src, so = os.path.join(d, "shim.c"), os.path.join(d, "shim.so")
    with open(src, "w") as f:
        f.write('#include "%s"\n' % os.path.join(ROOT, "oracle", "orlg_oracle.c"))
        f.write("void shim_philox(uint32_t *c, const uint64_t *key, int n) {\n"
                "    for (int i = 0; i < n; i++) philox4x32_10(c + 4 * i, (uint32_t)key[i], (uint32_t)(key[i] >> 32));\n}\n")
    subprocess.check_call([os.environ.get("CC", "cc"), "-O2", "-fPIC", "-ffp-contract=off", "-shared", "-o", so, src, "-lm",
                           "-lpthread"])
    L = C.CDLL(so)
    L.shim_philox.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    return L


def test_numpy_philox_equals_the_oracle_philox():
    rng = np.random.default_rng(5)
    n = 4096
    c = rng.integers(0, 2 ** 32, size=(n, 4), dtype=np.uint64).astype(np.uint32)
    c[:8] = [[0, 0, 0, 0], [1, 0, 0, 3], [0xFFFFFFFF] * 4, [7, 0, 1000, 3], [0, 0, 0xFFFFFFFF, 3], [1, 2, 3, 4], [5, 0, 6, 2],
             [0x80000000, 0, 1, 3]]
    key = rng.integers(0, 2 ** 63, size=n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=n, dtype=np.uint64)
    key[:4] = [0, 1, 2 ** 64 - 1, 41]
    want = np.ascontiguousarray(c.copy())
    _oracle_philox_shim().shim_philox(want.ctypes.data_as(C.c_void_p), np.ascontiguousarray(key).ctypes.data_as(C.c_void_p), n)
    got = np.stack(philox_np([c[:, i] for i in range(4)], key), 1)
    assert np.array_equal(got, want)


def test_reference_sampler_follows_the_softmax_on_a_grid():
    """u on the grid j 2^-16 (values the kernel's u takes): each action is picked on p_a of the grid, to one grid step."""
    G = 1 << 16
    u = np.arange(G, dtype=np.float64) / G
    rng = np.random.default_rng(1)
    for na in (1, 2, 5, 11, 15):
        logits = rng.normal(0.0, 2.0, size=na)
        p = np.exp(logits - logits.max())
        p /= p.sum()
        a, _ = reference_sample(np.broadcast_to(logits, (G, na)), u)
        freq = np.bincount(a, minlength=na) / G
        assert np.abs(freq - p).max() <= 1.0 / G + 1e-12, (na, freq, p)


# ------------------------------------------------------------------ critic loading and refusals (no GPU)
def _sb3_state_dict(obs_dim=54, n_actions=5, separate=True, seed=0):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    trunks = ("policy_net", "value_net") if separate else ("shared_net",)
    for t in trunks:
        d = obs_dim
        for i in range(5):
            sd["mlp_extractor.%s.%d.weight" % (t, 2 * i)] = torch.randn(128, d, generator=g) / d ** 0.5
            sd["mlp_extractor.%s.%d.bias" % (t, 2 * i)] = torch.randn(128, generator=g) * 0.1
            d = 128
    sd["action_net.weight"] = torch.randn(n_actions, 128, generator=g) * 0.1
    sd["action_net.bias"] = torch.zeros(n_actions)
    sd["value_net.weight"] = torch.randn(1, 128, generator=g) * 0.1
    sd["value_net.bias"] = torch.full((1,), 0.25)
    return sd


def test_critic_handle_spec_of_separate_and_shared_trunks():
    from optical_rl_gym_b200.policy import MlpPolicy

    sd = _sb3_state_dict(separate=True)
    pol = MlpPolicy.from_state_dict(sd)
    specs = pol._native_specs()
    lins, heads, obs_dim = specs["critic"]
    assert obs_dim == 54 and len(lins) == 5 and all(m.out_features == 128 for m in lins)
    for i, m in enumerate(lins):
        assert torch.equal(m.weight, sd["mlp_extractor.value_net.%d.weight" % (2 * i)])
        assert torch.equal(m.bias, sd["mlp_extractor.value_net.%d.bias" % (2 * i)])
    assert heads[0] is pol.value_net and heads[-1] is pol.value_net
    assert torch.equal(pol.value_net.weight, sd["value_net.weight"])
    alins, aheads, aobs = specs["actor"]
    assert aobs == 54 and aheads == [pol.action_net, pol.value_net]
    assert torch.equal(alins[0].weight, sd["mlp_extractor.policy_net.0.weight"])
    # its value is the critic trunk's: forward() agrees with the spec
    x = torch.randn(7, 54)
    h = x
    for m in lins:
        h = torch.tanh(m(h))
    assert torch.allclose(pol(x)[1], pol.value_net(h).squeeze(-1))

    shared = MlpPolicy.from_state_dict(_sb3_state_dict(separate=False))
    assert shared.critic_net is None and shared._native_specs()["critic"] is None


def test_native_refusals_that_need_no_device():
    from optical_rl_gym_b200 import _native as nat
    from optical_rl_gym_b200.policy import MlpPolicy

    L = nat.lib()
    with pytest.raises(nat.NativeError, match="null env or actor"):
        nat.check(L.orlg_rollout_policy(None, 4, None, None, 0, 0, None, None, None, None, None, None, None))
    draw = nat.PolicyDraw(seed=1)
    with pytest.raises(nat.NativeError, match="null policy"):
        nat.check(L.orlg_policy_sample(None, None, 4, C.byref(draw), None, None, None, None))
    assert L.orlg_request_index(None) == -1
    # an odd observation width (k even) does not fit the kernel's operand layout: refused by orlg_policy_create, also for
    # a policy with a separate critic trunk
    pol = MlpPolicy.from_state_dict(_sb3_state_dict(obs_dim=53, separate=True))
    with pytest.raises(nat.NativeError, match="fused policy kernel"):
        pol._native_handles(0)
    for obs_dim, n_actions in ((53, 5), (66, 5), (54, 16)):
        with pytest.raises(nat.NativeError, match="fused policy kernel"):
            _policy(obs_dim=obs_dim, n_actions=n_actions, device="cpu")._native_handles(0)


# ------------------------------------------------------------------ GPU: the sampling epilogue
def _sample(pol, obs, seed, counter, row_id_base=0, deterministic=False):
    """orlg_policy_sample with a scalar or per-row (int32 CUDA tensor) counter -> (actions [n], log_prob [n], value [n])."""
    from optical_rl_gym_b200 import _native as nat

    n = obs.shape[0]
    a = torch.empty(n, dtype=torch.int32, device="cuda")
    lp = torch.empty(n, dtype=torch.float32, device="cuda")
    v = torch.empty(n, dtype=torch.float32, device="cuda")
    per_row = torch.is_tensor(counter)
    draw = nat.PolicyDraw(seed=seed, counter_dev=counter.data_ptr() if per_row else None, counter=0 if per_row else counter,
                          deterministic=int(deterministic), row_id_base=row_id_base)
    actor, _ = pol._native_handles(obs.device.index)
    nat.check(nat.lib().orlg_policy_sample(actor, C.c_void_p(obs.data_ptr()), n, C.byref(draw), C.c_void_p(a.data_ptr()),
                                           C.c_void_p(lp.data_ptr()), C.c_void_p(v.data_ptr()),
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return a, lp, v


def _real_observations(j, n=65536):
    from optical_rl_gym_b200 import OpticalVecEnv

    env = OpticalVecEnv("DeepRMSA-v0", n, helpers.golden_tables(), seed=4, j=j)
    obs = env.rollout(30)[0][-1].clone()
    env.close()
    return obs


def _kernel_logits(pol, obs):
    n_actions = pol.action_net.out_features
    logits = torch.empty((obs.shape[0], n_actions + 1), dtype=torch.float32, device="cuda")
    act = pol.act_native(obs, logits=logits)
    return act[:, 0], logits


@pytest.mark.gpu
@pytest.mark.parametrize("j", [1, 2])
def test_sampled_actions_match_the_reference_sampler(j):
    obs = _real_observations(j)
    n = obs.shape[0]
    pol = _policy(seed=j, obs_dim=obs.shape[1])
    with torch.no_grad():
        pol.action_net.weight.mul_(0.3)            # logits a few units apart: every action has a real probability
    rng = np.random.default_rng(j)
    seed = int(rng.integers(0, 2 ** 63)) * 2 + 1
    counters = rng.integers(0, 2 ** 32, size=n, dtype=np.uint64)
    base = int(rng.integers(0, 2 ** 31))
    cdev = torch.from_numpy(counters.astype(np.uint32).view(np.int32)).cuda()
    a, lp, v = _sample(pol, obs, seed, cdev, row_id_base=base)
    _, klogits = _kernel_logits(pol, obs)
    ref = bf16_reference(pol, obs.double()).cpu().numpy()
    u = draw_u(seed, counters, base + np.arange(n, dtype=np.uint64))
    want, cdf = reference_sample(ref[:, :5], u)
    a, lp, v = a.cpu().numpy(), lp.cpu().numpy().astype(np.float64), v.cpu().numpy().astype(np.float64)
    clear = (np.abs(u[:, None] - cdf[:, :-1]) > CDF_DELTA).all(-1)
    assert clear.mean() > 0.5
    assert np.array_equal(a[clear], want[clear])
    agree = (a == want).mean()
    assert agree >= AGREEMENT_MIN, agree
    print("agreement j=%d: %.6f (clear rows %.4f)" % (j, agree, clear.mean()))
    ref_lsm = ref[:, :5] - ref[:, :5].max(-1, keepdims=True)
    ref_lsm -= np.log(np.exp(ref_lsm).sum(-1, keepdims=True))
    assert np.abs(lp - ref_lsm[np.arange(n), a]).max() < 0.04
    own = torch.log_softmax(klogits[:, :5].double(), -1).cpu().numpy()
    assert np.abs(lp - own[np.arange(n), a]).max() < 1e-5
    assert np.abs(v - ref[:, 5]).max() < BF16_LOGIT_ATOL
    assert np.array_equal(v, klogits[:, 5].cpu().numpy().astype(np.float64))


@pytest.mark.gpu
def test_sampled_distribution_of_one_observation():
    from scipy import stats

    obs_all = _real_observations(1, 4096)
    pol = _policy(seed=3)
    with torch.no_grad():
        pol.action_net.weight.mul_(0.2)
    _, logits = _kernel_logits(pol, obs_all)
    p_all = torch.softmax(logits[:, :5].double(), -1)
    row = int((-(p_all * p_all.log()).sum(-1)).argmax())          # the most uncertain observation
    n = 65536
    obs = obs_all[row:row + 1].repeat(n, 1).contiguous()
    p = p_all[row].cpu().numpy()
    a1 = _sample(pol, obs, 12345, 17)[0].cpu().numpy()
    counts = np.bincount(a1, minlength=5)
    exp = p * n
    keep = exp >= 5
    obs_c = np.append(counts[keep], counts[~keep].sum())
    exp_c = np.append(exp[keep], exp[~keep].sum())
    if exp_c[-1] == 0:
        obs_c, exp_c = obs_c[:-1], exp_c[:-1]
    pval = stats.chisquare(obs_c, exp_c * obs_c.sum() / exp_c.sum()).pvalue
    assert pval > 1e-3, (counts, exp, pval)
    a2 = _sample(pol, obs, 12345, 18)[0].cpu().numpy()
    same = (a1 == a2).mean()
    q = float((p * p).sum())
    assert abs(same - q) < 0.01 and q < 0.9, (same, q)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 129, 65536])
def test_deterministic_mode_is_the_argmax_of_policy_act(n):
    obs = _real_observations(1, max(n, 128))[:n].contiguous()
    pol = _policy(seed=5)
    act, logits = _kernel_logits(pol, obs)
    a, lp, v = _sample(pol, obs, 99, 3, deterministic=True)
    assert torch.equal(a, act)
    own = torch.log_softmax(logits[:, :5].double(), -1).gather(1, a.long()[:, None])[:, 0]
    assert (lp.double() - own).abs().max().item() < 1e-5
    assert torch.equal(v, logits[:, 5])
    # sample_native: the same through the Python API
    sa, slp, sv = pol.sample_native(obs, seed=99, counter=3, deterministic=True)
    assert torch.equal(sa[:, 0], a) and torch.equal(slp, lp) and torch.equal(sv, v)


@pytest.mark.gpu
def test_sample_native_checks_its_arguments():
    pol = _policy()
    obs = _real_observations(1, 256)
    with pytest.raises(ValueError, match="observations"):
        pol.sample_native(obs[:, :50].contiguous(), seed=1, counter=0)
    with pytest.raises(ValueError, match="observations"):
        pol.sample_native(obs.double(), seed=1, counter=0)
    with pytest.raises(ValueError, match="observations"):
        pol.act_native(obs.t())
    with pytest.raises(ValueError, match="observations"):
        pol.act_native(obs.cpu())
    with pytest.raises(ValueError, match="out"):
        pol.act_native(obs, out=torch.empty((255, 1), dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError, match="logits"):
        pol.act_native(obs, logits=torch.empty((256, 5), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError, match="log_prob"):
        pol.sample_native(obs, seed=1, counter=0, out=(torch.empty((256, 1), dtype=torch.int32, device="cuda"),
                                                        torch.empty(255, device="cuda"), torch.empty(256, device="cuda")))


# ------------------------------------------------------------------ GPU: the closed loop
CONFIGS = {   # name -> (topology, env_args); episode_length 10: dones and auto-resets inside every call
    "nsfnet_j1": ("nsfnet", dict()),
    "nsfnet_j2_rej": ("nsfnet", dict(j=2, allow_rejection=True)),
    "E20": ("E20", dict()),
    "small_xml_rej": ("small_xml", dict(allow_rejection=True)),
}
SEED, BASE = 77, 1000


def _env(config, n, base=BASE, **kw):
    from optical_rl_gym_b200 import OpticalVecEnv

    topo, args = CONFIGS[config]
    args = dict(dict(episode_length=10, mean_service_holding_time=40.0, num_spectrum_resources=64), **args, **kw)
    return OpticalVecEnv("DeepRMSA-v0", n, helpers.tables(topo), seed=SEED, env_id_base=base, **args)


def _env_policy(env, seed=0):
    t = env.tables
    return _policy(seed=seed, obs_dim=env.obs_dim, n_actions=t.k_paths * env.j + env.reject_action)


def _twin_loop(env, pol, T, deterministic):
    """The closed loop as a Python loop of sample_native + step_raw, keyed like orlg_rollout_policy."""
    obs = [env.observation().clone()]
    acts, lps, vals, rews, dones = [], [], [], [], []
    for _ in range(T):
        a, lp, v = pol.sample_native(obs[-1], seed=SEED, counter=env.request_index, row_id_base=BASE, deterministic=deterministic)
        o, r, d = env.step_raw(a)
        obs.append(o.clone()); acts.append(a[:, 0].clone()); lps.append(lp); vals.append(v); rews.append(r.clone()); dones.append(d.clone())
    vals.append(pol.sample_native(obs[-1], seed=SEED, counter=env.request_index, row_id_base=BASE)[2])
    return [torch.stack(x) for x in (obs, acts, lps, vals, rews, dones)]


def _state(env):
    m, _, now, nheap = env.export_state()
    return [env.counters(), m, now, nheap, env.error_flags()]


def _assert_same(got, want, what=""):
    for name, g, w in zip(("obs", "actions", "log_prob", "value", "reward", "done"), got, want):
        assert torch.equal(g, w), (what, name)


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("n,T", [(1, 64), (129, 7), (4097, 1), (4097, 64)])
def test_rollout_policy_equals_the_python_loop(config, deterministic, n, T):
    env, twin = _env(config, n), _env(config, n)
    pol = _env_policy(env, seed=n)
    ro = env.rollout_policy(pol, T, deterministic=deterministic)
    want = _twin_loop(twin, pol, T, deterministic)
    _assert_same(ro, want)
    assert int(ro.done.sum()) > 0 or T < 10
    for g, w in zip(_state(env), _state(twin)):
        assert torch.equal(g, w)
    assert env.request_index == twin.request_index
    assert int(env.error_flags().abs().sum()) == 0
    env.close(); twin.close()


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["nsfnet_j1", "nsfnet_j2_rej", "E20", "small_xml_rej"])
def test_rollout_policy_env_side_matches_the_oracle(config):
    from oracle import oracle

    n, T = 64, 40
    env = _env(config, n)
    pol = _env_policy(env, seed=1)
    ro = env.rollout_policy(pol, T)
    topo, args = CONFIGS[config]
    env_args = dict(dict(episode_length=10, mean_service_holding_time=40.0, num_spectrum_resources=64), **args)
    okw = helpers.sim_kwargs(dict(kind="DeepRMSA-v0", env_args=env_args))
    acts = ro.actions.cpu().numpy()
    obs, rew, done = ro.obs.cpu().numpy(), ro.reward.cpu().numpy(), ro.done.cpu().numpy()
    assert len(np.unique(acts)) > 1
    for i in range(n):
        o = oracle.OracleEnv("DeepRMSA-v0", helpers.tables(topo), **okw)
        o.set_philox(SEED, BASE + i)
        o.reset(full=True)
        np.testing.assert_allclose(obs[0, i], o.observation(), rtol=OBS_RTOL, atol=0)
        r = o.rollout(T, policy=0, actions=acts[:, i], want_obs=True)
        assert np.array_equal(rew[:, i].astype(np.float64), r["rewards"]), i
        assert np.array_equal(done[:, i], r["dones"]), i
        np.testing.assert_allclose(obs[1:, i], r["obs"], rtol=OBS_RTOL, atol=0, err_msg="env %d" % i)
        o.close()
    env.close()


@pytest.mark.gpu
def test_rollout_policy_split_into_calls():
    env_a, env_b = _env("nsfnet_j1", 300), _env("nsfnet_j1", 300)
    pol = _env_policy(env_a, seed=2)
    one = env_a.rollout_policy(pol, 30)
    parts = [env_b.rollout_policy(pol, 10) for _ in range(3)]
    for k in range(3):
        sl = slice(10 * k, 10 * k + 10)
        assert torch.equal(parts[k].obs, one.obs[10 * k:10 * k + 11])
        assert torch.equal(parts[k].value, one.value[10 * k:10 * k + 11])
        for f in ("actions", "log_prob", "reward", "done"):
            assert torch.equal(getattr(parts[k], f), getattr(one, f)[sl]), (k, f)


@pytest.mark.gpu
def test_rollout_policy_does_not_depend_on_sharding():
    whole = _env("nsfnet_j1", 256, base=0)
    halves = [_env("nsfnet_j1", 128, base=b) for b in (0, 128)]
    pol = _env_policy(whole, seed=3)
    a = whole.rollout_policy(pol, 25, seed=SEED)
    parts = [h.rollout_policy(pol, 25, seed=SEED) for h in halves]
    for f in a._fields:
        assert torch.equal(getattr(a, f), torch.cat([getattr(p, f) for p in parts], 1)), f


@pytest.mark.gpu
def test_rollout_policy_across_a_checkpoint():
    env, fresh, ref = _env("nsfnet_j1", 200), _env("nsfnet_j1", 200), _env("nsfnet_j1", 200)
    pol = _env_policy(env, seed=4)
    whole = ref.rollout_policy(pol, 30)
    env.rollout_policy(pol, 10)
    fresh.rollout(3)                                    # somewhere else entirely
    fresh.load_state_dict(env.state_dict())
    rest = fresh.rollout_policy(pol, 20)
    for f in ("actions", "log_prob", "reward", "done"):
        assert torch.equal(getattr(rest, f), getattr(whole, f)[10:]), f
    assert torch.equal(rest.obs, whole.obs[10:]) and torch.equal(rest.value, whole.value[10:])


@pytest.mark.gpu
def test_rollout_policy_between_persistent_rollouts_matches_the_oracle():
    from oracle import oracle

    n = 96
    env = _env("nsfnet_j1", n)
    pol = _env_policy(env, seed=6)
    _, r1, d1, a1 = env.rollout(20)
    assert env.kernel_info()["last_rollout_persistent"]
    ro = env.rollout_policy(pol, 20)
    _, r3, d3, a3 = env.rollout(20)
    acts = torch.cat([a1[..., 0], ro.actions, a3[..., 0]]).cpu().numpy()
    rew = torch.cat([r1, ro.reward, r3]).cpu().numpy()
    done = torch.cat([d1, ro.done, d3]).cpu().numpy()
    _, env_args = CONFIGS["nsfnet_j1"]
    okw = helpers.sim_kwargs(dict(kind="DeepRMSA-v0", env_args=dict(episode_length=10, mean_service_holding_time=40.0,
                                                                     num_spectrum_resources=64)))
    avail = env.available_slots().cpu().numpy()
    cnt = env.counters().cpu().numpy()
    _, _, now, nheap = env.export_state(masks=False)
    for i in range(n):
        o = oracle.OracleEnv("DeepRMSA-v0", helpers.tables("nsfnet"), **okw)
        o.set_philox(SEED, BASE + i)
        o.reset(full=True)
        r = o.rollout(60, policy=0, actions=acts[:, i])
        assert np.array_equal(rew[:, i].astype(np.float64), r["rewards"]) and np.array_equal(done[:, i], r["dones"]), i
        oa, _, onow, onh = o.state()
        assert np.array_equal(avail[i].reshape(oa.shape), oa), i
        assert np.array_equal(cnt[i], o.counters()) and now[i].item() == onow and nheap[i].item() == onh, i
        o.close()
    assert int(env.error_flags().abs().sum()) == 0


@pytest.mark.gpu
def test_critic_value_of_separate_and_shared_trunks():
    from optical_rl_gym_b200.policy import MlpPolicy

    obs = _real_observations(1, 4096)
    pol = MlpPolicy.from_state_dict(_sb3_state_dict(separate=True, seed=7)).cuda()
    a, lp, v = pol.sample_native(obs, seed=1, counter=2)
    critic = types.SimpleNamespace(shared_net=pol.critic_net, action_net=pol.value_net, value_net=pol.value_net)
    want = bf16_reference(critic, obs.double())[:, 1]
    assert (v.double() - want).abs().max().item() < BF16_LOGIT_ATOL
    actor_value = _kernel_logits(pol, obs)[1][:, 5]
    assert (v - actor_value).abs().max().item() > 10 * BF16_LOGIT_ATOL          # not the actor trunk's value
    env = _env("nsfnet_j1", 512)
    ro = env.rollout_policy(pol, 5)
    twin = _twin_loop(_env("nsfnet_j1", 512), pol, 5, False)
    _assert_same(ro, twin, "critic")

    shared = MlpPolicy.from_state_dict(_sb3_state_dict(separate=False, seed=8)).cuda()
    _, _, v = shared.sample_native(obs, seed=1, counter=2)
    assert torch.equal(v, _kernel_logits(shared, obs)[1][:, 5])


@pytest.mark.gpu
def test_native_weights_follow_optimizer_steps():
    from optical_rl_gym_b200.policy import MlpPolicy

    obs = _real_observations(1, 2048)
    pol = _policy(seed=9)
    before = pol.sample_native(obs, seed=5, counter=1)
    env_old = _env("nsfnet_j1", 256)
    ro_old = env_old.rollout_policy(pol, 8)
    opt = torch.optim.SGD(pol.parameters(), lr=0.05)
    logits, value = pol(obs)
    (logits.logsumexp(-1).mean() + value.square().mean()).backward()
    opt.step()
    after = pol.sample_native(obs, seed=5, counter=1)
    fresh = MlpPolicy(54, 5, (128,) * 5).cuda()
    fresh.load_state_dict(pol.state_dict())
    want = fresh.sample_native(obs, seed=5, counter=1)
    for g, w in zip(after, want):
        assert torch.equal(g, w)
    assert not torch.equal(after[1], before[1]) and not torch.equal(after[2], before[2])
    ro_new, ro_fresh = _env("nsfnet_j1", 256).rollout_policy(pol, 8), _env("nsfnet_j1", 256).rollout_policy(fresh, 8)
    _assert_same(ro_new, ro_fresh, "refresh")
    assert not torch.equal(ro_new.log_prob, ro_old.log_prob)
    # load_state_dict into the live policy is picked up as well
    pol.load_state_dict(MlpPolicy(54, 5, (128,) * 5).state_dict())
    again = pol.sample_native(obs, seed=5, counter=1)
    assert not torch.equal(again[2], after[2])


@pytest.mark.gpu
def test_rollout_policy_refusals():
    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200 import _native as nat

    pol = _policy()
    rmsa = OpticalVecEnv("RMSA-v0", 8, helpers.golden_tables(), seed=1)
    with pytest.raises(nat.NativeError, match="DeepRMSA-v0"):
        rmsa.rollout_policy(pol, 2)
    f64 = _env("nsfnet_j1", 8, obs_dtype=torch.float64)
    with pytest.raises(nat.NativeError, match="float32"):
        f64.rollout_policy(pol, 2)
    env = _env("nsfnet_j1", 8)
    with pytest.raises(nat.NativeError, match="actor obs_dim"):
        env.rollout_policy(_policy(obs_dim=64), 2)
    with pytest.raises(nat.NativeError, match="n_actions"):
        env.rollout_policy(_policy(n_actions=6), 2)
    bad_critic = _policy()
    bad_critic.critic_net = torch.nn.Sequential(*[m for i in range(5) for m in (torch.nn.Linear(64 if i == 0 else 128, 128),
                                                                                torch.nn.Tanh())]).cuda()
    with pytest.raises(nat.NativeError, match="critic obs_dim"):
        env.rollout_policy(bad_critic, 2)
    with pytest.raises(ValueError):
        env.rollout_policy(pol, -1)
    actor, _ = pol._native_handles(env._dev_index)
    with pytest.raises(nat.NativeError, match="steps"):
        nat.check(env._lib.orlg_rollout_policy(env._h, -1, actor, None, 1, 0, C.c_void_p(16), None, None, None, None, None, None))
    with pytest.raises(nat.NativeError, match="obs_dev"):
        nat.check(env._lib.orlg_rollout_policy(env._h, 1, actor, None, 1, 0, None, None, None, None, None, None, None))
    # nothing was stepped by the refused calls
    assert env.request_index == 1
