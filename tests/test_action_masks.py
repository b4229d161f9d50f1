"""Invalid-action masks of DeepRMSA-v0 (orlg_action_masks / OpticalVecEnv.action_masks) and masked PPO sampling
(orlg_policy_sample_masked / MlpPolicy.sample_native(action_masks=...), orlg_rollout_policy_masked /
OpticalVecEnv.rollout_policy(action_masks=True)), as sb3-contrib's MaskablePPO uses them.

References: what env.step does with every action (a twin loaded from state_dict, record_decisions=True), the observation's
length fields, the C oracle's integer observation on replayed envs, a float64 numpy MaskableCategorical on the kernel's own
logits with the Philox draw of test_policy_rollout, and a Python loop of action_masks + sample_native + step_raw on a twin."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

from test_policy_kernel import _policy  # noqa: E402
from test_policy_rollout import AGREEMENT_MIN, CDF_DELTA, draw_u  # noqa: E402

MASKED_LOGIT = -1e8           # MaskableCategorical's logit of an invalid action
SEED, BASE = 77, 1000


# ------------------------------------------------------------------ references and checks that need no device
def reference_masked_sample(logits, mask, u):
    """MaskableCategorical by inverse CDF in float64: the smallest a with u < p_0 + ... + p_a of softmax(l'), l' = l where
    the mask is set, else -1e8; when rounding leaves no action, the last action with p_a > 0."""
    lm = np.where(mask, np.asarray(logits, np.float64), MASKED_LOGIT)
    p = np.exp(lm - lm.max(-1, keepdims=True))
    cdf = np.cumsum(p / p.sum(-1, keepdims=True), -1)
    a = (u[:, None] >= cdf).sum(-1)
    last = p.shape[-1] - 1 - np.argmax(p[:, ::-1] > 0, -1)
    return np.minimum(a, last), cdf


def test_reference_masked_sampler_on_a_grid():
    """u on the grid j 2^-16: each valid action is drawn on its masked softmax share, a masked one never, and an all-zero
    mask is uniform."""
    G = 1 << 16
    u = np.arange(G, dtype=np.float64) / G
    rng = np.random.default_rng(2)
    for na in (2, 5, 11, 15):
        logits = rng.normal(0.0, 2.0, size=na)
        for mask in (rng.random(na) < 0.5, np.zeros(na, bool), np.ones(na, bool)):
            a, _ = reference_masked_sample(np.broadcast_to(logits, (G, na)), np.broadcast_to(mask, (G, na)), u)
            freq = np.bincount(a, minlength=na) / G
            if mask.any():
                p = np.where(mask, np.exp(logits - logits[mask].max()), 0.0)
            else:
                p = np.ones(na)
            p /= p.sum()
            assert np.abs(freq - p).max() <= 1.0 / G + 1e-12, (na, mask, freq, p)


def test_new_symbols_are_exported_and_refuse_null_handles():
    from optical_rl_gym_b200 import _native as nat

    L = nat.lib()
    for name in ("orlg_action_mask_dim", "orlg_action_masks", "orlg_policy_sample_masked", "orlg_rollout_policy_masked"):
        assert name in nat.EXPORTED and hasattr(L, name), name
    assert L.orlg_action_mask_dim(None) == 0
    with pytest.raises(nat.NativeError, match="null handle"):
        nat.check(L.orlg_action_masks(None, None, None))
    draw = nat.PolicyDraw(seed=1)
    with pytest.raises(nat.NativeError, match="null policy"):
        nat.check(L.orlg_policy_sample_masked(None, None, 4, C.byref(draw), None, None, None, None, None))
    with pytest.raises(nat.NativeError, match="null env or actor"):
        nat.check(L.orlg_rollout_policy_masked(None, 4, None, None, 0, 0, None, None, None, None, None, None, None, None, None))


# ------------------------------------------------------------------ environments
def _germany50():
    from optical_rl_gym_b200.topology import TopologyTables

    return TopologyTables.load(os.path.join(helpers.GOLDEN_DIR, "topo_germany50_tables.npz"))


# name -> (topology, env_args, float64 observation, trace traffic).  A small spectrum at a high load: rows with some and
# with no valid action occur.  nsfnet_wide160 is a wide handle (more than 128 slots: the 16-bit block cache) whose
# observation still fits the policy kernel; germany50's (126 wide) does not.
_BASE_ARGS = dict(episode_length=10, mean_service_holding_time=60.0, num_spectrum_resources=24)
MASK_CONFIGS = {
    "nsfnet_j1": ("nsfnet", dict(), False, False),
    "nsfnet_j2_rej": ("nsfnet", dict(j=2, allow_rejection=True), False, False),
    "nsfnet_j2_rej_f64": ("nsfnet", dict(j=2, allow_rejection=True), True, False),
    "nsfnet_j1_trace": ("nsfnet", dict(), False, True),
    "small_xml": ("small_xml", dict(), False, False),
    "E20": ("E20", dict(), False, False),
    "germany50": ("germany50", dict(), False, False),
    "nsfnet_wide160": ("nsfnet", dict(num_spectrum_resources=160, mean_service_holding_time=400.0), False, False),
}
LOOP_CONFIGS = ["nsfnet_j1", "nsfnet_j2_rej", "E20", "small_xml_rej", "nsfnet_wide160"]
MASK_CONFIGS["small_xml_rej"] = ("small_xml", dict(allow_rejection=True), False, False)


def _tables(topo):
    return _germany50() if topo == "germany50" else helpers.tables(topo)


def _env_args(config):
    return dict(_BASE_ARGS, **MASK_CONFIGS[config][1])


def _trace(env, length=400, seed=11):
    """A recorded request sequence per env (arrival, holding, src, dst, bit rate), the same for every env built from it."""
    rng = np.random.default_rng(seed)
    n, nodes = env.num_envs, env.tables.num_nodes
    arrival = np.cumsum(rng.exponential(0.1, size=(n, length)), 1)
    holding = rng.exponential(_env_args("nsfnet_j1_trace")["mean_service_holding_time"], size=(n, length))
    src = rng.integers(0, nodes, size=(n, length))
    dst = (src + rng.integers(1, nodes, size=(n, length))) % nodes
    return arrival, holding, src, dst, rng.integers(25, 101, size=(n, length))


def _env(config, n, base=BASE, **kw):
    from optical_rl_gym_b200 import OpticalVecEnv

    topo, _, f64, trace = MASK_CONFIGS[config]
    env = OpticalVecEnv("DeepRMSA-v0", n, _tables(topo), seed=SEED, env_id_base=base,
                        obs_dtype=torch.float64 if f64 else torch.float32, traffic="trace" if trace else "philox",
                        **_env_args(config), **kw)
    if trace:
        env.set_trace(*_trace(env))
        env.reset(full=True)
    return env


def _assert_no_errors(env):
    """No error flag but ORLG_ERR_NO_SUCH_PATH: a random action, or one drawn from an all-zero mask, may name a path the
    request's pair does not have (the reference's IndexError, blocked here)."""
    from optical_rl_gym_b200 import _native as nat

    assert int((env.error_flags() & ~nat.ERR_NO_SUCH_PATH).abs().sum()) == 0


def _n_actions(env):
    return env.k_paths * env.j + env.reject_action


# ------------------------------------------------------------------ GPU: the mask is what env.step accepts
def _check_mask(config, env, twin, actions_so_far):
    """mask == accepted of env.step(a) for every non-reject a (twin loaded from env's state); the reject action is valid;
    the observation's length fields and the C oracle's integer observation (replayed envs) agree.  Returns the mask."""
    n, A, k, j = env.num_envs, _n_actions(env), env.k_paths, env.j
    mask = env.action_masks()
    assert mask.dtype == torch.bool and tuple(mask.shape) == (n, A) and mask.device == env.device
    m = mask.cpu().numpy()
    # the observation: length field of (path p, block b) is -1 exactly when the block is absent
    obs = env.observation().cpu().numpy()
    base = 1 + 2 * env.tables.num_nodes
    lens = np.stack([obs[:, base + p * (2 * j + 3) + 2 * b + 1] for p in range(k) for b in range(j)], 1)
    assert np.array_equal(m[:, :k * j], lens != -1)
    oi = env.observation_int().cpu().numpy()
    assert np.array_equal(m[:, :k * j], oi[:, :, 0:2 * j:2].reshape(n, k * j) != -1)
    # every action on a twin
    sd = env.state_dict()
    for a in range(A):
        twin.load_state_dict(sd)
        twin.step_raw(torch.full((n, 1), a, dtype=torch.int32, device=env.device))
        accepted = twin.decisions[:, 0].cpu().numpy() == 1
        if a == k * j:
            assert m[:, a].all() and not accepted.any()
        else:
            assert np.array_equal(accepted, m[:, a]), (a, int((accepted != m[:, a]).sum()))
    # the C oracle, replaying the first envs' actions since the full reset
    from oracle import oracle

    topo, _, _, trace = MASK_CONFIGS[config]
    okw = helpers.sim_kwargs(dict(kind="DeepRMSA-v0", env_args=_env_args(config)))
    acts = np.stack(actions_so_far) if actions_so_far else np.zeros((0, n), np.int32)
    tr = _trace(env) if trace else None
    for i in range(min(n, 12)):
        o = oracle.OracleEnv("DeepRMSA-v0", _tables(topo), **okw)
        if trace:
            o.set_trace(*[x[i] for x in tr])
        else:
            o.set_philox(SEED, BASE + i)
        o.reset(full=True)
        if len(acts):
            o.rollout(len(acts), policy=0, actions=acts[:, i])
        starts = o.observation_int()[:, 0:2 * j:2].reshape(k * j)
        assert np.array_equal(m[i, :k * j], starts != -1), i
        o.close()
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(MASK_CONFIGS))
def test_mask_is_what_the_step_accepts(config):
    n = 300
    env, twin = _env(config, n), _env(config, n, record_decisions=True)
    A = _n_actions(env)
    assert env._lib.orlg_action_mask_dim(env._h) == A == env.action_space.n
    rng = np.random.default_rng(len(config))
    history, rows = [], []
    rows.append(_check_mask(config, env, twin, history))               # after the full reset
    wide = config in ("germany50", "nsfnet_wide160")
    for _ in range(300 if wide else 120):                              # steps across auto-resets (episode_length 10),
        a = env.heuristic("sap_ff")                                    # first fit: the spectrum fills up
        env.step_raw(a)
        history.append(a[:, 0].cpu().numpy())
    rows.append(_check_mask(config, env, twin, history))
    acts = rng.integers(0, A, size=(20, n, 1)).astype(np.int32)       # a rollout: the persistent kernel where it applies
    env.rollout(20, "replay", actions=torch.from_numpy(acts).cuda())
    if config == "nsfnet_j1":
        assert env.kernel_info()["last_rollout_persistent"]
    history += list(acts[..., 0])
    rows.append(_check_mask(config, env, twin, history))
    m = np.concatenate(rows)
    valid = m[:, :env.k_paths * env.j].sum(1)
    assert ((valid > 0) & (valid < env.k_paths * env.j)).any(), "no partial rows"
    if not env.allow_rejection and not wide:        # the 24-slot NSFNET-class configurations saturate
        assert (valid == 0).any(), "no all-zero rows"
    assert env.kernel_info()["wide"] == wide
    _assert_no_errors(env)
    env.close(); twin.close()


# ------------------------------------------------------------------ GPU: the masked sampler
ARCHS = {"5x128": (5, 128), "2x64": (2, 64)}


def _arch_policy(arch, obs_dim, n_actions, seed=0, critic=False):
    from optical_rl_gym_b200.policy import MlpPolicy

    L, H = ARCHS[arch]
    if (L, H) == (5, 128) and not critic:
        return _policy(seed=seed, obs_dim=obs_dim, n_actions=n_actions)
    torch.manual_seed(seed)
    pol = MlpPolicy(obs_dim, n_actions, (H,) * L)
    with torch.no_grad():
        for m in pol.shared_net:
            if isinstance(m, torch.nn.Linear):
                torch.nn.init.orthogonal_(m.weight, gain=2 ** 0.5)
        torch.nn.init.orthogonal_(pol.action_net.weight, gain=1.0)
    if critic:                      # SB3 >= 1.8: a separate critic trunk of the same shape
        layers = []
        for i in range(L):
            lin = torch.nn.Linear(obs_dim if i == 0 else H, H)
            torch.nn.init.orthogonal_(lin.weight, gain=2 ** 0.5)
            layers += [lin, torch.nn.Tanh()]
        pol.critic_net = torch.nn.Sequential(*layers)
    return pol.cuda()


_REAL = {}


def _real(j, n=65536):
    """Real observations and their masks at a high load (24 slots): (obs f32 [n, 54], mask bool [n, A])."""
    if (j, n) not in _REAL:
        from optical_rl_gym_b200 import OpticalVecEnv

        env = OpticalVecEnv("DeepRMSA-v0", n, helpers.golden_tables(), seed=4, j=j, allow_rejection=j == 2,
                            num_spectrum_resources=24, mean_service_holding_time=60.0)
        env.rollout(60, "sap_ff", want_obs=False, want_actions=False)
        _REAL[(j, n)] = (env.observation().clone(), env.action_masks().clone())
        env.close()
    return _REAL[(j, n)]


def _kernel_logits(pol, obs):
    logits = torch.empty((obs.shape[0], pol.action_net.out_features + 1), dtype=torch.float32, device="cuda")
    pol.act_native(obs, logits=logits)
    return logits


@pytest.mark.gpu
@pytest.mark.parametrize("arch", list(ARCHS))
@pytest.mark.parametrize("j", [1, 2])
def test_all_ones_mask_is_bit_identical_to_unmasked(arch, j):
    obs, mask = _real(j, 4099)
    pol = _arch_policy(arch, obs.shape[1], mask.shape[1], seed=j)
    ones = torch.ones_like(mask)
    for det in (False, True):
        for counter, base in ((0, 0), (7, 123456), (2 ** 32 - 1, 2 ** 40)):
            want = pol.sample_native(obs, seed=SEED, counter=counter, row_id_base=base, deterministic=det)
            got = pol.sample_native(obs, seed=SEED, counter=counter, row_id_base=base, deterministic=det, action_masks=ones)
            got8 = pol.sample_native(obs, seed=SEED, counter=counter, row_id_base=base, deterministic=det,
                                     action_masks=ones.to(torch.uint8))
            for g, g8, w in zip(got, got8, want):
                assert torch.equal(g, w) and torch.equal(g8, w)


@pytest.mark.gpu
@pytest.mark.parametrize("arch", list(ARCHS))
@pytest.mark.parametrize("j", [1, 2])
def test_masked_sampler_matches_maskable_categorical(arch, j):
    obs, mask = _real(j)
    n, A = mask.shape
    m = mask.cpu().numpy()
    valid = m.sum(1)
    assert ((valid > 0) & (valid < A)).mean() > 0.05
    pol = _arch_policy(arch, obs.shape[1], A, seed=10 + j)
    with torch.no_grad():
        pol.action_net.weight.mul_(0.3)            # logits a few units apart: every valid action has a real probability
    logits = _kernel_logits(pol, obs)[:, :A].cpu().numpy()
    rng = np.random.default_rng(j)
    for _ in range(3):
        seed, counter, base = int(rng.integers(0, 2 ** 63)), int(rng.integers(0, 2 ** 32)), int(rng.integers(0, 2 ** 31))
        a, lp, v = pol.sample_native(obs, seed=seed, counter=counter, row_id_base=base, action_masks=mask)
        a, lp = a[:, 0].cpu().numpy(), lp.cpu().numpy().astype(np.float64)
        u = draw_u(seed, counter, base + np.arange(n, dtype=np.uint64))
        want, cdf = reference_masked_sample(logits, m, u)
        clear = (np.abs(u[:, None] - cdf[:, :-1]) > CDF_DELTA).all(-1)
        assert np.array_equal(a[clear], want[clear])
        assert (a == want).mean() >= AGREEMENT_MIN
        # never a masked action while the row has a valid one; an all-zero row draws from all A actions
        assert m[np.arange(n), a][valid > 0].all()
        lm = np.where(m, logits.astype(np.float64), MASKED_LOGIT)
        lsm = lm - lm.max(-1, keepdims=True)
        lsm -= np.log(np.exp(lsm).sum(-1, keepdims=True))
        assert np.abs(lp - lsm[np.arange(n), a]).max() < 1e-5
        assert np.allclose(lp[valid == 0], -np.log(A), atol=1e-6)
        assert torch.equal(v, pol.sample_native(obs, seed=seed, counter=counter, row_id_base=base)[2])


@pytest.mark.gpu
@pytest.mark.parametrize("arch", list(ARCHS))
def test_masked_deterministic_is_the_argmax_of_the_masked_logits(arch):
    obs, mask = _real(2)
    pol = _arch_policy(arch, obs.shape[1], mask.shape[1], seed=5)
    logits = _kernel_logits(pol, obs)[:, :mask.shape[1]]
    want = torch.where(mask, logits, torch.full_like(logits, MASKED_LOGIT)).argmax(-1)
    a, lp, _ = pol.sample_native(obs, seed=1, counter=2, deterministic=True, action_masks=mask)
    assert torch.equal(a[:, 0].long(), want)
    assert (a[mask.sum(1) == 0] == 0).all()
    # the same mask in a row with no valid action but with rejection: covered by j = 2; without rejection:
    obs1, mask1 = _real(1)
    pol1 = _arch_policy(arch, obs1.shape[1], mask1.shape[1], seed=6)
    a1, _, _ = pol1.sample_native(obs1, seed=1, counter=2, deterministic=True, action_masks=mask1)
    l1 = _kernel_logits(pol1, obs1)[:, :mask1.shape[1]]
    assert torch.equal(a1[:, 0].long(), torch.where(mask1, l1, torch.full_like(l1, MASKED_LOGIT)).argmax(-1))
    assert (mask1.sum(1) == 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("arch", list(ARCHS))
def test_masked_distribution_of_one_observation(arch):
    from scipy import stats

    obs_all, _ = _real(1, 4096)
    pol = _arch_policy(arch, obs_all.shape[1], 5, seed=3)
    with torch.no_grad():
        pol.action_net.weight.mul_(0.2)
    logits = _kernel_logits(pol, obs_all)[:, :5].double()
    p_all = torch.softmax(logits, -1)
    row = int((-(p_all * p_all.log()).sum(-1)).argmax())          # the most uncertain observation
    n = 65536
    obs = obs_all[row:row + 1].repeat(n, 1).contiguous()
    for valid in ([True, False, True, True, False], [False] * 5):
        mask = torch.tensor(valid, device="cuda").repeat(n, 1).contiguous()
        a = pol.sample_native(obs, seed=12345, counter=17, action_masks=mask)[0][:, 0].cpu().numpy()
        counts = np.bincount(a, minlength=5)
        v = np.array(valid)
        if v.any():
            lv = np.where(v, logits[row].cpu().numpy(), -np.inf)
            p = np.exp(lv - lv.max())
            p /= p.sum()
            assert counts[~v].sum() == 0
        else:
            p = np.full(5, 0.2)
        keep = p > 0
        pval = stats.chisquare(counts[keep], p[keep] * n).pvalue
        assert pval > 1e-3, (valid, counts, p * n, pval)


@pytest.mark.gpu
def test_sample_native_checks_the_mask():
    obs, mask = _real(1, 256)
    pol = _policy()
    for bad in (torch.ones((256, 6), dtype=torch.bool, device="cuda"), torch.ones((255, 5), dtype=torch.bool, device="cuda"),
                torch.ones((256, 5), dtype=torch.int32, device="cuda"), torch.ones((256, 5), dtype=torch.float32, device="cuda"),
                mask.cpu(), torch.ones((5, 256), dtype=torch.bool, device="cuda").t()):
        with pytest.raises(ValueError, match="action_masks"):
            pol.sample_native(obs, seed=1, counter=0, action_masks=bad)


# ------------------------------------------------------------------ GPU: the closed loop
def _loop_env(config, n, base=BASE, **kw):
    return _env(config, n, base=base, **kw)


def _loop_policy(env, critic, seed=0):
    return _arch_policy("2x64" if critic else "5x128", env.obs_dim, _n_actions(env), seed=seed, critic=critic)


def _twin_masked_loop(env, pol, T, deterministic):
    """rollout_policy(action_masks=True) as a Python loop of action_masks + sample_native + step_raw, keyed the same way;
    also every step's info counters."""
    obs = [env.observation().clone()]
    acts, lps, vals, rews, dones, masks, counters = [], [], [], [], [], [], []
    for _ in range(T):
        m = env.action_masks().clone()
        a, lp, v = pol.sample_native(obs[-1], seed=SEED, counter=env.request_index, row_id_base=BASE,
                                     deterministic=deterministic, action_masks=m)
        o, r, d = env.step_raw(a)
        obs.append(o.clone()); acts.append(a[:, 0].clone()); lps.append(lp); vals.append(v); rews.append(r.clone())
        dones.append(d.clone()); masks.append(m); counters.append(env._info.clone())
    vals.append(pol.sample_native(obs[-1], seed=SEED, counter=env.request_index, row_id_base=BASE)[2])
    out = [torch.stack(x) for x in (obs, acts, lps, vals, rews, dones)]
    return out, (torch.stack(masks) if masks else None), (torch.stack(counters) if counters else None)


def _state(env):
    m, _, now, nheap = env.export_state()
    return [env.counters(), m, now, nheap, env.error_flags()]


def _check_invariant(env, ro, masks):
    """A valid action provisions (reward 1); while a row has a valid action, the drawn one is valid."""
    chosen = masks.gather(2, ro.actions.long().unsqueeze(-1))[..., 0]
    assert (ro.reward[chosen & (ro.actions != env.k_paths * env.j)] == 1).all()
    assert chosen[masks.any(-1)].all()
    assert (ro.reward[ro.actions < env.k_paths * env.j] == 1).sum() == (chosen & (ro.actions < env.k_paths * env.j)).sum()


@pytest.mark.gpu
@pytest.mark.parametrize("config", LOOP_CONFIGS)
@pytest.mark.parametrize("critic", [False, True])
@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("T", [1, 64])
def test_masked_rollout_policy_equals_the_python_loop(config, critic, deterministic, T):
    n = 257
    env, twin = _loop_env(config, n), _loop_env(config, n)
    pol = _loop_policy(env, critic, seed=T)
    ro, masks = env.rollout_policy(pol, T, deterministic=deterministic, action_masks=True)
    want, want_masks, _ = _twin_masked_loop(twin, pol, T, deterministic)
    assert masks.dtype == torch.bool and tuple(masks.shape) == (T, n, _n_actions(env))
    for name, g, w in zip(ro._fields, ro, want):
        assert torch.equal(g, w), name
    assert torch.equal(masks, want_masks)
    for g, w in zip(_state(env), _state(twin)):
        assert torch.equal(g, w)
    assert env.request_index == twin.request_index
    _check_invariant(env, ro, masks)
    _assert_no_errors(env)
    env.close(); twin.close()


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["nsfnet_j1", "nsfnet_j2_rej"])
def test_masked_rollout_policy_with_info(config):
    n, T = 300, 40
    env, twin = _loop_env(config, n), _loop_env(config, n)
    pol = _loop_policy(env, False, seed=3)
    ro, info, masks = env.rollout_policy(pol, T, action_masks=True, want_info=True)
    want, want_masks, want_counters = _twin_masked_loop(twin, pol, T, False)
    for name, g, w in zip(ro._fields, ro, want):
        assert torch.equal(g, w), name
    assert torch.equal(masks, want_masks) and torch.equal(info.counters, want_counters)
    assert int(ro.done.sum()) > 0
    _check_invariant(env, ro, masks)


@pytest.mark.gpu
def test_masked_rollout_policy_split_checkpoint_and_shards():
    pol_env = _loop_env("nsfnet_j2_rej", 256)
    pol = _loop_policy(pol_env, True, seed=2)
    whole, wmasks = _loop_env("nsfnet_j2_rej", 256).rollout_policy(pol, 30, action_masks=True)
    # split into calls
    env = _loop_env("nsfnet_j2_rej", 256)
    parts = [env.rollout_policy(pol, 10, action_masks=True) for _ in range(3)]
    for k, (p, m) in enumerate(parts):
        sl = slice(10 * k, 10 * k + 10)
        assert torch.equal(p.obs, whole.obs[10 * k:10 * k + 11]) and torch.equal(p.value, whole.value[10 * k:10 * k + 11])
        for f in ("actions", "log_prob", "reward", "done"):
            assert torch.equal(getattr(p, f), getattr(whole, f)[sl]), (k, f)
        assert torch.equal(m, wmasks[sl])
    # across a checkpoint
    first, fresh = _loop_env("nsfnet_j2_rej", 256), _loop_env("nsfnet_j2_rej", 256)
    first.rollout_policy(pol, 10, action_masks=True)
    fresh.rollout(3)
    fresh.load_state_dict(first.state_dict())
    rest, rmasks = fresh.rollout_policy(pol, 20, action_masks=True)
    for f in ("actions", "log_prob", "reward", "done"):
        assert torch.equal(getattr(rest, f), getattr(whole, f)[10:]), f
    assert torch.equal(rest.obs, whole.obs[10:]) and torch.equal(rest.value, whole.value[10:]) and torch.equal(rmasks, wmasks[10:])
    # two shards
    halves = [_loop_env("nsfnet_j2_rej", 128, base=b) for b in (BASE, BASE + 128)]
    res = [h.rollout_policy(pol, 30, action_masks=True) for h in halves]
    for i, f in enumerate(whole._fields):
        assert torch.equal(whole[i], torch.cat([r[0][i] for r in res], 1)), f
    assert torch.equal(wmasks, torch.cat([r[1] for r in res], 1))


# ------------------------------------------------------------------ GPU: refusals and VecMonitor
@pytest.mark.gpu
def test_refusals():
    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200 import _native as nat

    pol = _policy()
    for kind, kw in (("RMSA-v0", {}), ("RWA-v0", {}), ("RMCSA-v0", dict(num_spectrum_resources=64))):
        other = OpticalVecEnv(kind, 8, helpers.golden_tables(), seed=1, **kw)
        assert other._lib.orlg_action_mask_dim(other._h) == 0
        with pytest.raises(nat.NativeError, match="DeepRMSA-v0"):
            other.action_masks()
        with pytest.raises(nat.NativeError, match="DeepRMSA-v0"):
            other.rollout_policy(pol, 2, action_masks=True)
        other.close()
    env = _loop_env("nsfnet_j1", 8)
    with pytest.raises(nat.NativeError, match="n_actions"):
        env.rollout_policy(_policy(n_actions=6), 2, action_masks=True)
    for bad in (torch.empty((8, 6), dtype=torch.bool, device="cuda"), torch.empty((8, 5), dtype=torch.int32, device="cuda")):
        with pytest.raises(ValueError, match="out"):
            env.action_masks(out=bad)
    m8 = torch.empty((8, 5), dtype=torch.uint8, device="cuda")
    assert env.action_masks(out=m8) is m8 and torch.equal(m8.bool(), env.action_masks())
    actor, _ = pol._native_handles(env._dev_index)
    obs = torch.empty((3, 8, env.obs_dim), dtype=torch.float32, device="cuda")
    with pytest.raises(nat.NativeError, match="masks_dev"):
        nat.check(env._lib.orlg_rollout_policy_masked(env._h, 2, actor, None, 1, 0, C.c_void_p(obs.data_ptr()), None, None, None,
                                                      None, None, None, None, None))
    draw = nat.PolicyDraw(seed=1)
    with pytest.raises(nat.NativeError, match="mask_dev"):
        nat.check(env._lib.orlg_policy_sample_masked(actor, C.c_void_p(obs.data_ptr()), 8, C.byref(draw), None, None, None, None,
                                                     None))
    with pytest.raises(nat.NativeError, match="null mask"):
        nat.check(env._lib.orlg_action_masks(env._h, None, None))
    assert env.request_index == 1               # nothing was stepped by the refused calls
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("info_keywords", [(), ("episode_service_blocking_rate",)])
def test_vec_monitor_masked_rollout_policy(info_keywords):
    from optical_rl_gym_b200.monitor import VecMonitor
    from optical_rl_gym_b200.vec_env import PolicyRollout

    n, T = 64, 35
    env, twin = _loop_env("nsfnet_j1", n), _loop_env("nsfnet_j1", n)
    pol = _loop_policy(env, False, seed=8)
    mon, mon_twin = VecMonitor(env, info_keywords=info_keywords), VecMonitor(twin, info_keywords=info_keywords)
    res = mon.rollout_policy(pol, T, action_masks=True)
    assert isinstance(res, tuple) and len(res) == 2 and isinstance(res[0], PolicyRollout)
    ro, masks = res
    assert masks.dtype == torch.bool and tuple(masks.shape) == (T, n, 5)
    obs = twin.observation()
    for t in range(T):
        m = twin.action_masks()
        assert torch.equal(m, masks[t])
        a = pol.sample_native(obs, seed=SEED, counter=twin.request_index, row_id_base=BASE, action_masks=m)[0]
        obs, r, d, _ = mon_twin.step(a)
        assert torch.equal(r, ro.reward[t]) and torch.equal(d, ro.done[t])
    assert len(mon.episode_returns) > 0
    assert mon.episode_returns == mon_twin.episode_returns and mon.episode_lengths == mon_twin.episode_lengths
    assert mon.episode_infos == mon_twin.episode_infos
    res3 = mon.rollout_policy(pol, 5, action_masks=True, want_info=True)
    assert len(res3) == 3 and isinstance(res3[0], PolicyRollout) and tuple(res3[2].shape) == (5, n, 5)
    assert tuple(res3[1].counters.shape) == (5, n, 8)
