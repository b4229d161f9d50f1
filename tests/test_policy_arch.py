"""The fused policy kernel at other hidden widths and depths than the shipped agent's 5 x 128: any trunk of one width H (a
multiple of 16 in 16..128) whose weights fit in shared memory, in particular the trunk Stable-Baselines3 gives PPO and A2C by
default (separate actor and critic trunks of 2 x 64).

References as in test_policy_kernel / test_policy_rollout: the float64 forward with the kernel's roundings (bf16_reference),
the inverse-CDF sampler on its softmax, a Python loop of sample_native + step_raw on a twin env, and the C oracle replaying
the sampled actions."""
import ctypes as C
import io
import types
import zipfile

import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

from test_policy_kernel import BF16_LOGIT_ATOL, _bf16, _policy, bf16_reference  # noqa: E402
from test_policy_rollout import (AGREEMENT_MIN, BASE, CDF_DELTA, CONFIGS, OBS_RTOL, SEED, _assert_same, _env,  # noqa: E402
                                 _real_observations, _state, _twin_loop, draw_u, reference_sample)

SMEM_MAX = 232448             # dynamic shared memory a block may opt in to on sm_100
# Against bf16_reference.  Measured on an NVIDIA B200 (1000 W power limit) over GPU_ARCHS, real observations 54 and 64 wide
# and 1 .. 65536 rows (biases up to 0.5): the largest logit / value error grows with depth -- 4.1e-3 at 2 x 64, 1.0e-2 at
# 6 x 112, 1.19e-2 at 8 x 64 -- so the 5 x 128 tolerance (largest error 9.4e-3 there) still leaves a margin of 1.7.
ARCH_ATOL = BF16_LOGIT_ATOL
GPU_ARCHS = [(1, 16), (2, 32), (2, 64), (3, 48), (8, 64), (6, 112), (4, 128)]     # (hidden layers, width)


def _arch_policy(L, H, seed=0, obs_dim=54, n_actions=5, device="cuda"):
    """An MlpPolicy with a trunk of L layers of width H, initialised like test_policy_kernel._policy but with biases up to
    0.5 (so that a bias read from the wrong place moves the logits well beyond the tolerance)."""
    from optical_rl_gym_b200.policy import MlpPolicy

    torch.manual_seed(seed)
    pol = MlpPolicy(obs_dim, n_actions, (H,) * L).to(device)
    with torch.no_grad():
        for m in pol.shared_net:
            if isinstance(m, torch.nn.Linear):
                torch.nn.init.orthogonal_(m.weight, gain=2 ** 0.5)
                m.bias.uniform_(-0.5, 0.5)
        torch.nn.init.orthogonal_(pol.action_net.weight, gain=1.0)
    return pol


def _sb3_state_dict(obs_dim=54, n_actions=5, pi=(64, 64), vf=(64, 64), seed=0):
    """policy.pth of an SB3 >= 1.8 ActorCriticPolicy with separate trunks (net_arch=dict(pi=..., vf=...)); SB3's PPO and
    A2C default is pi = vf = [64, 64]."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for t, widths in (("policy_net", pi), ("value_net", vf)):
        d = obs_dim
        for i, w in enumerate(widths):
            sd["mlp_extractor.%s.%d.weight" % (t, 2 * i)] = torch.randn(w, d, generator=g) * (2.0 / d) ** 0.5
            sd["mlp_extractor.%s.%d.bias" % (t, 2 * i)] = torch.randn(w, generator=g) * 0.1
            d = w
    sd["action_net.weight"] = torch.randn(n_actions, pi[-1], generator=g) * 0.3
    sd["action_net.bias"] = torch.zeros(n_actions)
    sd["value_net.weight"] = torch.randn(1, vf[-1], generator=g) * 0.3
    sd["value_net.bias"] = torch.full((1,), 0.25)
    return sd


def _hand_forward(sd, x):
    """The SB3 forward of a separate-trunk state dict, written out: (logits, value)."""
    def trunk(name):
        h, i = x, 0
        while "mlp_extractor.%s.%d.weight" % (name, i) in sd:
            h = torch.tanh(h @ sd["mlp_extractor.%s.%d.weight" % (name, i)].T + sd["mlp_extractor.%s.%d.bias" % (name, i)])
            i += 2
        return h
    logits = trunk("policy_net") @ sd["action_net.weight"].T + sd["action_net.bias"]
    value = (trunk("value_net") @ sd["value_net.weight"].T + sd["value_net.bias"])[:, 0]
    return logits, value


def _critic_view(pol):
    """The critic handle's network (critic trunk, value_net as its one-row action head) for bf16_reference."""
    return types.SimpleNamespace(shared_net=pol.critic_net, action_net=pol.value_net, value_net=pol.value_net)


# ------------------------------------------------------------------ shapes and loading (no GPU)
@pytest.mark.parametrize("L,H", [(2, 8), (2, 24), (2, 144), (2, 256)])
def test_widths_outside_the_kernel_are_refused(L, H):
    from optical_rl_gym_b200._native import NativeError

    with pytest.raises(NativeError, match="fused policy kernel.*multiple of 16 in 16..128"):
        _arch_policy(L, H, device="cpu")._native_handles(0)


@pytest.mark.parametrize("L,H,smem", [(6, 128, 253056), (7, 112, 237248)])
def test_architectures_that_do_not_fit_in_shared_memory_are_refused(L, H, smem):
    from optical_rl_gym_b200._native import NativeError

    with pytest.raises(NativeError, match="fused policy kernel needs %d bytes of shared memory, %d available" % (smem, SMEM_MAX)):
        _arch_policy(L, H, device="cpu")._native_handles(0)


def test_observation_rule_is_kept_for_narrow_trunks():
    from optical_rl_gym_b200._native import NativeError

    for obs_dim in (66, 53):
        with pytest.raises(NativeError, match="fused policy kernel.*obs_dim <= 64"):
            _arch_policy(2, 64, obs_dim=obs_dim, device="cpu")._native_handles(0)


@pytest.mark.parametrize("L,H", [(1, 16), (2, 64), (8, 64), (6, 112), (5, 128)])
def test_accepted_architectures_reach_the_device_query(L, H):
    """Every shape check passes before the device query: a device that does not exist refuses them."""
    from optical_rl_gym_b200._native import NativeError
    from optical_rl_gym_b200.policy import MlpPolicy

    pol = _arch_policy(L, H, device="cpu")
    with pytest.raises(NativeError, match="no such CUDA device"):
        MlpPolicy._create_handle(999, pol._native_specs()["actor"])


@pytest.mark.parametrize("net_arch", [(128, 128, 128, 128, 64), (64, 128), ()])
def test_non_uniform_or_empty_trunks_are_refused_before_the_library(net_arch, monkeypatch):
    """orlg_policy_create takes one width: anything else would be read past the end of the weight array."""
    from optical_rl_gym_b200 import _native as nat
    from optical_rl_gym_b200.policy import MlpPolicy

    def no_library():
        raise AssertionError("the library was called")

    monkeypatch.setattr(nat, "lib", no_library)
    pol = MlpPolicy(54, 5, net_arch)
    with pytest.raises(ValueError, match="fused policy kernel"):
        pol._native_handles(0)


def test_sb3_checkpoint_with_critic_wider_than_actor_loads():
    """net_arch=dict(pi=[64, 64], vf=[128, 128]): value_net is sized from the checkpoint, forward() is SB3's, the critic spec
    carries the 128-wide trunk and both handles pass every shape check."""
    from optical_rl_gym_b200._native import NativeError
    from optical_rl_gym_b200.policy import MlpPolicy

    sd = _sb3_state_dict(pi=(64, 64), vf=(128, 128), seed=3)
    pol = MlpPolicy.from_state_dict(sd)
    assert pol.value_net.in_features == 128 and torch.equal(pol.value_net.weight, sd["value_net.weight"])
    x = torch.randn(33, 54, dtype=torch.float64)
    logits, value = pol.double()(x)
    want_logits, want_value = _hand_forward({k: v.double() for k, v in sd.items()}, x)
    assert torch.allclose(logits, want_logits, rtol=0, atol=1e-12) and torch.allclose(value, want_value, rtol=0, atol=1e-12)
    pol = pol.float()
    specs = pol._native_specs()
    clins, cheads, cobs = specs["critic"]
    assert cobs == 54 and [m.out_features for m in clins] == [128, 128] and cheads == [pol.value_net, pol.value_net]
    for i, m in enumerate(clins):
        assert torch.equal(m.weight, sd["mlp_extractor.value_net.%d.weight" % (2 * i)])
    alins, aheads, _ = specs["actor"]
    assert [m.out_features for m in alins] == [64, 64] and aheads[0] is pol.action_net
    assert aheads[1].in_features == 64 and torch.isnan(aheads[1].bias).all() and not aheads[1].weight.any()
    for spec in (specs["actor"], specs["critic"]):
        with pytest.raises(NativeError, match="no such CUDA device"):
            MlpPolicy._create_handle(999, spec)


def _flat_bias(pol):
    """The kernel's bias array: L * H hidden biases, then the output row's (logits, value), padded to 16."""
    lins = [m for m in pol.shared_net if isinstance(m, torch.nn.Linear)]
    out = torch.cat([pol.action_net.bias, pol.value_net.bias]).double()
    return torch.cat([m.bias.double() for m in lins] + [out, torch.zeros(16 - out.numel(), dtype=torch.float64)])


@torch.no_grad()
def _narrow_reference(pol, obs, bug=None):
    """bf16_reference written against the kernel's bias array, with a defect a narrow-width epilogue could have:
    "stale_chunk" (a hidden layer's last 16 output columns never written: zeros in the next A operand) or "bias_stride_128"
    (layer l's bias read at l * 128 instead of l * H)."""
    lins = [m for m in pol.shared_net if isinstance(m, torch.nn.Linear)]
    H, bias = lins[0].out_features, _flat_bias(pol)
    bias = torch.cat([bias, torch.zeros(128 * len(lins) + 16, dtype=torch.float64)])        # reads past the end see zeros
    h = _bf16(obs)
    for i, lin in enumerate(lins):
        b = bias[(128 if bug == "bias_stride_128" else H) * i:][:H]
        h = _bf16(torch.tanh(h @ _bf16(lin.weight).T + b))
        if bug == "stale_chunk" and i == 0:
            h[:, H - 16:] = 0.0
    w = _bf16(torch.cat([pol.action_net.weight, pol.value_net.weight]))
    na = pol.action_net.out_features
    return h @ w.T + bias[len(lins) * H:][:na + 1]


def test_bf16_reference_catches_narrow_epilogue_bugs():
    """For 2 x 64 on real observations each defect moves the logits by many times the tolerance."""
    from test_policy_kernel import _oracle_observations

    obs = _oracle_observations(1)
    pol = _arch_policy(2, 64, device="cpu")
    ref = bf16_reference(pol, obs)
    assert torch.allclose(_narrow_reference(pol, obs), ref, rtol=0, atol=1e-12)
    for bug in ("stale_chunk", "bias_stride_128"):
        moved = (_narrow_reference(pol, obs, bug) - ref).abs().max().item()
        assert moved > 10 * ARCH_ATOL, (bug, moved)


# ------------------------------------------------------------------ GPU: act_native and sample_native
_OBS = {}


def _observations(j, n):
    """Real DeepRMSA observations of n envs of a partly filled NSFNET (j = 1: 54 wide, j = 2: 64), own allocation."""
    if (j, n) not in _OBS:
        from optical_rl_gym_b200 import OpticalVecEnv

        env = OpticalVecEnv("DeepRMSA-v0", n, helpers.golden_tables(), seed=4, j=j)
        _OBS[(j, n)] = env.rollout(30)[0][-1].clone()
        env.close()
    return _OBS[(j, n)]


def _check_arch(pol, obs):
    n_actions = pol.action_net.out_features
    logits = torch.full((obs.shape[0], n_actions + 1), float("nan"), dtype=torch.float32, device="cuda")
    act = pol.act_native(obs, logits=logits)
    ref = bf16_reference(pol, obs.double())
    torch.cuda.synchronize()
    err = (logits.double() - ref).abs().max().item()
    assert err < ARCH_ATOL, err
    assert torch.equal(act[:, 0].long(), logits[:, :n_actions].argmax(-1))
    top2 = ref[:, :n_actions].topk(2, dim=-1).values
    clear = (top2[:, 0] - top2[:, 1]) > 2 * ARCH_ATOL
    assert torch.equal(act[clear, 0].long(), ref[clear, :n_actions].argmax(-1))
    return err


@pytest.mark.gpu
@pytest.mark.parametrize("L,H", GPU_ARCHS)
@pytest.mark.parametrize("j", [1, 2])
@pytest.mark.parametrize("n", [1, 127, 129, 65536])
def test_act_native_matches_bf16_reference(L, H, j, n):
    obs = _observations(j, n)
    assert obs.shape[1] == (54 if j == 1 else 64) and obs.data_ptr() % 16 == 0
    err = _check_arch(_arch_policy(L, H, seed=L * 1000 + H, obs_dim=obs.shape[1]), obs)
    print("%d x %d, j = %d, n = %d: max error %.2e" % (L, H, j, n, err))


@pytest.mark.gpu
@pytest.mark.parametrize("L,H", [(2, 64), (3, 48)])
def test_unaligned_observations_bit_for_bit_at_narrow_widths(L, H):
    """Rows that start off a 16-byte boundary take the scalar load path: the same results as the aligned batch."""
    n = 1000
    obs = _observations(1, 1001)
    sub = obs.view(-1)[54:].view(n, 54)                          # 216-byte offset
    assert sub.is_contiguous() and sub.data_ptr() % 16 != 0
    pol = _arch_policy(L, H, seed=H)
    la = torch.empty((n + 1, 6), dtype=torch.float32, device="cuda")
    lb = torch.empty((n, 6), dtype=torch.float32, device="cuda")
    aa, ab = pol.act_native(obs, logits=la), pol.act_native(sub, logits=lb)
    assert torch.equal(aa[1:], ab) and torch.equal(la[1:], lb)
    _check_arch(pol, sub)


@pytest.mark.gpu
def test_sampled_actions_of_a_2x64_policy_match_the_reference_sampler():
    obs = _real_observations(1)
    n = obs.shape[0]
    pol = _arch_policy(2, 64, seed=11)
    with torch.no_grad():
        pol.action_net.weight.mul_(0.3)            # logits a few units apart: every action has a real probability
    rng = np.random.default_rng(11)
    seed = int(rng.integers(0, 2 ** 63)) * 2 + 1
    base = int(rng.integers(0, 2 ** 31))
    a, lp, v = pol.sample_native(obs, seed=seed, counter=7, row_id_base=base)
    ref = bf16_reference(pol, obs.double()).cpu().numpy()
    u = draw_u(seed, 7, base + np.arange(n, dtype=np.uint64))
    want, cdf = reference_sample(ref[:, :5], u)
    a = a[:, 0].cpu().numpy()
    clear = (np.abs(u[:, None] - cdf[:, :-1]) > CDF_DELTA).all(-1)
    assert clear.mean() > 0.5
    assert np.array_equal(a[clear], want[clear])
    agree = (a == want).mean()
    assert agree >= AGREEMENT_MIN, agree
    assert np.abs(v.cpu().numpy() - ref[:, 5]).max() < ARCH_ATOL
    # deterministic mode is the argmax of act_native
    da, dlp, dv = pol.sample_native(obs, seed=seed, counter=7, deterministic=True)
    logits = torch.empty((n, 6), dtype=torch.float32, device="cuda")
    act = pol.act_native(obs, logits=logits)
    assert torch.equal(da, act) and torch.equal(dv, logits[:, 5])
    own = torch.log_softmax(logits[:, :5].double(), -1).gather(1, act.long())[:, 0]
    assert (dlp.double() - own).abs().max().item() < 1e-5


# ------------------------------------------------------------------ GPU: the SB3-default agent end to end
def _sb3_agent(env, vf=(64, 64), seed=0):
    from optical_rl_gym_b200.policy import MlpPolicy

    n_actions = env.tables.k_paths * env.j + env.reject_action
    return MlpPolicy.from_state_dict(_sb3_state_dict(env.obs_dim, n_actions, (64, 64), vf, seed)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("vf", [(64, 64), (128, 128)])
@pytest.mark.parametrize("config", ["nsfnet_j1", "E20"])
@pytest.mark.parametrize("deterministic", [False, True])
def test_sb3_default_agent_rollout_equals_the_python_loop(vf, config, deterministic):
    """Separate pi = [64, 64] and vf trunks: three launches per step (actor, critic, env), auto-resets inside the call."""
    n, T = 129, 25
    env, twin = _env(config, n), _env(config, n)
    pol = _sb3_agent(env, vf, seed=n)
    assert pol.critic_net is not None
    ro = env.rollout_policy(pol, T, deterministic=deterministic)
    want = _twin_loop(twin, pol, T, deterministic)
    _assert_same(ro, want)
    assert int(ro.done.sum()) > 0 and len(torch.unique(ro.actions)) > 1
    for g, w in zip(_state(env), _state(twin)):
        assert torch.equal(g, w)
    assert int(env.error_flags().abs().sum()) == 0
    # the value is the critic trunk's
    vals = bf16_reference(_critic_view(pol), ro.obs.reshape(-1, env.obs_dim).double())[:, 1]
    assert (ro.value.reshape(-1).double() - vals).abs().max().item() < ARCH_ATOL
    env.close(); twin.close()


@pytest.mark.gpu
def test_sb3_default_agent_env_side_matches_the_oracle(tmp_path):
    """An SB3-default PPO checkpoint (policy.pth in a zip) through from_sb3_zip and rollout_policy; the C oracle replays
    the sampled actions."""
    from oracle import oracle

    from optical_rl_gym_b200.policy import MlpPolicy

    n, T, config = 64, 40, "nsfnet_j2_rej"
    env = _env(config, n)
    n_actions = env.tables.k_paths * env.j + env.reject_action
    buf = io.BytesIO()
    torch.save(_sb3_state_dict(env.obs_dim, n_actions, seed=5), buf)
    path = tmp_path / "ppo_default.zip"
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
    pol = MlpPolicy.from_sb3_zip(path, device="cuda")
    ro = env.rollout_policy(pol, T)
    acts = ro.actions.cpu().numpy()
    assert len(np.unique(acts)) > 1
    topo, args = CONFIGS[config]
    env_args = dict(dict(episode_length=10, mean_service_holding_time=40.0, num_spectrum_resources=64), **args)
    okw = helpers.sim_kwargs(dict(kind="DeepRMSA-v0", env_args=env_args))
    obs, rew, done = ro.obs.cpu().numpy(), ro.reward.cpu().numpy(), ro.done.cpu().numpy()
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
def test_native_weights_of_a_2x64_policy_follow_optimizer_steps():
    from optical_rl_gym_b200.policy import MlpPolicy

    obs = _real_observations(1, 2048)
    pol = _arch_policy(2, 64, seed=9)
    before = pol.sample_native(obs, seed=5, counter=1)
    opt = torch.optim.SGD(pol.parameters(), lr=0.05)
    logits, value = pol(obs)
    (logits.logsumexp(-1).mean() + value.square().mean()).backward()
    opt.step()
    after = pol.sample_native(obs, seed=5, counter=1)
    fresh = MlpPolicy(54, 5, (64, 64)).cuda()
    fresh.load_state_dict(pol.state_dict())
    want = fresh.sample_native(obs, seed=5, counter=1)
    for g, w in zip(after, want):
        assert torch.equal(g, w)
    assert not torch.equal(after[1], before[1]) and not torch.equal(after[2], before[2])


@pytest.mark.gpu
def test_run_time_architecture_instance_equals_the_5x128_instance_bit_for_bit(monkeypatch):
    """5 x 128 runs a kernel instance compiled for it; ORLG_POLICY_GENERAL (read by orlg_policy_create) puts a handle on the
    instance that reads H and L at run time.  Both give the same bits: act_native, sample_native and rollout_policy."""
    def outputs():
        pol = _policy(seed=21)
        obs = _observations(1, 65536)
        logits = torch.empty((obs.shape[0], 6), dtype=torch.float32, device="cuda")
        res = [pol.act_native(obs, logits=logits), logits]
        res += list(pol.sample_native(obs, seed=3, counter=8, row_id_base=5))
        res += list(_env("nsfnet_j1", 300).rollout_policy(pol, 12))
        return res

    monkeypatch.delenv("ORLG_POLICY_GENERAL", raising=False)
    compiled = outputs()
    monkeypatch.setenv("ORLG_POLICY_GENERAL", "1")
    general = outputs()
    monkeypatch.delenv("ORLG_POLICY_GENERAL")
    assert len(compiled) == len(general) == 11
    for i, (c, g) in enumerate(zip(compiled, general)):
        assert torch.equal(c, g), i


@pytest.mark.gpu
def test_handles_of_different_sizes_on_one_device():
    """A small policy made after a large one (and the reverse) leaves both launchable: each kernel instance keeps the
    largest shared-memory size asked of it."""
    obs = _observations(1, 4096)
    big, small, mid = _arch_policy(6, 112, seed=1), _arch_policy(2, 64, seed=2), _policy(seed=3)
    for pol in (big, small, mid, big):
        _check_arch(pol, obs)
