"""The fused policy kernel for observations up to 256 wide (orlg_policy_create_wide / MlpPolicy(wide_observations=True)):
DeepRMSA-v0 on germany50 (126 inputs) and on the 100-node ring with k = 10 (251 inputs) run their agents on the device.

References: the float64 forward with the kernel's bf16 roundings (test_policy_kernel.bf16_reference, which pads nothing: the
wide kernel pads K to 16 with zeros), the narrow kernel itself (a wide handle at obs_dim <= 64 gives its results bit for
bit), a Python loop of action_masks / sample_native / step_raw on a twin env, and the step loop of VecMonitor."""
import copy
import ctypes as C
import io
import os
import zipfile

import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

from test_action_masks import BASE, SEED, _assert_no_errors, _n_actions, _state  # noqa: E402
from test_policy_kernel import BF16_LOGIT_ATOL, bf16_reference  # noqa: E402

SMEM_MAX = 232448
# tile groups per CTA (None: refused) of orlg_policy_create_wide, from weights(H, L, K0) + G x 32 KB + biases <= SMEM_MAX
GROUPS = {((2, 64), 126): 2, ((2, 64), 251): 2, ((5, 128), 126): 1, ((5, 128), 251): None,
          ((6, 112), 126): 2, ((6, 112), 251): 1, ((4, 128), 226): 2, ((4, 128), 251): 1, ((6, 112), 226): 1}


def smem_bytes(L, H, obs_dim, G):
    k0 = (obs_dim + 15) // 16 * 16
    return H * k0 * 2 + (L - 1) * H * H * 2 + 16 * H * 2 + G * 32768 + (L * H + 16) * 4 + 64


def _wide_policy(L, H, obs_dim, n_actions=5, seed=0, device="cuda", critic=False):
    """An MlpPolicy with wide handles, initialised like test_policy_arch (orthogonal, biases up to 0.5)."""
    from optical_rl_gym_b200.policy import MlpPolicy

    torch.manual_seed(seed)
    pol = MlpPolicy(obs_dim, n_actions, (H,) * L, wide_observations=True)
    with torch.no_grad():
        for m in pol.shared_net:
            if isinstance(m, torch.nn.Linear):
                torch.nn.init.orthogonal_(m.weight, gain=2 ** 0.5)
                m.bias.uniform_(-0.5, 0.5)
        torch.nn.init.orthogonal_(pol.action_net.weight, gain=1.0)
    if critic:                      # SB3 >= 1.8: a separate critic trunk (SB3's default shape, 2 x 64)
        layers, d = [], obs_dim
        for _ in range(2):
            lin = torch.nn.Linear(d, 64)
            torch.nn.init.orthogonal_(lin.weight, gain=2 ** 0.5)
            layers += [lin, torch.nn.Tanh()]
            d = 64
        pol.critic_net = torch.nn.Sequential(*layers)
        pol.value_net = torch.nn.Linear(64, 1)
    return pol.to(device)


def _create_wide(obs_dim, H, L, n_actions, device=999):
    from optical_rl_gym_b200 import _native as nat

    w = np.zeros(H * max(obs_dim, 1) + max(L - 1, 0) * H * H + (n_actions + 1) * H, np.float32)
    b = np.zeros(max(L, 1) * H + n_actions + 1, np.float32)
    h = C.c_void_p()
    nat.check(nat.lib().orlg_policy_create_wide(device, obs_dim, H, L, n_actions, w.ctypes.data_as(C.c_void_p),
                                                b.ctypes.data_as(C.c_void_p), C.byref(h)))
    return h


# ------------------------------------------------------------------ shapes and plumbing (no GPU)
def test_group_table_follows_the_shared_memory_formula():
    for ((L, H), obs), g in GROUPS.items():
        want = 2 if smem_bytes(L, H, obs, 2) <= SMEM_MAX else 1 if smem_bytes(L, H, obs, 1) <= SMEM_MAX else None
        assert want == g, (L, H, obs)
    assert smem_bytes(2, 64, 126, 2) == 92800 and smem_bytes(5, 128, 126, 1) == 203392
    assert smem_bytes(6, 112, 226, 1) == 218368 and smem_bytes(5, 128, 251, 1) == 236160


@pytest.mark.parametrize("obs_dim,H,L,n_actions,match", [
    (0, 64, 2, 5, "wide fused policy kernel is built for obs_dim 1..256"),
    (257, 64, 2, 5, "wide fused policy kernel is built for obs_dim 1..256"),
    (126, 64, 2, 16, "wide fused policy kernel is built for obs_dim 1..256, <= 15 actions"),
    (126, 8, 2, 5, "multiple of 16 in 16..128"),
    (126, 144, 2, 5, "multiple of 16 in 16..128"),
    (126, 24, 2, 5, "multiple of 16 in 16..128"),
    (126, 64, 0, 5, "at least one hidden layer"),
    (251, 128, 5, 5, "needs 236160 bytes of shared memory with one tile group, 232448 available, for obs_dim 251"),
])
def test_create_wide_refusals(obs_dim, H, L, n_actions, match):
    from optical_rl_gym_b200._native import NativeError

    with pytest.raises(NativeError, match=match):
        _create_wide(obs_dim, H, L, n_actions)


@pytest.mark.parametrize("obs_dim,L,H", [(1, 2, 64), (53, 2, 64), (126, 2, 64), (251, 2, 64), (256, 2, 64), (240, 5, 128),
                                         (126, 5, 128), (251, 6, 112)])
def test_accepted_wide_shapes_reach_the_device_query(obs_dim, L, H):
    """Every shape check passes before the device query: a device that does not exist refuses them."""
    from optical_rl_gym_b200._native import NativeError

    with pytest.raises(NativeError, match="no such CUDA device"):
        _create_wide(obs_dim, H, L, 15)


def test_default_policy_still_refuses_wide_observations():
    from optical_rl_gym_b200._native import NativeError
    from optical_rl_gym_b200.policy import MlpPolicy

    with pytest.raises(NativeError, match="fused policy kernel.*obs_dim <= 64"):
        MlpPolicy(126, 5, (64, 64))._native_handles(0)
    with pytest.raises(NativeError, match="no such CUDA device"):        # the same policy, opted in
        MlpPolicy(126, 5, (64, 64), wide_observations=True)._native_handles(999)


def _sb3_state_dict(obs_dim=126, n_actions=5, seed=0):
    """policy.pth of an SB3 >= 1.8 ActorCriticPolicy with separate trunks pi = [64, 64], vf = [64, 64] (SB3's default)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for t in ("policy_net", "value_net"):
        d = obs_dim
        for i in range(2):
            sd["mlp_extractor.%s.%d.weight" % (t, 2 * i)] = torch.randn(64, d, generator=g) * (2.0 / d) ** 0.5
            sd["mlp_extractor.%s.%d.bias" % (t, 2 * i)] = torch.randn(64, generator=g) * 0.1
            d = 64
    sd["action_net.weight"] = torch.randn(n_actions, 64, generator=g) * 0.3
    sd["action_net.bias"] = torch.zeros(n_actions)
    sd["value_net.weight"] = torch.randn(1, 64, generator=g) * 0.3
    sd["value_net.bias"] = torch.full((1,), 0.25)
    return sd


def test_wide_flag_reaches_both_handles_through_the_loaders(tmp_path, monkeypatch):
    """from_state_dict / from_sb3_zip pass wide_observations on; both the actor's and the critic's handle are made with it,
    and flipping it rebuilds them."""
    from optical_rl_gym_b200.policy import MlpPolicy

    sd = _sb3_state_dict()
    path = tmp_path / "model.zip"
    buf = io.BytesIO()
    torch.save(sd, buf)
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
    calls = []

    def fake_create(device_index, spec, wide=False):
        calls.append((device_index, spec[2], [m.out_features for m in spec[0]], wide))
        return object()

    monkeypatch.setattr(MlpPolicy, "_create_handle", staticmethod(fake_create))
    monkeypatch.setattr(MlpPolicy, "_destroy_handles", lambda self, handles, dev: None)
    for pol in (MlpPolicy.from_state_dict(sd, wide_observations=True), MlpPolicy.from_sb3_zip(str(path), wide_observations=True)):
        assert pol.wide_observations and pol.critic_net is not None
        calls.clear()
        actor, critic = pol._native_handles(7)
        assert critic is not None and calls == [(7, 126, [64, 64], True), (7, 126, [64, 64], True)]
        assert pol._native_handles(7) == (actor, critic) and len(calls) == 2          # cached
        pol.wide_observations = False
        pol._native_handles(7)
        assert calls[2:] == [(7, 126, [64, 64], False), (7, 126, [64, 64], False)]
        pol.__dict__["_native_cache"].clear()
    assert not MlpPolicy.from_state_dict(sd).wide_observations and not MlpPolicy.from_sb3_zip(str(path)).wide_observations


@pytest.mark.parametrize("obs_dim", [126, 251])
def test_bf16_reference_catches_a_lost_chunk(obs_dim):
    """A layer 0 that loses a chunk of 64 inputs, or its last 16-wide K block, moves the reference's logits by many times
    BF16_LOGIT_ATOL, so the GPU comparison would fail on it.  (No GPU: CPU weights and observations.)"""
    pol = _wide_policy(2, 64, obs_dim, device="cpu")
    obs = (torch.rand((512, obs_dim), generator=torch.Generator().manual_seed(obs_dim)) * 2 - 1).double()
    ref = bf16_reference(pol, obs)
    last16 = (obs_dim - 1) // 16 * 16
    for cols in (slice(64, 128), slice(last16, obs_dim)):
        bad = copy.deepcopy(pol)
        with torch.no_grad():
            bad.shared_net[0].weight[:, cols] = 0.0
        moved = (bf16_reference(bad, obs) - ref).abs().max().item()
        assert moved > 10 * BF16_LOGIT_ATOL, (cols, moved)


# ------------------------------------------------------------------ GPU: against the reference and the narrow kernel
WIDE_TRUNKS = [(1, 16), (2, 64), (2, 128), (5, 128)]
WIDE_OBS = [2, 53, 54, 63, 64, 65, 66, 126, 127, 128, 129, 192, 251, 256]
WIDE_CASES = [(obs, t) for obs in WIDE_OBS for t in WIDE_TRUNKS if smem_bytes(*t, obs, 1) <= SMEM_MAX]     # 5 x 128: obs <= 240


def _check(pol, obs, n_actions):
    logits = torch.full((obs.shape[0], n_actions + 1), float("nan"), dtype=torch.float32, device="cuda")
    act = pol.act_native(obs, logits=logits)
    ref = bf16_reference(pol, obs.double())
    torch.cuda.synchronize()
    err = (logits.double() - ref).abs().max().item()
    assert err < BF16_LOGIT_ATOL, err
    assert torch.equal(act[:, 0].long(), logits[:, :n_actions].argmax(-1))
    return logits


@pytest.mark.gpu
@pytest.mark.parametrize("obs_dim,trunk", WIDE_CASES, ids=["%d-%dx%d" % (o, *t) for o, t in WIDE_CASES])
def test_wide_kernel_matches_bf16_reference(obs_dim, trunk):
    """n = 1, 127, 128, 129 and 300 (ragged tiles), and the same 300 rows starting 4 bytes into a buffer: the same bits."""
    L, H = trunk
    n_actions = 15 if obs_dim % 2 else 5
    pol = _wide_policy(L, H, obs_dim, n_actions, seed=obs_dim + L)
    gen = torch.Generator(device="cuda").manual_seed(obs_dim * 10 + L)
    for n in (1, 127, 128, 129, 300):
        obs = torch.rand((n, obs_dim), generator=gen, device="cuda") * 2 - 1
        aligned = _check(pol, obs, n_actions)
    buf = torch.zeros(300 * obs_dim + 1, device="cuda")
    buf[1:].copy_(obs.reshape(-1))
    sub = buf[1:].view(300, obs_dim)
    assert sub.data_ptr() % 16 == 4
    assert torch.equal(_check(pol, sub, n_actions), aligned)


@pytest.mark.gpu
@pytest.mark.parametrize("trunk", [(5, 128), (2, 64)], ids=["5x128", "2x64"])
@pytest.mark.parametrize("obs_dim", [54, 64])
def test_wide_equals_narrow_bit_for_bit(obs_dim, trunk):
    L, H = trunk
    narrow = _wide_policy(L, H, obs_dim, seed=obs_dim)
    narrow.wide_observations = False
    wide = copy.deepcopy(narrow)
    wide.wide_observations = True
    from optical_rl_gym_b200 import _native as nat

    assert nat.lib().orlg_policy_tile_groups(wide._native_handle(0)) == 2
    n = 4099
    gen = torch.Generator(device="cuda").manual_seed(obs_dim)
    obs = torch.rand((n, obs_dim), generator=gen, device="cuda") * 2 - 1
    mask = torch.rand((n, 5), generator=gen, device="cuda") < 0.6
    ln, lw = torch.empty((n, 6), device="cuda"), torch.empty((n, 6), device="cuda")
    assert torch.equal(narrow.act_native(obs, logits=ln), wide.act_native(obs, logits=lw)) and torch.equal(ln, lw)
    for det in (False, True):
        for m in (None, mask):
            kw = dict(seed=SEED, counter=5, row_id_base=BASE, deterministic=det, action_masks=m)
            for g, w in zip(wide.sample_native(obs, **kw), narrow.sample_native(obs, **kw)):
                assert torch.equal(g, w)


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(GROUPS), ids=["%dx%d-%d" % (k[0][0], k[0][1], k[1]) for k in GROUPS])
def test_tile_groups_follow_the_table(key):
    from optical_rl_gym_b200 import _native as nat

    (L, H), obs_dim = key
    pol = _wide_policy(L, H, obs_dim, seed=L * H)
    if GROUPS[key] is None:
        with pytest.raises(nat.NativeError, match="%d bytes" % smem_bytes(L, H, obs_dim, 1)):
            pol._native_handle(0)
        return
    assert nat.lib().orlg_policy_tile_groups(pol._native_handle(0)) == GROUPS[key]
    obs = torch.rand((1000, obs_dim), generator=torch.Generator(device="cuda").manual_seed(L), device="cuda") * 2 - 1
    _check(pol, obs, 5)


# ------------------------------------------------------------------ GPU: the closed loop on germany50 and the 100-node ring
TOPOS = ["germany50", "ring100"]
_ARGS = dict(episode_length=10, mean_service_holding_time=60.0, num_spectrum_resources=24)


def _topology(name):
    from optical_rl_gym_b200.topology import TopologyTables

    f = "topo_germany50_tables.npz" if name == "germany50" else "topo_c3_ring100_chords200_k10.npz"
    return TopologyTables.load(os.path.join(helpers.GOLDEN_DIR, f))


def _env(topo, n, base=BASE):
    from optical_rl_gym_b200 import OpticalVecEnv

    env = OpticalVecEnv("DeepRMSA-v0", n, _topology(topo), seed=SEED, env_id_base=base, **_ARGS)
    assert env.obs_dim == (126 if topo == "germany50" else 251) and env.kernel_info()["wide"]
    return env


def _loop_policy(env, seed=0):
    """A 5 x 128 actor where it fits (germany50), else 2 x 64, with a separate 2 x 64 critic."""
    L, H = (5, 128) if env.obs_dim <= 240 else (2, 64)
    return _wide_policy(L, H, env.obs_dim, _n_actions(env), seed=seed, critic=True)


def _twin_loop(env, pol, T, deterministic, masked):
    """rollout_policy as a Python loop of action_masks + sample_native + step_raw, keyed the same way."""
    obs = [env.observation().clone()]
    acts, lps, vals, rews, dones, masks, counters = [], [], [], [], [], [], []
    for _ in range(T):
        m = env.action_masks().clone() if masked else None
        a, lp, v = pol.sample_native(obs[-1], seed=SEED, counter=env.request_index, row_id_base=BASE,
                                     deterministic=deterministic, action_masks=m)
        o, r, d = env.step_raw(a)
        obs.append(o.clone()); acts.append(a[:, 0].clone()); lps.append(lp); vals.append(v); rews.append(r.clone())
        dones.append(d.clone()); masks.append(m); counters.append(env._info.clone())
    vals.append(pol.sample_native(obs[-1], seed=SEED, counter=env.request_index, row_id_base=BASE)[2])
    out = [torch.stack(x) for x in (obs, acts, lps, vals, rews, dones)]
    return out, (torch.stack(masks) if masked else None), torch.stack(counters)


@pytest.mark.gpu
@pytest.mark.parametrize("topo", TOPOS)
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("deterministic", [False, True])
def test_wide_rollout_policy_equals_the_python_loop(topo, masked, deterministic):
    n, T = 257, 24
    env, twin = _env(topo, n), _env(topo, n)
    pol = _loop_policy(env, seed=3)
    res = env.rollout_policy(pol, T, deterministic=deterministic, action_masks=masked, want_info=True)
    ro, info = res[0], res[1]
    want, want_masks, want_counters = _twin_loop(twin, pol, T, deterministic, masked)
    for name, g, w in zip(ro._fields, ro, want):
        assert torch.equal(g, w), name
    assert torch.equal(info.counters, want_counters)
    for g, w in zip(_state(env), _state(twin)):
        assert torch.equal(g, w)
    if masked:
        masks = res[2]
        assert torch.equal(masks, want_masks)
        chosen = masks.gather(2, ro.actions.long().unsqueeze(-1))[..., 0]
        assert chosen[masks.any(-1)].all()                               # never a masked action while a valid one exists
        assert (~masks).any() and masks.any()
    _assert_no_errors(env)
    env.close(); twin.close()


@pytest.mark.gpu
@pytest.mark.parametrize("topo", TOPOS)
def test_wide_rollout_policy_split_and_checkpoint(topo):
    n = 256
    pol = _loop_policy(_env(topo, 8), seed=2)
    whole, wmasks = _env(topo, n).rollout_policy(pol, 30, action_masks=True)
    env = _env(topo, n)
    for k in range(3):
        p, m = env.rollout_policy(pol, 10, action_masks=True)
        sl = slice(10 * k, 10 * k + 10)
        assert torch.equal(p.obs, whole.obs[10 * k:10 * k + 11]) and torch.equal(p.value, whole.value[10 * k:10 * k + 11])
        for f in ("actions", "log_prob", "reward", "done"):
            assert torch.equal(getattr(p, f), getattr(whole, f)[sl]), (k, f)
        assert torch.equal(m, wmasks[sl])
    first, fresh = _env(topo, n), _env(topo, n)
    first.rollout_policy(pol, 10, action_masks=True)
    fresh.rollout(3)
    fresh.load_state_dict(first.state_dict())
    rest, rmasks = fresh.rollout_policy(pol, 20, action_masks=True)
    for f in ("actions", "log_prob", "reward", "done"):
        assert torch.equal(getattr(rest, f), getattr(whole, f)[10:]), f
    assert torch.equal(rest.obs, whole.obs[10:]) and torch.equal(rest.value, whole.value[10:]) and torch.equal(rmasks, wmasks[10:])


@pytest.mark.gpu
@pytest.mark.parametrize("topo", TOPOS)
def test_vec_monitor_wide_rollout_policy(topo):
    from optical_rl_gym_b200.monitor import VecMonitor

    n, T = 64, 35
    env, twin = _env(topo, n), _env(topo, n)
    pol = _loop_policy(env, seed=8)
    mon, mon_twin = VecMonitor(env), VecMonitor(twin)
    ro, masks = mon.rollout_policy(pol, T, action_masks=True)
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
