"""SB3 agents of PathOnlyFirstFitAction(SimpleMatrixObservation(env)) on RMSA-v0 / RWA-v0: packed matrix observations,
the MATRIX instances of the fused policy kernel (orlg_policy_create_matrix: layer 0 streamed through a shared-memory ring)
and rollout_policy through the path-only wrapper.

CPU: the packing / unpacking against numpy and the oracle (and the golden wrapper run), every refusal that needs no device,
and that the bf16 reference catches a misplaced layer-0 block.  GPU: packed rows against matrix_observation() bit for bit,
the kernel against the bf16 reference, sampling against the reference sampler, and rollout_policy against a Python loop."""
import ctypes as C
import io
import os
import zipfile

import numpy as np
import pytest

import helpers
from oracle import oracle

torch = pytest.importorskip("torch")

from test_policy_kernel import BF16_LOGIT_ATOL, bf16_reference  # noqa: E402
from test_policy_rollout import _sb3_state_dict, draw_u, reference_sample  # noqa: E402

SEED, BASE = 31, 500


# ------------------------------------------------------------------ numpy restatement of the packed row
def words(nodes, links, slots):
    return 4 + 4 * ((slots + 127) // 128) * links


def pack_np(src, dst, avail, nodes):
    """Rows of (src [R], dst [R], available_slots uint8 [R, links, slots]) -> int32 [R, W] as orlg_matrix_observation_packed."""
    R, links, slots = avail.shape
    nwv = (slots + 127) // 128
    W = words(nodes, links, slots)
    out = np.zeros((R, W), np.uint32)
    out[:, 0] = np.minimum(src, dst) | (np.maximum(src, dst) << 8)
    bits = np.zeros((R, links, 128 * nwv), np.uint8)
    bits[:, :, :slots] = avail
    w = np.packbits(bits.reshape(R, links, -1, 32), axis=-1, bitorder="little").view("<u4")[..., 0]    # [R, links, 4 nwv]
    out[:, 4:] = w.reshape(R, -1)
    return out.view(np.int32)


def unpacked_np(src, dst, avail, nodes):
    R = len(src)
    lo, hi = np.zeros((R, nodes), np.uint8), np.zeros((R, nodes), np.uint8)
    lo[np.arange(R), np.minimum(src, dst)] = 1
    hi[np.arange(R), np.maximum(src, dst)] = 1
    return np.concatenate([lo, hi, avail.reshape(R, -1)], 1)


def _random_rows(rng, R, nodes, links, slots, p=0.5):
    src = rng.integers(0, nodes, R)
    dst = (src + rng.integers(1, nodes, R)) % nodes
    avail = (rng.random((R, links, slots)) < p).astype(np.uint8)
    return src, dst, avail


@pytest.mark.parametrize("slots", [1, 31, 32, 33, 100, 127, 128, 129, 320, 512])
@pytest.mark.parametrize("nodes", [2, 14, 50, 255])
def test_unpack_inverts_the_numpy_packing(slots, nodes):
    from optical_rl_gym_b200.vec_env import matrix_obs_words, unpack_matrix_observation

    rng = np.random.default_rng(slots * 1000 + nodes)
    links = 3
    src, dst, avail = _random_rows(rng, 40, nodes, links, slots)
    packed = pack_np(src, dst, avail, nodes)
    assert packed.shape[1] == matrix_obs_words((nodes, links, slots)) and packed.shape[1] % 4 == 0
    got = unpack_matrix_observation(torch.from_numpy(packed), (nodes, links, slots))
    assert got.dtype == torch.uint8
    assert np.array_equal(got.numpy(), unpacked_np(src, dst, avail, nodes))
    got3 = unpack_matrix_observation(torch.from_numpy(packed).reshape(4, 10, -1), (nodes, links, slots), dtype=torch.float32)
    assert np.array_equal(got3.reshape(40, -1).numpy(), unpacked_np(src, dst, avail, nodes).astype(np.float32))


def _oracle_rows(e, nodes):
    avail, _, _, _ = e.state()
    r = e.request()
    return np.array([r["src"]]), np.array([r["dst"]]), avail[0][None].astype(np.uint8)


@pytest.mark.parametrize("name", ["wrap_rmsa_matrix_pathonly"])
def test_unpacked_oracle_packing_is_the_golden_matrix_observation(name):
    """At every step of the golden wrapper run: unpack(pack(oracle state)) == oracle.simple_matrix_observation == the
    reference's bits."""
    from optical_rl_gym_b200.vec_env import unpack_matrix_observation

    g = helpers.load_golden(name)
    meta = g["meta"]
    assert meta["matrix"]
    tables = helpers.golden_tables()
    nodes, links, slots = tables.num_nodes, tables.num_links, int(meta["env_args"].get("num_spectrum_resources", 100))
    for i in range(meta["n_envs"]):
        e = oracle.OracleEnv(meta["kind"], tables, **helpers.sim_kwargs(meta))
        e.set_trace(g["req_arrival"][i], g["req_holding"][i], g["req_src"][i], g["req_dst"][i], g["req_bit_rate"][i])
        e.reset(full=True)
        e.reset(full=False)
        for t in range(meta["T"] + 1):
            want = oracle.simple_matrix_observation(e, nodes)
            packed = pack_np(*_oracle_rows(e, nodes), nodes)
            got = unpack_matrix_observation(torch.from_numpy(packed), (nodes, links, slots))[0].numpy()
            assert np.array_equal(got, want.astype(np.uint8)), (i, t)
            assert np.array_equal(np.packbits(got, bitorder="little"), g["matrix_bits"][i, t]), (i, t)
            if t == meta["T"]:
                break
            a = oracle.path_only_first_fit(e, tables, int(g["path_action"][i, t])) if meta["path_only"] else g["actions"][i, t]
            o, rc = e.step(a)
            assert rc == 0
            if o.done:
                e.reset(full=False)
        e.close()


# ------------------------------------------------------------------ refusals without a device
def _create_matrix(nodes, links, slots, H, L, n_actions, device=999):
    from optical_rl_gym_b200 import _native as nat

    obs = 2 * nodes + links * slots
    w = np.zeros(H * obs + (L - 1) * H * H + (n_actions + 1) * H, np.float32)
    b = np.zeros(L * H + n_actions + 1, np.float32)
    h = C.c_void_p()
    nat.check(nat.lib().orlg_policy_create_matrix(device, nodes, links, slots, H, L, n_actions, w.ctypes.data_as(C.c_void_p),
                                                  b.ctypes.data_as(C.c_void_p), C.byref(h)))
    return h


@pytest.mark.parametrize("nodes,links,slots,H,L,n_actions,match", [
    (14, 22, 100, 8, 2, 6, "hidden width"), (14, 22, 100, 72, 2, 6, "hidden width"), (14, 22, 100, 144, 2, 6, "hidden width"),
    (14, 22, 100, 64, 0, 6, "hidden layer"),
    (14, 22, 100, 64, 2, 0, "1..15 actions"), (14, 22, 100, 64, 2, 16, "1..15 actions"),
    (1, 22, 100, 64, 2, 6, "2..255 nodes"), (256, 22, 100, 64, 2, 6, "2..255 nodes"),
    (14, 22, 0, 64, 2, 6, "1..512 slots"), (14, 22, 513, 64, 2, 6, "1..512 slots"),
    (14, 0, 100, 64, 2, 6, "links"),
    (14, 22, 100, 128, 7, 6, "bytes of shared memory"),
])
def test_create_matrix_refusals(nodes, links, slots, H, L, n_actions, match):
    from optical_rl_gym_b200._native import NativeError

    with pytest.raises(NativeError, match=match):
        _create_matrix(nodes, links, slots, H, L, n_actions)


@pytest.mark.parametrize("layout,trunk", [((14, 22, 100), (2, 64)), ((14, 22, 100), (5, 128)), ((50, 88, 100), (2, 64)),
                                          ((20, 42, 512), (2, 128)), ((255, 1, 1), (1, 16))])
def test_accepted_matrix_shapes_reach_the_device_query(layout, trunk):
    from optical_rl_gym_b200._native import NativeError

    with pytest.raises(NativeError, match="no such CUDA device"):
        _create_matrix(*layout, trunk[1], trunk[0], 6)


def test_python_refusals():
    from optical_rl_gym_b200.policy import MlpPolicy

    layout = (14, 22, 100)
    with pytest.raises(ValueError, match="exclude"):
        MlpPolicy(2228, 6, (64, 64), wide_observations=True, matrix_observation=layout)
    with pytest.raises(ValueError, match="obs_dim is 2227"):
        MlpPolicy(2227, 6, (64, 64), matrix_observation=layout)
    sd = _sb3_state_dict(obs_dim=2228, n_actions=6, separate=True)
    pol = MlpPolicy.from_state_dict(sd, matrix_observation=layout)
    assert pol.matrix_observation == layout and pol.critic_net is not None
    with pytest.raises(ValueError, match="inputs"):
        MlpPolicy.from_state_dict(sd, matrix_observation=(14, 22, 64))
    with pytest.raises(ValueError, match="packed observations"):            # float rows, CPU rows: refused before any launch
        pol.act_native(torch.zeros((4, 2228)))
    with pytest.raises(ValueError, match="packed observations"):
        pol.sample_native(torch.zeros((4, words(*layout)), dtype=torch.int32), seed=1, counter=0)
    pol.wide_observations = True
    with pytest.raises(ValueError, match="exclude"):
        pol._native_handles(0)


def _matrix_policy(layout, L, H, n_actions=6, seed=0, device="cuda", critic=False):
    from optical_rl_gym_b200.policy import MlpPolicy

    nodes, links, slots = layout
    obs_dim = 2 * nodes + links * slots
    torch.manual_seed(seed)
    pol = MlpPolicy(obs_dim, n_actions, (H,) * L, matrix_observation=layout)
    with torch.no_grad():
        for m in pol.shared_net:
            if isinstance(m, torch.nn.Linear):
                torch.nn.init.orthogonal_(m.weight, gain=2 ** 0.5)
                m.bias.uniform_(-0.1, 0.1)
        torch.nn.init.orthogonal_(pol.action_net.weight, gain=1.0)
        if critic:
            pol.critic_net = torch.nn.Sequential(torch.nn.Linear(obs_dim, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh())
            pol.value_net = torch.nn.Linear(64, 1)
    return pol.to(device)


@pytest.mark.parametrize("bug", ["drop_link", "shift_link"])
def test_bf16_reference_catches_a_misplaced_layer0_block(bug):
    """A kernel that lost one link's block of layer 0, or read a link's columns one slot off, moves the logits on random
    bit rows by more than 10 x BF16_LOGIT_ATOL: the GPU comparison would see it."""
    layout = (14, 22, 100)
    pol = _matrix_policy(layout, 2, 64, device="cpu")
    rng = np.random.default_rng(3)
    x = torch.from_numpy(unpacked_np(*_random_rows(rng, 256, *layout), 14)).double()
    ref = bf16_reference(pol, x)
    l, off = 7, 28 + 7 * 100
    bad = x.clone()
    if bug == "drop_link":
        bad[:, off:off + 100] = 0
    else:
        bad[:, off:off + 100] = torch.roll(x[:, off:off + 100], 1, dims=1)
    moved = (bf16_reference(pol, bad) - ref).abs().max().item()
    assert moved > 10 * BF16_LOGIT_ATOL, (bug, l, moved)


# ------------------------------------------------------------------ GPU: packed rows
def _assert_packed_equals_matrix(env):
    packed = env.packed_matrix_observation()
    assert packed.dtype == torch.int32 and packed.shape == (env.num_envs, words(*env.matrix_layout))
    assert torch.equal(env.unpack_matrix_observation(packed), env.matrix_observation())
    S = env.num_spectrum_resources
    nwv = (S + 127) // 128
    w = packed[:, 4:].reshape(env.num_envs, env.tables.num_links, 4 * nwv).cpu().numpy().view(np.uint32)
    bits = np.unpackbits(w.view(np.uint8), axis=-1, bitorder="little")
    assert not bits[..., S:].any()                                      # bits at and above S are 0
    assert not packed[:, 1:4].any()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["wrap_rmsa_matrix_pathonly"])
def test_packed_rows_on_the_golden_run(name):
    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200.wrappers import PathOnlyFirstFitAction, SimpleMatrixObservation

    g = helpers.load_golden(name)
    meta = g["meta"]
    base = OpticalVecEnv(meta["kind"], meta["n_envs"], helpers.golden_tables(), traffic="trace", **meta["env_args"])
    base.set_trace(g["req_arrival"], g["req_holding"], g["req_src"], g["req_dst"], g["req_bit_rate"])
    env = PathOnlyFirstFitAction(SimpleMatrixObservation(base))
    base.reset(full=True)
    env.reset()
    for t in range(meta["T"] + 1):
        packed = env.packed_matrix_observation()                        # through the wrappers' attribute pass-through
        got = np.packbits(env.unpack_matrix_observation(packed).cpu().numpy(), axis=1, bitorder="little")
        assert np.array_equal(got, g["matrix_bits"][:, t]), t
        _assert_packed_equals_matrix(base)
        if t < meta["T"]:
            env.step(torch.as_tensor(g["path_action"][:, t], device="cuda"))
    base.close()


def _layout_env(which, n, kind="RMSA-v0", **kw):
    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200.topology import synthetic_ring_chords

    if which == "nsfnet":
        tables, args = helpers.golden_tables(), dict(num_spectrum_resources=kw.pop("slots", 100))
    elif which == "ring200":
        tables, args = synthetic_ring_chords(num_nodes=20, num_chords=22, k_paths=6, seed=11), dict(num_spectrum_resources=200)
    elif which == "ring512":
        tables, args = synthetic_ring_chords(num_nodes=20, num_chords=22, k_paths=4, seed=5), dict(num_spectrum_resources=512)
    else:
        from optical_rl_gym_b200.topology import TopologyTables

        tables = TopologyTables.load(os.path.join(helpers.GOLDEN_DIR, "topo_germany50_tables.npz"))
        args = dict(num_spectrum_resources=100)
    if kind == "RWA-v0":
        args = dict(num_spectrum_resources=args["num_spectrum_resources"])
    args.update(episode_length=10, load=kw.pop("load", 250), mean_service_holding_time=25)
    args.update(kw)
    return OpticalVecEnv(kind, n, tables, seed=SEED, env_id_base=BASE, **args)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["nsfnet", "ring200", "germany50", "ring512"])
@pytest.mark.parametrize("kind", ["RMSA-v0", "RWA-v0"])
def test_packed_rows_equal_matrix_observation(which, kind):
    env = _layout_env(which, 300, kind)
    assert env.kernel_info()["wide"] == (which != "nsfnet")               # both mask layouts
    _assert_packed_equals_matrix(env)
    env.rollout(17, "sp_ff" if kind == "RMSA-v0" else "sap_ff")
    _assert_packed_equals_matrix(env)
    env.close()


# ------------------------------------------------------------------ GPU: the kernel
def _random_packed(layout, n, seed):
    rng = np.random.default_rng(seed)
    src, dst, avail = _random_rows(rng, n, *layout, p=rng.uniform(0.2, 0.8))
    packed = torch.from_numpy(pack_np(src, dst, avail, layout[0])).cuda()
    return packed, torch.from_numpy(unpacked_np(src, dst, avail, layout[0])).cuda()


TRUNKS = [(1, 16), (2, 64), (2, 128), (5, 128)]
LAYOUTS = [(14, 22, 64), (14, 22, 100), (50, 88, 100), (20, 42, 512)]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("trunk", TRUNKS)
@pytest.mark.parametrize("n", [1, 127, 128, 129, 300])
def test_matrix_kernel_matches_bf16_reference(layout, trunk, n):
    pol = _matrix_policy(layout, *trunk, seed=n)
    packed, x = _random_packed(layout, n, seed=n + trunk[1])
    logits = torch.full((n, 7), float("nan"), device="cuda")
    act = pol.act_native(packed, logits=logits)
    ref = bf16_reference(pol, x.double())
    err = (logits.double() - ref).abs().max().item()
    assert err < BF16_LOGIT_ATOL, err
    assert torch.equal(act[:, 0].long(), logits[:, :6].argmax(-1))
    top2 = ref[:, :6].topk(2, dim=-1).values
    clear = (top2[:, 0] - top2[:, 1]) > 2 * BF16_LOGIT_ATOL
    assert torch.equal(act[clear, 0].long(), ref[clear, :6].argmax(-1))


@pytest.mark.gpu
@pytest.mark.parametrize("layout,trunk", [((14, 22, 100), (2, 64)), ((14, 22, 100), (5, 128)), ((50, 88, 100), (2, 64))])
def test_matrix_sampling_matches_the_reference_sampler(layout, trunk):
    n = 4096
    pol = _matrix_policy(layout, *trunk, seed=7)
    with torch.no_grad():
        pol.action_net.weight.mul_(0.3)
    packed, x = _random_packed(layout, n, seed=11)
    a, lp, v = pol.sample_native(packed, seed=123, counter=9, row_id_base=77)
    ref = bf16_reference(pol, x.double()).cpu().numpy()
    u = draw_u(123, 9, 77 + np.arange(n, dtype=np.uint64))
    want, cdf = reference_sample(ref[:, :6], u)
    got = a[:, 0].cpu().numpy()
    clear = (np.abs(u[:, None] - cdf[:, :-1]) > 0.041).all(-1)
    assert clear.mean() > 0.5 and np.array_equal(got[clear], want[clear])
    assert np.abs(v.cpu().numpy() - ref[:, 6]).max() < BF16_LOGIT_ATOL
    logits = torch.empty((n, 7), device="cuda")
    act = pol.act_native(packed, logits=logits)
    da, dlp, dv = pol.sample_native(packed, seed=123, counter=9, deterministic=True)
    assert torch.equal(da, act) and torch.equal(dv, logits[:, 6])
    own = torch.log_softmax(logits[:, :6].double(), -1).gather(1, a.long())[:, 0]
    assert (lp.double() - own).abs().max().item() < 1e-5
    with pytest.raises(ValueError, match="masked"):
        pol.sample_native(packed, seed=1, counter=0, action_masks=torch.ones((n, 6), dtype=torch.bool, device="cuda"))
    with pytest.raises(ValueError, match="packed"):
        pol.act_native(x.float())
    with pytest.raises(ValueError, match="packed"):
        pol.act_native(torch.zeros((n, packed.shape[1] + 4), dtype=torch.int32, device="cuda")[:, 1:-3])


# ------------------------------------------------------------------ GPU: the closed loop
def _twin_loop(env, pol, T, deterministic):
    """rollout_policy as a Python loop: packed_matrix_observation + sample_native + path_only_first_fit + step_raw."""
    obs = [env.packed_matrix_observation().clone()]
    acts, lps, vals, rews, dones = [], [], [], [], []
    for _ in range(T):
        a, lp, v = pol.sample_native(obs[-1], seed=SEED, counter=env.request_index, row_id_base=BASE, deterministic=deterministic)
        _, r, d = env.step_raw(env.path_only_first_fit(a[:, 0]))
        obs.append(env.packed_matrix_observation().clone())
        acts.append(a[:, 0].clone()); lps.append(lp); vals.append(v); rews.append(r.clone()); dones.append(d.clone())
    vals.append(pol.sample_native(obs[-1], seed=SEED, counter=env.request_index, row_id_base=BASE)[2])
    return [torch.stack(x) for x in (obs, acts, lps, vals, rews, dones)]


def _state(env):
    m, _, now, nheap = env.export_state()
    return [env.counters(), m, now, nheap, env.error_flags()]


def _assert_same(got, want):
    for name, g, w in zip(("obs", "actions", "log_prob", "value", "reward", "done"), got, want):
        assert torch.equal(g, w), name


def _loop_policy(env, critic=False, L=2, H=64, seed=0):
    pol = _matrix_policy(env.matrix_layout, L, H, n_actions=env.k_paths + env.reject_action, seed=seed, critic=critic)
    with torch.no_grad():
        pol.action_net.weight.mul_(0.3)
    return pol


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["RMSA-v0", "RWA-v0"])
@pytest.mark.parametrize("which", ["nsfnet", "ring200"])
@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("critic", [False, True])
def test_matrix_rollout_policy_equals_the_python_loop(kind, which, deterministic, critic):
    n, T = 300, 24
    env, twin = _layout_env(which, n, kind, allow_rejection=True), _layout_env(which, n, kind, allow_rejection=True)
    pol = _loop_policy(env, critic=critic)
    ro, info = env.rollout_policy(pol, T, deterministic=deterministic, want_info=True)
    assert ro.obs.dtype == torch.int32 and ro.obs.shape == (T + 1, n, words(*env.matrix_layout))
    want = _twin_loop(twin, pol, T, deterministic)
    _assert_same(ro, want)
    assert int(ro.done.sum()) > 0 and (deterministic or len(torch.unique(ro.actions)) > 1)
    for g, w in zip(_state(env), _state(twin)):
        assert torch.equal(g, w)
    assert env.request_index == twin.request_index
    for key in info.keys():
        assert info[key].shape[:2] == (T, n), key
    assert int(env.error_flags().abs().sum()) == 0
    env.close(); twin.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["RMSA-v0", "RWA-v0"])
def test_matrix_rollout_info_equals_step_info(kind):
    n, T = 200, 12
    env, twin = _layout_env("nsfnet", n, kind), _layout_env("nsfnet", n, kind)
    pol = _loop_policy(env)
    ro, info = env.rollout_policy(pol, T, want_info=True)
    obs = twin.packed_matrix_observation()
    for t in range(T):
        a = pol.sample_native(obs, seed=SEED, counter=twin.request_index, row_id_base=BASE)[0]
        obs_, r, d, tinfo = twin.step(twin.path_only_first_fit(a[:, 0]))
        obs = twin.packed_matrix_observation()
        for key in tinfo.keys():
            assert torch.equal(info[key][t], tinfo[key]), (key, t)
    env.close(); twin.close()


@pytest.mark.gpu
def test_matrix_rollout_split_checkpoint_and_monitor():
    from optical_rl_gym_b200.monitor import VecMonitor

    n = 257
    a, b, c = (_layout_env("nsfnet", n, "RMSA-v0") for _ in range(3))
    pol = _loop_policy(a, critic=True)
    one = a.rollout_policy(pol, 20)
    first = b.rollout_policy(pol, 8)
    sd = b.state_dict()
    c.load_state_dict(sd)
    second = c.rollout_policy(pol, 12)
    assert torch.equal(one.obs[:9], first.obs) and torch.equal(one.obs[8:], second.obs)
    assert torch.equal(one.actions, torch.cat([first.actions, second.actions]))
    assert torch.equal(one.log_prob, torch.cat([first.log_prob, second.log_prob]))
    assert torch.equal(one.reward, torch.cat([first.reward, second.reward]))
    mon_env, loop_env = _layout_env("nsfnet", n, "RWA-v0"), _layout_env("nsfnet", n, "RWA-v0")
    pol2 = _loop_policy(mon_env, seed=4)
    mon = VecMonitor(mon_env)
    ro = mon.rollout_policy(pol2, 30)
    loop = VecMonitor(loop_env)
    obs = loop_env.packed_matrix_observation()
    for t in range(30):
        act = pol2.sample_native(obs, seed=SEED, counter=loop_env.request_index, row_id_base=BASE)[0]
        loop.step(loop_env.path_only_first_fit(act[:, 0]))
        obs = loop_env.packed_matrix_observation()
        assert torch.equal(act[:, 0], ro.actions[t])
    assert mon.episode_returns == loop.episode_returns and mon.episode_lengths == loop.episode_lengths
    assert len(mon.episode_returns) > 0
    for e in (a, b, c, mon_env, loop_env):
        e.close()


@pytest.mark.gpu
def test_sb3_zip_drives_the_loop(tmp_path):
    from optical_rl_gym_b200.policy import MlpPolicy

    env, twin = _layout_env("nsfnet", 128, "RMSA-v0"), _layout_env("nsfnet", 128, "RMSA-v0")
    k1 = env.k_paths + env.reject_action
    g = torch.Generator().manual_seed(2)
    sd = {}
    for t in ("policy_net", "value_net"):
        d = 2228
        for i in range(2):
            sd["mlp_extractor.%s.%d.weight" % (t, 2 * i)] = torch.randn(64, d, generator=g) / d ** 0.5
            sd["mlp_extractor.%s.%d.bias" % (t, 2 * i)] = torch.randn(64, generator=g) * 0.1
            d = 64
    sd["action_net.weight"] = torch.randn(k1, 64, generator=g) * 0.1
    sd["action_net.bias"] = torch.zeros(k1)
    sd["value_net.weight"] = torch.randn(1, 64, generator=g) * 0.1
    sd["value_net.bias"] = torch.full((1,), 0.25)
    buf = io.BytesIO()
    torch.save(sd, buf)
    path = tmp_path / "ppo_rmsa.zip"
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
    pol = MlpPolicy.from_sb3_zip(path, device="cuda", matrix_observation=env.matrix_layout)
    assert pol.action_net.out_features == k1 and pol.critic_net is not None
    ro = env.rollout_policy(pol, 16)
    _assert_same(ro, _twin_loop(twin, pol, 16, False))
    # forward on unpacked rows is the float32 reference of the same policy
    logits, value = pol(env.unpack_matrix_observation(ro.obs[3], torch.float32))
    assert (value - ro.value[3]).abs().max().item() < 0.06
    env.close(); twin.close()


@pytest.mark.gpu
def test_matrix_rollout_refusals():
    from optical_rl_gym_b200 import OpticalVecEnv
    from optical_rl_gym_b200 import _native as nat
    from optical_rl_gym_b200.policy import MlpPolicy

    env = _layout_env("nsfnet", 8, "RMSA-v0")
    pol = _loop_policy(env)
    deep = OpticalVecEnv("DeepRMSA-v0", 8, helpers.golden_tables(), seed=1)
    with pytest.raises(nat.NativeError, match="matrix-observation policy"):
        deep.rollout_policy(pol, 2)
    rmcsa = OpticalVecEnv("RMCSA-v0", 8, helpers.golden_tables(), seed=1, num_spectrum_resources=64)
    with pytest.raises(nat.NativeError, match="DeepRMSA-v0"):
        rmcsa.rollout_policy(pol, 2)
    assert rmcsa._lib.orlg_matrix_obs_words(rmcsa._h) == 0
    buf = torch.empty((8, 4), dtype=torch.int32, device="cuda")
    with pytest.raises(nat.NativeError, match="packed matrix observations exist"):
        nat.check(rmcsa._lib.orlg_matrix_observation_packed(rmcsa._h, C.c_void_p(buf.data_ptr()), None))
    plain = MlpPolicy(54, 6, (64, 64)).cuda()
    with pytest.raises(nat.NativeError, match="DeepRMSA-v0"):
        env.rollout_policy(plain, 2)
    other = _matrix_policy((14, 22, 64), 2, 64, n_actions=env.k_paths + env.reject_action)
    with pytest.raises(nat.NativeError, match="actor matrix layout"):
        env.rollout_policy(other, 2)
    wrong_n = _matrix_policy(env.matrix_layout, 2, 64, n_actions=env.k_paths + env.reject_action + 1)
    with pytest.raises(nat.NativeError, match="n_actions"):
        env.rollout_policy(wrong_n, 2)
    actor = _loop_policy(env)._native_handles(0)[0]
    crit_other = _matrix_policy((14, 22, 64), 2, 64, n_actions=1)._native_handles(0)[0]
    with pytest.raises(nat.NativeError, match="critic matrix layout"):
        nat.check(nat.lib().orlg_rollout_policy(env._h, 1, actor, crit_other, 1, 0, None, None, None, None, None, None, None))
    with pytest.raises(nat.NativeError, match="DeepRMSA-v0"):
        env.rollout_policy(pol, 2, action_masks=True)
    for e in (env, deep, rmcsa):
        e.close()
