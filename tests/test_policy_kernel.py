"""The fused tensor-core policy kernel (orlg_policy_act: bf16 tcgen05.mma, TMEM accumulators) against two references.

* The plain PyTorch float32 forward of the same MLP.  The operands are rounded to bf16 (8-bit mantissa) in every one of
  the six layers and tanh is the hardware approximation, so logits agree to a few 1e-2 absolute; the action (argmax)
  must be identical wherever the float32 top-2 margin exceeds twice that tolerance.
* A float64 forward with the kernel's roundings (bf16_reference): weights and every layer's input rounded to bf16 (round
  to nearest even, like the weight packing and __floats2bfloat162_rn), exact tanh.  What is left is tanh.approx and the
  fp32 accumulation order, so the tolerance is three times tighter; a CPU test shows that it still catches the kernel
  bugs one would expect (a lost K block, a shifted bias, swapped output rows)."""
import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

LOGIT_ATOL = 0.06          # against the float32 forward
# Against bf16_reference.  Measured on an NVIDIA B200 (1000 W power limit): over real DeepRMSA observations (54 and 64 wide,
# 129 and 65536 envs, three weight seeds) and the shape limits below, the largest logit / value error was 9.4e-3 (mean
# 2.4e-4): a tanh.approx result on the other side of a bf16 rounding boundary, carried through the later layers.  The same
# runs differ from the float32 forward by up to 1.7e-2.
BF16_LOGIT_ATOL = 0.02


def _policy(seed=0, obs_dim=54, n_actions=5, device="cuda"):
    from optical_rl_gym_b200.policy import MlpPolicy

    torch.manual_seed(seed)
    pol = MlpPolicy(obs_dim, n_actions, (128,) * 5).to(device)
    with torch.no_grad():                       # weights at the scale of a trained SB3 policy (orthogonal init, gain sqrt(2) / 0.01)
        for m in pol.shared_net:
            if isinstance(m, torch.nn.Linear):
                torch.nn.init.orthogonal_(m.weight, gain=2 ** 0.5)
                m.bias.uniform_(-0.1, 0.1)
        torch.nn.init.orthogonal_(pol.action_net.weight, gain=1.0)
    return pol


def _bf16(x):
    """Round to the nearest bf16 (ties to even) through float32, as the kernel rounds its float32 values; float64 result."""
    return x.to(torch.float32).to(torch.bfloat16).to(torch.float64)


@torch.no_grad()
def bf16_reference(pol, obs, bug=None):
    """float64 forward with the fused kernel's roundings -> [n, n_actions + 1] (logits, then value).  `bug` applies a known
    defect to the reference itself: "drop_k_block" (layer 0 loses the last 16-wide K block of the padded 64), "shift_bias"
    (every bias read one column late), "swap_value" (the value row and the last logit row of the output layer swapped)."""
    lins = [m for m in pol.shared_net if isinstance(m, torch.nn.Linear)]
    h = _bf16(obs)
    for i, lin in enumerate(lins):
        w, b = _bf16(lin.weight).clone(), lin.bias.to(torch.float64)
        if bug == "drop_k_block" and i == 0:
            w[:, 48:] = 0.0
        if bug == "shift_bias":
            b = torch.roll(b, 1)
        h = _bf16(torch.tanh(h @ w.T + b))
    w = _bf16(torch.cat([pol.action_net.weight, pol.value_net.weight])).clone()
    b = torch.cat([pol.action_net.bias, pol.value_net.bias]).to(torch.float64)
    if bug == "shift_bias":
        b = torch.roll(b, 1)
    if bug == "swap_value":
        na = pol.action_net.out_features
        w[[na - 1, na]] = w[[na, na - 1]]
        b[[na - 1, na]] = b[[na, na - 1]]
    return h @ w.T + b


def _oracle_observations(j, n=96, seed=4):
    """Real DeepRMSA observations of partly filled NSFNET networks (j = 1: 54 wide, j = 2: 64) from the C oracle."""
    from oracle import oracle

    tables = helpers.golden_tables()
    rows = []
    for i in range(n):
        o = oracle.OracleEnv("DeepRMSA-v0", tables, num_slots=100, episode_length=1000, j=j)
        o.set_philox(seed, i)
        o.reset(full=True)
        o.rollout(20 + i, policy=1)
        rows.append(o.observation())
    return torch.tensor(np.array(rows))


@pytest.mark.parametrize("j", [1, 2])
def test_bf16_reference_tolerance_catches_kernel_bugs(j):
    """The defects a packing or epilogue bug of the kernel would cause, applied to the reference: each moves the logits by
    many times BF16_LOGIT_ATOL, so the GPU comparison would fail on them.  (No GPU: oracle observations, CPU weights.)"""
    bits = np.random.default_rng(0).standard_normal(4096).astype(np.float32)
    u = bits.view(np.uint32).astype(np.uint64)
    rne = (((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16).astype(np.uint32).view(np.float32)      # f32_to_bf16 of orlg_api.cu
    assert np.array_equal(_bf16(torch.from_numpy(bits)).numpy(), rne.astype(np.float64))
    obs = _oracle_observations(j)
    assert obs.shape[1] == (54 if j == 1 else 64)
    pol = _policy(obs_dim=obs.shape[1], device="cpu")
    ref = bf16_reference(pol, obs)
    for bug in ("drop_k_block", "shift_bias", "swap_value"):
        moved = (bf16_reference(pol, obs, bug) - ref).abs().max().item()
        assert moved > 10 * BF16_LOGIT_ATOL, (bug, moved)


def test_policy_create_refuses_shapes_outside_the_kernel():
    """Odd or > 64 observation widths and more than 15 actions do not fit the kernel's operand layout: refused up front."""
    from optical_rl_gym_b200._native import NativeError

    for obs_dim, n_actions in ((53, 5), (66, 5), (54, 16)):
        pol = _policy(obs_dim=obs_dim, n_actions=n_actions, device="cpu")
        with pytest.raises(NativeError, match="fused policy kernel"):
            pol._native_handle(0)


def _check_against_bf16_reference(pol, obs, n_actions):
    logits = torch.full((obs.shape[0], n_actions + 1), float("nan"), dtype=torch.float32, device="cuda")
    act = pol.act_native(obs, logits=logits)
    ref = bf16_reference(pol, obs.double())
    torch.cuda.synchronize()
    err = (logits.double() - ref).abs().max().item()
    assert err < BF16_LOGIT_ATOL, err
    assert torch.equal(act[:, 0].long(), logits[:, :n_actions].argmax(-1))
    top2 = ref[:, :n_actions].topk(min(2, n_actions), dim=-1).values
    clear = (top2[:, 0] - top2[:, -1]) > 2 * BF16_LOGIT_ATOL if n_actions > 1 else torch.ones_like(top2[:, 0], dtype=torch.bool)
    assert torch.equal(act[clear, 0].long(), ref[clear, :n_actions].argmax(-1))
    return err


@pytest.mark.gpu
@pytest.mark.parametrize("j", [1, 2])
@pytest.mark.parametrize("n", [1, 127, 129, 65536])
def test_fused_policy_kernel_matches_bf16_reference(j, n):
    """Real DeepRMSA observations, 54 wide (j = 1) and 64 wide (j = 2: the 16 KB staging area of the vectorised load is
    full and layer 0 uses all four K blocks)."""
    from optical_rl_gym_b200 import OpticalVecEnv

    env = OpticalVecEnv("DeepRMSA-v0", n, helpers.golden_tables(), seed=4, j=j)
    obs = env.rollout(30)[0][-1].clone()                      # own allocation: 16-byte aligned rows, the staged load path
    assert obs.shape[1] == (54 if j == 1 else 64) and obs.data_ptr() % 16 == 0
    _check_against_bf16_reference(_policy(obs_dim=obs.shape[1]), obs, 5)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("obs_dim,n_actions", [(54, 1), (54, 15), (2, 5), (64, 15)])
def test_fused_policy_kernel_at_the_shape_limits(obs_dim, n_actions):
    """The smallest and largest shapes orlg_policy_create accepts, on uniform random observations (n = 300: a ragged tile)."""
    gen = torch.Generator(device="cuda").manual_seed(obs_dim * 100 + n_actions)
    obs = torch.rand((300, obs_dim), generator=gen, device="cuda") * 2 - 1
    _check_against_bf16_reference(_policy(seed=n_actions, obs_dim=obs_dim, n_actions=n_actions), obs, n_actions)


@pytest.mark.gpu
@pytest.mark.parametrize("obs_dim", [54, 64])
def test_unaligned_observations_take_the_scalar_load_path_bit_for_bit(obs_dim):
    """Rows that do not start on a 16-byte boundary are read by the kernel's per-thread float2 loads instead of the staged
    16-byte loads: the same bf16 operands, so actions and logits equal those of the aligned batch bit for bit."""
    n = 1000
    gen = torch.Generator(device="cuda").manual_seed(obs_dim)
    buf = torch.rand(n * obs_dim + 2, generator=gen, device="cuda") * 2 - 1
    obs = buf[:n * obs_dim].view(n, obs_dim).clone()
    if obs_dim == 54:
        sub = obs[1:]                                             # 216-byte offset
        want = slice(1, None)
    else:
        buf[2:].view(-1)[:n * obs_dim].copy_(obs.view(-1))        # the same rows starting 8 bytes into the buffer
        sub = buf[2:2 + n * obs_dim].view(n, obs_dim)
        want = slice(None)
    assert sub.is_contiguous() and sub.data_ptr() % 16 != 0
    pol = _policy(obs_dim=obs_dim)
    la = torch.empty((n, 6), dtype=torch.float32, device="cuda")
    lb = torch.empty((sub.shape[0], 6), dtype=torch.float32, device="cuda")
    aa, ab = pol.act_native(obs, logits=la), pol.act_native(sub, logits=lb)
    assert torch.equal(aa[want], ab) and torch.equal(la[want], lb)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129, 5000, 65536])
def test_fused_policy_kernel_matches_float32_forward(n):
    from optical_rl_gym_b200 import OpticalVecEnv

    pol = _policy()
    env = OpticalVecEnv("DeepRMSA-v0", n, helpers.golden_tables(), seed=4)
    obs = env.rollout(30)[0][-1].contiguous()              # real observations of a partly filled network
    logits = torch.empty((n, 6), dtype=torch.float32, device="cuda")
    act = pol.act_native(obs, logits=logits)
    ref_logits, ref_value = pol(obs)
    torch.cuda.synchronize()
    err = (logits[:, :5] - ref_logits).abs().max().item()
    assert err < LOGIT_ATOL, err
    assert (logits[:, 5] - ref_value).abs().max().item() < LOGIT_ATOL
    top2 = ref_logits.topk(2, dim=-1).values
    clear = (top2[:, 0] - top2[:, 1]) > 2 * LOGIT_ATOL
    assert torch.equal(act[clear, 0].long(), ref_logits.argmax(-1)[clear])
    assert torch.equal(act[:, 0].long(), logits[:, :5].argmax(-1))          # the action IS the argmax of the kernel's own logits
    if n >= 5000:
        assert (act[:, 0].long() == ref_logits.argmax(-1)).float().mean().item() > 0.97
    env.close()


@pytest.mark.gpu
def test_policy_drives_the_env_like_the_notebook_loop():
    """obs -> fused policy -> env.step, 50 steps: same trajectory as the float32 torch policy wherever its argmax is clear
    (checked by stepping a twin env with the kernel's actions and comparing rewards with an oracle-free invariant)."""
    from optical_rl_gym_b200 import OpticalVecEnv

    pol = _policy(1)
    n = 4096
    env = OpticalVecEnv("DeepRMSA-v0", n, helpers.golden_tables(), seed=9, episode_length=40)
    obs = env.reset()
    acc = 0
    for t in range(50):
        a = pol.act_native(obs.contiguous())
        assert int(a.min()) >= 0 and int(a.max()) <= 4
        obs, reward, done, info = env.step(a)
        acc += int((reward > 0).sum())
    assert int(env.error_flags().abs().sum()) == 0
    assert acc > 0.3 * n * 50
    env.close()
