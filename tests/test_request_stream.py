"""The end of a recorded trace on every step-kernel family, and the trace bit-rate cap of the persistent rollout kernel.

Past the end of its trace an env keeps stepping on the request (now, holding 0, node 0 -> node 1) with ORLG_ERR_TRACE_EXHAUSTED
set.  Its bit rate is the lower bound of the bit-rate range, except on the persistent RWA rollout, where requests carry none.
Each case asserts through kernel_info() which kernel ran."""
import numpy as np
import pytest

import helpers

torch = pytest.importorskip("torch")

ERR_TRACE_EXHAUSTED, ERR_TRACE_RANGE = 1, 32
N_ENVS, TRACE_LEN, STEPS = 64, 6, 10
BR_LO = 25                        # bit_rate_lower_bound's default


def _trace(kind, n, length, seed, bit_rate=None):
    """Seeded requests [n, length] on NSFNET: increasing arrivals, short holding times, src != dst."""
    rng = np.random.default_rng(seed)
    arrival = np.cumsum(rng.exponential(0.1, size=(n, length)), axis=1)
    holding = rng.exponential(1.0, size=(n, length))
    src = rng.integers(0, 14, size=(n, length)).astype(np.int32)
    dst = ((src + rng.integers(1, 14, size=(n, length))) % 14).astype(np.int32)
    if bit_rate is None:
        bit_rate = np.zeros((n, length), np.int32) if kind == "RWA-v0" else rng.integers(25, 101, size=(n, length)).astype(np.int32)
    return arrival, holding, src, dst, bit_rate


def _env(kind, n, trace, **args):
    from optical_rl_gym_b200 import OpticalVecEnv

    env = OpticalVecEnv(kind, n, helpers.golden_tables(), traffic="trace", seed=5, **args)
    env.set_trace(*trace)
    env.reset(full=True)
    return env


def _assert_exhausted(env, trace, bit_rate):
    flags = env.error_flags().cpu().numpy()
    assert np.all(flags == ERR_TRACE_EXHAUSTED), flags
    req, _ = env.current_requests()
    assert np.array_equal(req["arrival"], trace[0][:, -1])          # the clock stays at the last recorded arrival
    assert np.all(req["holding"] == 0.0)
    assert np.all(req["src"] == 0) and np.all(req["dst"] == 1)
    assert np.all(req["bit_rate"] == bit_rate), req["bit_rate"]


# name -> (kind, env_args, which kernel: "generic" step_kernel, "wide" step_wide_kernel, "fast" deeprmsa_fast_kernel)
PER_STEP = {
    "rmsa_generic": ("RMSA-v0", dict(num_spectrum_resources=64), "generic"),
    "rmsa_wide": ("RMSA-v0", dict(num_spectrum_resources=160), "wide"),
    "deeprmsa_fast": ("DeepRMSA-v0", dict(), "fast"),
    "rwa_generic": ("RWA-v0", dict(num_spectrum_resources=16), "generic"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PER_STEP))
def test_exhausted_trace_per_step(name):
    """orlg_step past the end of the trace: the flag and the fallback request, on each per-step kernel family."""
    kind, args, kernel = PER_STEP[name]
    trace = _trace(kind, N_ENVS, TRACE_LEN, seed=3)
    env = _env(kind, N_ENVS, trace, **args)
    info = env.kernel_info()
    assert info["wide"] == (kernel == "wide") and info["fast"] == (kernel == "fast"), info
    for t in range(STEPS):
        env.step(env.sample_actions())
        if t == TRACE_LEN - 2:                                           # the last recorded request is pending
            assert int(env.error_flags().abs().sum()) == 0
    _assert_exhausted(env, trace, BR_LO)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["DeepRMSA-v0", "RMSA-v0", "RWA-v0"])
def test_exhausted_trace_rollout(kind):
    """The persistent rollout kernel replaying given actions past the end of the trace."""
    trace = _trace(kind, N_ENVS, TRACE_LEN, seed=4)
    args = dict(num_spectrum_resources=16) if kind == "RWA-v0" else {}
    env = _env(kind, N_ENVS, trace, **args)
    info = env.kernel_info()
    assert info["rollout_kernel"] and not info["wide"], info
    rng = np.random.default_rng(6)
    actions = rng.integers(0, 5, size=(STEPS, N_ENVS, env.action_dim)).astype(np.int32)
    if kind != "DeepRMSA-v0":
        actions[..., 1] = rng.integers(0, env.num_spectrum_resources, size=(STEPS, N_ENVS))
    env.rollout(STEPS, "replay", actions=torch.as_tensor(actions, device="cuda"))
    assert env.kernel_info()["last_rollout_persistent"]
    _assert_exhausted(env, trace, 0 if kind == "RWA-v0" else BR_LO)
    env.close()


@pytest.mark.gpu
def test_rollout_caps_trace_bit_rates_at_127():
    """A recorded bit rate above 127 Gb/s reaches the persistent kernel as 127 with ORLG_ERR_TRACE_RANGE set."""
    kind, T = "RMSA-v0", 4
    n = N_ENVS
    bit_rate = np.full((n, T + 2), 100, np.int32)
    bit_rate[:, T] = 200                                                 # the request pending after T steps
    trace = _trace(kind, n, T + 2, seed=7, bit_rate=bit_rate)
    env = _env(kind, n, trace)
    assert env.kernel_info()["rollout_kernel"]
    actions = np.full((T, n, 2), 5, np.int32)                            # path 5 of k = 5: rejected, nothing provisioned
    env.rollout(T, "replay", actions=torch.as_tensor(actions, device="cuda"))
    assert env.kernel_info()["last_rollout_persistent"]
    flags = env.error_flags().cpu().numpy()
    assert np.all(flags == ERR_TRACE_RANGE), flags
    req, _ = env.current_requests()
    assert np.all(req["bit_rate"] == 127), req["bit_rate"]
    assert np.array_equal(req["arrival"], trace[0][:, T])
    env.close()
