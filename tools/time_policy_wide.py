"""Cost of the wide policy kernel (MlpPolicy(wide_observations=True), orlg_policy_create_wide), 65536 rows:
  * narrow against wide instance at obs_dim 54 (one chunk: the cost of opting in), 5 x 128 and 2 x 64;
  * the wide instance at obs_dim 126 and 251 for 2 x 64 (two tile groups), and 5 x 128 at 126 (one tile group);
  * rollout_policy per step on DeepRMSA-v0 germany50 (126 inputs, wide step kernels), SB3's default agent (actor 2 x 64 and
    a separate critic 2 x 64), masked and unmasked.
Kernel timings are sample_native calls (the sampling epilogue rollout_policy runs) on uniform random observations: the kernel's
work does not depend on the values.  CUDA events behind a queued torch.cuda._sleep, the median of 7 repetitions of K calls
after a warm-up call; the variants of a line alternate, twice.  Prints the GPU name and power limit beside the numbers, and
the time it takes just to read the observations at 7.7 TB/s (a floor, not a prediction)."""
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "optical-rl-gym_b200")):
    sys.path.insert(0, p)
import torch

from optical_rl_gym_b200 import OpticalVecEnv
from optical_rl_gym_b200 import _native as nat
from optical_rl_gym_b200.policy import MlpPolicy
from optical_rl_gym_b200.topology import TopologyTables

N = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
T, K, REPS, ROUNDS = 64, 200, 7, 2
HBM_BPS = 7.7e12


def policy(L, H, obs_dim, wide, critic=False, n_actions=5):
    torch.manual_seed(L * 1000 + H)
    pol = MlpPolicy(obs_dim, n_actions, (H,) * L, wide_observations=wide)
    for m in pol.shared_net:
        if isinstance(m, torch.nn.Linear):
            torch.nn.init.orthogonal_(m.weight, gain=2 ** 0.5)
    if critic:                      # SB3 >= 1.8 layout: a separate critic trunk of the same shape
        layers = []
        for i in range(L):
            lin = torch.nn.Linear(obs_dim if i == 0 else H, H)
            torch.nn.init.orthogonal_(lin.weight, gain=2 ** 0.5)
            layers += [lin, torch.nn.Tanh()]
        pol.critic_net = torch.nn.Sequential(*layers)
    return pol.cuda()


def timed(fn, reps=REPS):
    """median over `reps` of the device time of one fn() in us (CUDA events, queued behind a sleep so the host runs ahead)."""
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(20_000_000)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) * 1e3)
    return statistics.median(out)


def per_call(pol, obs, bufs):
    return timed(lambda: [pol.sample_native(obs, seed=1, counter=i, out=bufs) for i in range(K)]) / K


def main():
    assert torch.cuda.is_available(), "needs a CUDA device"
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        gpu = torch.cuda.get_device_name()
    print("GPU: %s; %d rows, median of %d, %d alternating rounds" % (gpu, N, REPS, ROUNDS))
    gen = torch.Generator(device="cuda").manual_seed(0)
    obs = {d: torch.rand((N, d), generator=gen, device="cuda") * 2 - 1 for d in (54, 126, 251)}
    bufs = (torch.empty((N, 1), dtype=torch.int32, device="cuda"), torch.empty(N, device="cuda"), torch.empty(N, device="cuda"))
    pairs = [(L, H, policy(L, H, 54, False), policy(L, H, 54, True)) for L, H in ((5, 128), (2, 64))]
    wides = [(2, 64, 126), (2, 64, 251), (5, 128, 126)]
    wide_pols = [(L, H, d, policy(L, H, d, True)) for L, H, d in wides]
    for rnd in range(ROUNDS):
        print("-- round %d" % rnd)
        for L, H, narrow, wide in pairs:
            a = per_call(narrow, obs[54], bufs)
            b = per_call(wide, obs[54], bufs)
            print("obs 54, %d x %-3d  narrow %8.2f  wide %8.2f us/call  (%+.1f %%)" % (L, H, a, b, 100.0 * (b / a - 1.0)))
        for L, H, d, pol in wide_pols:
            g = nat.lib().orlg_policy_tile_groups(pol._native_handle(0))
            t = per_call(pol, obs[d], bufs)
            print("obs %d, %d x %-3d wide (%d tile group%s) %8.2f us/call; reading the observations at %.1f TB/s: %.2f us" % (
                d, L, H, g, "s" if g > 1 else "", t, HBM_BPS / 1e12, N * d * 4 / HBM_BPS * 1e6))
    g50 = TopologyTables.load(os.path.join(ROOT, "tests", "golden", "topo_germany50_tables.npz"))
    env = OpticalVecEnv("DeepRMSA-v0", N, g50, seed=1, collect_info=False, episode_length=1000)
    env.rollout(200, "sap_ff", want_obs=False, want_actions=False)
    pol = policy(2, 64, env.obs_dim, True, critic=True)
    buf = env.rollout_policy(pol, T)
    mask = env.action_masks()
    print("germany50 (obs %d, %d envs, 200 fill steps): rows with an invalid action %.4f" % (
        env.obs_dim, N, (~mask).any(1).float().mean().item()))
    for rnd in range(ROUNDS):
        plain = timed(lambda: env.rollout_policy(pol, T, out=buf)) / T
        masked = timed(lambda: env.rollout_policy(pol, T, out=buf, action_masks=True)) / T
        print("round %d: rollout_policy SB3 default actor 2 x 64 + critic 2 x 64  unmasked %8.2f  masked %8.2f us/step" % (
            rnd, plain, masked))
    print("germany50 error flags:", int((env.error_flags() != 0).sum()))
    env.close()


if __name__ == "__main__":
    main()
