"""The fused policy kernel across trunk architectures, at the headline configuration (DeepRMSA-v0 NSFNET, 250 Erlang, 65536
envs, 1000 fill steps: real observations, 54 wide):
  * orlg_policy_act and orlg_policy_sample (sampled actions) per architecture (L hidden layers of width H), us per 65536 rows;
  * rollout_policy in us per step for the SB3-default PPO agent (separate actor and critic trunks of 2 x 64: actor, critic
    and env launches per step) and for the shipped agent (one 5 x 128 trunk: policy and env launches per step).
CUDA events behind a queued torch.cuda._sleep, the median of 7 repetitions after a warm-up call.  Prints the GPU name and
power limit beside the numbers."""
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "optical-rl-gym_b200")):
    sys.path.insert(0, p)
import torch

from optical_rl_gym_b200 import OpticalVecEnv, nsfnet
from optical_rl_gym_b200.policy import MlpPolicy

N = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
ARCHS = [(2, 64), (2, 128), (4, 64), (8, 64), (6, 112), (5, 128)]      # (hidden layers, width)
T, K, REPS = 64, 200, 7


def policy(L, H, obs_dim=54, n_actions=5, critic=False):
    torch.manual_seed(L * 1000 + H)
    pol = MlpPolicy(obs_dim, n_actions, (H,) * L)
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


def main():
    assert torch.cuda.is_available(), "needs a CUDA device"
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        gpu = torch.cuda.get_device_name()
    print("GPU: %s; DeepRMSA-v0 NSFNET 250 E, %d envs, 1000 fill steps, median of %d" % (gpu, N, REPS))
    env = OpticalVecEnv("DeepRMSA-v0", N, nsfnet(), seed=1, collect_info=False, episode_length=1000)
    env.rollout(1000, want_obs=False, want_actions=False)
    obs = env.observation().contiguous()
    act = torch.empty((N, 1), dtype=torch.int32, device="cuda")
    lp, val = torch.empty(N, device="cuda"), torch.empty(N, device="cuda")
    print("%-8s %10s %10s %12s %9s" % ("L x H", "act us", "sample us", "GFLOP/call", "TFLOP/s"))
    for L, H in ARCHS:
        pol = policy(L, H)

        def act_only():
            for _ in range(K):
                pol.act_native(obs, out=act)

        def sample_only():
            for i in range(K):
                pol.sample_native(obs, seed=1, counter=i, out=(act, lp, val))

        ta, ts = timed(act_only) / K, timed(sample_only) / K
        flop = 2.0 * N * (54 * H + (L - 1) * H * H + 6 * H)
        print("%d x %-4d %10.2f %10.2f %12.3f %9.1f" % (L, H, ta, ts, flop / 1e9, flop / ta / 1e6))
    agents = [("SB3 default: actor 2 x 64 + critic 2 x 64", policy(2, 64, critic=True)), ("shipped: 5 x 128 shared trunk", policy(5, 128))]
    buf = env.rollout_policy(agents[0][1], T)
    for name, pol in agents:
        us = timed(lambda: env.rollout_policy(pol, T, out=buf)) / T
        print("rollout_policy, sampled, %-44s %8.2f us/step  %.3e env-steps/s" % (name, us, N / us * 1e6))
    print("env error flags:", int((env.error_flags() != 0).sum()))


if __name__ == "__main__":
    main()
