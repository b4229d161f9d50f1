"""PPO rollout collection at the headline configuration (DeepRMSA-v0 NSFNET, 250 Erlang, 65536 envs, 1000 fill steps):
per-step time of
  (a) the Python loop act_native + step_raw (argmax actions, nothing kept),
  (b) rollout_policy, deterministic mode,
  (c) rollout_policy, sampled actions,
  (d) rollout_policy, sampled actions and a separate critic trunk (SB3 >= 1.8 agents),
and the sampling kernel alone against orlg_policy_act alone.  CUDA events behind a queued torch.cuda._sleep; T = 64 steps
per repetition, the median of 7 repetitions.  Prints the GPU name and power limit beside the numbers."""
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
T, REPS = 64, 7


def policy(separate_critic):
    torch.manual_seed(0)
    pol = MlpPolicy(54, 5, (128,) * 5)
    for m in pol.shared_net:
        if isinstance(m, torch.nn.Linear):
            torch.nn.init.orthogonal_(m.weight, gain=2 ** 0.5)
    if separate_critic:
        layers = []
        for i in range(5):
            lin = torch.nn.Linear(54 if i == 0 else 128, 128)
            torch.nn.init.orthogonal_(lin.weight, gain=2 ** 0.5)
            layers += [lin, torch.nn.Tanh()]
        pol.critic_net = torch.nn.Sequential(*layers)
    return pol.cuda()


def timed(fn, reps=REPS):
    """median over `reps` of the device time of one fn() (CUDA events, queued behind a sleep so the host runs ahead)."""
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(20_000_000)                 # ~10 ms: the host enqueues the whole window behind it
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
    print("GPU: %s; DeepRMSA-v0 NSFNET 250 E, %d envs, 1000 fill steps, T = %d steps per call, median of %d" % (gpu, N, T, REPS))
    env = OpticalVecEnv("DeepRMSA-v0", N, nsfnet(), seed=1, collect_info=False, episode_length=1000)
    env.rollout(1000, want_obs=False, want_actions=False)
    actor, critic = policy(False), policy(True)
    act = torch.empty((N, 1), dtype=torch.int32, device="cuda")

    def loop():
        obs = env.observation()
        for _ in range(T):
            actor.act_native(obs, out=act)
            obs = env.step_raw(act)[0]

    buf = env.rollout_policy(actor, T)
    rows = [("(a) Python loop act_native + step_raw", loop),
            ("(b) rollout_policy, deterministic", lambda: env.rollout_policy(actor, T, deterministic=True, out=buf)),
            ("(c) rollout_policy, sampled", lambda: env.rollout_policy(actor, T, out=buf)),
            ("(d) rollout_policy, sampled + critic trunk", lambda: env.rollout_policy(critic, T, out=buf))]
    for name, fn in rows:
        us = timed(fn) / T
        print("%-44s %8.2f us/step  %.3e env-steps/s" % (name, us, N / us * 1e6))
    obs = buf.obs[-1]
    K = 200

    def act_only():
        for _ in range(K):
            actor.act_native(obs, out=act)

    def sample_only():
        for i in range(K):
            actor.sample_native(obs, seed=1, counter=i, out=(act, buf.log_prob[0], buf.value[0]))

    ta, ts = timed(act_only) / K, timed(sample_only) / K
    print("%-44s %8.2f us per %d rows" % ("orlg_policy_act alone", ta, N))
    print("%-44s %8.2f us per %d rows (%+.2f us)" % ("orlg_policy_sample alone (sampled)", ts, N, ts - ta))
    print("env error flags:", int((env.error_flags() != 0).sum()))


if __name__ == "__main__":
    main()
