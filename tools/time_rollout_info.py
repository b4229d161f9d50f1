"""Cost of keeping every step's info in a rollout (want_info=True: the int64 counters, 64 bytes per env-step) at bench.py's
configuration (DeepRMSA-v0 NSFNET, 250 Erlang, 65536 envs, episodes of 1000, 1000 fill steps):
  * rollout (the persistent kernel, observations, rewards, dones and actions written) at launches of 20 and 200 steps;
  * rollout_policy for the shipped 5 x 128 agent.
ms per step with the counters off and on, CUDA events behind a queued torch.cuda._sleep, the median of 7 repetitions after a
warm-up call; off and on alternate within each repetition.  Prints the GPU name and power limit beside the numbers."""
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
REPS, STEPS = 7, 400          # env steps per timed repetition of rollout (20-step launches: 20 of them)


def device_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(20_000_000)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def compare(off, on, steps):
    """(ms per step off, ms per step on): medians over REPS alternating repetitions."""
    off(); on()
    torch.cuda.synchronize()
    t_off, t_on = [], []
    for _ in range(REPS):
        t_off.append(device_ms(off) / steps)
        t_on.append(device_ms(on) / steps)
    return statistics.median(t_off), statistics.median(t_on)


def main():
    assert torch.cuda.is_available(), "needs a CUDA device"
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        gpu = torch.cuda.get_device_name()
    print("GPU: %s; DeepRMSA-v0 NSFNET 250 E, %d envs, 1000 fill steps, median of %d" % (gpu, N, REPS))
    env = OpticalVecEnv("DeepRMSA-v0", N, nsfnet(), seed=1, episode_length=1000)
    env.rollout(1000, want_obs=False, want_actions=False)
    for T in (20, 200):
        obs = torch.empty((T, N, env.obs_dim), dtype=torch.float32, device="cuda")
        rew = torch.empty((T, N), dtype=torch.float32, device="cuda")
        done = torch.empty((T, N), dtype=torch.uint8, device="cuda")
        act = torch.empty((T, N, 1), dtype=torch.int32, device="cuda")

        def run(want_info):
            def fn():
                for _ in range(STEPS // T):
                    env.rollout(T, obs=obs, reward=rew, done=done, actions=act, want_info=want_info)
            return fn

        off, on = compare(run(False), run(True), STEPS)
        assert env.kernel_info()["last_rollout_persistent"]
        print("rollout, %3d-step launches: %.4f ms/step counters off, %.4f on (%+.1f %%)" % (T, off, on, 100 * (on / off - 1)))
    torch.manual_seed(0)
    pol = MlpPolicy(env.obs_dim, 5, (128,) * 5).cuda()
    T = 64
    buf = env.rollout_policy(pol, T)
    off, on = compare(lambda: env.rollout_policy(pol, T, out=buf), lambda: env.rollout_policy(pol, T, out=buf, want_info=True), T)
    print("rollout_policy 5 x 128, %d steps per call: %.4f ms/step counters off, %.4f on (%+.1f %%)" % (T, off, on, 100 * (on / off - 1)))
    print("env error flags:", int((env.error_flags() != 0).sum()))


if __name__ == "__main__":
    main()
