"""Cost of invalid-action masking on the device, at the headline configuration (DeepRMSA-v0 NSFNET, 250 Erlang, 65536 envs,
1000 fill steps: real observations and masks):
  * rollout_policy masked against unmasked, us per step, for the shipped agent (one 5 x 128 trunk) and for SB3's default PPO
    agent (separate actor and critic trunks of 2 x 64);
  * action_masks() alone, and sample_native masked against unmasked, us per call;
  * action_masks() on germany50 (a wide handle; its 126-wide observation is beyond the policy kernel's 64 inputs, so
    rollout_policy does not run there).
CUDA events behind a queued torch.cuda._sleep, the median of 7 repetitions after a warm-up call; masked and unmasked
alternate.  Prints the GPU name and power limit beside the numbers."""
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
from optical_rl_gym_b200.topology import TopologyTables

N = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
T, K, REPS, ROUNDS = 64, 200, 7, 2


def policy(L, H, critic=False, obs_dim=54, n_actions=5):
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
    print("GPU: %s; DeepRMSA-v0 NSFNET 250 E, %d envs, 1000 fill steps, median of %d, %d alternating rounds" % (gpu, N, REPS, ROUNDS))
    env = OpticalVecEnv("DeepRMSA-v0", N, nsfnet(), seed=1, collect_info=False, episode_length=1000)
    env.rollout(1000, want_obs=False, want_actions=False)
    obs = env.observation().contiguous()
    mask = env.action_masks()
    print("rows with an invalid action: %.4f, with no valid action: %.4f" % ((~mask).any(1).float().mean().item(),
                                                                            (~mask.any(1)).float().mean().item()))
    act = torch.empty((N, 1), dtype=torch.int32, device="cuda")
    lp, val = torch.empty(N, device="cuda"), torch.empty(N, device="cuda")
    mbuf = torch.empty_like(mask)
    agents = [("shipped: 5 x 128 shared trunk", policy(5, 128)), ("SB3 default: actor 2 x 64 + critic 2 x 64", policy(2, 64, critic=True))]
    buf = env.rollout_policy(agents[0][1], T)
    for rnd in range(ROUNDS):
        print("-- round %d" % rnd)
        masks_us = timed(lambda: [env.action_masks(out=mbuf) for _ in range(K)]) / K
        print("action_masks()                               %8.2f us/call" % masks_us)
        for name, pol in agents:
            plain = timed(lambda: [pol.sample_native(obs, seed=1, counter=i, out=(act, lp, val)) for i in range(K)]) / K
            masked = timed(lambda: [pol.sample_native(obs, seed=1, counter=i, out=(act, lp, val), action_masks=mask)
                                    for i in range(K)]) / K
            print("sample_native %-44s unmasked %8.2f  masked %8.2f us/call" % (name, plain, masked))
        for name, pol in agents:
            plain = timed(lambda: env.rollout_policy(pol, T, out=buf)) / T
            masked = timed(lambda: env.rollout_policy(pol, T, out=buf, action_masks=True)) / T
            print("rollout_policy %-43s unmasked %8.2f  masked %8.2f us/step  (+%.1f %%)" % (name, plain, masked,
                                                                                          100.0 * (masked / plain - 1.0)))
    print("env error flags:", int((env.error_flags() != 0).sum()))
    env.close()
    g50 = TopologyTables.load(os.path.join(ROOT, "tests", "golden", "topo_germany50_tables.npz"))
    genv = OpticalVecEnv("DeepRMSA-v0", N, g50, seed=1, collect_info=False, episode_length=1000)
    genv.rollout(200, "sap_ff", want_obs=False, want_actions=False)
    gm = genv.action_masks()
    print("germany50 (wide, %d envs, 200 fill steps): action_masks() %8.2f us/call; rows with an invalid action %.4f" % (
        N, timed(lambda: [genv.action_masks(out=gm) for _ in range(K)]) / K, (~gm).any(1).float().mean().item()))
    print("germany50 error flags:", int((genv.error_flags() != 0).sum()))


if __name__ == "__main__":
    main()
