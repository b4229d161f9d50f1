"""Cost of the MATRIX policy kernel (MlpPolicy(matrix_observation=...), orlg_policy_create_matrix), 65536 rows:
  * sample_native per call on packed rows: 2 x 64 and 5 x 128 on NSFNET / 100 slots (2228 inputs), 2 x 64 on germany50 /
    100 slots (8900 inputs);
  * rollout_policy per step on RMSA-v0 NSFNET with SB3's default agent (actor 2 x 64, separate critic 2 x 64), next to what
    a user has without it: per step matrix_observation() (uint8), a float32 torch forward of actor and critic on those rows,
    a multinomial draw, path_only_first_fit and step_raw.
Kernel timings run on random packed rows (the kernel's work does not depend on the bits).  CUDA events behind a queued
torch.cuda._sleep, the median of 7 repetitions after a warm-up call; the variants of a line alternate, twice.  Prints the GPU
name and power limit beside the numbers."""
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
from optical_rl_gym_b200.vec_env import matrix_obs_words

N = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
T, K, REPS, ROUNDS = 16, 50, 7, 2


def policy(L, H, layout, critic=False, n_actions=6):
    nodes, links, slots = layout
    obs_dim = 2 * nodes + links * slots
    torch.manual_seed(L * 1000 + H)
    pol = MlpPolicy(obs_dim, n_actions, (H,) * L, matrix_observation=layout)
    for m in pol.shared_net:
        if isinstance(m, torch.nn.Linear):
            torch.nn.init.orthogonal_(m.weight, gain=2 ** 0.5)
    if critic:
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


def random_packed(layout, gen):
    nodes, links, slots = layout
    W = matrix_obs_words(layout)
    x = torch.randint(-2 ** 31, 2 ** 31 - 1, (N, W), generator=gen, device="cuda", dtype=torch.int64).to(torch.int32)
    nwv = (slots + 127) // 128
    keep = torch.zeros(128 * nwv, dtype=torch.int64)
    keep[:slots] = 1
    mask = (keep.reshape(-1, 32) << torch.arange(32)).sum(1).to(torch.int64)
    mask = torch.where(mask >= 2 ** 31, mask - 2 ** 32, mask).to(torch.int32).cuda()
    x[:, 4:] &= mask.repeat(links)
    src = torch.randint(0, nodes, (N,), generator=gen, device="cuda")
    dst = (src + torch.randint(1, nodes, (N,), generator=gen, device="cuda")) % nodes
    x[:, 0] = (torch.minimum(src, dst) | (torch.maximum(src, dst) << 8)).to(torch.int32)
    x[:, 1:4] = 0
    return x


def main():
    assert torch.cuda.is_available(), "needs a CUDA device"
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        gpu = torch.cuda.get_device_name()
    print("GPU: %s; %d rows, median of %d, %d alternating rounds" % (gpu, N, REPS, ROUNDS))
    nsf = TopologyTables.load(os.path.join(ROOT, "tests", "golden", "nsfnet_tables.npz"))
    g50 = TopologyTables.load(os.path.join(ROOT, "tests", "golden", "topo_germany50_tables.npz"))
    gen = torch.Generator(device="cuda").manual_seed(0)
    cases = []
    for name, tables, L, H in (("NSFNET", nsf, 2, 64), ("NSFNET", nsf, 5, 128), ("germany50", g50, 2, 64)):
        layout = (tables.num_nodes, tables.num_links, 100)
        cases.append((name, L, H, layout, policy(L, H, layout), random_packed(layout, gen)))
    bufs = (torch.empty((N, 1), dtype=torch.int32, device="cuda"), torch.empty(N, device="cuda"), torch.empty(N, device="cuda"))
    for rnd in range(ROUNDS):
        for name, L, H, layout, pol, x in cases:
            t = timed(lambda: [pol.sample_native(x, seed=1, counter=i, out=bufs) for i in range(K)]) / K
            g = nat.lib().orlg_policy_tile_groups(pol._native_handle(0))
            flop = 2.0 * N * (H * (2 * layout[0] + layout[1] * layout[2]) + (L - 1) * H * H + 7 * H)
            print("round %d: %-9s obs %5d, %d x %-3d (%d tile group%s)  sample_native %8.2f us/call  (%.0f TFLOP/s of the "
                  "unpadded MLP)" % (rnd, name, 2 * layout[0] + layout[1] * layout[2], L, H, g, "s" if g > 1 else "", t,
                                     flop / t * 1e-6))
    env = OpticalVecEnv("RMSA-v0", N, nsf, seed=1, collect_info=False, episode_length=1000, load=250,
                        mean_service_holding_time=25)
    env.rollout(100, "sp_ff", want_obs=False, want_actions=False)
    pol = policy(2, 64, env.matrix_layout, critic=True, n_actions=env.k_paths + env.reject_action)
    buf = env.rollout_policy(pol, T)

    def torch_step():
        with torch.no_grad():
            logits, value = pol(env.matrix_observation().float())
            a = torch.multinomial(torch.softmax(logits, -1), 1)[:, 0]
            env.step_raw(env.path_only_first_fit(a))

    for rnd in range(ROUNDS):
        native = timed(lambda: env.rollout_policy(pol, T, out=buf)) / T
        eager = timed(lambda: [torch_step() for _ in range(T)]) / T
        print("round %d: RMSA-v0 NSFNET, SB3 default actor 2 x 64 + critic 2 x 64: rollout_policy %8.2f us/step; "
              "torch forward on uint8 rows %8.2f us/step" % (rnd, native, eager))
    print("error flags:", int((env.error_flags() != 0).sum()))
    env.close()


if __name__ == "__main__":
    main()
