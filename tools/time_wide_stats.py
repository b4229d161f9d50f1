"""Per-step time of the wide step kernel with the float statistics of row f1 off and on (OpticalVecEnv(link_stats=...)):
  * C3: RMSA-v0 on the synthetic 100-node / 300-link topology, 320 slots, k = 10, 600 E, 131072 envs, device SAP-FF;
  * C4: RMCSA-v0 on NSFNET, 7 cores x 320 slots, 700 E, 262144 envs, device first-core first-fit;
  * germany50: RMSA-v0 (50 nodes, 88 links, k = 5), 320 slots, 600 E, 65536 envs, device SAP-FF.
Each: orlg_rollout of the heuristic (one fused heuristic + step launch per step), FILL steps first, then the median of 7 windows
of K steps timed with CUDA events behind a queued torch.cuda._sleep.  Prints the GPU name and power limit beside the numbers.
Usage: python tools/time_wide_stats.py [K] [FILL]"""
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "optical-rl-gym_b200")):
    sys.path.insert(0, p)
import torch

from optical_rl_gym_b200 import OpticalVecEnv, nsfnet
from optical_rl_gym_b200.topology import TopologyTables

K = int(sys.argv[1]) if len(sys.argv) > 1 else 20
FILL = int(sys.argv[2]) if len(sys.argv) > 2 else 600
REPS = 7
GOLDEN = os.path.join(ROOT, "tests", "golden")
RMSA320 = dict(episode_length=1000, load=600, mean_service_holding_time=25, num_spectrum_resources=320)
CONFIGS = [
    ("C3", "RMSA-v0", "topo_c3_ring100_chords200_k10.npz", 131072, RMSA320),
    ("C4", "RMCSA-v0", None, 262144, dict(episode_length=1000, load=700, mean_service_holding_time=25, num_spectrum_resources=320,
                                          num_spatial_resources=7, worst_xt=-84.7)),
    ("germany50", "RMSA-v0", "topo_germany50_tables.npz", 65536, RMSA320),
]


def step_ms(env):
    """median over REPS windows of K rollout steps, ms per step"""
    def run(k):
        left = k
        while left > 0:
            t = min(left, 64)
            env.rollout(t, "sap_ff", want_obs=False, want_actions=False)
            left -= t

    run(FILL)
    torch.cuda.synchronize()
    out = []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(20_000_000)
        a.record()
        run(K)
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) / K)
    return statistics.median(out), min(out), max(out)


def main():
    assert torch.cuda.is_available(), "needs a CUDA device"
    try:
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        gpu = torch.cuda.get_device_name()
    print("GPU: %s; %d fill steps, median of %d windows of %d steps" % (gpu, FILL, REPS, K))
    print("%-10s %8s %6s %12s %12s %12s %6s" % ("config", "envs", "stats", "ms/step", "min", "max", "errors"))
    for name, kind, topo, n, args in CONFIGS:
        tables = nsfnet() if topo is None else TopologyTables.load(os.path.join(GOLDEN, topo))
        for stats in (False, True):
            env = OpticalVecEnv(kind, n, tables, seed=1, collect_info=False, link_stats=stats, **args)
            med, lo, hi = step_ms(env)
            errors = int((env.error_flags() != 0).sum())
            print("%-10s %8d %6s %12.4f %12.4f %12.4f %6d" % (name, n, "on" if stats else "off", med, lo, hi, errors))
            env.close()
            del env
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
