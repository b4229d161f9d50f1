#!/usr/bin/env python
"""Benchmark of the batched step hot path (BASELINE.json metric: env-steps/s, DeepRMSA-v0 NSFNET,
65536 envs per GPU, obs + reward + done on device).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one env.step of the whole batch (one env-step for each of the 65536 envs of every rank)
with the uniform random policy drawn on the device.  The K timed steps run as ONE orlg_rollout call
(persistent kernel: K steps per launch, every step's observation / reward / done / action written to
[K, N, ...] device buffers), repeated R times; the median repetition is reported (the list is in the
line).  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for value / e2e / roofline /
cpu_baseline.

--dump-outputs DIR writes what the last timed step returned (rank 0's envs) as DIR/<name>.npy.  Traffic and
actions come from seeded Philox streams, so the same arguments give the same inputs on every run and two
builds can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True      # the benchmark may run from a read-only tree: it writes nothing there

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "optical-rl-gym_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

ENV_ID = "DeepRMSA-v0"
ENV_ARGS = dict(episode_length=1000)          # DeepRMSA defaults: k=5, j=1, 100 slots, holding 25 / iat 0.1 = 250 Erlang
ENVS_PER_GPU = 65536
FILL_STEPS = 1000                              # ~4 mean holding times: network in steady state before timing
# SURVEY.md 8(d): algorithmic bytes per env-step for this config (random policy, fp32 obs)
B_STEP = 868
WORKLOAD = "DeepRMSA-v0 NSFNET(14n/22l) k=5 j=1 S=100 250E, %d envs/GPU, uniform random policy, Philox traffic"


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback"


DUMP_LIMIT = 64 << 20           # bytes written by --dump-outputs


def dump_outputs(path, arrays):
    """Writes each [N, ...] device tensor as path/<name>.npy in float32 (the integer outputs are exact in it).  Above
    DUMP_LIMIT bytes the same fixed, seeded sample of envs is kept in every array; its indices go to env_index.npy."""
    arrays = {k: v.float().cpu().numpy() for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    budget = DUMP_LIMIT - 4096                  # room for the .npy headers
    if n * row_bytes > budget:
        keep = np.sort(np.random.default_rng(0).choice(n, budget // (row_bytes + 8), replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
        arrays["env_index"] = keep.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.01)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def oracle_kwargs():
    # stats=False: like the GPU arm, the CPU arm computes obs / reward / done / counters, not the float statistics of info
    return dict(num_slots=100, episode_length=ENV_ARGS["episode_length"], j=1, mean_holding=25.0,
                mean_iat=1 / float((25.0 / 0.1) / 25.0), stats=False)


def cpu_baseline(threads, seconds=12.0):
    """The oracle port on all host cores, on a bounded sample of the same workload."""
    from optical_rl_gym_b200 import nsfnet
    from oracle import oracle

    n_envs = max(64, 16 * threads)
    vec = oracle.OracleVec(ENV_ID, nsfnet(), n_envs, seed=1, threads=threads, **oracle_kwargs())
    vec.run(FILL_STEPS)                                     # steady state, untimed
    chunk, done_steps, t0 = 500, 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        vec.run(chunk)
        done_steps += chunk
    dt = time.perf_counter() - t0
    vec.close()
    return {"value": n_envs * done_steps / dt, "unit": "env-steps/s", "cores": threads, "kind": "port",
            "sample": "%d envs x %d steps after a %d-step fill, oracle/orlg_oracle.c with float64 observation, "
                      "%d pthreads" % (n_envs, done_steps, FILL_STEPS, threads)}


def python_reference_baseline(seconds=8.0):
    """The UNMODIFIED Python reference (baseline/_ref), one env per process over all host cores, pipe-driven like
    SB3's SubprocVecEnv (baseline/subproc_reference.py).  None when the install did not travel to this box."""
    try:
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import subproc_reference as sr

        if not sr.available():
            return None
        return sr.measure(ENV_ID, dict(ENV_ARGS), workers=os.cpu_count() or 1, seconds=seconds)
    except Exception as exc:  # noqa: BLE001
        return {"unavailable": "%s: %s" % (type(exc).__name__, exc)}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port: the reference is
    pure Python and cannot travel to the GPU box), all host threads, same config / metric / unit."""
    if rank != 0:
        return
    from optical_rl_gym_b200 import nsfnet
    from oracle import oracle

    threads = os.cpu_count() or 1
    n_envs = int(os.environ.get("ORLG_REF_ENVS", 8192))
    vec = oracle.OracleVec(ENV_ID, nsfnet(), n_envs, seed=1, threads=threads, **oracle_kwargs())
    vec.run(FILL_STEPS)
    if args.warmup:
        vec.run(args.warmup)
    # the --steps chunk is repeated until the timed window is at least 2 s (a 20-step chunk alone lasts ~2 ms: pure noise)
    chunks, t0 = 0, time.perf_counter()
    while True:
        vec.run(args.steps)
        chunks += 1
        dt = time.perf_counter() - t0
        if dt >= float(os.environ.get("ORLG_REF_MIN_SECONDS", 2.0)):
            break
    vec.close()
    value = n_envs * args.steps * chunks / dt
    dt = dt / chunks
    sample = "%d of %d envs, %d chunks of %d steps after a %d-step fill, %d pthreads" % (
        n_envs, ENVS_PER_GPU * args.gpus, chunks, args.steps, FILL_STEPS, threads)
    print(json.dumps({
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8/f64", "data": "synthetic",
        "config": {"workload": WORKLOAD % ENVS_PER_GPU, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample},
        "cpu_baseline_python": python_reference_baseline(),
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# The other BASELINE.json configs: secondary lines (`--config c0|c1|c3|c4`); the headline stays configs[2].
# B_step = SURVEY.md 8(d) algorithmic bytes per env-step of each config.
SECONDARY = {
    "c0": dict(kind="RWA-v0", topo="nsfnet", envs=65536, policy="sap_ff", b_step=930, fill=1800,
               args=dict(episode_length=1000, load=450, mean_service_holding_time=25),
               workload="RWA-v0 NSFNET k=5 W=80 450E, %d envs/GPU, device shortest-available-path first-fit (configs[0] batched)"),
    "c1": dict(kind="RMSA-v0", topo="nsfnet", envs=4096, policy="sap_ff", b_step=800, fill=1000,
               args=dict(episode_length=1000, load=250, mean_service_holding_time=25),
               workload="RMSA-v0 NSFNET k=5 S=100 250E, %d envs/GPU, device SAP-FF (configs[1])"),
    "c1x": dict(kind="RMSA-v0", topo="nsfnet", envs=65536, policy="sap_ff", b_step=800, fill=1000,
                args=dict(episode_length=1000, load=250, mean_service_holding_time=25),
                workload="RMSA-v0 NSFNET k=5 S=100 250E, %d envs/GPU, device SAP-FF (configs[1] at 65536 envs)"),
    "c3": dict(kind="RMSA-v0", topo="c3", envs=131072, policy="sap_ff", b_step=1700, fill=600,
               args=dict(episode_length=1000, load=600, mean_service_holding_time=25, num_spectrum_resources=320),
               workload="RMSA-v0 synthetic 100 nodes / 300 links, S=320, k=10, 600E, %d envs/GPU, device SAP-FF (configs[3])"),
    "c4": dict(kind="RMCSA-v0", topo="nsfnet", envs=262144, policy="sap_ff", b_step=1000, fill=600,
               args=dict(episode_length=1000, load=700, mean_service_holding_time=25, num_spectrum_resources=320,
                         num_spatial_resources=7, worst_xt=-84.7),
               workload="RMCSA-v0 NSFNET 7 cores x 320 slots, 700E, %d envs/GPU, device first-core first-fit (configs[4])"),
}


def run_secondary(args):
    """One JSON line for another BASELINE config: K steps = orlg_rollout launches (persistent kernel for RMSA / RWA on
    NSFNET, per-step kernels for the wide layouts), R repetitions, CUDA events; single GPU."""
    import torch

    from optical_rl_gym_b200 import OpticalVecEnv, nsfnet
    from optical_rl_gym_b200.topology import TopologyTables

    c = SECONDARY[args.config]
    tables = nsfnet() if c["topo"] == "nsfnet" else TopologyTables.load(
        os.path.join(ROOT, "tests", "golden", "topo_c3_ring100_chords200_k10.npz"))
    torch.cuda.set_device(0)
    n, K = (args.envs if args.envs != ENVS_PER_GPU else c["envs"]), args.steps
    env = OpticalVecEnv(c["kind"], n, tables, seed=1, collect_info=False, **c["args"])
    chunk = min(K, 64)
    rew = torch.empty((chunk, n), dtype=torch.float32, device="cuda")
    done = torch.empty((chunk, n), dtype=torch.uint8, device="cuda")
    act = torch.empty((chunk, n, env.action_dim), dtype=torch.int32, device="cuda")

    def k_steps(k):
        left = k
        while left > 0:
            t = min(left, chunk)
            env.rollout(t, c["policy"], reward=rew[:t], done=done[:t], actions=act[:t], want_obs=False)
            left -= t

    k_steps(c["fill"])
    k_steps(max(args.warmup, 3))
    sampler = ClockSampler(0)
    rep_ms = []
    with sampler:
        for _ in range(args.reps):
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(400000)
            ev0.record()
            k_steps(K)
            ev1.record()
            torch.cuda.synchronize()
            rep_ms.append(ev0.elapsed_time(ev1))
        last = (K - 1) % chunk          # the last timed step, kept before the launches below overwrite the buffers
        dump = {"reward": rew[last].clone(), "done": done[last].clone(), "action": act[last].clone()} if args.dump_outputs else None
        t_end = time.perf_counter() + 0.25
        while time.perf_counter() < t_end:
            k_steps(chunk)
            torch.cuda.synchronize()
    ms = sorted(rep_ms)[len(rep_ms) // 2]
    peak, peak_src = read_peaks()
    achieved = c["b_step"] * n * K / (ms * 1e-3) / 1e9
    cnt = env.counters().sum(0).cpu().numpy()
    persistent = c["topo"] == "nsfnet" and c["kind"] in ("RMSA-v0", "RWA-v0")
    print(json.dumps({
        "metric": "env_steps_per_sec", "value": n * K / (ms * 1e-3), "unit": "env-steps/s", "n_gpus": 1, "steps": K,
        "warmup": args.warmup, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": c["workload"] % n, "secondary": args.config, "envs_per_gpu": n, "fill_steps": c["fill"],
                   "call": "orlg_rollout, %d steps per call (%s)" % (chunk, "persistent kernel" if persistent else
                                                                      "heuristic + step kernel per step")},
        "timing": {"reps": args.reps, "rep_ms": rep_ms, "stat": "median"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "algorithmic_bytes_per_env_step": c["b_step"], "peak_source": peak_src,
                     "note": "B_step of this config from SURVEY.md 8(d) (an estimate from the formula there)"},
        "cpu_baseline": None, "e2e": None, "gpu_launches": (K + chunk - 1) // chunk * (1 if persistent else 2 * chunk),
        "clocks": sampler.summary(), "accept_rate": float(cnt[1]) / float(cnt[0]),
        "envs_with_errors": int((env.error_flags() != 0).sum()), "state_MB": env.state_bytes / 1e6}))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dump)


E2E_CHUNK = int(os.environ.get("ORLG_E2E_CHUNK", "2"))   # steps per pipeline stage of the end-to-end leg (orlg_rollout_host)
ROLLOUT_CHUNK = 256      # steps per orlg_rollout launch (bounds the [chunk, N, 54] float32 output buffer: 3.6 GB)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7, help="repetitions of the --steps block (median reported)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="envs per GPU (default: BASELINE config)")
    ap.add_argument("--config", default="c2", choices=["c2"] + sorted(SECONDARY),
                    help="c2 = the headline (BASELINE configs[2]); the others print a secondary line for that config")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's obs / reward / done / action of rank 0's envs to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the device path; --impl reference has none")
    args.warmup = max(args.warmup, 3)
    args.reps = max(args.reps, 1)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.config != "c2":
        if rank == 0:
            run_secondary(args)
        return

    # The CPU baseline runs FIRST, on rank 0, while the other ranks are still blocked in the rendezvous of
    # init_process_group (a socket wait, no spinning): it has the host cores to itself.
    cpu = cpu_py = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = cpu_baseline(os.cpu_count() or 1)
        cpu_py = python_reference_baseline()

    import torch
    import torch.distributed as dist

    from optical_rl_gym_b200 import OpticalVecEnv, nsfnet, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    n, K = args.envs, args.steps
    env = OpticalVecEnv(ENV_ID, n, nsfnet(), device=dev, env_id_base=rank * n, seed=1, collect_info=False, **ENV_ARGS)
    chunk = min(K, ROLLOUT_CHUNK)
    obs = torch.empty((chunk, n, env.obs_dim), dtype=torch.float32, device=dev)
    rew = torch.empty((chunk, n), dtype=torch.float32, device=dev)
    done = torch.empty((chunk, n), dtype=torch.uint8, device=dev)
    act = torch.empty((chunk, n, 1), dtype=torch.int32, device=dev)
    launches = (K + chunk - 1) // chunk                 # kernel launches per K-step block

    def k_steps(k):
        """k env-steps of every env: orlg_rollout launches of <= chunk steps, all outputs written every step."""
        left = k
        while left > 0:
            t = min(left, chunk)
            env.rollout(t, "random", obs=obs[:t], reward=rew[:t], done=done[:t], actions=act[:t])
            left -= t

    k_steps(FILL_STEPS)                                 # bring the network to steady state (setup, untimed)
    k_steps(args.warmup)
    torch.cuda.synchronize()

    # ---- timed region: R repetitions of exactly K steps; each is bracketed by barrier + synchronize and timed with CUDA
    # events on the launching stream.  A short device-side sleep is queued first so that the host has enqueued
    # [start event, the block's launches, end event] before the GPU reaches them: no host jitter inside the region.
    sampler = ClockSampler(local_rank)
    rep_ms = []
    with sampler:
        for _ in range(args.reps):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(400000)
            ev0.record()
            k_steps(K)
            ev1.record()
            torch.cuda.synchronize()
            t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)        # max over ranks, per repetition
            rep_ms.append(float(t.item()))
        last = (K - 1) % chunk          # the last timed step, kept before the launches below overwrite the buffers
        dump = {"obs": obs[last].clone(), "reward": rew[last].clone(), "done": done[last].clone(),
                "action": act[last].clone()} if args.dump_outputs and rank == 0 else None
        # keep the GPU under the same load a little longer so that the clock sampler sees it
        t_end = time.perf_counter() + 0.25
        while time.perf_counter() < t_end:
            k_steps(chunk)
            torch.cuda.synchronize()
    elapsed_ms = sorted(rep_ms)[len(rep_ms) // 2]
    value = n * world * K / (elapsed_ms * 1e-3)
    stats = sharding.global_statistics(env.reduce_counters())      # the per-rollout NCCL all-reduce (8e)

    # ---- end to end through the public API with HOST buffers (pinned): H2D actions, step, D2H obs/reward/done.
    # Every rank runs it at the same time (they share the host's PCIe / memory), max over ranks.
    e2e_result = e2e_sync = None
    actions = torch.empty((n, 1), dtype=torch.int32, device=dev)
    env.sample_actions(out=actions)
    if not args.no_e2e:
        h_act = torch.zeros((n, 1), dtype=torch.int32).pin_memory()
        h_obs = torch.zeros((n, env.obs_dim), dtype=torch.float32).pin_memory()
        h_rew = torch.zeros(n, dtype=torch.float32).pin_memory()
        h_done = torch.zeros(n, dtype=torch.uint8).pin_memory()
        h_act.copy_(actions.cpu())
        k_e2e = max(20, min(K, 300))

        def e2e_step():
            d_act = h_act.to(dev, non_blocking=True)
            o, r, d, _ = env.step(d_act)
            h_obs.copy_(o, non_blocking=True)
            h_rew.copy_(r, non_blocking=True)
            h_done.copy_(d, non_blocking=True)
            torch.cuda.synchronize()            # the host policy needs the observation before it can act

        for _ in range(5):
            e2e_step()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(k_e2e):
            e2e_step()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_sync = {"value": n * world * k_e2e / float(dt.item()), "unit": "env-steps/s",
                    "h2d_bytes_per_step": h_act.numel() * 4 * world,
                    "d2h_bytes_per_step": (h_obs.numel() * 4 + h_rew.numel() * 4 + h_done.numel()) * world,
                    "steps": k_e2e, "n_gpus": world,
                    "note": "VecEnv.step with pinned host buffers on every rank concurrently, synchronised every step "
                            "(float32 rows cross PCIe: 14.5 MB per step and GPU)"}
        del h_obs, h_rew, h_done

        # ---- the headline end-to-end number: the same K-step rollout through the C ABI with HOST buffers on both sides
        # (orlg_rollout_host, ORLG_POLICY_REPLAY).  Input: the actions of every step, drawn beforehand on the host (the uniform
        # random policy does not look at observations), in pinned memory, copied to the device chunk by chunk.  Output: every
        # step's float32 observation row, reward and done in host memory.  Inside the call the device runs chunk c + 1 while
        # chunk c's 32-byte step records cross PCIe and the host threads expand them to the float32 rows (bit-identical to
        # what orlg_rollout writes on the device).  Wall clock around the calls, every rank at the same time, max over ranks.
        k_h = 40                               # steps per call (580 MB of float32 rows in host memory per rank)
        threads = max(1, (os.cpu_count() or 1) // world)
        rng = np.random.default_rng(1234 + rank)
        ha_t = torch.from_numpy(rng.integers(0, env.k_paths * env.j + 1, size=(k_h, n), dtype=np.int32)).pin_memory()
        ha = ha_t.numpy()
        ho = np.zeros((k_h, n, env.obs_dim), np.float32)
        hr = np.zeros((k_h, n), np.float32)
        hd = np.zeros((k_h, n), np.uint8)
        for _ in range(2):
            env.rollout_host(k_h, "replay", obs=ho, reward=hr, done=hd, actions=ha, chunk=E2E_CHUNK, threads=threads)
        if world > 1:
            dist.barrier()
        reps_h = 3
        t0 = time.perf_counter()
        for _ in range(reps_h):
            env.rollout_host(k_h, "replay", obs=ho, reward=hr, done=hd, actions=ha, chunk=E2E_CHUNK, threads=threads)
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_result = {"value": n * world * k_h * reps_h / float(dt.item()), "unit": "env-steps/s",
                      "h2d_bytes_per_step": n * 4 * world, "d2h_bytes_per_step": n * 32 * world,
                      "host_bytes_delivered_per_step": n * (env.obs_dim * 4 + 5) * world,
                      "steps": k_h * reps_h, "n_gpus": world, "host_threads_per_rank": threads, "chunk_steps": E2E_CHUNK,
                      "accepted_in_sample": float((hr > 0).mean()),
                      "note": "orlg_rollout_host(ORLG_POLICY_REPLAY): actions [steps, N] int32 from pinned host memory (H2D per "
                              "chunk), float32 observation rows + reward + done of every step delivered in host memory; the step "
                              "records cross PCIe packed (32 B per env-step) and are expanded by the library's host threads; "
                              "wall clock, every rank concurrently, max over ranks"}
        del ho, hr, hd

    # ---- the same K steps with the results delivered to the HOST as packed 32-byte records (orlg_rollout_packed: the
    # integer pre-image of the observation + request + action / accepted / done; orlg_expand_packed decodes them).  The
    # device policy needs no per-step input, so there is no H2D; chunks of 4 steps are double-buffered: the D2H copy of
    # chunk c (side stream) overlaps the kernel of chunk c + 1.
    e2e_packed = None
    if not args.no_e2e:
        ck = 4
        k_pk = max(20, min(K, 200)) // ck * ck
        d_pk = [torch.empty((ck, n, 8), dtype=torch.int32, device=dev) for _ in range(2)]
        h_pk = [torch.empty((ck, n, 8), dtype=torch.int32).pin_memory() for _ in range(2)]
        s_copy = torch.cuda.Stream(device=dev)
        ev_k = [torch.cuda.Event() for _ in range(2)]
        ev_c = [torch.cuda.Event() for _ in range(2)]

        def packed_block(k):
            cur = torch.cuda.current_stream(dev)
            for c in range(k // ck):
                b = c & 1
                if c >= 2:
                    cur.wait_event(ev_c[b])                 # the copy that last read d_pk[b] has finished
                env.rollout_packed(ck, "random", out=d_pk[b])
                ev_k[b].record(cur)
                s_copy.wait_event(ev_k[b])
                with torch.cuda.stream(s_copy):
                    h_pk[b].copy_(d_pk[b], non_blocking=True)
                    ev_c[b].record(s_copy)
                if c >= 1:
                    ev_c[1 - b].synchronize()               # the consumer now owns chunk c - 1 in h_pk[1 - b]
            ev_c[(k // ck - 1) & 1].synchronize()
            torch.cuda.synchronize()

        packed_block(2 * ck)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        packed_block(k_pk)
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_packed = {"value": n * world * k_pk / float(dt.item()), "unit": "env-steps/s", "h2d_bytes_per_step": 0,
                      "d2h_bytes_per_step": n * 32 * world, "steps": k_pk, "n_gpus": world,
                      "note": "orlg_rollout_packed (device policy) + pinned D2H of 32-byte step records, double-buffered in chunks "
                              "of %d steps; wall clock, max over ranks; decoding to float32 rows (orlg_expand_packed) is left to the consumer" % ck}

    out = None
    if rank == 0:
        # ---- roofline of the dominant kernel: the timed region IS that kernel (one launch per <= 256 steps)
        peak, peak_src = read_peaks()
        achieved = B_STEP * n * K / (elapsed_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": None, "kernel": "deeprmsa_rollout_kernel<22,0>", "kernel_ms": elapsed_ms / launches,
                    "steps_per_launch": chunk, "algorithmic_bytes_per_env_step": B_STEP,
                    "algorithmic_bytes_per_launch": B_STEP * n * chunk, "peak_source": peak_src,
                    "note": "achieved = 868 B x envs x steps of one launch / its CUDA-event duration; the kernel keeps masks and "
                            "scalars on chip across the steps of a launch, so its DRAM traffic is BELOW the algorithmic bytes"}
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
            # per launch like `achieved`: the ncu capture (65536 envs x 20 steps per launch) scaled to this launch's env-steps
            roofline["traffic"] = tj.get("rollout_kernel_bytes_per_env_step") * n * chunk
            roofline["traffic_source"] = "ncu --set full capture of a %s-step launch (profiles/r2d_rollout_ncu_full.csv), %.0f B per env-step" % (
                tj.get("rollout_kernel_steps_per_launch"), tj.get("rollout_kernel_bytes_per_env_step"))
        except Exception:  # noqa: BLE001
            pass

        # ---- the step-by-step path (one policy launch + one step launch per step), for comparison
        for _ in range(20):
            env.sample_actions(out=actions)
            env.step_raw(actions)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(400000)
        a.record()
        for _ in range(200):
            env.sample_actions(out=actions)
            env.step_raw(actions)
        b.record()
        torch.cuda.synchronize()
        step_path_ms = a.elapsed_time(b) / 200

        # ---- the "PPO-policy actions" variant of this config (DeepRMSA.ipynb cell 13): obs -> shipped agent's MLP
        # (54 -> 5 x 128 tanh -> 5 logits, random-init weights of that architecture) -> env.step, all on the device
        ppo = None
        try:
            from optical_rl_gym_b200.policy import MlpPolicy

            torch.manual_seed(0)
            pol = MlpPolicy(env.obs_dim, 5, (128,) * 5).to(dev)
            env.observation()

            def ppo_step():
                pol.act_native(env._obs, out=actions)
                env.step_raw(actions)

            for _ in range(20):
                ppo_step()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(400000)
            a.record()
            for _ in range(200):
                ppo_step()
            b.record()
            torch.cuda.synchronize()
            ppo_ms = a.elapsed_time(b) / 200
            a.record()
            for _ in range(200):
                pol.act_native(env._obs, out=actions)
            b.record()
            torch.cuda.synchronize()
            pol_ms = a.elapsed_time(b) / 200
            flop = 2.0 * n * (env.obs_dim * 128 + 4 * 128 * 128 + 6 * 128)
            ppo = {"value": n / (ppo_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ppo_ms, "policy_kernel_ms": pol_ms,
                   "policy_tflops": flop / (pol_ms * 1e-3) / 1e12, "policy_kernel": "mlp_policy_kernel (bf16 tcgen05.mma, TMEM accumulators)",
                   "note": "per step: fused policy kernel + per-step env kernel, chained by programmatic dependent launch; 1 GPU"}
        except Exception as exc:  # noqa: BLE001
            ppo = {"unavailable": "%s: %s" % (type(exc).__name__, exc)}

        out = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": K, "warmup": args.warmup, "ms_per_step": elapsed_ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": WORKLOAD % n, "envs_per_gpu": n, "fill_steps": FILL_STEPS,
                       "obs": "float32 [steps, N, 54] on device, every step written",
                       "call": "orlg_rollout: %d steps per launch, %d launch(es) per timed block" % (chunk, launches),
                       "l2": "no flush: the %d-step output block (%.0f MB) and the event storage (%.0f MB) exceed the 126 MB L2; "
                             "masks and scalars stay on chip by design" % (chunk, chunk * n * (env.obs_dim * 4 + 9) / 1e6,
                                                                            env.state_bytes / 1e6),
                       "parallelism": "env-sharded x%d, no data-path collective" % world},
            "timing": {"reps": args.reps, "rep_ms": rep_ms, "stat": "median of the repetitions (each: max over ranks)"},
            "roofline": roofline, "cpu_baseline": cpu, "cpu_baseline_python": cpu_py, "e2e": e2e_result, "e2e_step_sync": e2e_sync, "e2e_packed": e2e_packed,
            "gpu_launches": launches,
            "clocks": sampler.summary(), "step_path_ms_per_step": step_path_ms, "ppo_policy_variant": ppo,
            "accept_rate": 1.0 - stats["service_blocking_rate"], "envs_with_errors": stats["envs_with_errors"],
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if dump is not None:
        dump_outputs(args.dump_outputs, dump)
    if out is not None:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
