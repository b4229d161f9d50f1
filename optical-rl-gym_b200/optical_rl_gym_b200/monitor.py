"""Episode bookkeeping for a batched env in the format Stable-Baselines3's ``Monitor`` writes
(SURVEY.md row f4; the reference trains through ``Monitor(env, log_dir + 'training',
info_keywords=('episode_service_blocking_rate', 'episode_bit_rate_blocking_rate'))``,
examples/stable_baselines3/DeepRMSA.ipynb cell 13, and ships such a file:
examples/stable_baselines3/bkp/deeprmsa-ppo-trained/training.monitor.csv).

File layout: ``#{"t_start": ..., "env_id": ...}`` then a CSV with header ``r,l,t,<info_keywords>``; one
row per finished episode = sum of rewards, number of steps, seconds since ``t_start`` and the value of each
info keyword at the terminal step.  Sums and lengths accumulate on the device; the host is only touched
when an episode ends (one 1-byte read per step to learn whether any did).  ``rollout`` and ``rollout_policy``
write the same rows as the equivalent ``step`` loop, from every step's reward, done and info of the rollout.
"""
from __future__ import annotations

import json
import time
from typing import Optional, Sequence

import numpy as np
import torch

from .wrappers import VecWrapper


class VecMonitor(VecWrapper):
    EXT = "monitor.csv"

    def __init__(self, venv, filename: Optional[str] = None, info_keywords: Sequence[str] = ()):
        super().__init__(venv)
        self.info_keywords = tuple(info_keywords)
        if self.info_keywords:           # fail at construction, not at the first episode end
            base0 = self.unwrapped
            if getattr(base0, "_info", None) is None:
                raise ValueError("info_keywords need the venv's info: construct it with collect_info=True")
            known = set(getattr(base0, "info_keys", ()) or ())
            missing = [k for k in self.info_keywords if known and k not in known]
            if missing:
                raise ValueError("info_keywords %s are not in this env's info (%s)" % (missing, sorted(known)))
        self.t_start = time.time()
        base = self.unwrapped
        n, dev = base.num_envs, base.device
        self._ret = torch.zeros(n, dtype=torch.float64, device=dev)
        self._len = torch.zeros(n, dtype=torch.int64, device=dev)
        self.episode_returns, self.episode_lengths, self.episode_times = [], [], []
        self.episode_infos = {k: [] for k in self.info_keywords}
        self.total_steps = 0
        self._fh = None
        if filename is not None:
            if not filename.endswith(self.EXT):
                filename = filename + "." + self.EXT
            self._fh = open(filename, "wt")
            self._fh.write("#%s\n" % json.dumps({"t_start": self.t_start, "env_id": base.env_id}))
            self._fh.write(",".join(("r", "l", "t") + self.info_keywords) + "\n")
            self._fh.flush()

    def reset(self, **kwargs):
        self._ret.zero_()
        self._len.zero_()
        return self.venv.reset(**kwargs)

    def step_wait(self):
        obs, reward, done, info = self.venv.step_wait()
        self._ret += reward.to(torch.float64)
        self._len += 1
        self.total_steps += int(self._len.shape[0])
        if bool(done.any()):
            idx = torch.nonzero(done, as_tuple=False).flatten()
            self._record(self._ret[idx], self._len[idx], [info[k][idx] for k in self.info_keywords])
            self._ret[idx] = 0.0
            self._len[idx] = 0
        return obs, reward, done, info

    def _record(self, r, l, cols):
        """Appends the rows of finished episodes: returns, lengths and info keyword values (device tensors, in row order)."""
        r, l = r.cpu().numpy(), l.cpu().numpy()
        t = round(time.time() - self.t_start, 6)
        cols = [np.asarray(c.cpu().numpy(), np.float64) for c in cols]
        self.episode_returns.extend(r.tolist())
        self.episode_lengths.extend(l.tolist())
        self.episode_times.extend([t] * len(r))
        for k, c in zip(self.info_keywords, cols):
            self.episode_infos[k].extend(c.tolist())
        if self._fh is not None:
            # every finished episode gets its row (SB3's Monitor writes one per episode): one buffered write per call
            self._fh.write("".join(",".join([repr(float(r[i])), str(int(l[i])), repr(t)] + [repr(float(c[i])) for c in cols]) + "\n"
                                   for i in range(len(r))))
            self._fh.flush()

    def _base(self, method):
        from .vec_env import OpticalVecEnv

        if not isinstance(self.venv, OpticalVecEnv):
            # a wrapper in between (UseInfoReward, ...) would be bypassed by the native rollout: its rows would be wrong
            raise TypeError("VecMonitor.%s needs the OpticalVecEnv itself as its venv, not %s" % (method, type(self.venv).__name__))
        return self.venv

    def _record_rollout(self, reward, done, info):
        """The rows a ``step`` loop over the rollout's T steps would write, from reward / done ``[T, N]`` and ``info``."""
        T, n = done.shape
        self.total_steps += T * n
        if T == 0:
            return
        d = done.bool()
        csum = torch.cumsum(reward.to(torch.float64), 0)         # rewards are -1 / 0 / 1: exact in any order of addition
        steps = torch.arange(T, device=d.device).unsqueeze(1).expand(T, n)
        last = torch.where(d, steps, torch.full_like(steps, -1)).cummax(0).values      # last episode end at or before t
        idx = torch.nonzero(d, as_tuple=False)                    # (t, env) in the step loop's row order
        if idx.shape[0]:
            t, e = idx[:, 0], idx[:, 1]
            prev = torch.where(t > 0, last[(t - 1).clamp(min=0), e], torch.full_like(t, -1))   # the env's previous end
            first = prev < 0                                      # the episode began before this call
            before = torch.where(first, torch.zeros_like(csum[t, e]), csum[prev.clamp(min=0), e])
            r = torch.where(first, self._ret[e], torch.zeros_like(before)) + (csum[t, e] - before)
            l = torch.where(first, self._len[e], torch.zeros_like(t)) + (t - prev)
            self._record(r, l, [info[k][t, e] for k in self.info_keywords])
        end = last[T - 1]
        ended = end >= 0
        self._ret = torch.where(ended, csum[T - 1] - csum[end.clamp(min=0), torch.arange(n, device=d.device)], self._ret + csum[T - 1])
        self._len = torch.where(ended, T - 1 - end, self._len + T)

    def rollout(self, steps, policy="random", **kw):
        """:meth:`OpticalVecEnv.rollout` that logs the episodes it finishes like the equivalent ``step`` loop; returns what
        the env returns (with the info only when ``want_info=True`` is passed)."""
        want = kw.pop("want_info", False)
        with_info = want or bool(self.info_keywords)
        res = self._base("rollout").rollout(steps, policy, want_info=with_info, **kw)
        self._record_rollout(res[1], res[2], res[4] if with_info else None)
        return res if want or not with_info else res[:4]

    def rollout_policy(self, agent, steps, **kw):
        """:meth:`OpticalVecEnv.rollout_policy` that logs the episodes it finishes like the equivalent ``step`` loop; returns
        what the env returns (``action_masks=True`` appends the masks, the info only comes with ``want_info=True``)."""
        want = kw.pop("want_info", False)
        with_info = want or bool(self.info_keywords)
        res = self._base("rollout_policy").rollout_policy(agent, steps, want_info=with_info, **kw)
        parts = list(res) if with_info or kw.get("action_masks", False) else [res]     # [PolicyRollout, StepInfo?, masks?]
        out, info = parts[0], (parts[1] if with_info else None)
        self._record_rollout(out.reward, out.done, info)
        if want or not with_info:
            return res
        rest = parts[2:]                  # the masks, after the info this call added for its own rows
        return (out, *rest) if rest else out

    def get_episode_rewards(self):
        return self.episode_returns

    def get_episode_lengths(self):
        return self.episode_lengths

    def get_episode_times(self):
        return self.episode_times

    def get_total_steps(self):
        return self.total_steps

    def close(self):
        if self._fh is not None:
            self._fh.close()
            self._fh = None
        self.venv.close()


def load_monitor_csv(path):
    """(header dict, {column: numpy array}) of a monitor file (ours or Stable-Baselines3's)."""
    with open(path) as f:
        first = f.readline()
        assert first.startswith("#"), "not a monitor file"
        header = json.loads(first[1:])
        names = f.readline().strip().split(",")
        rows = [ln.strip().split(",") for ln in f if ln.strip()]
    cols = {nm: np.array([float(r[i]) for r in rows]) for i, nm in enumerate(names)}
    return header, cols
