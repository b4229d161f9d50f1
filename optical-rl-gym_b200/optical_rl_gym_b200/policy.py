"""On-device MLP policy for the "PPO-policy actions" variant of the headline config (SURVEY.md row f4).

Architecture of the agent the reference trains and ships
(examples/stable_baselines3/DeepRMSA.ipynb: ``PPO(MlpPolicy, env, policy_kwargs=dict(net_arch=5*[128]))``;
examples/stable_baselines3/bkp/deeprmsa-ppo-trained/best_model.zip): observation 54 -> 5 x (Linear 128 + tanh)
shared trunk -> ``action_net`` (5 logits) and ``value_net`` (1).  ``from_sb3_zip`` reads ``policy.pth`` out of
such an archive (a plain ``state_dict``; Stable-Baselines3 itself is not needed).

Two forward paths: :meth:`forward` (plain torch float32, the numerics reference) and :meth:`act_native` -- the whole
``model.predict(obs, deterministic=True)`` as ONE fused sm_100a kernel of liborlg.so (``orlg_policy_act``: bf16
``tcgen05.mma`` with TMEM accumulators, weights resident in shared memory, tanh + argmax epilogue, int32 actions out).
:meth:`sample_native` is the same kernel with a sampling epilogue (``orlg_policy_sample``): sampled or argmax actions, their
log-probabilities and the value estimate, as PPO's rollout collection needs them.  The native weights follow the module:
an in-place update (``optimizer.step()``, ``load_state_dict``) rebuilds them at the next call.
"""
from __future__ import annotations

import io
import zipfile
from typing import Sequence

import torch


class MlpPolicy(torch.nn.Module):
    def __init__(self, obs_dim: int = 54, n_actions: int = 5, net_arch: Sequence[int] = (128,) * 5):
        super().__init__()
        layers, d = [], obs_dim
        for width in net_arch:
            layers += [torch.nn.Linear(d, width), torch.nn.Tanh()]
            d = width
        self.shared_net = torch.nn.Sequential(*layers)
        self.action_net = torch.nn.Linear(d, n_actions)
        self.value_net = torch.nn.Linear(d, 1)
        self.critic_net = None          # the critic's own trunk when the checkpoint has separate ones (SB3 >= 1.8)

    @classmethod
    def from_state_dict(cls, sd) -> "MlpPolicy":
        """``policy.pth`` of an SB3 ``ActorCriticPolicy`` with a shared trunk (keys ``mlp_extractor.shared_net.<2i>``)
        or with separate actor/critic trunks (``mlp_extractor.policy_net`` / ``mlp_extractor.value_net``, SB3 >= 1.8: the
        actor's trunk becomes ``shared_net``, the critic's is kept as ``critic_net``: ``forward``, :meth:`sample_native` and
        ``OpticalVecEnv.rollout_policy`` return its value (a second native handle evaluates it); the value column of
        :meth:`act_native`'s ``logits`` is the actor trunk's)."""
        shared = any(k.startswith("mlp_extractor.shared_net.") for k in sd)
        trunk = "mlp_extractor.shared_net." if shared else "mlp_extractor.policy_net."
        idx = sorted({int(k[len(trunk):].split(".")[0]) for k in sd if k.startswith(trunk)})
        widths = [sd["%s%d.weight" % (trunk, i)].shape[0] for i in idx]
        obs_dim = sd["%s%d.weight" % (trunk, idx[0])].shape[1]
        pol = cls(obs_dim, sd["action_net.weight"].shape[0], widths)
        mine = {}
        for j, i in enumerate(idx):
            mine["shared_net.%d.weight" % (2 * j)] = sd["%s%d.weight" % (trunk, i)]
            mine["shared_net.%d.bias" % (2 * j)] = sd["%s%d.bias" % (trunk, i)]
        for k in ("action_net.weight", "action_net.bias", "value_net.weight", "value_net.bias"):
            mine[k] = sd[k]
        pol.load_state_dict(mine)
        vtrunk = "mlp_extractor.value_net."
        if not shared and any(k.startswith(vtrunk) for k in sd):
            vidx = sorted({int(k[len(vtrunk):].split(".")[0]) for k in sd if k.startswith(vtrunk)})
            layers = []
            for i in vidx:
                w = sd["%s%d.weight" % (vtrunk, i)]
                lin = torch.nn.Linear(w.shape[1], w.shape[0])
                lin.load_state_dict({"weight": w, "bias": sd["%s%d.bias" % (vtrunk, i)]})
                layers += [lin, torch.nn.Tanh()]
            pol.critic_net = torch.nn.Sequential(*layers)
        return pol

    @classmethod
    def from_sb3_zip(cls, path, device=None) -> "MlpPolicy":
        with zipfile.ZipFile(path) as z:
            sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
        pol = cls.from_state_dict(sd)
        return pol.to(device) if device is not None else pol

    # ------------------------------------------------------------------ fused native kernel (csrc/orlg_policy.cuh)
    def _native_specs(self):
        """What the native handles are built from: ``{"actor": spec, "critic": spec | None}`` with ``spec`` =
        ``(trunk Linear layers, head Linear layers, obs_dim)``.  The actor's heads are ``action_net`` then ``value_net``.  With
        a separate critic trunk (SB3 >= 1.8) the critic handle evaluates that trunk; its one-row action head is ``value_net``
        as well (its actions are never requested), so its value output is ``value_net(critic_net(obs))``."""
        lins = [m for m in self.shared_net if isinstance(m, torch.nn.Linear)]
        specs = {"actor": (lins, [self.action_net, self.value_net], lins[0].in_features), "critic": None}
        if self.critic_net is not None:
            clins = [m for m in self.critic_net if isinstance(m, torch.nn.Linear)]
            specs["critic"] = (clins, [self.value_net, self.value_net], clins[0].in_features)
        return specs

    @staticmethod
    def _create_handle(device_index: int, spec):
        import ctypes as C

        import numpy as np

        from . import _native as nat

        lins, heads, obs_dim = spec
        mats = list(lins) + list(heads)
        w = np.concatenate([m.weight.detach().float().cpu().numpy().reshape(-1) for m in mats]).astype(np.float32)
        b = np.concatenate([m.bias.detach().float().cpu().numpy().reshape(-1) for m in mats]).astype(np.float32)
        h = C.c_void_p()
        nat.check(nat.lib().orlg_policy_create(device_index, obs_dim, lins[0].out_features, len(lins), heads[0].out_features,
                                               w.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), C.byref(h)))
        return h

    def _weights_key(self):
        """Identity of the weights the native handles are built from.  optimizer.step() and load_state_dict() write the
        parameters in place, which bumps their ``_version``; ``.to()`` and replaced parameters or layers change the storage
        (a data pointer also identifies the device).  Read straight from the module dicts: this runs before every launch,
        and ``self.parameters()`` alone would cost several times the rest of the call."""
        key = []
        for seq in (self._modules["shared_net"], self._modules.get("critic_net")):
            if seq is not None:
                for m in seq._modules.values():
                    if isinstance(m, torch.nn.Linear):
                        w, b = m._parameters["weight"], m._parameters["bias"]
                        key += (w._version, w.data_ptr(), b._version, b.data_ptr())
        for name in ("action_net", "value_net"):
            w, b = self._modules[name]._parameters["weight"], self._modules[name]._parameters["bias"]
            key += (w._version, w.data_ptr(), b._version, b.data_ptr())
        return tuple(key)

    def _destroy_handles(self, handles, device_index):
        from . import _native as nat

        if any(h is not None for h in handles):
            if torch.cuda.is_available() and device_index is not None:
                torch.cuda.current_stream(device_index).synchronize()      # launches queued with the old weights finish first
            for h in handles:
                if h is not None:
                    nat.lib().orlg_policy_destroy(h)

    def _native_handles(self, device_index: int):
        """(actor handle, critic handle | None) holding the CURRENT weights: rebuilt when a parameter was changed in place
        (optimizer step, load_state_dict) or moved since the handles were made."""
        cache = self.__dict__.setdefault("_native_cache", {})
        key = self._weights_key()
        entry = cache.get(device_index)
        if entry is not None and entry[0] == key:
            return entry[1], entry[2]
        if entry is not None:
            del cache[device_index]
            self._destroy_handles(entry[1:], device_index)
        specs = self._native_specs()
        actor = self._create_handle(device_index, specs["actor"])
        try:
            critic = None if specs["critic"] is None else self._create_handle(device_index, specs["critic"])
        except Exception:
            self._destroy_handles((actor,), device_index)
            raise
        cache[device_index] = (key, actor, critic)
        return actor, critic

    def _native_handle(self, device_index: int):
        """The actor's native handle (``orlg_policy_act`` / ``orlg_policy_sample``) with the current weights."""
        return self._native_handles(device_index)[0]

    def __del__(self):
        try:
            cache = self.__dict__.get("_native_cache") or {}
            for dev, entry in list(cache.items()):
                self._destroy_handles(entry[1:], dev)
            cache.clear()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass

    def _check_obs(self, obs: torch.Tensor):
        d = self.shared_net[0].in_features
        if not (torch.is_tensor(obs) and obs.is_cuda and obs.dtype == torch.float32 and obs.dim() == 2 and obs.shape[1] == d
                and obs.is_contiguous()):
            raise ValueError("observations must be a contiguous float32 CUDA tensor [N, %d], got %s %s %s%s" % (
                d, tuple(obs.shape), obs.dtype, obs.device, "" if obs.is_contiguous() else " (not contiguous)"))
        return obs.shape[0]

    @staticmethod
    def _check_out(name, t, shape, dtype, device):
        if t is not None and (tuple(t.shape) != shape or t.dtype != dtype or t.device != device or not t.is_contiguous()):
            raise ValueError("%s must be a contiguous %s tensor %s on %s, got %s %s %s" % (
                name, dtype, shape, device, tuple(t.shape), t.dtype, t.device))

    @torch.no_grad()
    def act_native(self, obs: torch.Tensor, out: torch.Tensor = None, logits: torch.Tensor = None) -> torch.Tensor:
        """Deterministic actions int32 ``[N, 1]`` from float32 CUDA observations ``[N, obs_dim]`` through the fused tensor-core
        kernel; ``logits`` (optional float32 ``[N, n_actions + 1]``) receives the logits and the value estimate."""
        import ctypes as C

        from . import _native as nat

        n = self._check_obs(obs)
        if out is None:
            out = torch.empty((n, 1), dtype=torch.int32, device=obs.device)
        self._check_out("out", out, (n, 1), torch.int32, obs.device)
        self._check_out("logits", logits, (n, self.action_net.out_features + 1), torch.float32, obs.device)
        h = self._native_handle(obs.device.index)
        stream = C.c_void_p(torch.cuda.current_stream(obs.device).cuda_stream)
        nat.check(nat.lib().orlg_policy_act(h, C.c_void_p(obs.data_ptr()), n, C.c_void_p(out.data_ptr()),
                                            None if logits is None else C.c_void_p(logits.data_ptr()), stream))
        return out

    @torch.no_grad()
    def sample_native(self, obs: torch.Tensor, *, seed: int, counter: int, row_id_base: int = 0, deterministic: bool = False,
                      out=None):
        """What PPO collects per observation, from the fused kernel: ``(actions int32 [N, 1], log_prob f32 [N], value f32 [N])``.
        Sampled actions come from softmax(logits) with one Philox4x32-10 draw per row (key ``seed``, counter
        ``(counter, 0, row_id_base + row, 3)``); ``deterministic=True`` gives the argmax of :meth:`act_native`.  ``log_prob`` is
        log softmax(logits)[action]; ``value`` is the critic's (``critic_net``) when the policy has a separate one.
        ``out`` = the three tensors to fill."""
        import ctypes as C

        from . import _native as nat

        n = self._check_obs(obs)
        if out is None:
            out = (torch.empty((n, 1), dtype=torch.int32, device=obs.device), torch.empty(n, dtype=torch.float32, device=obs.device),
                   torch.empty(n, dtype=torch.float32, device=obs.device))
        actions, log_prob, value = out
        self._check_out("actions", actions, (n, 1), torch.int32, obs.device)
        self._check_out("log_prob", log_prob, (n,), torch.float32, obs.device)
        self._check_out("value", value, (n,), torch.float32, obs.device)
        actor, critic = self._native_handles(obs.device.index)
        stream = C.c_void_p(torch.cuda.current_stream(obs.device).cuda_stream)
        draw = nat.PolicyDraw(seed=int(seed) & (2 ** 64 - 1), counter_dev=None, counter=int(counter) & 0xFFFFFFFF,
                              deterministic=int(bool(deterministic)), row_id_base=int(row_id_base))
        L, o = nat.lib(), C.c_void_p(obs.data_ptr())
        nat.check(L.orlg_policy_sample(actor, o, n, C.byref(draw), C.c_void_p(actions.data_ptr()), C.c_void_p(log_prob.data_ptr()),
                                       None if critic is not None else C.c_void_p(value.data_ptr()), stream))
        if critic is not None:
            nat.check(L.orlg_policy_sample(critic, o, n, C.byref(draw), None, None, C.c_void_p(value.data_ptr()), stream))
        return actions, log_prob, value

    def forward(self, obs: torch.Tensor):
        """(logits [N, n_actions], value [N]) -- observations are used as they are (SB3 ``preprocess_obs`` of a
        Box space is a cast to float)."""
        x = obs.to(self.action_net.weight.dtype)
        latent = self.shared_net(x)
        latent_vf = latent if self.critic_net is None else self.critic_net(x)
        return self.action_net(latent), self.value_net(latent_vf).squeeze(-1)

    @torch.no_grad()
    def act(self, obs: torch.Tensor, deterministic: bool = True, generator=None) -> torch.Tensor:
        """int32 actions [N, 1] ready for ``OpticalVecEnv.step_raw`` (``model.predict(obs, deterministic=...)``)."""
        logits, _ = self.forward(obs)
        if deterministic:
            a = logits.argmax(dim=-1)
        else:
            a = torch.multinomial(torch.softmax(logits.float(), dim=-1), 1, generator=generator).squeeze(-1)
        return a.to(torch.int32).unsqueeze(-1)
