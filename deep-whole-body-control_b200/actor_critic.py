"""Flat-buffer ActorCritic: the parameters of `rsl_rl.modules.ActorCritic`
(rsl_rl/rsl_rl/modules/actor_critic.py:86-298, cited AC:line) in ONE fp32 device buffer.

Tensors are laid out in `ActorCritic.parameters()` order (std first, AC:296) with each tensor
start aligned to 32 floats (128 B) so every GEMM operand is 16-byte aligned; the padding holds
zeros, receives zero gradient and is inert under Adam.  `state_dict()` / `load_state_dict()`
use the reference's key names and shapes, so checkpoints written by
`OnPolicyRunner.save` (rsl_rl/runners/on_policy_runner.py:276-282) round-trip.
"""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import List, Tuple

import torch

from . import _lib as L

ALIGN = 32


def manifest(num_prop=76, num_priv=24, num_hist=10, priv_dims=(64, 20), actor_dims=(128,), critic_dims=(128,),
             leg_dims=(128, 128), arm_dims=(128, 128), n_leg=12, n_arm=6) -> List[Tuple[str, tuple]]:
    """(name, shape) in ActorCritic.parameters() order (AC:186-298)."""
    m = [("std", (1, n_leg + n_arm))]

    def lin(prefix, idx, o, i):
        m.append((f"{prefix}.{idx}.weight", (o, i)))
        m.append((f"{prefix}.{idx}.bias", (o,)))
    d = num_priv
    for k, o in enumerate(priv_dims):
        lin("actor.priv_encoder", 2 * k, o, d)
        d = o
    latent = d
    lin("actor.history_encoder.encoder", 0, 30, num_prop)                               # AC:49-51
    m += [("actor.history_encoder.conv_layers.0.weight", (20, 30, 4)), ("actor.history_encoder.conv_layers.0.bias", (20,)),
          ("actor.history_encoder.conv_layers.2.weight", (10, 20, 2)), ("actor.history_encoder.conv_layers.2.bias", (10,))]  # AC:58-62
    lin("actor.history_encoder.linear_output", 0, latent, 30)                           # AC:71-73
    d = num_prop + latent
    for k, o in enumerate(actor_dims):
        lin("actor.actor_backbone", 2 * k, o, d)
        d = o
    for head, dims, n_out in (("actor.actor_leg_control_head", leg_dims, n_leg), ("actor.actor_arm_control_head", arm_dims, n_arm)):
        dd = d
        for k, o in enumerate(list(dims) + [n_out]):
            lin(head, 2 * k, o, dd)
            dd = o
    d = num_prop + num_priv
    for k, o in enumerate(critic_dims):
        lin("critic.critic_backbone", 2 * k, o, d)
        d = o
    for head, dims in (("critic.critic_leg_control_head", leg_dims), ("critic.critic_arm_control_head", arm_dims)):
        dd = d
        for k, o in enumerate(list(dims) + [1]):
            lin(head, 2 * k, o, dd)
            dd = o
    return m


class FlatActorCritic:
    is_recurrent = False

    def __init__(self, num_actor_obs=76, num_critic_obs=76, num_actions=18, actor_hidden_dims=(128,), critic_hidden_dims=(128,),
                 priv_encoder_dims=(64, 20), activation="elu", init_std=None, device="cuda:0", seed=None, **kwargs):
        if activation not in L.ACTIVATIONS:
            raise L.DwbcError(f"activation={activation!r}: rsl_rl's get_activation offers {sorted(L.ACTIVATIONS)}")
        self.activation = activation
        if kwargs.get("adaptive_arm_gains", False):
            raise L.DwbcError("adaptive_arm_gains=True is outside the hot path (WGC:168: False)")
        self.num_prop = kwargs.get("num_prop", num_actor_obs)
        self.num_priv, self.num_hist = kwargs.get("num_priv", 24), kwargs.get("num_hist", 10)
        self.num_leg_actions, self.num_arm_actions = kwargs.get("num_leg_actions", 12), kwargs.get("num_arm_actions", 6)
        self.leg_dims = tuple(kwargs.get("leg_control_head_hidden_dims", (128, 128)))
        self.arm_dims = tuple(kwargs.get("arm_control_head_hidden_dims", (128, 128)))
        self.priv_dims, self.actor_dims, self.critic_dims = tuple(priv_encoder_dims), tuple(actor_hidden_dims), tuple(critic_hidden_dims)
        self.num_obs = self.num_prop * (self.num_hist + 1) + self.num_priv
        self.device = torch.device(device)
        self.manifest = manifest(self.num_prop, self.num_priv, self.num_hist, self.priv_dims, self.actor_dims, self.critic_dims,
                                 self.leg_dims, self.arm_dims, self.num_leg_actions, self.num_arm_actions)
        self.offsets, off = OrderedDict(), 0
        for name, shape in self.manifest:
            self.offsets[name] = off
            off += (math.prod(shape) + ALIGN - 1) // ALIGN * ALIGN
        self.num_params = off
        self.num_real_params = sum(math.prod(s) for _, s in self.manifest)
        self.flat = torch.zeros(self.num_params, device=self.device)
        self.views = OrderedDict((n, self.flat[self.offsets[n]:self.offsets[n] + math.prod(s)].view(s)) for n, s in self.manifest)
        self.reset_parameters(init_std, seed)
        self.net_cfg = self._make_net_cfg()

    # -- torch default init of nn.Linear / nn.Conv1d (kaiming_uniform(a=sqrt 5) == U(+-1/sqrt(fan_in))), AC relies on it
    def reset_parameters(self, init_std=None, seed=None):
        g = torch.Generator(device="cpu")
        if seed is not None:
            g.manual_seed(seed)
        prev_fan = 1
        for name, shape in self.manifest:
            if name == "std":
                std = torch.tensor(init_std if init_std is not None else [[1.0] * shape[1]], dtype=torch.float).reshape(shape)
                self.views[name].copy_(std)
                continue
            if len(shape) > 1:
                prev_fan = math.prod(shape[1:])
            b = 1.0 / math.sqrt(prev_fan)
            self.views[name].copy_((torch.rand(shape, generator=g) * 2 - 1) * b)

    def _make_net_cfg(self) -> L.NetCfg:
        c, o = L.NetCfg(), self.offsets
        c.abi_version = L.ABI_VERSION
        c.num_prop, c.num_priv, c.num_hist, c.num_obs = self.num_prop, self.num_priv, self.num_hist, self.num_obs
        c.n_leg, c.n_arm = self.num_leg_actions, self.num_arm_actions

        def dims(n_attr, d_attr, d):
            if len(d) > L.MAX_LAYERS:
                raise L.DwbcError("too many layers for the ABI struct")
            setattr(c, n_attr, len(d))
            for i, v in enumerate(d):
                getattr(c, d_attr)[i] = v
        dims("n_priv_layers", "priv_dims", self.priv_dims)
        dims("n_actor_layers", "actor_dims", self.actor_dims)
        dims("n_critic_layers", "critic_dims", self.critic_dims)
        dims("n_leg_layers", "leg_dims", self.leg_dims)
        dims("n_arm_layers", "arm_dims", self.arm_dims)
        c.hist_proj, c.hist_c1, c.hist_k1, c.hist_s1, c.hist_c2, c.hist_k2, c.hist_s2 = 30, 20, 4, 2, 10, 2, 1
        c.num_params, c.off_std = self.num_params, o["std"]
        c.activation = L.ACTIVATIONS[self.activation]

        def offs(w_attr, b_attr, prefix, n):
            for i in range(n):
                getattr(c, w_attr)[i] = o[f"{prefix}.{2 * i}.weight"]
                getattr(c, b_attr)[i] = o[f"{prefix}.{2 * i}.bias"]
        offs("off_priv_w", "off_priv_b", "actor.priv_encoder", len(self.priv_dims))
        for i, k in enumerate(("encoder.0", "conv_layers.0", "conv_layers.2", "linear_output.0")):
            c.off_hist_w[i] = o[f"actor.history_encoder.{k}.weight"]
            c.off_hist_b[i] = o[f"actor.history_encoder.{k}.bias"]
        offs("off_actor_w", "off_actor_b", "actor.actor_backbone", len(self.actor_dims))
        offs("off_aleg_w", "off_aleg_b", "actor.actor_leg_control_head", len(self.leg_dims) + 1)
        offs("off_aarm_w", "off_aarm_b", "actor.actor_arm_control_head", len(self.arm_dims) + 1)
        offs("off_critic_w", "off_critic_b", "critic.critic_backbone", len(self.critic_dims))
        offs("off_cleg_w", "off_cleg_b", "critic.critic_leg_control_head", len(self.leg_dims) + 1)
        offs("off_carm_w", "off_carm_b", "critic.critic_arm_control_head", len(self.arm_dims) + 1)
        return c

    @property
    def hist_range(self) -> Tuple[int, int]:
        """[first, first+count) of the history-encoder parameters in the flat buffer (contiguous)."""
        names = [n for n, _ in self.manifest if n.startswith("actor.history_encoder.")]
        first = self.offsets[names[0]]
        last, shape = names[-1], dict(self.manifest)[names[-1]]
        end = self.offsets[last] + (math.prod(shape) + ALIGN - 1) // ALIGN * ALIGN
        return first, end - first

    # -- nn.Module-like surface the runner touches (OPR:203-205,277-279,286; PPO:293-296)
    @property
    def std(self):
        return self.views["std"]

    def state_dict(self):
        return OrderedDict((k, v.detach().clone()) for k, v in self.views.items())

    def load_state_dict(self, sd, strict=True):
        missing = [k for k in self.views if k not in sd]
        unexpected = [k for k in sd if k not in self.views]
        if strict and (missing or unexpected):
            raise KeyError(f"missing {missing}, unexpected {unexpected}")
        for k, v in sd.items():
            if k in self.views:
                self.views[k].copy_(torch.as_tensor(v).to(self.device).reshape(self.views[k].shape))

    def parameters(self):
        return list(self.views.values())

    def named_parameters(self):
        return list(self.views.items())

    def flat_from(self, values: dict) -> torch.Tensor:
        """Pack {name: tensor} (reference layout) into a new padded flat buffer."""
        out = torch.zeros_like(self.flat)
        for n, s in self.manifest:
            out[self.offsets[n]:self.offsets[n] + math.prod(s)] = torch.as_tensor(values[n]).to(self.device).reshape(-1)
        return out

    def unflat(self, flat: torch.Tensor) -> "OrderedDict[str, torch.Tensor]":
        return OrderedDict((n, flat[self.offsets[n]:self.offsets[n] + math.prod(s)].view(s)) for n, s in self.manifest)

    def to(self, device):
        return self

    def train(self):
        return self

    def eval(self):
        return self

    def reset(self, dones=None):
        pass
