"""TEST INFRASTRUCTURE ONLY -- the ActorCritic of oracle/ppo_oracle.py with rsl_rl's other hidden activations.

`get_activation` (AC) maps a name to the module every hidden layer applies: the privileged encoder, the four history-encoder stages, the
backbones and the heads' hidden layers; the actor heads end in tanh, the critic heads are linear.  The functions below restate
ppo_oracle's network functions with that activation as a parameter and apply torch's own function for it (F.selu, F.relu, F.leaky_relu,
torch.tanh, torch.sigmoid), so torch's arithmetic is the reference.  Everything that does not involve the activation (log-prob, entropy,
schedules, gather, clip, Adam) is ppo_oracle's.  With act="elu" every function returns exactly what its ppo_oracle namesake returns
(tests/test_activations_cpu.py holds that), which ties this module to the oracle the golden vectors pin.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle import ppo_oracle as PO

# rsl_rl `get_activation`: the torch function of the module each name builds ("crelu" is a plain nn.ReLU() there)
ACTIVATIONS = dict(elu=F.elu, selu=F.selu, relu=F.relu, crelu=F.relu, lrelu=F.leaky_relu, tanh=torch.tanh, sigmoid=torch.sigmoid)


def _mlp(P, prefix, x, last_act, act):
    """Linear(+act) blocks prefix.{0,2,4..}; the last one is followed by `last_act` in {"act", "tanh", None}."""
    f, n = ACTIVATIONS[act], PO._count(P, prefix)
    for k in range(n):
        x = F.linear(x, P[f"{prefix}.{2 * k}.weight"], P[f"{prefix}.{2 * k}.bias"])
        if k < n - 1 or last_act == "act":
            x = f(x)
        elif last_act == "tanh":
            x = torch.tanh(x)
    return x


def priv_latent(P, obs, act, num_prop=76, num_priv=24):
    return _mlp(P, "actor.priv_encoder", obs[:, num_prop:num_prop + num_priv], "act", act)                    # AC:219-221


def hist_latent(P, obs, act, num_prop=76, num_hist=10):
    f = ACTIVATIONS[act]
    h = obs[:, -num_hist * num_prop:].reshape(-1, num_hist, num_prop)                                          # AC:223-225
    nd = h.shape[0]
    pre = "actor.history_encoder"
    proj = f(F.linear(h.reshape(nd * num_hist, -1), P[pre + ".encoder.0.weight"], P[pre + ".encoder.0.bias"]))   # AC:80
    x = proj.reshape(nd, num_hist, -1).permute(0, 2, 1)
    x = f(F.conv1d(x, P[pre + ".conv_layers.0.weight"], P[pre + ".conv_layers.0.bias"], stride=2))            # AC:59
    x = f(F.conv1d(x, P[pre + ".conv_layers.2.weight"], P[pre + ".conv_layers.2.bias"], stride=1))            # AC:60
    return f(F.linear(x.flatten(1), P[pre + ".linear_output.0.weight"], P[pre + ".linear_output.0.bias"]))    # AC:72


def actor_mean(P, obs, act, hist_encoding=False, num_prop=76):
    z = hist_latent(P, obs, act) if hist_encoding else priv_latent(P, obs, act)                                # AC:204-217
    h = _mlp(P, "actor.actor_backbone", torch.cat([obs[:, :num_prop], z], dim=1), "act", act)
    return torch.cat([_mlp(P, "actor.actor_leg_control_head", h, "tanh", act), _mlp(P, "actor.actor_arm_control_head", h, "tanh", act)], dim=-1)


def critic_values(P, obs, act, num_prop=76, num_priv=24):
    h = _mlp(P, "critic.critic_backbone", obs[:, :num_prop + num_priv], "act", act)                           # AC:280-286
    return torch.cat([_mlp(P, "critic.critic_leg_control_head", h, None, act), _mlp(P, "critic.critic_arm_control_head", h, None, act)], dim=-1)


def policy_act(P, obs, eps, act, hist_encoding=False):
    """PPO.act (PPO:115-127) with the standard-normal draw `eps` supplied by the caller."""
    with torch.no_grad():
        mean = actor_mean(P, obs, act, hist_encoding)
        sigma = mean * 0.0 + P["std"]
        actions = mean + sigma * eps
        return dict(actions=actions, values=critic_values(P, obs, act), log_prob=PO.log_prob2(mean, P["std"], actions), mean=mean, sigma=sigma)


def minibatch_loss(P, mb, hp, counter, act):
    """ppo_oracle.minibatch_loss (PPO:166-221) with the hidden activation `act`; the torque-supervision branch is not restated here."""
    assert not hp.get("torque_supervision", False)
    obs = mb["obs"]
    mean = actor_mean(P, obs, act)
    logp = PO.log_prob2(mean, P["std"], mb["actions"])
    value = critic_values(P, obs, act)
    ent = PO.entropy2(mean, P["std"])
    zp = priv_latent(P, obs, act)
    with torch.no_grad():
        zh = hist_latent(P, obs, act)
    reg = (zp - zh.detach()).norm(p=2, dim=1).mean()
    rho = PO.value_mixing_ratio(counter, hp["mixing_schedule"])
    adv = mb["advantages"]
    mix = torch.zeros_like(adv)
    mix[..., 0] = adv[..., 0] + rho * adv[..., 1]
    mix[..., 1] = adv[..., 1] + rho * adv[..., 0]
    ratio = torch.exp(logp - mb["old_log_prob"])
    clip = hp["clip_param"]
    surr = torch.max(-mix * ratio, -mix * torch.clamp(ratio, 1.0 - clip, 1.0 + clip)).mean()
    if hp.get("use_clipped_value_loss", True):
        vclip = mb["values"] + (value - mb["values"]).clamp(-clip, clip)
        vloss = torch.max((value - mb["returns"]).pow(2), (vclip - mb["returns"]).pow(2)).mean()
    else:
        vloss = (mb["returns"] - value).pow(2).mean()
    creg = PO.priv_reg_coef(counter, hp["priv_reg_coef_schedual"])
    loss = surr + hp["value_loss_coef"] * vloss - hp["entropy_coef"] * ent.mean() + creg * reg
    return loss, dict(surrogate=surr.detach(), value=vloss.detach(), priv_reg=reg.detach(), ratio=ratio.detach())


def ppo_update(P, opt, storage, indices, hp, counter, act):
    """ppo_oracle.ppo_update (PPO:152-263, min-std PPO:293-296) with the hidden activation `act`."""
    names = list(P.keys())
    nmb, nep = hp["num_mini_batches"], hp["num_learning_epochs"]
    mbs = indices.numel() // nmb
    for _ in range(nep):
        for i in range(nmb):
            mb = PO.gather(storage, indices[i * mbs:(i + 1) * mbs])
            for n in names:
                P[n].requires_grad_(True)
                P[n].grad = None
            loss, _ = minibatch_loss(P, mb, hp, counter, act)
            loss.backward()
            G = {n: (P[n].grad.detach() if P[n].grad is not None else None) for n in names}
            for n in names:
                P[n].requires_grad_(False)
            PO.clip_grad_norm(G, names, hp["max_grad_norm"])
            with torch.no_grad():
                opt.step(P, G)
    if hp.get("min_policy_std") is not None:
        P["std"] = torch.max(P["std"], torch.tensor(hp["min_policy_std"]))
