"""The reference's OWN driver, unmodified (rsl_rl/runners/on_policy_runner.py from baseline/_ref: __init__ OPR:48-91, learn OPR:93-177, save
OPR:276-282), running on the fused classes: FusedActorCritic / FusedPPO resolved through OPR's eval() of the class names, a VecEnv whose step()
is the fused post-physics kernel behind synthetic physics.  Two iterations: it = 0 is a student iteration (hist_encoding = it % 20 == 0 ->
update_dagger), it = 1 a teacher iteration (update).  Checked: the checkpoint the runner writes loads STRICTLY into the reference's own
ActorCritic, and that reference module (CPU, torch) reproduces the fused policy's act_inference / evaluate on fresh observations."""
import os
import sys
import types

import numpy as np
import pytest
import torch

import envstate as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")
pytestmark = pytest.mark.gpu


class SyntheticWidowGo1(object):
    """VecEnv surface (rsl_rl/env/vec_env.py:36-59, WG:1156-1199) over FusedWidowGo1Core; the physics between pre- and post-physics is a
    pool of synthetic simulator states."""

    def __init__(self, n_envs, device, seed=3):
        from dwbc_b200 import synth
        from dwbc_b200.env import FusedWidowGo1Core
        p = E.make_params("flat", n_envs)
        self.core = FusedWidowGo1Core(p, device, state=E.initial(p, seed), seed=77)
        self.p, self.device, self.seed, self.t = p, device, seed, 0
        self.num_envs, self.num_obs, self.num_privileged_obs, self.num_actions = n_envs, p.num_obs, None, p.num_actions
        self.max_episode_length = p.max_episode_length
        self.cfg = types.SimpleNamespace(env=types.SimpleNamespace(num_proprio=p.num_prop, num_priv=p.num_priv, history_len=p.history_len))
        self.p_gains, self.d_gains = torch.tensor(p.p_gains, device=device), torch.tensor(p.d_gains, device=device)
        self.default_dof_pos = torch.tensor(p.default_dof_pos, device=device)
        self.synth = synth

    episode_length_buf = property(lambda s: s.core.episode_length_buf, lambda s, v: setattr(s.core, "episode_length_buf", v))

    def update_command_curriculum(self):
        self.core.update_command_curriculum()

    def get_observations(self):
        return self.core.obs_buf

    def get_privileged_observations(self):
        return None

    def _physics(self, core):
        self.t += 1
        sim = self.synth.sim_state(self.p, self.seed, self.t, rp_sigma=0.05, z_lo=0.327)
        for k, dst in (("root_states", core._root_states), ("dof_state", core.dof_state), ("rigid_body_state", core._rigid_body_state),
                       ("contact_forces", core._contact_forces), ("force_sensor", core.force_sensor_tensor), ("torques", core.torques)):
            dst.copy_(torch.from_numpy(sim[k]).to(self.device))

    def reset(self):
        self.step(torch.zeros(self.num_envs, self.num_actions, device=self.device))
        return self.core.obs_buf, None

    def step(self, actions):
        return self.core.step(actions, physics=self._physics)


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "rsl_rl")), reason="baseline/_ref (unmodified rsl_rl) is absent: run baseline/install_reference.sh")
def test_unmodified_on_policy_runner_drives_the_fused_classes(tmp_path):
    import json
    for pth in (REF, os.path.join(ROOT, "tests", "fakes")):
        if pth not in sys.path:
            sys.path.insert(0, pth)
    import rsl_rl.runners.on_policy_runner as opr                     # the reference's file, unmodified (wandb / torchinfo: tests/fakes)
    from rsl_rl.modules import ActorCritic
    import torchinfo
    from dwbc_b200 import runner_compat as RC
    cfg = json.load(open(os.path.join(ROOT, "baseline", "widowgo1_train_cfg.json")))
    names = RC.install(opr)
    train_cfg = dict(policy=dict(cfg["policy"]), algorithm=dict(cfg["algorithm"], num_learning_epochs=2, num_mini_batches=2, precision="tf32x3"),
                     runner=dict(cfg["runner"], num_steps_per_env=8, save_interval=100, **names))
    dev = "cuda:0"
    N = 256
    env = SyntheticWidowGo1(N, dev)
    runner = opr.OnPolicyRunner(env, train_cfg, log_dir=str(tmp_path), device=dev)
    assert torchinfo.last["params"] == runner.alg.actor_critic.num_real_params == 168698       # summary() saw the nn.Module (OPR:78)
    assert isinstance(runner.alg.actor_critic, torch.nn.Module) and type(runner.alg).__name__ == "FusedPPO"
    p0 = runner.alg.actor_critic.flat.clone()
    runner.learn(2, init_at_random_ep_len=True)                        # it 0: hist_encoding -> update_dagger; it 1: update
    assert runner.current_learning_iteration == 2 and runner.alg.counter == 2
    moved = (runner.alg.actor_critic.flat - p0).abs()
    hf, hc = runner.alg.actor_critic.hist_range
    assert float(moved[hf:hf + hc].max()) > 0 and float(moved[:hf].max()) > 0          # both optimizers stepped
    ck = torch.load(os.path.join(str(tmp_path), "model_2.pt"), map_location="cpu", weights_only=False)
    a = cfg["actor_critic_args"]
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        ref_ac = ActorCritic(a["num_actor_obs"], a["num_critic_obs"], a["num_actions"], **cfg["policy"], num_priv=a["num_priv"], num_hist=a["num_hist"],
                             num_prop=a["num_prop"])
    ref_ac.load_state_dict(ck["model_state_dict"], strict=True)       # reference key names and shapes (OPR:276-290 round trip)
    assert "optimizer_state_dict" in ck and ck["iter"] == 2
    obs = torch.randn(777, 860, generator=torch.Generator().manual_seed(1)).clamp(-3, 3)
    with torch.no_grad():
        for hist in (False, True):
            want = ref_ac.act_inference(obs, hist_encoding=hist)
            got = runner.alg.actor_critic.act_inference(obs.to(dev), hist_encoding=hist).cpu()
            np.testing.assert_allclose(got.numpy(), want.numpy(), rtol=0, atol=2e-5)
        np.testing.assert_allclose(runner.alg.actor_critic.evaluate(obs.to(dev)).cpu().numpy(), ref_ac.evaluate(obs).numpy(), rtol=0, atol=2e-5)
