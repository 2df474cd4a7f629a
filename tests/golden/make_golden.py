"""Generate the golden vectors under tests/golden/ by EXECUTING THE UNMODIFIED REFERENCE.

Needs a checkout of the original Deep-Whole-Body-Control repository, named by DWBC_REFERENCE:

    DWBC_REFERENCE=<checkout> python tests/golden/make_golden.py

For each fixture the script (1) runs the reference's own Python on CPU (env half through the
fake isaacgym of tests/fakes, update half straight from its rsl_rl), (2) runs the
restatement in oracle/ on the same inputs and ASSERTS it reproduces the reference (this is
what pins the oracle), (3) stores the reference outputs.  Inputs are not stored: they are
regenerated from (seed, stream) by dwbc_b200.synth (integer-hash, machine independent).
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, ".."))
import ref_harness as H  # noqa: E402
import envstate as E  # noqa: E402
from dwbc_b200 import synth  # noqa: E402
from oracle import ppo_oracle as PO  # noqa: E402
from oracle.env_oracle import EnvOracle, heights_obs as EO_heights_obs  # noqa: E402

ENV_N, ENV_STEPS, ENV_SEED, ENV_COUNTER0 = 48, 20, 3, 143
PPO_N, PPO_T, PPO_SEED, PPO_COUNTER = 64, 40, 7, 1500


def _close(a, b, tol, what):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    d = float((a - b).abs().max()) if a.numel() else 0.0
    assert d <= tol, f"oracle != reference for {what}: max|diff|={d}"
    return d


def _ref_heights_obs(ref):
    """Perceptive observation columns of the BASE class (LR:205-226; WidowGo1.compute_observations, WG:966-1001, does not append
    them): run LeggedRobot.compute_observations on the reference object and keep the last 187 columns."""
    from legged_gym.envs.base.legged_robot import LeggedRobot
    keep = ref.obs_buf
    ref.projected_gravity, ref.add_noise = torch.zeros(ref.num_envs, 3), False
    LeggedRobot.compute_observations(ref)
    h = ref.obs_buf[:, -ref.measured_heights.shape[1]:].clone()
    ref.obs_buf = keep
    return h


def gen_env(name):
    p = E.make_params(name, ENV_N)
    st = E.initial(p, ENV_SEED)
    ref = H.make_reference_env(p, st, ENV_SEED)
    orc = EnvOracle(p, E.oracle_state(p, st))
    rt = E.runtime(p)
    ref.update_command_curriculum()
    ref.common_step_counter = orc.common_step_counter = ENV_COUNTER0
    out = {k: [] for k in ("obs100", "rew", "arm_rew", "reset", "time_out", "commands", "ee_goal_sphere",
                           "goal_timer", "ep_len", "heights", "ep_stats", "env_origins_pre", "env_origins", "terrain_levels",
                           "heights_obs")}
    worst = 0.0
    for t in range(1, ENV_STEPS + 1):
        out["env_origins_pre"].append(ref.env_origins.numpy().copy())
        sim = E.sim_state(p, ENV_SEED, t, ref.env_origins)
        H.load_sim_into_reference(ref, p, sim)
        E.load_sim_into_oracle(orc, p, sim)
        tab = torch.from_numpy(synth.rand_table(p, ENV_SEED, t))
        ref._rr.table = tab
        ref.post_physics_step()
        robs = torch.clip(ref.obs_buf, -p.clip_observations, p.clip_observations)        # WG:1195-1196
        obs, rew, arew, rst, ex = orc.post_physics_step(tab, rt)
        pairs = [(robs, obs, "obs"), (ref.rew_buf, rew, "rew"), (ref.arm_rew_buf, arew, "arm_rew"),
                 (ref.reset_buf, rst, "reset"), (ref.time_out_buf, orc.s.time_out_buf, "time_out"),
                 (ref.obs_history_buf, orc.s.obs_history_buf, "hist"), (ref._root_states, orc.s.root_states_full, "root"),
                 (ref.dof_state, orc.s.dof_state, "dof"), (ref.commands, orc.s.commands, "commands"),
                 (ref.ee_goal_sphere, orc.s.ee_goal_sphere, "goal"), (ref.ee_start_sphere, orc.s.ee_start_sphere, "start"),
                 (ref.ee_goal_cart, orc.s.ee_goal_cart, "goal_cart"), (ref.goal_timer, orc.s.goal_timer, "timer"),
                 (ref.curr_ee_goal_cart, orc.s.curr_ee_goal_cart, "curr_cart"),
                 (ref.curr_ee_goal_sphere, orc.s.curr_ee_goal_sphere, "curr_sphere"),
                 (ref.last_root_vel, orc.s.last_root_vel, "last_root_vel"), (ref.last_dof_vel, orc.s.last_dof_vel, "last_dof_vel"),
                 (ref.last_actions, orc.s.last_actions, "last_actions"), (ref.base_lin_vel, orc.s.base_lin_vel, "blv"),
                 (ref.base_yaw_quat, orc.s.base_yaw_quat, "byq"),
                 (ref.episode_length_buf, orc.s.episode_length_buf, "ep_len"),
                 (ref.action_history_buf, orc.s.action_history_buf, "ahist"),
                 (ref.ee_goal_orn_euler, orc.s.ee_goal_orn_euler, "goal_orn"), (ref.feet_air_time, orc.s.feet_air_time, "fat")]
        pairs += [(ref.episode_sums[k], orc.s.episode_sums[k], "sum_" + k) for k in ref.episode_sums]
        pairs += [(ref.episode_metric_sums[k], orc.s.episode_metric_sums[k], "metric_" + k) for k in ref.episode_metric_sums]
        if p.measure_heights:
            pairs.append((ref.measured_heights, orc.measured_heights, "heights"))
            ref_ho = _ref_heights_obs(ref)                                   # LR:221-223 executed by the base class itself
            pairs.append((ref_ho, EO_heights_obs(orc.root[:, 2], orc.measured_heights, p.obs_scale_height), "heights_obs"))
        if p.terrain_curriculum:
            pairs += [(ref.terrain_levels, orc.s.terrain_levels, "terrain_levels"), (ref.env_origins, orc.s.env_origins, "env_origins")]
        stats = []
        if int(rst.sum()):
            for k in [k for k in ref.extras["episode"] if not k.startswith("coeff")]:
                pairs.append((ref.extras["episode"][k], ex["episode"][k], "extras_" + k))
                stats.append(float(ref.extras["episode"][k]))
        worst = max([worst] + [_close(a, b, 0.0, f"{name}/step{t}/{w}") for a, b, w in pairs])
        out["obs100"].append(robs[:, :100].numpy().copy())
        out["rew"].append(ref.rew_buf.numpy().copy())
        out["arm_rew"].append(ref.arm_rew_buf.numpy().copy())
        out["reset"].append(ref.reset_buf.numpy().copy())
        out["time_out"].append(ref.time_out_buf.numpy().copy())
        out["commands"].append(ref.commands.numpy().copy())
        out["ee_goal_sphere"].append(ref.ee_goal_sphere.numpy().copy())
        out["goal_timer"].append(ref.goal_timer.numpy().copy())
        out["ep_len"].append(ref.episode_length_buf.numpy().copy())
        out["heights"].append(ref.measured_heights.numpy().copy() if p.measure_heights else np.zeros((0,), np.float32))
        out["heights_obs"].append(ref_ho.numpy().copy() if p.measure_heights else np.zeros((0,), np.float32))
        out["env_origins"].append(ref.env_origins.numpy().copy())
        out["terrain_levels"].append(ref.terrain_levels.numpy().copy() if p.terrain_curriculum else np.zeros((0,), np.int64))
        out["ep_stats"].append(np.array(stats if stats else [np.nan] * (len(ref.episode_sums) + len(ref.episode_metric_sums)),
                                        np.float32))
    arrs = {k: np.stack(v) for k, v in out.items()}
    arrs.update(final_obs=robs.numpy(), final_hist=ref.obs_history_buf.numpy(), final_root=ref._root_states.numpy(),
                final_dof=ref.dof_state.numpy(), final_ahist=ref.action_history_buf.numpy(),
                final_sums=np.stack([ref.episode_sums[k].numpy() for k in ref.episode_sums]),
                final_metrics=np.stack([ref.episode_metric_sums[k].numpy() for k in ref.episode_metric_sums]),
                sum_names=np.array(list(ref.episode_sums.keys())),
                stat_names=np.array([k for k in ref.extras["episode"] if not k.startswith("coeff")]),
                meta=np.array([ENV_N, ENV_STEPS, ENV_SEED, ENV_COUNTER0]))
    np.savez_compressed(os.path.join(HERE, f"env_{name}.npz"), **arrs)
    extra = ""
    if p.terrain_curriculum:
        lv = arrs["terrain_levels"]
        d = np.diff(np.concatenate([np.asarray(st["terrain_levels"])[None], lv]), axis=0)
        extra = f"; terrain levels: {int((d > 0).sum())} promotions, {int((d < 0).sum())} demotions / wraps, final range {lv[-1].min()}..{lv[-1].max()}"
    print(f"env_{name}: oracle == reference (max diff {worst}) over {ENV_STEPS} steps; resets/step "
          f"{arrs['reset'].sum(1).tolist()}, timeouts {int(arrs['time_out'].sum())}{extra}")


# ----------------------------------------------------------------------------------------------

def _make_reference_alg(N, T, hp_over=None):
    with contextlib.redirect_stdout(io.StringIO()):
        from rsl_rl.modules import ActorCritic
        from rsl_rl.algorithms import PPO
        from legged_gym.utils.helpers import class_to_dict
        _, _, CfgPPO = H.import_reference_env()
        train = class_to_dict(CfgPPO())
        ac = ActorCritic(76, 76, 18, **train["policy"], num_priv=24, num_hist=10, num_prop=76)
        alg = PPO(ac, device="cpu", **train["algorithm"])
    alg.init_storage(N, T, [860], [None], [18])
    return alg, train


def _load_params(alg, seed):
    manifest = [(n, tuple(p.shape)) for n, p in alg.actor_critic.named_parameters()]
    assert manifest == PO.param_manifest(), "oracle manifest != reference named_parameters()"
    vals = synth.policy_params(manifest, seed)
    sd = {}
    for (n, shape), v in zip(manifest, vals):
        sd[n] = alg.actor_critic.state_dict()[n].clone() if v is None else torch.from_numpy(v).clone()
    alg.actor_critic.load_state_dict(sd)
    return {n: sd[n].clone() for n, _ in manifest}


def _fill(alg, inp, hist_encoding, seed):
    T = inp["rew"].shape[0]
    obs = torch.from_numpy(inp["obs"])
    torch.manual_seed(seed)
    with torch.inference_mode():
        for t in range(T):
            alg.act(obs[t], obs[t], hist_encoding)
            alg.process_env_step(torch.from_numpy(inp["rew"][t]), torch.from_numpy(inp["arm_rew"][t]),
                                 torch.from_numpy(inp["dones"][t]), {"time_outs": torch.from_numpy(inp["time_outs"][t])})
        alg.compute_returns(obs[T])
    s = alg.storage
    return {k: getattr(s, k).clone() for k in ("observations", "actions", "rewards", "dones", "values", "actions_log_prob",
                                                "mu", "sigma", "returns", "advantages")}


def gen_ppo():
    N, T = PPO_N, PPO_T
    alg, train = _make_reference_alg(N, T)
    hp = dict(train["algorithm"])
    P = _load_params(alg, PPO_SEED)
    inp = synth.rollout_inputs(N, T, 860, PPO_SEED)
    st = _fill(alg, inp, False, 11)

    # ---- oracle: rollout forward, bootstrap, GAE ----
    obs = torch.from_numpy(inp["obs"])
    worst = 0.0
    o_vals = []
    for t in range(T):
        eps = (st["actions"][t] - st["mu"][t]) / st["sigma"][t]
        a = PO.policy_act(P, obs[t], eps)
        worst = max(worst, _close(a["mean"], st["mu"][t], 2e-6, "act.mean"), _close(a["values"], st["values"][t], 2e-6, "act.values"),
                    _close(a["log_prob"], st["actions_log_prob"][t], 2e-5, "act.log_prob"))
        r = PO.bootstrap_rewards(torch.from_numpy(inp["rew"][t]), torch.from_numpy(inp["arm_rew"][t]), st["values"][t],
                                 torch.from_numpy(inp["time_outs"][t]), hp["gamma"])
        _close(r, st["rewards"][t], 0.0, "bootstrapped rewards")
        o_vals.append(a["values"])
    last_values = alg.actor_critic.evaluate(obs[T]).detach()
    ret, adv = PO.compute_returns(st["rewards"], st["values"], st["dones"], last_values, hp["gamma"], hp["lam"])
    _close(ret, st["returns"], 0.0, "returns")
    _close(adv, st["advantages"], 0.0, "advantages")

    # ---- reference update() with recorded permutation, grads and params ----
    alg.counter = PPO_COUNTER
    rec = {}

    def hook(opt, args, kwargs):
        k = rec.setdefault("n", 0)
        if k == 0:
            rec["grad1"] = {n: (p.grad.clone() if p.grad is not None else None) for n, p in alg.actor_critic.named_parameters()}
        rec["n"] = k + 1
        if k == 0:
            rec["want_post1"] = True

    def post_hook(opt, args, kwargs):
        if rec.pop("want_post1", False):
            rec["param1"] = {n: p.detach().clone() for n, p in alg.actor_critic.named_parameters()}

    alg.optimizer.register_step_pre_hook(hook)
    alg.optimizer.register_step_post_hook(post_hook)
    torch.manual_seed(123)
    perm = torch.randperm(N * T)
    torch.manual_seed(123)
    res = alg.update()
    ref_params20 = {n: p.detach().clone() for n, p in alg.actor_critic.named_parameters()}

    # ---- oracle update ----
    Po = {n: v.clone() for n, v in P.items()}
    opt = PO.Adam(list(Po.keys()), hp["learning_rate"])
    snap = {}

    def record(k, Pn, G, when):
        if k == 0 and when == "pre_step":
            snap["grad1"] = {n: (g.clone() if g is not None else None) for n, g in G.items()}
        if k == 0 and when == "post_step":
            snap["param1"] = {n: v.detach().clone() for n, v in Pn.items()}

    logs = PO.ppo_update(Po, opt, st, perm, hp, PPO_COUNTER, record)
    for n in P:
        if rec["grad1"][n] is None:
            assert snap["grad1"][n] is None
        else:
            worst = max(worst, _close(snap["grad1"][n], rec["grad1"][n], 1e-7, "grad1/" + n))
        worst = max(worst, _close(snap["param1"][n], rec["param1"][n], 1e-7, "param1/" + n),
                    _close(Po[n], ref_params20[n], 2e-6, "param20/" + n))
    mv = float(torch.stack([l["value"] for l in logs]).mean())
    ms = float(torch.stack([l["surrogate"] for l in logs]).mean())
    mr = float(torch.stack([l["priv_reg"] for l in logs]).mean())
    _close(mv, res[0], 1e-5, "mean value loss")
    _close(ms, res[1], 1e-5, "mean surrogate loss")
    _close(mr, res[5], 1e-5, "mean priv reg loss")
    assert abs(logs[0]["mixing_ratio"] - res[3]) < 1e-12 and abs(logs[0]["priv_reg_coef"] - res[6]) < 1e-12

    # ---- dagger iteration (hist_encoding rollouts, update_dagger) ----
    inp2 = synth.rollout_inputs(N, T, 860, PPO_SEED + 1)
    alg.storage.clear()
    Pd_start = {n: p.detach().clone() for n, p in alg.actor_critic.named_parameters()}
    st2 = _fill(alg, inp2, True, 12)
    eps2 = (st2["actions"][0] - st2["mu"][0]) / st2["sigma"][0]
    a2 = PO.policy_act(Pd_start, torch.from_numpy(inp2["obs"][0]), eps2, hist_encoding=True)
    _close(a2["mean"], st2["mu"][0], 2e-6, "act(hist).mean")
    torch.manual_seed(321)
    perm2 = torch.randperm(N * T)
    torch.manual_seed(321)
    dag = alg.update_dagger()
    ref_dag = {n: p.detach().clone() for n, p in alg.actor_critic.named_parameters()}
    Pd = {n: v.clone() for n, v in Pd_start.items()}
    hnames = [n for n in Pd if n.startswith(PO.HIST_PREFIX)]
    dl = PO.dagger_update(Pd, PO.Adam(hnames, hp["learning_rate"]), st2, perm2, hp)
    _close(float(torch.stack(dl).mean()), dag, 1e-5, "mean hist latent loss")
    for n in Pd:
        worst = max(worst, _close(Pd[n], ref_dag[n], 2e-6, "dagger/" + n))

    flat = lambda d: torch.cat([d[n].reshape(-1) for n in P]).numpy()  # noqa: E731
    g1 = torch.cat([(rec["grad1"][n] if rec["grad1"][n] is not None else torch.zeros_like(P[n])).reshape(-1) for n in P]).numpy()
    np.savez_compressed(
        os.path.join(HERE, "ppo.npz"),
        meta=np.array([N, T, PPO_SEED, PPO_COUNTER]), names=np.array(list(P.keys())),
        actions=st["actions"].numpy(), values=st["values"].numpy(), log_prob=st["actions_log_prob"].numpy(),
        mu0=st["mu"][0].numpy(), rewards=st["rewards"].numpy(), last_values=last_values.numpy(),
        returns=st["returns"].numpy(), advantages=st["advantages"].numpy(), perm=perm.numpy().astype(np.int32),
        update_result=np.array([float(x) for x in res], np.float64), grad1=g1, param1=flat(rec["param1"]),
        param20=flat(ref_params20),
        mb_losses=np.array([[float(l["surrogate"]), float(l["value"]), float(l["priv_reg"]), float(l["grad_norm"])] for l in logs]),
        dag_actions0=st2["actions"][0].numpy(), dag_mu0=st2["mu"][0].numpy(), dag_perm=perm2.numpy().astype(np.int32),
        dag_loss=np.array([dag], np.float64), dag_mb_losses=np.array([float(x) for x in dl]), dag_params=flat(ref_dag),
    )
    print(f"ppo: oracle == reference (worst abs diff {worst:.3g}); update() -> {res}; update_dagger() -> {dag}")


if __name__ == "__main__":
    which = sys.argv[1:] or ["env_flat", "env_full", "ppo"]
    if "env_flat" in which:
        gen_env("flat")
    if "env_full" in which:
        gen_env("full")
    if "ppo" in which:
        gen_ppo()
