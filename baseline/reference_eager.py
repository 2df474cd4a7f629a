"""The reference's own update half (unmodified rsl_rl from baseline/_ref: PPO.act / process_env_step / compute_returns / update,
rsl_rl/algorithms/ppo.py:115-263, storage/rollout_storage.py:95-205, modules/actor_critic.py) run as eager PyTorch on a device --
the "same box" comparison SURVEY.md 8d asks for: the reference has no Blackwell kernels, its GPU path IS eager PyTorch.

Only bench.py calls this (report-only block `reference_eager_b200`, and the `--impl reference` CPU arm); none of this repo's kernels,
models or engine are on that path.  The env half of the reference (legged_gym WidowGo1) needs Isaac Gym and cannot run here: the
observations / rewards / dones fed to the reference PPO are synthetic tensors of the metric's shapes (4096 envs x 40 steps x 860).
"""
from __future__ import annotations

import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "_ref")


def available() -> str | None:
    """None if the reference install is usable, else a one-line reason."""
    if not os.path.isdir(os.path.join(REF, "rsl_rl")):
        return "baseline/_ref/rsl_rl is absent (run baseline/install_reference.sh with DWBC_REFERENCE set to a checkout of the original project)"
    return None


def make_reference_alg(device: str, n_envs: int, T: int):
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from rsl_rl.algorithms import PPO            # the reference's classes, unmodified
    from rsl_rl.modules import ActorCritic
    import contextlib
    import io
    cfg = json.load(open(os.path.join(HERE, "widowgo1_train_cfg.json")))
    a = cfg["actor_critic_args"]
    with contextlib.redirect_stdout(io.StringIO()):          # the reference prints its modules; bench.py must print ONE json line
        ac = _make_ac(ActorCritic, a, cfg, device)
    alg = PPO(ac, device=device, **cfg["algorithm"])
    alg.init_storage(n_envs, T, [a["num_prop"] * (a["num_hist"] + 1) + a["num_priv"]], [None], [a["num_actions"]])
    alg.counter = 1500                          # same schedules as the fused arm: priv-reg coefficient 0.5, mixing ratio 1
    return alg


def _make_ac(ActorCritic, a, cfg, device):
    return ActorCritic(a["num_actor_obs"], a["num_critic_obs"], a["num_actions"], **cfg["policy"], num_priv=a["num_priv"], num_hist=a["num_hist"],
                       num_prop=a["num_prop"]).to(device)


def time_iterations(device: str, n_envs: int, T: int, steps: int, warmup: int, allow_tf32: bool | None = None):
    """`steps` timed PPO iterations of the reference's update half on synthetic rollout data; returns per-iteration ms of
    (rollout policy part: T x (act + process_env_step), compute_returns, update)."""
    import torch
    if allow_tf32 is not None:
        torch.backends.cuda.matmul.allow_tf32 = allow_tf32
        torch.backends.cudnn.allow_tf32 = allow_tf32
    alg = make_reference_alg(device, n_envs, T)
    g = torch.Generator(device=device)
    g.manual_seed(3)
    obs = torch.randn(T + 1, n_envs, 860, device=device, generator=g)
    rew = torch.randn(T, n_envs, device=device, generator=g)
    arew = torch.randn(T, n_envs, device=device, generator=g)
    dones = torch.rand(T, n_envs, device=device, generator=g) < 0.05
    touts = torch.rand(T, n_envs, device=device, generator=g) < 0.02
    cuda = device.startswith("cuda")

    def sync():
        if cuda:
            torch.cuda.synchronize()

    def iteration():
        t0 = time.perf_counter()
        with torch.inference_mode():             # OPR:131
            for t in range(T):
                alg.act(obs[t], obs[t], False)
                alg.process_env_step(rew[t], arew[t], dones[t], {"time_outs": touts[t]})
            sync()
            t1 = time.perf_counter()
            alg.compute_returns(obs[T])
            sync()
        t2 = time.perf_counter()
        alg.update()
        sync()
        t3 = time.perf_counter()
        return (t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3

    for _ in range(warmup):
        iteration()
    out = [iteration() for _ in range(steps)]
    n = len(out)
    return dict(rollout_policy_ms=sum(o[0] for o in out) / n, compute_returns_ms=sum(o[1] for o in out) / n, update_ms=sum(o[2] for o in out) / n,
                iteration_ms=sum(sum(o) for o in out) / n)
