"""update() and rollout time per hidden activation at the flat-config shape (4096 envs x 40 steps, 5 epochs x 4 mini-batches, tf32x3), each
activation measured in alternation with ELU in the same process.  Reports only: CUDA events around whole calls that end in a synchronise.

    python tools/activation_timing.py [--reps 5] [--precision tf32x3] [--out FILE]

rollout_ms: the 40 policy forwards (dwbc_policy_act) of one iteration; update_ms: one update() over the 40 x 4096 storage."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from dwbc_b200.actor_critic import FlatActorCritic  # noqa: E402
from dwbc_b200.ppo import FusedPPO  # noqa: E402

N, T = 4096, 40
HP = dict(num_learning_epochs=5, num_mini_batches=4, clip_param=0.2, gamma=0.99, lam=0.95, learning_rate=2e-4, max_grad_norm=1.0,
          mixing_schedule=[1.0, 0, 1], priv_reg_coef_schedual=[0, 1, 1000, 1000])


def make(act, precision):
    ac = FlatActorCritic(device="cuda:0", seed=0, init_std=[[0.8, 1.0, 1.0] * 4 + [1.0] * 6], num_priv=24, num_hist=10, num_prop=76, activation=act)
    alg = FusedPPO(ac, device="cuda:0", precision=precision, **HP)
    alg.init_storage(N, T, [860], [None], [18])
    alg.counter = 1500
    gen = torch.Generator(device="cuda").manual_seed(0)
    s = alg.storage
    s._obs_all.normal_(generator=gen)
    for k in ("actions", "values", "returns", "advantages"):
        getattr(s, k).normal_(generator=gen)
    s.actions_log_prob.normal_(generator=gen).sub_(20.0)
    return alg


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def rollout(alg):
    obs = alg.storage._obs_all
    for t in range(T):
        alg.storage.step = t
        alg.act(obs[t], obs[t], False)
    alg.storage.step = 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--precision", default="tf32x3", choices=["fp32", "tf32", "tf32x3"])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    algs = {act: make(act, a.precision) for act in ("elu", "selu", "relu", "lrelu", "tanh", "sigmoid")}
    for alg in algs.values():                    # warm-up of every shape
        rollout(alg)
        alg.update()
        alg.storage.step = 0
    res = {act: dict(rollout_ms=[], update_ms=[]) for act in algs}
    elu_pair = {act: dict(rollout_ms=[], update_ms=[]) for act in algs if act != "elu"}
    for _ in range(a.reps):
        for act in elu_pair:                     # ELU, then the other activation, back to back
            for who, dst in (("elu", elu_pair[act]), (act, res[act])):
                alg = algs[who]
                dst["rollout_ms"].append(timed(lambda: rollout(alg)))
                dst["update_ms"].append(timed(lambda: alg.update()))
                alg.storage.step = 0
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    rows = []
    for act, r in elu_pair.items():
        rows.append(dict(activation=act, rollout_ms=round(med(res[act]["rollout_ms"]), 3), update_ms=round(med(res[act]["update_ms"]), 3),
                         elu_rollout_ms=round(med(r["rollout_ms"]), 3), elu_update_ms=round(med(r["update_ms"]), 3),
                         update_ms_spread=[round(min(res[act]["update_ms"]), 3), round(max(res[act]["update_ms"]), 3)],
                         elu_update_ms_spread=[round(min(r["update_ms"]), 3), round(max(r["update_ms"]), 3)]))
    out = dict(gpu=q, precision=a.precision, envs=N, steps=T, reps=a.reps, statistic="median over reps", results=rows)
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
