"""GPU: the ActorCritic with every rsl_rl hidden activation (DwbcNetCfg.activation) against the CPU oracle (tests/activation_oracle.py: torch's own F.selu / F.relu /
F.leaky_relu / torch.tanh / torch.sigmoid, autograd for the gradients), on the three precisions: rollout act() on teacher and student
latents, the history latent, the unclipped mini-batch gradient over many tiles with a ragged tail, the DAgger gradient, the parameters after
a 20-step update(), and the stock 512/256/128 trunk that runs layer by layer.

Tolerances.  ELU, tanh and sigmoid are smooth: on 'fp32' / 'tf32x3' they get the fp32 tolerances of tests/test_gpu_ppo.py.  ReLU, leaky
ReLU and SELU have a kink at 0: a pre-activation within rounding of 0 takes the other branch of the derivative under any other summation
order, so their gradients are bounded by the relative norm ||g - g_ref|| <= tol ||g_ref|| (per parameter tensor) at 2 x the error measured
on a B200, as TF32_TOL does; so are all 'tf32' results.  The measured values are printed."""
import ctypes as C
import functools
import json
import os
import sys

import numpy as np
import pytest
import torch

from dwbc_b200 import _lib as L, synth
import activation_oracle as AO
from oracle import ppo_oracle as PO
from test_oracle_golden import golden_params, ppo_hp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
REF = os.path.join(ROOT, "baseline", "_ref")
ACTS = ("elu", "selu", "relu", "lrelu", "tanh", "sigmoid")
PRECISIONS = ("fp32", "tf32x3", "tf32")
SMOOTH = ("elu", "tanh", "sigmoid")
# today's fp32 tolerances (tests/test_gpu_ppo.py): forward outputs, log-prob, per-tensor max |dg| / max |g|, parameters after update()
FP32_TOL = dict(fwd=1e-5, logp=1e-4, grad_max=2e-3, param20=2e-5)
# 2 x the largest errors measured on B200 (NVIDIA B200, 1000 W; printed by the tests) for the kinked activations on fp32 / tf32x3 and for
# every activation on tf32.  fwd: max abs of means, values and the history latent; grad / dagger: worst per-tensor ||dg|| / ||g||; param20:
# RMS and max abs over all parameters after the 20 steps.  logp: a = mu + sigma eps, so its log-prob does not depend on the precision of mu
MEASURED_TOL = {
    "fp32": dict(grad=8e-4, dagger=1.1e-4, param20_rms=1.1e-5, param20_max=8.2e-4),         # measured 3.9e-4 relu, 5.2e-5, 5.4e-6, 4.1e-4 selu
    "tf32x3": dict(grad=1.2e-2, dagger=1.1e-4, param20_rms=2.1e-5, param20_max=1e-3),       # 5.9e-3 lrelu, 5.2e-5 selu, 1.0e-5, 4.9e-4 relu
    "tf32": dict(fwd=5.1e-3, logp=1e-4, grad=8e-2, dagger=2.1e-2, param20_rms=1.7e-4, param20_max=7e-3),   # 2.5e-3, -, 4.0e-2, 1.0e-2, 8.1e-5, 3.5e-3
}
ROWS = 40960 + 77                       # 320 full tiles and a ragged one: every CTA takes several tile pairs


def exact(act, precision):
    return precision != "tf32" and act in SMOOTH


def params(seed, **dims):
    manifest = PO.param_manifest(**dims)
    vals = synth.policy_params(manifest, seed)
    return {n: (torch.tensor([[0.8, 1.0, 1.0] * 4 + [1.0] * 6]) if v is None else torch.from_numpy(v).clone()) for (n, _), v in zip(manifest, vals)}


def make_alg(P, act, precision, N, T, dims=None, **over):
    from dwbc_b200.actor_critic import FlatActorCritic
    from dwbc_b200.ppo import FusedPPO
    dims = dims or {}
    ac = FlatActorCritic(device="cuda:0", num_priv=24, num_hist=10, num_prop=76, activation=act, **dims)
    ac.load_state_dict(P)
    hp = ppo_hp()
    hp.update(over)
    alg = FusedPPO(ac, device="cuda:0", precision=precision, **hp)
    alg.init_storage(N, T, [860], [None], [18])
    return alg


def rel_norms(got, ref):
    """worst per-tensor ||got - ref|| / ||ref|| (tensors with a non-zero reference) and worst max |got - ref| / max |ref|"""
    worst_n, worst_m = 0.0, 0.0
    for n, r in ref.items():
        g = got[n].detach().double().cpu()
        r = r.double()
        assert torch.isfinite(g).all(), n
        if float(r.norm()) > 1e-9:
            worst_n = max(worst_n, float((g - r).norm() / r.norm()))
            worst_m = max(worst_m, float((g - r).abs().max() / r.abs().max()))
    return worst_n, worst_m


def report(**kw):
    print("MEASURED " + json.dumps(kw))


# ---- rollout act() and the history latent ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("act", ACTS)
def test_rollout_and_history_latent_match_oracle(act, precision):
    N = 4096
    P = params(7)
    alg = make_alg(P, act, precision, N, 1)
    gen = torch.Generator().manual_seed(3)
    obs = torch.randn(N, 860, generator=gen)
    eps = torch.randn(N, 18, generator=gen)
    errs = {}
    for hist in (False, True):
        ref = AO.policy_act(P, obs, eps, act, hist)
        alg.storage.step = 0
        alg.act(obs.cuda(), obs.cuda(), hist, eps=eps.cuda())
        s = alg.storage
        errs[f"mean{int(hist)}"] = float((s.mu[0].cpu() - ref["mean"]).abs().max())
        errs[f"value{int(hist)}"] = float((s.values[0].cpu() - ref["values"]).abs().max())
        errs[f"logp{int(hist)}"] = float((s.actions_log_prob[0].cpu() - ref["log_prob"]).abs().max())
    ac = alg.actor_critic
    Lld = 20
    out = torch.zeros(N, Lld, device="cuda")
    oc = obs.cuda()
    L.check(L.lib().dwbc_hist_latent(C.addressof(ac.net_cfg), L.ptr(ac.flat), L.ptr(oc), oc.stride(0), L.ptr(out), Lld, N, L.ptr(alg._workspace(N)),
                                     L.stream_ptr()), "dwbc_hist_latent")
    errs["hist"] = float((out.cpu() - AO.hist_latent(P, obs, act)).abs().max())
    report(test="rollout", act=act, precision=precision, **errs)
    tol = MEASURED_TOL["tf32"] if precision == "tf32" else FP32_TOL        # the forward is continuous: fp32 tolerances on fp32 / tf32x3
    for k, e in errs.items():
        assert e < (tol["logp"] if k.startswith("logp") else tol["fwd"]), (k, e)


# ---- the unclipped mini-batch gradient and the DAgger gradient ---------------------------------------------------------------------------
def _storage_inputs(N, seed):
    gen = torch.Generator().manual_seed(seed)
    return dict(observations=torch.randn(1, N, 860, generator=gen), actions=torch.randn(1, N, 18, generator=gen),
                values=torch.randn(1, N, 2, generator=gen), returns=torch.randn(1, N, 2, generator=gen),
                actions_log_prob=torch.randn(1, N, 2, generator=gen) - 20.0, advantages=torch.randn(1, N, 2, generator=gen))


@functools.lru_cache(maxsize=None)
def _oracle_grads(act):
    P = params(21)
    st = _storage_inputs(ROWS, 4)
    idx = torch.randperm(ROWS, generator=torch.Generator().manual_seed(8))
    for n in P:
        P[n].requires_grad_(True)
    loss, _ = AO.minibatch_loss(P, PO.gather(st, idx), ppo_hp(), 1500, act)
    loss.backward()
    g = {n: (P[n].grad.clone() if P[n].grad is not None else torch.zeros_like(P[n])) for n in P}
    for n in P:
        P[n].grad = None
    obs = st["observations"].flatten(0, 1)[idx]
    with torch.no_grad():
        zp = AO.priv_latent(P, obs, act)
    zh = AO.hist_latent(P, obs, act)
    (zp - zh).norm(p=2, dim=1).mean().backward()
    gd = {n: P[n].grad.clone() for n in P if n.startswith(PO.HIST_PREFIX)}
    return {n: v.detach() for n, v in P.items()}, st, idx, g, gd


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("act", ACTS)
def test_minibatch_and_dagger_gradients_match_oracle(act, precision):
    P, st, idx, g_ref, gd_ref = _oracle_grads(act)
    alg = make_alg(P, act, precision, ROWS, 1, num_mini_batches=1, num_learning_epochs=1)
    alg.counter = 1500
    s = alg.storage
    s._obs_all[0].copy_(st["observations"][0].cuda())
    for k in ("actions", "values", "returns", "actions_log_prob", "advantages"):
        getattr(s, k).copy_(st[k].cuda())
    ac, lib, di = alg.actor_critic, L.lib(), idx.cuda()
    h = alg._fill_hp()
    alg._losses.zero_()
    L.check(lib.dwbc_ppo_minibatch_grad(C.addressof(ac.net_cfg), L.ptr(ac.flat), s.c_struct_ptr(), L.ptr(di), ROWS, C.addressof(h), L.ptr(alg.grad),
                                        L.ptr(alg._losses), L.ptr(alg._workspace(ROWS)), L.stream_ptr()), "dwbc_ppo_minibatch_grad")
    g_norm, g_max = rel_norms(ac.unflat(alg.grad), g_ref)
    L.check(lib.dwbc_dagger_minibatch_grad(C.addressof(ac.net_cfg), L.ptr(ac.flat), s.c_struct_ptr(), L.ptr(di), ROWS, L.ptr(alg.grad),
                                           L.ptr(alg._losses), L.ptr(alg._workspace(ROWS)), L.stream_ptr()), "dwbc_dagger_minibatch_grad")
    got = ac.unflat(alg.grad)
    d_norm, d_max = rel_norms(got, gd_ref)
    assert all(float(got[n].abs().max()) == 0.0 for n in got if n not in gd_ref)        # DAgger touches the history encoder only
    report(test="gradient", act=act, precision=precision, grad_rel_norm=g_norm, grad_max_rel=g_max, dagger_rel_norm=d_norm, dagger_max_rel=d_max)
    if exact(act, precision):
        assert g_max < FP32_TOL["grad_max"] and d_max < FP32_TOL["grad_max"], (g_max, d_max)
    else:
        tol = MEASURED_TOL[precision]
        assert g_norm < tol["grad"] and d_norm < tol["dagger"], (g_norm, d_norm)


# ---- parameters after a 20-step update() (5 epochs x 4 mini-batches of BASELINE.json configs[0]) -----------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("act", ACTS)
def test_update_parameters_match_oracle(act, precision):
    g = np.load(os.path.join(G, "ppo.npz"))
    N, T, seed, counter = [int(x) for x in g["meta"]]
    P = golden_params(g, seed)
    inp = synth.rollout_inputs(N, T, 860, seed)
    st = dict(observations=torch.from_numpy(inp["obs"][:T]), actions=torch.from_numpy(g["actions"]), values=torch.from_numpy(g["values"]),
              actions_log_prob=torch.from_numpy(g["log_prob"]), returns=torch.from_numpy(g["returns"]), advantages=torch.from_numpy(g["advantages"]))
    hp = ppo_hp()
    perm = torch.from_numpy(g["perm"]).long()
    Po = {k: v.clone() for k, v in P.items()}
    AO.ppo_update(Po, PO.Adam(list(Po.keys()), hp["learning_rate"]), st, perm, hp, counter, act)
    alg = make_alg(P, act, precision, N, T)
    alg.counter = counter
    s = alg.storage
    s._obs_all.copy_(torch.from_numpy(inp["obs"]).cuda())
    for k, src in (("actions", "actions"), ("values", "values"), ("actions_log_prob", "log_prob"), ("returns", "returns"), ("advantages", "advantages")):
        getattr(s, k).copy_(torch.from_numpy(g[src]).cuda())
    res = alg.update(indices=perm.cuda())
    assert all(np.isfinite(x) for x in res), res
    got = alg.actor_critic.state_dict()
    d = torch.cat([(got[n].cpu() - Po[n]).reshape(-1) for n in Po])
    e_rms, e_max = float(d.pow(2).mean().sqrt()), float(d.abs().max())
    report(test="update20", act=act, precision=precision, param_rms=e_rms, param_max=e_max)
    if exact(act, precision):
        assert e_max < FP32_TOL["param20"], e_max
    else:
        tol = MEASURED_TOL[precision]
        assert e_rms < tol["param20_rms"] and e_max < tol["param20_max"], (e_rms, e_max)


# ---- the stock legged_gym trunk (512, 256, 128): layers wider than 128 run layer by layer ---------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("act", ACTS)
def test_stock_trunk_layerwise_matches_oracle(act, precision):
    N, T = 256, 8
    dims = dict(actor_dims=(512, 256, 128), critic_dims=(512, 256, 128))
    P = params(33, **dims)
    alg = make_alg(P, act, precision, N, T, dims=dict(actor_hidden_dims=dims["actor_dims"], critic_hidden_dims=dims["critic_dims"]),
                   num_mini_batches=1, num_learning_epochs=1)
    alg.counter = 1500
    st = _storage_inputs(N * T, 11)
    st = {k: v.reshape(T, N, *v.shape[2:]) for k, v in st.items()}
    eps = torch.randn(N, 18, generator=torch.Generator().manual_seed(2))
    obs0 = st["observations"][0]
    ref = AO.policy_act(P, obs0, eps, act)
    alg.act(obs0.cuda(), obs0.cuda(), False, eps=eps.cuda())
    s = alg.storage
    e_fwd = max(float((s.mu[0].cpu() - ref["mean"]).abs().max()), float((s.values[0].cpu() - ref["values"]).abs().max()))
    s._obs_all[:T].copy_(st["observations"].cuda())
    for k in ("actions", "values", "returns", "actions_log_prob", "advantages"):
        getattr(s, k).copy_(st[k].cuda())
    idx = torch.randperm(N * T, generator=torch.Generator().manual_seed(6))
    Pg = {n: v.clone().requires_grad_(True) for n, v in P.items()}
    loss, _ = AO.minibatch_loss(Pg, PO.gather(st, idx), ppo_hp(), 1500, act)
    loss.backward()
    g_ref = {n: (v.grad if v.grad is not None else torch.zeros_like(v)) for n, v in Pg.items()}
    ac = alg.actor_critic
    h = alg._fill_hp()
    alg._set_precision()
    alg._losses.zero_()
    L.check(L.lib().dwbc_ppo_minibatch_grad(C.addressof(ac.net_cfg), L.ptr(ac.flat), s.c_struct_ptr(), L.ptr(idx.cuda()), N * T, C.addressof(h),
                                            L.ptr(alg.grad), L.ptr(alg._losses), L.ptr(alg._workspace(N * T)), L.stream_ptr()), "grad")
    g_norm, g_max = rel_norms(ac.unflat(alg.grad), g_ref)
    report(test="stock", act=act, precision=precision, fwd=e_fwd, grad_rel_norm=g_norm, grad_max_rel=g_max)
    if precision == "tf32":
        tol = MEASURED_TOL["tf32"]
        assert e_fwd < tol["fwd"] and g_norm < tol["grad"], (e_fwd, g_norm)
    else:
        assert e_fwd < 2e-5, e_fwd                       # (the stock-trunk tolerance of tests/test_gpu_ppo.py)
        if act in SMOOTH:
            assert g_max < FP32_TOL["grad_max"], g_max
        else:
            assert g_norm < MEASURED_TOL[precision]["grad"], g_norm


# ---- the reference's own ActorCritic with a non-ELU activation --------------------------------------------------------------------------
@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "rsl_rl")),
                    reason="needs the unmodified rsl_rl under baseline/_ref: set DWBC_REFERENCE to a checkout of the original project and build")
@pytest.mark.parametrize("act", ["selu", "lrelu"])
def test_reference_actor_critic_with_activation_matches(act):
    """The fused policy built with activation=`act` saves a checkpoint that loads STRICTLY into rsl_rl's ActorCritic(activation=`act`), and
    that module reproduces act_inference (teacher and student latents) and evaluate: where the activation sits is the reference's."""
    import contextlib
    import io
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from rsl_rl.modules import ActorCritic
    from dwbc_b200 import runner_compat as RC
    cfg = json.load(open(os.path.join(ROOT, "baseline", "widowgo1_train_cfg.json")))
    a = cfg["actor_critic_args"]
    pol = dict(cfg["policy"], activation=act)
    ac = RC.FusedActorCritic(a["num_actor_obs"], a["num_critic_obs"], a["num_actions"], **pol, num_priv=a["num_priv"], num_hist=a["num_hist"],
                             num_prop=a["num_prop"], device="cuda:0")
    sd = {k: v + 0.05 * torch.randn(v.shape, generator=torch.Generator().manual_seed(i), device="cpu").to(v.device)
          for i, (k, v) in enumerate(ac.state_dict().items())}
    ac.load_state_dict(sd)
    ac.net_cfg.precision = L.PRECISIONS["tf32x3"]
    with contextlib.redirect_stdout(io.StringIO()):
        ref_ac = ActorCritic(a["num_actor_obs"], a["num_critic_obs"], a["num_actions"], **pol, num_priv=a["num_priv"], num_hist=a["num_hist"],
                             num_prop=a["num_prop"])
    ref_ac.load_state_dict({k: v.cpu() for k, v in ac.state_dict().items()}, strict=True)
    obs = torch.randn(777, 860, generator=torch.Generator().manual_seed(1)).clamp(-3, 3)
    with torch.no_grad():
        for hist in (False, True):
            np.testing.assert_allclose(ac.act_inference(obs.cuda(), hist_encoding=hist).cpu().numpy(),
                                       ref_ac.act_inference(obs, hist_encoding=hist).numpy(), rtol=0, atol=2e-5)
        np.testing.assert_allclose(ac.evaluate(obs.cuda()).cpu().numpy(), ref_ac.evaluate(obs).numpy(), rtol=0, atol=2e-5)
