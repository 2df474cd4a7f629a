"""CPU: the hidden-layer activation of the ActorCritic (rsl_rl `get_activation` names) -- name map, the DwbcNetCfg.activation field, and
the layer-chain programs each activation builds (dwbc_debug_describe_chain, host code only)."""
import ctypes as C
import os
import re

import pytest
import torch

from dwbc_b200 import _lib as L
from dwbc_b200.actor_critic import FlatActorCritic
import activation_oracle as AO
from oracle import ppo_oracle as PO

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
NAMES = ("elu", "selu", "relu", "crelu", "lrelu", "tanh", "sigmoid")
# activation codes the kernels put into a layer op (gemm_simt.cuh: ACT_*)
OP_CODE = dict(elu=1, selu=3, relu=4, crelu=4, lrelu=5, tanh=2, sigmoid=6)
ACT_NONE, ACT_ELU, ACT_TANH = 0, 1, 2


def make(act):
    return FlatActorCritic(device="cpu", num_priv=24, num_hist=10, num_prop=76, activation=act)


def test_activation_names_map_to_the_abi_enum():
    hdr = open(os.path.join(ROOT, "include", "dwbc.h")).read()
    enum = {k.lower(): int(v) for k, v in re.findall(r"DWBC_ACT_([A-Z]+) = (\d+)", hdr)}
    assert enum == dict(elu=0, selu=1, relu=2, lrelu=3, tanh=4, sigmoid=5)
    assert L.ACTIVATIONS == dict(enum, crelu=enum["relu"])          # rsl_rl's "crelu" builds a plain nn.ReLU()
    assert int(re.search(r"#define DWBC_ABI_VERSION (\d+)", hdr).group(1)) == L.ABI_VERSION == 4
    for name in NAMES:
        assert make(name).net_cfg.activation == L.ACTIVATIONS[name]
    for bad in ("gelu", "ELU", "", None, "softplus"):
        with pytest.raises(L.DwbcError):
            make(bad)


def test_elu_net_cfg_is_byte_identical_to_a_zeroed_activation_field():
    """The field took the place of the zero-filled `reserved_` word: same struct size, same offset, ELU == 0, so a caller that never sets
    it keeps the ELU network."""
    assert L.NetCfg.activation.offset == C.sizeof(L.NetCfg) - 4 and L.NetCfg.activation.size == 4
    default, elu = FlatActorCritic(device="cpu", num_priv=24, num_hist=10, num_prop=76).net_cfg, make("elu").net_cfg
    assert bytes(elu) == bytes(default)
    blank = L.NetCfg.from_buffer_copy(bytes(elu))
    blank.activation = 0
    assert bytes(blank) == bytes(elu)
    for name in NAMES[1:]:
        other = bytes(make(name).net_cfg)
        assert other[:-4] == bytes(elu)[:-4] and other[-4:] != bytes(elu)[-4:]


def test_fused_actor_critic_takes_the_name():
    from dwbc_b200 import runner_compat as RC
    ac = RC.FusedActorCritic(76, 76, 18, actor_hidden_dims=[128], critic_hidden_dims=[128], activation="crelu", num_priv=24, num_hist=10,
                             num_prop=76, device="cpu")
    assert ac.net_cfg.activation == L.ACTIVATIONS["relu"] and ac.core.activation == "crelu"
    with pytest.raises(L.DwbcError):
        RC.FusedActorCritic(76, 76, 18, activation="swish", num_priv=24, num_hist=10, num_prop=76, device="cpu")


def test_library_rejects_unknown_activation_codes():
    lib = L.lib()
    lib.dwbc_workspace_bytes.argtypes = [C.c_void_p, C.c_int64]
    cfg = make("elu").net_cfg
    assert lib.dwbc_workspace_bytes(C.addressof(cfg), 16) > 0
    for code in (6, 7, -1, 1000):
        cfg.activation = code
        assert lib.dwbc_workspace_bytes(C.addressof(cfg), 16) == -1      # DWBC_ERR_ARG


def describe(cfg, rows, what, hist, precision="tf32x3"):
    lib = L.lib()
    lib.dwbc_debug_describe_chain.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_int32]
    cfg.precision = L.PRECISIONS[precision]
    out = (C.c_int32 * 1024)()
    k = lib.dwbc_debug_describe_chain(C.addressof(cfg), rows, what, hist, 148, out, 1024)
    assert k > 0, k
    v, i, progs = list(out[:k]), 2, []
    for _ in range(v[0]):
        n_ops, n_loads = v[i], v[i + 1]
        i += 2
        progs.append((n_loads, [dict(zip(("N", "kpad", "act", "fin", "fin_c", "out_col0", "y", "y_img"), v[i + 8 * j:i + 8 * j + 8]))
                                for j in range(n_ops)]))
        i += 8 * n_ops
    assert i == k
    return v[1], progs


@pytest.mark.parametrize("precision", ["tf32x3", "tf32"])
@pytest.mark.parametrize("name", NAMES[1:])
def test_chain_programs_carry_the_hidden_activation(name, precision):
    """Rollout (what 0), bootstrap values (1), update forward + loss (2) and backward (3), teacher and student latents: every op that carries
    ELU in the ELU network carries the configured activation, the heads' outputs keep tanh (actor) / none (critic), and everything else
    (programs, ops, loads, widths, K padding, loss hooks, outputs and tile images) is the ELU network's."""
    ref_cfg, cfg = make("elu").net_cfg, make(name).net_cfg
    seen = set()
    for what in range(4):
        for hist in (0, 1):
            for rows in (4096, 40960 + 77):
                npack0, progs0 = describe(ref_cfg, rows, what, hist, precision)
                npack, progs = describe(cfg, rows, what, hist, precision)
                assert npack == npack0 and len(progs) == len(progs0)
                for (nl0, ops0), (nl, ops) in zip(progs0, progs):
                    assert nl == nl0 and len(ops) == len(ops0)
                    for o0, o in zip(ops0, ops):
                        assert {k: v for k, v in o.items() if k != "act"} == {k: v for k, v in o0.items() if k != "act"}
                        assert o0["act"] in (ACT_NONE, ACT_ELU, ACT_TANH)
                        assert o["act"] == (OP_CODE[name] if o0["act"] == ACT_ELU else o0["act"])
                        seen.add(o0["act"])
                        if o0["fin"] in (1, 2):                  # action heads' last op: tanh whatever the hidden activation
                            assert o["act"] == ACT_TANH
                        if o0["fin"] == 3:                       # value heads' last op: linear
                            assert o["act"] == ACT_NONE
    assert seen == {ACT_NONE, ACT_ELU, ACT_TANH}


def test_activation_oracle_is_the_pinned_oracle_for_elu():
    """tests/activation_oracle.py with act="elu" reproduces oracle/ppo_oracle.py (pinned to the reference by the golden vectors) bit for bit:
    networks, history latent, loss and its gradient, and a 20-step update()."""
    from test_oracle_golden import ppo_hp
    P = {n: torch.randn(s, generator=torch.Generator().manual_seed(i)) * 0.3 for i, (n, s) in enumerate(PO.param_manifest())}
    P["std"] = torch.full((1, 18), 0.8)
    gen = torch.Generator().manual_seed(9)
    obs = torch.randn(64, 860, generator=gen)
    eps = torch.randn(64, 18, generator=gen)
    for hist in (False, True):
        a, b = AO.policy_act(P, obs, eps, "elu", hist), PO.policy_act(P, obs, eps, hist)
        assert all(torch.equal(a[k], b[k]) for k in b)
    assert torch.equal(AO.hist_latent(P, obs, "elu"), PO.hist_latent(P, obs)) and torch.equal(AO.priv_latent(P, obs, "elu"), PO.priv_latent(P, obs))
    T, N = 4, 16
    st = dict(observations=torch.randn(T, N, 860, generator=gen), actions=torch.randn(T, N, 18, generator=gen),
              values=torch.randn(T, N, 2, generator=gen), returns=torch.randn(T, N, 2, generator=gen),
              actions_log_prob=torch.randn(T, N, 2, generator=gen) - 20.0, advantages=torch.randn(T, N, 2, generator=gen))
    hp = dict(ppo_hp(), num_mini_batches=2, num_learning_epochs=2)
    perm = torch.randperm(T * N, generator=gen)
    grads = []
    for f in (lambda Q, mb: AO.minibatch_loss(Q, mb, hp, 1500, "elu")[0], lambda Q, mb: PO.minibatch_loss(Q, mb, hp, 1500)[0]):
        Q = {n: v.clone().requires_grad_(True) for n, v in P.items()}
        f(Q, PO.gather(st, perm)).backward()
        grads.append({n: v.grad for n, v in Q.items()})
    assert all((grads[0][n] is None and grads[1][n] is None) or torch.equal(grads[0][n], grads[1][n]) for n in P)
    Pa, Pb = {n: v.clone() for n, v in P.items()}, {n: v.clone() for n, v in P.items()}
    AO.ppo_update(Pa, PO.Adam(list(Pa), 2e-4), st, perm, hp, 1500, "elu")
    PO.ppo_update(Pb, PO.Adam(list(Pb), 2e-4), st, perm, hp, 1500)
    assert all(torch.equal(Pa[n], Pb[n]) for n in P)


def test_activation_oracle_applies_torch_functions_where_rsl_rl_puts_them():
    """Each name applies torch's own function to the layers AC builds `activation` into; the action means keep their tanh."""
    P = {n: torch.randn(s, generator=torch.Generator().manual_seed(i)) * 0.3 for i, (n, s) in enumerate(PO.param_manifest())}
    obs = torch.randn(5, 860, generator=torch.Generator().manual_seed(9))
    assert torch.equal(AO.critic_values(P, obs, "crelu"), AO.critic_values(P, obs, "relu"))
    h = torch.nn.functional.linear(obs[:, 76:100], P["actor.priv_encoder.0.weight"], P["actor.priv_encoder.0.bias"])
    z = torch.sigmoid(torch.nn.functional.linear(torch.sigmoid(h), P["actor.priv_encoder.2.weight"], P["actor.priv_encoder.2.bias"]))
    assert torch.equal(AO.priv_latent(P, obs, "sigmoid"), z)
    m = AO.actor_mean(P, obs, "relu")
    assert float(m.abs().max()) <= 1.0 and not torch.equal(m, PO.actor_mean(P, obs))
