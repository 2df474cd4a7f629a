"""Host-side logic of the reference mirror that needs no GPU: schedules, checkpoint layout (SURVEY 8f row f3), storage bookkeeping."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import dwbc_b200  # noqa: E402,F401
from dwbc_b200.actor_critic import FlatActorCritic  # noqa: E402
from dwbc_b200.ppo import FusedPPO  # noqa: E402
from oracle import ppo_oracle as PO  # noqa: E402
from test_oracle_golden import G, golden_params, ppo_hp  # noqa: E402


def make_cpu_alg(**over):
    ac = FlatActorCritic(device="cpu", num_priv=24, num_hist=10, num_prop=76)
    hp = ppo_hp()
    hp.update(over)
    return FusedPPO(ac, device="cpu", **hp)


def test_schedules_match_reference_formulas():
    """PPO:178-179 (priv_reg_coef) and PPO:301-302 (value mixing ratio) as restated by the oracle, over the whole counter range."""
    alg = make_cpu_alg(mixing_schedule=[0.5, 2000, 4000], priv_reg_coef_schedual=[0, 0.1, 3000, 7000])
    for c in (0, 1, 1999, 2000, 2001, 3000, 4000, 5999, 6000, 6500, 10000, 20000):
        alg.counter = c
        assert alg.get_value_mixing_ratio() == PO.value_mixing_ratio(c, [0.5, 2000, 4000])
        assert alg.get_priv_reg_coef() == PO.priv_reg_coef(c, [0, 0.1, 3000, 7000])


def test_unsupported_reference_switches_fail_loudly():
    from dwbc_b200 import _lib as L
    with pytest.raises(L.DwbcError):
        make_cpu_alg(adaptive_arm_gains=True)
    with pytest.raises(L.DwbcError):
        make_cpu_alg(schedule="adaptive")


def test_torque_supervision_host_side():
    """PPO:304-310, RS:82-84, PPO:136-142 on the host mirror: schedule, coefficient broadcast, storage rows, loud failure without coefficients."""
    from dwbc_b200 import _lib as L
    alg = make_cpu_alg(torque_supervision=True, torque_supervision_schedule=[0.1, 1000, 1000])
    for c in (0, 999, 1000, 1400, 2000, 5000):
        alg.counter = c
        assert alg.get_torque_supervision_weight() == PO.torque_supervision_weight(c, [0.1, 1000, 1000])
    alg.counter = 1400
    with pytest.raises(L.DwbcError):
        alg._fill_hp()                                    # OPR:91 has not run
    alg.set_arm_default_coeffs(torch.arange(6.0) + 5, torch.full((6,), 0.5), torch.zeros(1, 6))
    assert alg._arm_coefs.shape == (3, 6) and alg._arm_coefs[0].tolist() == [5, 6, 7, 8, 9, 10]
    hp = alg._fill_hp()
    assert abs(hp.torque_supervision_weight - 0.06) < 1e-7 and hp.arm_coefs == alg._arm_coefs.data_ptr()
    with pytest.raises(L.DwbcError):
        alg.set_arm_default_coeffs(torch.zeros(4, 6), torch.zeros(6), torch.zeros(6))      # per-env coefficients
    with pytest.raises(L.DwbcError):
        alg.set_arm_default_coeffs(torch.zeros(6), torch.zeros(6), torch.zeros(1, 20))     # OPR:91 hands `default_dof_pos[-7:-2]` of a [1, 20] tensor
    alg.set_arm_default_coeffs(5.0, torch.tensor(0.5), torch.zeros(6))                      # scalars broadcast
    assert alg._arm_coefs[0].tolist() == [5.0] * 6
    alg.set_arm_default_coeffs(torch.arange(6.0) + 5, torch.full((6,), 0.5), torch.zeros(1, 6))
    alg.init_storage(4, 3, [860], [None], [18])
    s = alg.storage
    assert s.target_arm_torques.shape == s.current_arm_dof_pos.shape == s.current_arm_dof_vel.shape == (3, 4, 6)
    assert s._c.target_arm_torques == s.target_arm_torques.data_ptr() and s._c.current_arm_dof_vel == s.current_arm_dof_vel.data_ptr()
    off = make_cpu_alg()
    off.init_storage(4, 3, [860], [None], [18])
    assert off.storage.target_arm_torques is None and not off.storage._c.target_arm_torques and off._fill_hp().arm_coefs is None


def test_chain_work_item_planner_host_logic():
    """launch_chain2n's planner (mlp_chain2.cuh, host code): every tile of every program is covered exactly once by the two-tile items
    [0, 2 np2) and the one-tile items behind them; one-tile items are only used when the simulated queue gets shorter; the bench shape
    (320 tiles x {actor, critic} on 148 SMs) gets a tail of one-tile items, small launches get one tile per item."""
    import ctypes as C
    from dwbc_b200 import _lib as L
    lib = L.lib()
    lib.dwbc_debug_chain_plan.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                          C.POINTER(C.c_double), C.POINTER(C.c_double)]

    def plan(tiles, costs, sms=148):
        c = (C.c_double * 4)(*(list(costs) + [0.0] * (4 - len(costs))))
        np2, ns1, span, span0 = C.c_int(), C.c_int(), C.c_double(), C.c_double()
        assert lib.dwbc_debug_chain_plan(tiles, len(costs), c, sms, C.byref(np2), C.byref(ns1), C.byref(span), C.byref(span0)) == 0
        return np2.value, ns1.value, span.value, span0.value

    for tiles in (1, 2, 37, 74, 75, 149, 299, 320, 321, 640, 1000):
        for costs in ((9.6, 7.65), (9.0,), (6.0, 6.0, 4.0, 4.0)):
            np2, ns1, span, span0 = plan(tiles, costs)
            if tiles * len(costs) <= 148:
                assert (np2, ns1) == (0, tiles)                     # one tile per item, spread over the SMs
                continue
            assert ns1 == 0 or 2 * np2 + ns1 == tiles               # whole pairs in front of the one-tile items
            assert 2 * np2 + ns1 >= tiles and 2 * (np2 - 1) + ns1 < tiles
            assert span <= span0 * (1 + 1e-12)
    np2, ns1, span, span0 = plan(320, (9.6, 7.65))                  # the flat-config mini-batch: 40 960 rows
    assert ns1 >= 48 and span < 0.92 * span0
    assert plan(320, (9.6, 7.65), sms=160)[1] == 0                  # 160 pairs per program on 160 CTAs: two full waves, nothing to fill
    assert lib.dwbc_debug_chain_plan(0, 2, None, 148, None, None, None, None) == -1


def test_chain_programs_host_logic():
    """The layer-chain PROGRAMS the entry points build (mlp.cu: build_forward / build_backward; host code, described by
    dwbc_debug_describe_chain without a GPU): a 4096-row rollout is four programs, one per head, of at most 6 ops (AC:204-217, 280-286); above
    37 tiles the heads share a program; update(): the loss hooks sit on the heads' last ops (PPO:166-221); fp32 precision does not use the chains."""
    import ctypes as C
    from dwbc_b200 import _lib as L
    lib = L.lib()
    lib.dwbc_debug_describe_chain.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_int32]
    ac = FlatActorCritic(device="cpu", num_priv=24, num_hist=10, num_prop=76)
    FIN_ACT, FIN_PPO, FIN_VALUE, FIN_REG, ELU, TANH = 1, 2, 3, 4, 1, 2

    def describe(rows, what, hist=0, precision="tf32x3", sms=148):
        ac.net_cfg.precision = L.PRECISIONS[precision]
        out = (C.c_int32 * 512)()
        k = lib.dwbc_debug_describe_chain(C.addressof(ac.net_cfg), rows, what, hist, sms, out, 512)
        if k < 0:
            return k
        v, i, progs = list(out[:k]), 2, []
        for _ in range(out[0]):
            n_ops, n_loads = v[i], v[i + 1]
            i += 2
            progs.append((n_loads, [dict(zip(("N", "kpad", "act", "fin", "fin_c", "out_col0", "y", "y_img"), v[i + 8 * j:i + 8 * j + 8])) for j in range(n_ops)]))
            i += 8 * n_ops
        assert i == k
        return v[1], progs

    widths = lambda prog: [o["N"] for o in prog[1]]  # noqa: E731
    fins = lambda prog: [(o["fin"], o["fin_c"]) for o in prog[1] if o["fin"]]  # noqa: E731
    # ---- rollout, 4096 rows: one program per head ----
    npack, progs = describe(4096, 0)
    assert npack == 20 and len(progs) == 4
    assert sorted(map(widths, progs)) == sorted([[64, 20, 128, 128, 128, 12], [64, 20, 128, 128, 128, 6], [128, 128, 128, 1], [128, 128, 128, 1]])
    assert sorted(f for p in progs for f in fins(p)) == [(FIN_ACT, 0), (FIN_ACT, 1)]          # sampling + log-prob on the two action heads only
    assert all(o["y"] == 0 or o["N"] <= 2 for p in progs for o in p[1])                         # nothing but the values leaves a rollout program by stores
    assert [o["act"] for o in progs[0][1]] == [ELU] * 5 + [TANH]                                # AC:157,170: tanh on the action means
    # ---- the same with the history-encoder latent (student rollouts): no privileged encoder in the programs ----
    _, progs_h = describe(4096, 0, hist=1)
    assert sorted(map(widths, progs_h)) == sorted([[128, 128, 128, 12], [128, 128, 128, 6], [128, 128, 128, 1], [128, 128, 128, 1]])
    # ---- 8192 rows (ROA): 64 tiles x 4 programs would not fit the SMs -> the heads share a program again ----
    npack, progs = describe(8192, 0)
    assert npack == 16 and list(map(widths, progs)) == [[64, 20, 128, 128, 128, 12, 128, 128, 6], [128, 128, 128, 1, 128, 128, 1]]
    assert progs[0][0] == 3 and progs[1][0] == 2                                                # gathers + the trunk reload of the second head
    assert len(describe(4096, 0, sms=100)[1]) == 2                                              # (the split follows the SM count)
    # ---- bootstrap values: the critic alone, split by head ----
    npack, progs = describe(4096, 1)
    assert npack == 8 and list(map(widths, progs)) == [[128, 128, 128, 1]] * 2
    # ---- update(): forward + loss, backward ----
    npack, (actor, critic) = describe(40960, 2)
    assert npack == 30 and widths(actor) == [64, 20, 128, 128, 128, 12, 128, 128, 6] and widths(critic) == [128, 128, 128, 1, 128, 128, 1]
    assert [(i, o["fin"], o["fin_c"]) for i, o in enumerate(actor[1]) if o["fin"]] == [(1, FIN_REG, 0), (5, FIN_PPO, 0), (8, FIN_PPO, 1)]
    assert [(i, o["fin"], o["fin_c"]) for i, o in enumerate(critic[1]) if o["fin"]] == [(3, FIN_VALUE, 0), (6, FIN_VALUE, 1)]
    assert all(o["y_img"] == (o["N"] == 128) for o in actor[1] + critic[1] if o["y"])          # 128-wide activations are kept as tile images
    _, (actor_b, critic_b) = describe(40960, 3)
    assert widths(actor_b) == [128] * 6 + [20, 64] and widths(critic_b) == [128] * 6
    assert describe(40960, 2, precision="fp32") == -2 and describe(0, 0) == -1


def test_checkpoint_round_trip_keeps_reference_names_and_shapes():
    """OPR:276-290: model_state_dict / optimizer_state_dict.  Names and order are the reference ActorCritic's (pinned by the golden file)."""
    g = np.load(os.path.join(G, "ppo.npz"))
    P = golden_params(g, int(g["meta"][2]))
    alg = make_cpu_alg()
    ac = alg.actor_critic
    ac.load_state_dict(P)
    sd = ac.state_dict()
    assert list(sd.keys()) == list(g["names"]) and list(sd.keys())[0] == "std"
    for k in P:
        assert sd[k].shape == P[k].shape and torch.equal(sd[k], P[k])
    assert sum(v.numel() for v in sd.values()) == 168698 and ac.num_params == ac.flat.numel() == 168928      # padded flat length
    # padded flat buffer: every tensor starts on a 32-float boundary, pads stay zero
    for n, off in ac.offsets.items():
        assert off % 32 == 0
    used = torch.zeros_like(ac.flat, dtype=torch.bool)
    for n, v in ac.views.items():
        used[ac.offsets[n]:ac.offsets[n] + v.numel()] = True
    assert float(ac.flat[~used].abs().max()) == 0.0
    # a second model loaded from the checkpoint is identical
    ac2 = FlatActorCritic(device="cpu", num_priv=24, num_hist=10, num_prop=76)
    ac2.load_state_dict(sd)
    assert torch.equal(ac2.flat, ac.flat)
    with pytest.raises(KeyError):
        ac2.load_state_dict({k: v for k, v in list(sd.items())[1:]})
    # optimizer: torch.optim.Adam layout (state[i] = {step, exp_avg, exp_avg_sq}, param_groups[0]['params'] = indices)
    opt = alg.optimizer
    assert opt.state_dict()["state"] == {}
    opt.step = 3
    opt.m.normal_()
    opt.v.uniform_()
    osd = opt.state_dict()
    names = list(sd.keys())
    assert sorted(osd["state"].keys()) == list(range(len(names))) and osd["param_groups"][0]["params"] == list(range(len(names)))
    for i, n in enumerate(names):
        st = osd["state"][i]
        assert st["exp_avg"].shape == sd[n].shape and st["exp_avg_sq"].shape == sd[n].shape and float(st["step"]) == 3.0
    alg2 = make_cpu_alg()
    alg2.optimizer.load_state_dict(osd)
    assert alg2.optimizer.step == 3
    for n in names:
        o, k = ac.offsets[n], sd[n].numel()
        assert torch.equal(alg2.optimizer.m[o:o + k], opt.m[o:o + k]) and torch.equal(alg2.optimizer.v[o:o + k], opt.v[o:o + k])
    assert osd["param_groups"][0]["lr"] == ppo_hp()["learning_rate"] and osd["param_groups"][0]["betas"] == (0.9, 0.999)


def test_storage_shapes_follow_reference():
    """RS:65-84 field names and shapes; observations are a view of the [T+1, N, n_obs] buffer the env kernel writes into."""
    alg = make_cpu_alg()
    alg.init_storage(8, 5, [860], [None], [18])
    s = alg.storage
    assert s.observations.shape == (5, 8, 860) and s.obs_row(5).shape == (8, 860)
    assert s.observations.data_ptr() == s.obs_row(0).data_ptr()
    for k, shp, dt in (("rewards", (5, 8, 2), torch.float32), ("actions", (5, 8, 18), torch.float32), ("dones", (5, 8, 1), torch.uint8),
                       ("values", (5, 8, 2), torch.float32), ("returns", (5, 8, 2), torch.float32), ("advantages", (5, 8, 2), torch.float32),
                       ("actions_log_prob", (5, 8, 2), torch.float32), ("mu", (5, 8, 18), torch.float32), ("sigma", (5, 8, 18), torch.float32)):
        t = getattr(s, k)
        assert tuple(t.shape) == shp and t.dtype == dt, k
    idx, mbs = s.draw_indices(4)
    assert mbs == 10 and sorted(idx.tolist()) == list(range(40))
    batches = list(s.mini_batch_generator(4, 3, idx))
    assert len(batches) == 12 and all(b.numel() == 10 for b in batches) and torch.equal(batches[0], batches[4])     # RS:182-188 order


@pytest.mark.skipif(not (os.environ.get("DWBC_REFERENCE") and os.path.isdir(os.path.join(os.environ["DWBC_REFERENCE"], "legged_gym"))),
                    reason="needs the original project's legged_gym config module: set DWBC_REFERENCE to a checkout of it")
def test_default_params_equal_the_reference_config():
    """`WidowGo1Params()` hard-codes the widowGo1 constants so that the kernels can run without legged_gym; this pins every one of them
    (dims, ranges, thresholds, curricula, PD gains, action scale, active reward terms and scales) to `WidowGo1RoughCfg` as shipped, read
    through `WidowGo1Params.from_legged_gym` (the path a real integration takes).  URDF-derived inputs are passed through."""
    import dataclasses
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import ref_harness as RH
    from dwbc_b200.config import DOF_NAMES_IG, WidowGo1Params
    _, Cfg, _ = RH.import_reference_env()
    cfg = Cfg()
    d = WidowGo1Params()
    scales = lambda o: {k: getattr(o, k) for k in dir(o) if not k.startswith("_")}  # noqa: E731  (class_to_dict of legged_gym/utils/helpers.py)
    p = WidowGo1Params.from_legged_gym(
        cfg, num_envs=d.num_envs, dt=cfg.control.decimation * cfg.sim.dt, dof_names=DOF_NAMES_IG, num_bodies=d.num_bodies, gripper_idx=d.gripper_idx,
        feet_indices=d.feet_indices, penalized_contact_indices=d.penalized_contact_indices, termination_contact_indices=d.termination_contact_indices,
        dof_pos_limits=d.dof_pos_limits, dof_vel_limits=d.dof_vel_limits, torque_limits=d.torque_limits, default_dof_pos=d.default_dof_pos,
        base_init_state=d.base_init_state, reward_scales=scales(cfg.rewards.scales), arm_reward_scales=scales(cfg.rewards.arm_scales))
    nz = lambda t: {k: v for k, v in t.items() if v != 0}  # noqa: E731  (zero-scale terms are dropped, WG:130-136)
    for f in dataclasses.fields(d):
        a, b = getattr(d, f.name), getattr(p, f.name)
        if f.name in ("reward_scales", "arm_reward_scales"):
            a, b = nz(a), nz(b)
        assert a == b, (f.name, a, b)


def test_fused_actor_critic_is_an_nn_module_over_the_flat_buffer():
    """What OnPolicyRunner.__init__ needs from the policy object (OPR:63-91), checked without a GPU: reference constructor signature, nn.Module
    parameters that alias the flat buffer, reference state_dict keys, .to() / .train(), every key of the reference's algorithm cfg accepted."""
    import json
    import os
    import torch.nn as nn
    from dwbc_b200 import runner_compat as RC
    from dwbc_b200.ppo import FusedPPO
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cfg = json.load(open(os.path.join(root, "baseline", "widowgo1_train_cfg.json")))
    ac = RC.FusedActorCritic(76, 76, 18, **cfg["policy"], num_priv=24, num_hist=10, num_prop=76, device="cpu")
    assert isinstance(ac, nn.Module) and ac.to("cpu") is ac and ac.train() is ac
    assert sum(p.numel() for p in ac.parameters()) == 168698
    keys = list(ac.state_dict())
    assert keys[0] == "std" and "actor.history_encoder.conv_layers.2.weight" in keys and "critic.critic_arm_control_head.4.bias" in keys
    ac.flat[ac.offsets["std"] + 3] = 0.5                                   # a kernel writing the flat buffer ...
    assert float(next(iter(ac.parameters())).view(-1)[3]) == 0.5           # ... is what torch sees through the Parameter
    sd = {k: v + 1.0 for k, v in ac.state_dict().items()}
    ac.load_state_dict(sd)
    assert abs(float(ac.std.view(-1)[3]) - 1.5) < 1e-6
    alg = FusedPPO(ac, device="cpu", **cfg["algorithm"])
    assert alg.actor_critic is ac and alg.precision == "tf32x3" and alg.actor_critic.net_cfg.precision == 2
    alg.precision = "fp32"
    assert ac.net_cfg.precision == 0

    class Mod:
        pass
    names = RC.install(Mod)
    assert Mod.FusedPPO is FusedPPO and Mod.FusedActorCritic is RC.FusedActorCritic and names["algorithm_class_name"] == "FusedPPO"
