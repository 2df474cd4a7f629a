"""Golden vectors of `WidowGo1._compute_torques` (WG:1262-1295): the UNMODIFIED reference method is called on a stub object
holding exactly the attributes it reads; asserts oracle == reference and writes tests/golden/torques.npz.
Run with a checkout of the original repository:  DWBC_REFERENCE=<checkout> python tests/golden/make_golden_torques.py"""
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness as RH  # noqa: E402  (sets up sys.path, the fake isaacgym and the import stubs)
from dwbc_b200 import synth  # noqa: E402
from dwbc_b200.config import WidowGo1Params  # noqa: E402
from oracle import env_oracle as EO  # noqa: E402

wg_mod, _, _ = RH.import_reference_env()
p = WidowGo1Params(num_envs=64)
N, nd, na, seed = p.num_envs, p.num_dofs, p.num_actions, 77
actions = torch.from_numpy(synth.normal(seed, 1, (N, na), 0.0, 1.5))
dof_pos = torch.tensor(p.default_dof_pos) + torch.from_numpy(synth.normal(seed, 2, (N, nd), 0.0, 0.6))
dof_pos[:, 10] += torch.from_numpy(synth.normal(seed, 3, (N,), 0.0, 4.0))       # column -8 of the 18-wide tensor leaves (-pi, pi] for some envs
dof_vel = torch.from_numpy(synth.normal(seed, 4, (N, nd), 0.0, 3.0))
motor = torch.from_numpy(0.7 + 0.6 * synth.uniform(seed, 5, (N, na)))
obj = SimpleNamespace(
    cfg=SimpleNamespace(control=SimpleNamespace(adaptive_arm_gains=False, torque_supervision=False)),
    motor_strength=motor.clone(), action_scale=torch.tensor(p.action_scale), p_gains=torch.tensor(p.p_gains), d_gains=torch.tensor(p.d_gains),
    dof_pos_wo_gripper=dof_pos[:, :na].clone(), dof_pos_wo_gripper_wrapped=torch.zeros(N, na), dof_vel_wo_gripper=dof_vel[:, :na].clone(),
    default_dof_pos_wo_gripper=torch.tensor(p.default_dof_pos)[:na].unsqueeze(0), gripper_torques_zero=torch.zeros(N, nd - na),
    torque_limits=torch.tensor(p.torque_limits))
ref = wg_mod.WidowGo1._compute_torques(obj, actions.clone())
orc = EO.compute_torques(actions, dof_pos, dof_vel, motor, torch.tensor(p.p_gains), torch.tensor(p.d_gains), torch.tensor(p.action_scale),
                         torch.tensor(p.default_dof_pos), torch.tensor(p.torque_limits))
assert ref.shape == (N, nd)
assert torch.equal(ref, orc), float((ref - orc).abs().max())
assert int((ref.abs() == torch.tensor(p.torque_limits)).sum()) > 0 and int((ref.abs() < torch.tensor(p.torque_limits) - 1e-3).sum()) > 0
np.savez_compressed(os.path.join(HERE, "torques.npz"), actions=actions.numpy(), dof_pos=dof_pos.numpy(), dof_vel=dof_vel.numpy(), motor=motor.numpy(),
                    torques=ref.numpy(), meta=np.array([N, seed]))
print("torques.npz written: oracle == reference (max |diff| = 0.0), clipped entries:", int((ref.abs() == torch.tensor(p.torque_limits)).sum()))
