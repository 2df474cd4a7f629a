"""Executes the UNMODIFIED reference on CPU for golden-vector generation: the checkout of the original
Deep-Whole-Body-Control repository (legged_gym/, rsl_rl/) that the environment variable DWBC_REFERENCE names.

The tests proper read the .npz files this produces; only the check of the default parameters against the
reference config (tests/test_host_cpu.py) imports it, and it skips without DWBC_REFERENCE.

Recipe = SURVEY.md Appendix A: fake `isaacgym` (tests/fakes), `WidowGo1.__new__`, synthetic
state tensors, then the reference's own `post_physics_step()`.  The reference draws randoms
with `torch_rand_float` over sparse `env_ids`; to make them reproducible the *harness* (not
the reference) wraps the resampling/reset methods so each call site reads its slice of one
dense uniform table rand[N, RAND_COLS] (column map: config.py).  The arithmetic executed is
still the reference's.
"""
import contextlib
import io
import os
import sys
import types
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
REF = os.environ.get("DWBC_REFERENCE", "")
if not (REF and os.path.isdir(os.path.join(REF, "legged_gym"))):
    raise ImportError("set DWBC_REFERENCE to a checkout of the original Deep-Whole-Body-Control repository (legged_gym/, rsl_rl/)")
for pth in (ROOT, os.path.join(ROOT, "tests", "fakes"), os.path.join(REF, "legged_gym"), os.path.join(REF, "rsl_rl")):
    if pth not in sys.path:
        sys.path.insert(0, pth)

for name in ("torchinfo", "matplotlib", "matplotlib.pyplot"):
    if name not in sys.modules:
        m = types.ModuleType(name)
        m.summary = lambda *a, **k: None
        sys.modules[name] = m

import dwbc_b200  # noqa: E402
from dwbc_b200 import config as C, synth  # noqa: E402


def import_reference_env():
    with contextlib.redirect_stdout(io.StringIO()):
        import isaacgym  # noqa: F401  (fake)
        from legged_gym.envs.widowGo1 import widowGo1 as wg_mod
        from legged_gym.envs.widowGo1.widowGo1_config import WidowGo1RoughCfg, WidowGo1RoughCfgPPO
    return wg_mod, WidowGo1RoughCfg, WidowGo1RoughCfgPPO


class _Gym:
    def __getattr__(self, name):
        return lambda *a, **k: None


class RandRedirect:
    """Context shared by the wrappers; `table` is the current step's rand[N, RAND_COLS]."""

    def __init__(self):
        self.table = None
        self.ids = None
        self.col = None
        self.in_reset = False
        self.goal_cols = None
        self.try_idx = 0

    def rand_float(self, lower, upper, shape, device):
        n = shape[1]
        r = self.table[self.ids, self.col:self.col + n]
        assert tuple(r.shape) == tuple(shape), (r.shape, shape, self.col)
        self.col += n
        return (upper - lower) * r + lower


def make_reference_env(p, st, seed, overrides=None):
    """Build a reference WidowGo1 with `WidowGo1.__new__` and fill the attributes of SURVEY
    Appendix A.2 from the dict `st` (numpy, synth.initial_env_state + synth.sim_state)."""
    wg_mod, Cfg, _ = import_reference_env()
    W = wg_mod.WidowGo1
    e = W.__new__(W)
    cfg = Cfg()
    N = p.num_envs
    for obj, d in ((cfg.rewards.scales, p.reward_scales), (cfg.rewards.arm_scales, p.arm_reward_scales)):
        for k in [k for k in dir(obj) if not k.startswith("_")]:
            setattr(obj, k, 0)
        for k, v in d.items():
            setattr(obj, k, v)
    cfg.rewards.only_positive_rewards = p.only_positive_rewards
    cfg.terrain.measure_heights = p.measure_heights
    cfg.terrain.curriculum = bool(p.terrain_curriculum)          # mesh_type stays 'trimesh' (WGC:290), so WG:115-116 keeps it
    e.cfg = cfg
    e.sim_params = SimpleNamespace(dt=0.005)
    e.num_envs, e.device, e.num_dofs, e.num_bodies, e.num_actions = N, "cpu", p.num_dofs, p.num_bodies, p.num_actions
    e.up_axis_idx = 2
    with contextlib.redirect_stdout(io.StringIO()):
        e._parse_cfg(cfg)
    e.dof_names = list(p.dof_names)
    e.dof_wo_gripper_names = e.dof_names[:-2]
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).clone()  # noqa: E731
    e._root_states = T(st["root_states"])
    e.root_states = e._root_states[:, 0, :]
    e.box_root_state = e._root_states[:, 1, :]
    e.base_quat = e.root_states[:, 3:7]
    e.dof_state = T(st["dof_state"])
    e.dof_pos = e.dof_state.view(N, p.num_dofs, 2)[..., 0]
    e.dof_vel = e.dof_state.view(N, p.num_dofs, 2)[..., 1]
    e.dof_pos_wrapped = e.dof_pos.clone()
    e._rigid_body_state = T(st["rigid_body_state"])
    e.rigid_body_state = e._rigid_body_state[:, :-1, :]
    e.gripper_idx = p.gripper_idx
    e.ee_pos = e.rigid_body_state[:, e.gripper_idx, :3]
    e.ee_orn = e.rigid_body_state[:, e.gripper_idx, 3:7]
    e._contact_forces = T(st["contact_forces"])
    e.contact_forces = e._contact_forces[:, :-1, :]
    e.force_sensor_tensor = T(st["force_sensor"])
    e.termination_contact_indices = torch.tensor(p.termination_contact_indices, dtype=torch.long)
    e.penalized_contact_indices = torch.tensor(p.penalized_contact_indices, dtype=torch.long)
    e.feet_indices = torch.tensor(p.feet_indices, dtype=torch.long)
    e.torques = T(st["torques"])
    e.action_history_buf = T(st["action_history_buf"])
    e.actions = e.action_history_buf[:, -3].clone()
    e.base_lin_vel = torch.zeros(N, 3)
    e.base_ang_vel = torch.zeros(N, 3)
    e.base_yaw_euler = torch.zeros(N, 3)
    e.base_yaw_quat = torch.zeros(N, 4)
    e.commands = T(st["commands"])
    e.commands_scale = torch.tensor([p.obs_scale_lin_vel, p.obs_scale_lin_vel, p.obs_scale_ang_vel])
    e.default_dof_pos = torch.tensor(p.default_dof_pos, dtype=torch.float)
    e.z_invariant_offset = torch.tensor([p.z_invariant_offset]).repeat(N, 1)
    for k in ("goal_timer", "traj_timesteps", "traj_total_timesteps", "ee_start_sphere", "ee_goal_sphere",
              "ee_goal_cart", "curr_ee_goal_sphere", "curr_ee_goal_cart", "ee_goal_delta_orn_euler",
              "ee_goal_orn_euler", "obs_history_buf", "last_actions", "last_dof_vel", "last_root_vel",
              "feet_air_time", "last_contacts", "env_origins", "box_env_origins_delta_y"):
        setattr(e, k, T(st[k]))
    e.curr_ee_goal = e.curr_ee_goal_sphere                     # alias, WG:590-593
    e.sphere_error_scale = torch.tensor(cfg.goal_ee.sphere_error_scale)
    e.orn_error_scale = torch.tensor(cfg.goal_ee.orn_error_scale)
    e.collision_lower_limits = torch.tensor(cfg.goal_ee.collision_lower_limits, dtype=torch.float)
    e.collision_upper_limits = torch.tensor(cfg.goal_ee.collision_upper_limits, dtype=torch.float)
    e.underground_limit = cfg.goal_ee.underground_limit
    e.num_collision_check_samples = cfg.goal_ee.num_collision_check_samples
    e.collision_check_t = torch.linspace(0, 1, e.num_collision_check_samples)[None, None, :]
    e.mass_params_tensor = T(st["mass_params"])
    e.friction_coeffs_tensor = T(st["friction"])
    e.motor_strength = T(st["motor_strength"])
    e.episode_length_buf = T(st["episode_length_buf"])
    e.rew_buf = torch.zeros(N)
    e.arm_rew_buf = torch.zeros(N)
    e.reset_buf = torch.ones(N, dtype=torch.long)
    e.time_out_buf = torch.zeros(N, dtype=torch.bool)
    e.obs_buf = torch.zeros(N, p.num_obs)
    e.privileged_obs_buf = None
    e.base_init_state = torch.tensor(p.base_init_state, dtype=torch.float)
    e.box_env_origins_x = p.box_env_origins_x
    e.box_env_origins_z = p.box_env_origins_z
    e.dof_pos_limits = torch.tensor(p.dof_pos_limits, dtype=torch.float)
    e.dof_vel_limits = torch.tensor(p.dof_vel_limits, dtype=torch.float)
    e.torque_limits = torch.tensor(p.torque_limits, dtype=torch.float)
    e.extras = {"episode": {}}
    e.common_step_counter = 0
    e.viewer = None
    e.gym = _Gym()
    e.sim = None
    e.init_done = True
    if p.measure_heights or p.terrain_curriculum:
        e.terrain = SimpleNamespace(cfg=cfg.terrain, env_length=p.terrain_env_length)
    if p.measure_heights:
        e.height_samples = T(st["height_samples"])
        e.height_points = e._init_height_points()
    if p.terrain_curriculum:
        # base-class wiring of LR:717-731 (WidowGo1._get_env_origins, WG:207-228, does not create these tensors; SURVEY 8a row a21)
        assert cfg.terrain.curriculum, "WG:115-116 switched the terrain curriculum off"
        e.terrain_levels, e.terrain_types = T(st["terrain_levels"]), T(st["terrain_types"])
        e.terrain_origins = T(st["terrain_origins"])
        e.max_terrain_level = p.max_terrain_level
    e.measured_heights = 0
    e._prepare_reward_function()

    # ---- RNG redirection (harness-side wrappers; see module docstring) ----
    rr = RandRedirect()
    wg_mod.torch_rand_float = rr.rand_float
    allids = torch.arange(N)

    def wrap(name, pre):
        orig = getattr(e, name)

        def f(*a, **k):
            pre(*a, **k)
            return orig(*a, **k)
        setattr(e, name, f)

    def pre_goal(env_ids, is_init=False):
        rr.goal_cols = (C.RAND_RST_GOAL_ORN, C.RAND_RST_GOAL_SPH) if is_init else (C.RAND_GOAL_ORN, C.RAND_GOAL_SPH)
        rr.try_idx = 0

    def pre_orn(env_ids):
        rr.ids, rr.col = env_ids, rr.goal_cols[0]

    def pre_sph(env_ids):
        rr.ids, rr.col = env_ids, rr.goal_cols[1] + 3 * rr.try_idx
        rr.try_idx += 1

    def pre_cmd(env_ids):
        rr.ids, rr.col = env_ids, (C.RAND_RST_CMD if rr.in_reset else C.RAND_CMD)

    def pre_push():
        rr.ids, rr.col = allids, C.RAND_PUSH

    def pre_dofs(env_ids):
        rr.ids, rr.col = env_ids, C.RAND_RST_DOF

    def pre_root(env_ids):
        rr.ids, rr.col = env_ids, C.RAND_RST_XY

    if p.terrain_curriculum:
        # LR:438 draws with torch.randint_like (not torch_rand_float): for the duration of the reference's own
        # _update_terrain_curriculum the harness serves that draw from column RAND_TERRAIN of the step's table,
        # floor(u * max_level) clamped to max_level - 1 (the integer the oracle and the kernel derive from the same uniform)
        orig_tc = e._update_terrain_curriculum

        def terrain_curriculum(env_ids):
            real = torch.randint_like

            def from_table(t, high, **kw):
                r = (rr.table[env_ids, C.RAND_TERRAIN] * high).long().clamp(max=high - 1)
                assert r.shape == t.shape
                return r.to(t.dtype)
            torch.randint_like = from_table
            try:
                return orig_tc(env_ids)
            finally:
                torch.randint_like = real
        e._update_terrain_curriculum = terrain_curriculum
    wrap("_resample_ee_goal", pre_goal)
    wrap("_resample_ee_goal_orn_once", pre_orn)
    wrap("_resample_ee_goal_sphere_once", pre_sph)
    wrap("_resample_commands", pre_cmd)
    wrap("_push_robots", pre_push)
    wrap("_reset_dofs", pre_dofs)
    wrap("_reset_root_states", pre_root)
    orig_reset = e.reset_idx

    def reset_idx(env_ids, start=False):
        rr.in_reset = True
        try:
            return orig_reset(env_ids, start)
        finally:
            rr.in_reset = False
    e.reset_idx = reset_idx
    e._rr = rr
    return e


def load_sim_into_reference(e, p, sim):
    """Overwrite the Isaac-Gym-owned tensors in place (views stay valid) and emulate the
    pre-physics half of `step` (WG:1162-1173): permute+clip+delay the policy action."""
    e._root_states.copy_(torch.from_numpy(sim["root_states"]))
    e.dof_state.copy_(torch.from_numpy(sim["dof_state"]))
    e._rigid_body_state.copy_(torch.from_numpy(sim["rigid_body_state"]))
    e._contact_forces.copy_(torch.from_numpy(sim["contact_forces"]))
    e.force_sensor_tensor.copy_(torch.from_numpy(sim["force_sensor"]))
    e.torques = torch.from_numpy(sim["torques"]).clone()
    a = torch.from_numpy(sim["policy_actions"])[:, p.raisim2ig(p.num_actions)]
    a = torch.clip(a, -100.0, 100.0)
    e.action_history_buf = torch.cat([e.action_history_buf[:, 1:], a[:, None, :]], dim=1)
    e.actions = e.action_history_buf[:, -3].clone()
