"""ctypes binding of libdwbc.so (include/dwbc.h).  This is the thin host<->C-ABI seam: struct
mirrors, argument marshalling (`tensor.data_ptr()`, current CUDA stream) and error mapping.

There is NO fallback: if the shared library is missing or a call fails the binding raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdwbc.so")

ABI_VERSION = 4
MAX_DOF, MAX_TERMS, MAX_IDX, MAX_SLOTS, NUM_METRICS, RAND_COLS, MAX_LAYERS = 24, 40, 8, 64, 10, 104, 4
GS, DS = 28, 72
GS_COL = dict(commands=0, goal_timer=3, traj_timesteps=4, traj_total_timesteps=5, ee_start_sphere=6, ee_goal_sphere=9,
              ee_goal_cart=12, curr_ee_goal_sphere=15, curr_ee_goal_cart=18, ee_goal_delta_orn_euler=21, ee_goal_orn_euler=24)
DS_COL = dict(base_lin_vel=0, base_ang_vel=3, base_yaw_euler=6, base_yaw_quat=9, last_root_vel=13, feet_air_time=19,
              last_contacts=23, last_actions=28, last_dof_vel=48)

i32, i64, f32, u64, vp = C.c_int32, C.c_int64, C.c_float, C.c_uint64, C.c_void_p


class EnvCfg(C.Structure):
    _fields_ = [
        ("abi_version", i32),
        ("num_envs", i32), ("num_dofs", i32), ("num_actions", i32), ("num_bodies_p1", i32), ("gripper_idx", i32),
        ("num_prop", i32), ("num_priv", i32), ("history_len", i32), ("num_obs", i32), ("action_hist_len", i32),
        ("feet_idx", i32 * 4), ("feet_perm", i32 * 4),
        ("n_penalized", i32), ("penalized_idx", i32 * MAX_IDX),
        ("n_term_contact", i32), ("term_contact_idx", i32 * MAX_IDX),
        ("ig2raisim", i32 * MAX_DOF),
        ("waist_dof", i32), ("goal_is_cart", i32), ("max_episode_length", i32), ("resample_interval", i32),
        ("n_collision_samples", i32), ("max_goal_tries", i32), ("only_positive_rewards", i32),
        ("n_leg_terms", i32), ("leg_term", i32 * MAX_TERMS), ("leg_slot", i32 * MAX_TERMS),
        ("n_arm_terms", i32), ("arm_term", i32 * MAX_TERMS), ("arm_slot", i32 * MAX_TERMS),
        ("termination_slot", i32), ("n_sum_slots", i32), ("sums_stride", i32),
        ("measure_heights", i32), ("n_height_x", i32), ("n_height_y", i32), ("terrain_rows", i32), ("terrain_cols", i32),
        ("terrain_curriculum", i32), ("max_terrain_level", i32), ("terrain_n_types", i32),
        ("default_dof_pos", f32 * MAX_DOF),
        ("dof_pos_lower", f32 * MAX_DOF), ("dof_pos_upper", f32 * MAX_DOF), ("dof_vel_limits", f32 * MAX_DOF),
        ("torque_limits", f32 * MAX_DOF),
        ("obs_scale_lin_vel", f32), ("obs_scale_ang_vel", f32), ("obs_scale_dof_pos", f32), ("obs_scale_dof_vel", f32),
        ("obs_scale_height", f32), ("clip_obs", f32),
        ("term_roll", f32), ("term_pitch", f32), ("term_z", f32), ("lin_vel_x_clip", f32), ("ang_vel_yaw_clip", f32),
        ("collision_lower", f32 * 3), ("collision_upper", f32 * 3), ("underground_limit", f32), ("collision_t", f32 * 16),
        ("sphere_error_scale", f32 * 3), ("orn_error_scale", f32 * 3), ("z_invariant_offset", f32),
        ("tracking_sigma", f32), ("tracking_ee_sigma", f32), ("base_height_target", f32), ("max_contact_force", f32),
        ("soft_dof_vel_limit", f32), ("soft_torque_limit", f32), ("dt", f32), ("max_episode_length_s", f32),
        ("base_init_state", f32 * 13), ("origin_perturb", f32 * 2), ("init_vel_perturb", f32 * 2),
        ("box_x", f32), ("box_z", f32), ("push_vel", f32 * 2), ("dof_reset", f32 * 2),
        ("delta_orn_lo", f32 * 3), ("delta_orn_span", f32 * 3),
        ("height_x", f32 * 24), ("height_y", f32 * 16), ("border_size", f32), ("horizontal_scale", f32),
        ("vertical_scale", f32), ("terrain_env_length", f32),
    ]


class EnvBuffers(C.Structure):
    _fields_ = [(n, vp) for n in (
        "root_states", "dof_state", "rigid_body_state", "contact_forces", "force_sensor", "torques", "actions",
        "action_history", "mass_params", "friction", "motor_strength", "env_origins", "box_env_origins_delta_y",
        "goal_state", "derived_state", "episode_length", "obs_history", "episode_sums", "height_samples",
        "measured_heights", "heights_obs", "terrain_levels", "terrain_types", "terrain_origins", "obs_buf")] + \
        [("obs_stride", i64)] + [(n, vp) for n in ("rew_buf", "arm_rew_buf", "reset_buf", "time_out_buf", "episode_stats",
                                                   "store_values", "store_rewards", "store_dones")] + [("store_gamma", f32), ("reserved_", i32)]


class StepArgs(C.Structure):
    _fields_ = [("rand_uniform", vp), ("seed", u64), ("step", u64), ("do_push", i32),
                ("lin_vel_x", f32 * 2), ("ang_vel_yaw", f32 * 2), ("goal_l", f32 * 2), ("goal_p", f32 * 2), ("goal_y", f32 * 2),
                ("leg_scale", f32 * MAX_TERMS), ("arm_scale", f32 * MAX_TERMS),
                ("leg_termination_scale", f32), ("arm_termination_scale", f32), ("generic_kernel", i32), ("reserved_", i32)]


class NetCfg(C.Structure):
    _fields_ = [
        ("abi_version", i32),
        ("num_prop", i32), ("num_priv", i32), ("num_hist", i32), ("num_obs", i32), ("n_leg", i32), ("n_arm", i32),
        ("n_priv_layers", i32), ("priv_dims", i32 * MAX_LAYERS),
        ("n_actor_layers", i32), ("actor_dims", i32 * MAX_LAYERS),
        ("n_critic_layers", i32), ("critic_dims", i32 * MAX_LAYERS),
        ("n_leg_layers", i32), ("leg_dims", i32 * MAX_LAYERS),
        ("n_arm_layers", i32), ("arm_dims", i32 * MAX_LAYERS),
        ("hist_proj", i32), ("hist_c1", i32), ("hist_k1", i32), ("hist_s1", i32), ("hist_c2", i32), ("hist_k2", i32), ("hist_s2", i32),
        ("num_params", i64), ("off_std", i64),
        ("off_priv_w", i64 * MAX_LAYERS), ("off_priv_b", i64 * MAX_LAYERS),
        ("off_hist_w", i64 * 4), ("off_hist_b", i64 * 4),
        ("off_actor_w", i64 * MAX_LAYERS), ("off_actor_b", i64 * MAX_LAYERS),
        ("off_aleg_w", i64 * (MAX_LAYERS + 1)), ("off_aleg_b", i64 * (MAX_LAYERS + 1)),
        ("off_aarm_w", i64 * (MAX_LAYERS + 1)), ("off_aarm_b", i64 * (MAX_LAYERS + 1)),
        ("off_critic_w", i64 * MAX_LAYERS), ("off_critic_b", i64 * MAX_LAYERS),
        ("off_cleg_w", i64 * (MAX_LAYERS + 1)), ("off_cleg_b", i64 * (MAX_LAYERS + 1)),
        ("off_carm_w", i64 * (MAX_LAYERS + 1)), ("off_carm_b", i64 * (MAX_LAYERS + 1)),
        ("precision", i32), ("activation", i32),
    ]


PRECISIONS = {"fp32": 0, "tf32": 1, "tf32x3": 2}
# rsl_rl `get_activation` names (AC) -> DwbcActivation; "crelu" is rsl_rl's name for a plain nn.ReLU()
ACTIVATIONS = {"elu": 0, "selu": 1, "relu": 2, "crelu": 2, "lrelu": 3, "tanh": 4, "sigmoid": 5}


class PpoHyper(C.Structure):
    _fields_ = [("clip_param", f32), ("value_loss_coef", f32), ("entropy_coef", f32), ("priv_reg_coef", f32),
                ("mixing_ratio", f32), ("use_clipped_value_loss", i32), ("max_grad_norm", f32), ("lr", f32),
                ("beta1", f32), ("beta2", f32), ("adam_eps", f32), ("grad_scale", f32),
                ("torque_supervision_weight", f32), ("arm_coefs", vp)]


class Storage(C.Structure):
    _fields_ = [("observations", vp), ("obs_stride", i64), ("actions", vp), ("values", vp), ("returns", vp),
                ("advantages", vp), ("log_prob", vp), ("hist_latent", vp), ("hist_latent_ld", i64),
                ("target_arm_torques", vp), ("current_arm_dof_pos", vp), ("current_arm_dof_vel", vp)]


class PdCfg(C.Structure):
    _fields_ = [("n_dof", i32), ("n_act", i32), ("wrap_dof", i32)] + \
               [(k, C.c_float * MAX_DOF) for k in ("p_gains", "d_gains", "action_scale", "default_dof_pos", "torque_limits")]


class DwbcError(RuntimeError):
    pass


_ERR = {-1: "DWBC_ERR_ARG (null pointer / bad dimension)", -2: "DWBC_ERR_UNSUPPORTED (configuration not implemented)",
        -3: "DWBC_ERR_LAUNCH (CUDA launch failed)"}
_lib = None

_SIGS = {
    "dwbc_post_physics_step": [vp, vp, vp, vp],
    "dwbc_fill_uniform": [vp, i32, u64, u64, vp],
    "dwbc_pre_physics_actions": [vp, vp, f32, vp, vp, i32, i32, i32, i32, vp],
    "dwbc_store_rewards": [vp, vp, vp, vp, vp, f32, vp, vp, i32, vp],
    "dwbc_gae": [vp, vp, vp, vp, vp, vp, vp, i32, i32, f32, f32, i32, vp],
    "dwbc_normalize_advantages": [vp, vp, i64, vp],
    "dwbc_policy_act": [vp, vp, vp, i64, vp, i32, vp, vp, vp, vp, vp, i32, i32, vp, vp],
    "dwbc_critic_values": [vp, vp, vp, i64, vp, i32, vp, vp],
    "dwbc_hist_latent": [vp, vp, vp, i64, vp, i64, i32, vp, vp],
    "dwbc_compute_torques": [vp, vp, vp, vp, vp, i32, vp],
    "dwbc_ppo_minibatch_grad": [vp, vp, vp, vp, i32, vp, vp, vp, vp, vp],
    "dwbc_dagger_minibatch_grad": [vp, vp, vp, vp, i32, vp, vp, vp, vp],
    "dwbc_clip_adam_step": [vp, vp, vp, vp, i64, i64, vp, i32, vp, vp, vp],
    "dwbc_enforce_min_std": [vp, i64, vp, i32, vp],
}
EXPORTS = sorted(list(_SIGS) + ["dwbc_workspace_bytes", "dwbc_version", "dwbc_struct_sizes", "dwbc_launch_count"])


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libdwbc.so in-tree with nvcc for sm_100a (no GPU needed)."""
    csrc = os.path.join(_HERE, "csrc")
    if force:
        subprocess.run(["make", "-C", csrc, "clean"], check=True, capture_output=not verbose)
    r = subprocess.run(["make", "-C", csrc, "-j4"], capture_output=not verbose, text=True)
    if r.returncode != 0:
        raise DwbcError("building libdwbc.so failed:\n" + (r.stdout or "") + (r.stderr or ""))
    return LIB_PATH


def lib():
    """Load libdwbc.so (once).  Raises if it is absent: there is no CPU / PyTorch fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DwbcError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(or make -C deep-whole-body-control_b200/csrc). The dwbc_b200 product path has no fallback.")
    L = C.CDLL(LIB_PATH)
    for name, sig in _SIGS.items():
        fn = getattr(L, name)
        fn.argtypes = sig
        fn.restype = C.c_int
    L.dwbc_workspace_bytes.argtypes = [vp, i64]
    L.dwbc_workspace_bytes.restype = i64
    L.dwbc_version.restype = C.c_char_p
    L.dwbc_launch_count.restype = C.c_uint64
    L.dwbc_struct_sizes.argtypes = [C.POINTER(i64 * 6)]
    L.dwbc_struct_sizes.restype = None
    sizes = (i64 * 6)()
    L.dwbc_struct_sizes(C.byref(sizes))
    mine = [C.sizeof(s) for s in (EnvCfg, EnvBuffers, StepArgs, NetCfg, PpoHyper, Storage)]
    if list(sizes) != mine:
        raise DwbcError(f"struct layout mismatch between include/dwbc.h and _lib.py: C {list(sizes)} vs ctypes {mine}")
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        raise DwbcError(f"{what} failed: {_ERR.get(rc, rc)}")


def ptr(t, dtype=None):
    """Device pointer of a contiguous CUDA torch tensor (None -> NULL).  The kernels reinterpret raw memory, so a tensor of the
    wrong dtype or on the host must fail here, loudly, instead of being misread (`dtype`: expected torch dtype or tuple)."""
    if t is None:
        return None
    if not t.is_contiguous():
        raise DwbcError("dwbc kernels need contiguous buffers")
    if not t.is_cuda:
        raise DwbcError("dwbc kernels need CUDA tensors (got a host tensor)")
    if dtype is not None and t.dtype not in (dtype if isinstance(dtype, tuple) else (dtype,)):
        raise DwbcError(f"dwbc kernel argument has dtype {t.dtype}, expected {dtype}")
    return t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream
