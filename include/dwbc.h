/*
 * dwbc.h -- C ABI of the B200-native widowGo1 hot path (libdwbc.so, sm_100a).
 *
 * The reference (MarkFzp/Deep-Whole-Body-Control) has NO FFI / plugin interface: the path
 * sits behind four Python surfaces (SURVEY.md section 8b).  Each entry point below replaces
 * the body of one of those Python methods; the reference-side binding a maintainer adds is
 * the ctypes stub shown in INTEGRATION.md.  File:line citations are relative to the reference
 * tree (WG = legged_gym/legged_gym/envs/widowGo1/widowGo1.py, LR = envs/base/legged_robot.py,
 * RS = rsl_rl/rsl_rl/storage/rollout_storage.py, PPO = rsl_rl/rsl_rl/algorithms/ppo.py,
 * AC = rsl_rl/rsl_rl/modules/actor_critic.py).
 *
 * Conventions: every pointer is a DEVICE pointer into a caller-owned, contiguous, row-major
 * buffer (fp32 unless the type says otherwise).  The library allocates nothing, keeps no
 * global state (except a launch counter and the tuning defaults of include/dwbc_debug.h), never synchronises and never throws: every function enqueues its kernels on
 * the given stream and returns DWBC_OK or a negative error code.  Structs are passed by
 * pointer to HOST memory and are read before the call returns.
 */
#ifndef DWBC_H
#define DWBC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dwbc_stream_t; /* cudaStream_t */

enum {
  DWBC_OK = 0,
  DWBC_ERR_ARG = -1,         /* null pointer / bad dimension */
  DWBC_ERR_UNSUPPORTED = -2, /* configuration outside what the kernels implement */
  DWBC_ERR_LAUNCH = -3       /* cudaGetLastError() != cudaSuccess after the launch */
};

#define DWBC_ABI_VERSION 4
#define DWBC_MAX_DOF 24
#define DWBC_MAX_TERMS 40   /* active reward terms per channel */
#define DWBC_MAX_IDX 8      /* penalised / termination contact bodies */
#define DWBC_MAX_SLOTS 64   /* episode_sums + episode_metric_sums columns */
#define DWBC_NUM_METRICS 10 /* WG:164 */
#define DWBC_RAND_COLS 104  /* uniform table columns, see DwbcRandCol */

/* Columns of the per-step uniform table rand[N, DWBC_RAND_COLS]; one per element the
 * reference draws with torch_rand_float at the cited call site. */
enum DwbcRandCol {
  DWBC_RAND_GOAL_ORN = 0,       /* 3   WG:1307-1313 (timer expiry) */
  DWBC_RAND_GOAL_SPH = 3,       /* 30  WG:1303-1306 x <=10 tries (WG:1325-1330) */
  DWBC_RAND_CMD = 33,           /* 2   WG:837-839 via WG:922-925 */
  DWBC_RAND_PUSH = 35,          /* 2   WG:808 */
  DWBC_RAND_RST_DOF = 37,       /* 20  WG:824 */
  DWBC_RAND_RST_XY = 57,        /* 2   WG:767 */
  DWBC_RAND_RST_VEL = 59,       /* 6   WG:774 */
  DWBC_RAND_RST_CMD = 65,       /* 2   WG:726-727 */
  DWBC_RAND_RST_GOAL_ORN = 67,  /* 3 */
  DWBC_RAND_RST_GOAL_SPH = 70,  /* 30 */
  DWBC_RAND_TERRAIN = 100       /* 1   LR:438 */
};

/* Reward terms (WG:1352-1469, LR:832-922), alphabetical = the reference's dir() order. */
enum DwbcTerm {
  DWBC_TERM_action_rate = 0, DWBC_TERM_ang_vel_xy, DWBC_TERM_arm_energy_abs_sum, DWBC_TERM_base_height,
  DWBC_TERM_collision, DWBC_TERM_dof_acc, DWBC_TERM_dof_pos_limits, DWBC_TERM_dof_vel, DWBC_TERM_dof_vel_limits,
  DWBC_TERM_energy_square, DWBC_TERM_feet_air_time, DWBC_TERM_feet_contact_forces, DWBC_TERM_foot_contacts_z,
  DWBC_TERM_hip_action_l2, DWBC_TERM_leg_action_l2, DWBC_TERM_leg_energy, DWBC_TERM_leg_energy_abs_sum,
  DWBC_TERM_leg_energy_sum_abs, DWBC_TERM_lin_vel_z, DWBC_TERM_stand_still, DWBC_TERM_stumble, DWBC_TERM_survive,
  DWBC_TERM_termination, DWBC_TERM_torque_limits, DWBC_TERM_torques, DWBC_TERM_tracking_ang_vel,
  DWBC_TERM_tracking_ang_vel_yaw_exp, DWBC_TERM_tracking_ang_vel_yaw_l1, DWBC_TERM_tracking_ee_cart,
  DWBC_TERM_tracking_ee_orn, DWBC_TERM_tracking_ee_orn_ry, DWBC_TERM_tracking_ee_sphere, DWBC_TERM_tracking_lin_vel,
  DWBC_TERM_tracking_lin_vel_x_exp, DWBC_TERM_tracking_lin_vel_x_l1, DWBC_TERM_tracking_lin_vel_y_l2,
  DWBC_TERM_tracking_lin_vel_z_l2, DWBC_TERM_COUNT
};

/* Column layout of goal_state[N, DWBC_GS] (task state the kernel reads AND writes). */
enum {
  DWBC_GS_COMMANDS = 0, DWBC_GS_GOAL_TIMER = 3, DWBC_GS_TRAJ_T = 4, DWBC_GS_TRAJ_TOTAL = 5, DWBC_GS_START_SPH = 6,
  DWBC_GS_GOAL_SPH = 9, DWBC_GS_GOAL_CART = 12, DWBC_GS_CURR_SPH = 15, DWBC_GS_CURR_CART = 18, DWBC_GS_DELTA_ORN = 21,
  DWBC_GS_GOAL_ORN = 24, DWBC_GS = 28
};
/* Column layout of derived_state[N, DWBC_DS] (written every step; the feet/last_* columns are
 * read back only when a term that needs them is active). */
enum {
  DWBC_DS_BASE_LIN_VEL = 0, DWBC_DS_BASE_ANG_VEL = 3, DWBC_DS_YAW_EULER = 6, DWBC_DS_YAW_QUAT = 9,
  DWBC_DS_LAST_ROOT_VEL = 13, DWBC_DS_FEET_AIR_TIME = 19, DWBC_DS_LAST_CONTACTS = 23, DWBC_DS_LAST_ACTIONS = 28,
  DWBC_DS_LAST_DOF_VEL = 48, DWBC_DS = 72
};

/* Static task description, snapshotted from the reference config at start-up
 * (widowGo1_config.py) plus the URDF-derived tables of WG:255-420 / LR:279-305. */
typedef struct DwbcEnvCfg {
  int32_t abi_version;
  int32_t num_envs, num_dofs, num_actions, num_bodies_p1 /* n_body + box */, gripper_idx;
  int32_t num_prop, num_priv, history_len, num_obs, action_hist_len;
  int32_t feet_idx[4], feet_perm[4];
  int32_t n_penalized, penalized_idx[DWBC_MAX_IDX];
  int32_t n_term_contact, term_contact_idx[DWBC_MAX_IDX];
  int32_t ig2raisim[DWBC_MAX_DOF]; /* obs column j <- Isaac Gym dof (WG:1010-1028) */
  int32_t waist_dof;               /* dof wrapped to (-pi,pi] (WG:970: column -8) */
  int32_t goal_is_cart;            /* cfg.goal_ee.command_mode == 'cart' (WG:589-593) */
  int32_t max_episode_length;      /* WG:118 */
  int32_t resample_interval;       /* WG:922 */
  int32_t n_collision_samples, max_goal_tries;
  int32_t only_positive_rewards;
  /* reward tables: active terms per channel in summation order, and their episode_sums slot */
  int32_t n_leg_terms, leg_term[DWBC_MAX_TERMS], leg_slot[DWBC_MAX_TERMS];
  int32_t n_arm_terms, arm_term[DWBC_MAX_TERMS], arm_slot[DWBC_MAX_TERMS];
  int32_t termination_slot;        /* slot of episode_sums['termination'] or -1 */
  int32_t n_sum_slots;             /* episode_sums columns; metrics follow at [n_sum_slots, +10) */
  int32_t sums_stride;             /* row stride of episode_sums (>= n_sum_slots + 10) */
  /* terrain */
  int32_t measure_heights, n_height_x, n_height_y, terrain_rows, terrain_cols;
  int32_t terrain_curriculum, max_terrain_level, terrain_n_types;
  float default_dof_pos[DWBC_MAX_DOF];
  float dof_pos_lower[DWBC_MAX_DOF], dof_pos_upper[DWBC_MAX_DOF], dof_vel_limits[DWBC_MAX_DOF], torque_limits[DWBC_MAX_DOF];
  float obs_scale_lin_vel, obs_scale_ang_vel, obs_scale_dof_pos, obs_scale_dof_vel, obs_scale_height;
  float clip_obs;                  /* <= 0 disables the +-clip of WG:1195-1196 */
  float term_roll, term_pitch, term_z;
  float lin_vel_x_clip, ang_vel_yaw_clip;
  float collision_lower[3], collision_upper[3], underground_limit, collision_t[16];
  float sphere_error_scale[3], orn_error_scale[3], z_invariant_offset;
  float tracking_sigma, tracking_ee_sigma, base_height_target, max_contact_force;
  float soft_dof_vel_limit, soft_torque_limit, dt, max_episode_length_s;
  float base_init_state[13], origin_perturb[2] /* lo, span */, init_vel_perturb[2];
  float box_x, box_z, push_vel[2];
  float dof_reset[2];              /* 0.8, (1.2-0.8) : WG:824 */
  float delta_orn_lo[3], delta_orn_span[3];
  float height_x[24], height_y[16], border_size, horizontal_scale, vertical_scale, terrain_env_length;
} DwbcEnvCfg;

/* Device buffers of one env shard. */
typedef struct DwbcEnvBuffers {
  /* Isaac-Gym-owned tensors, layouts of WG:523-558 */
  float* root_states;            /* [N,2,13] robot row 0, box row 1; written on reset / push */
  float* dof_state;              /* [N*n_dof,2] (pos, vel); written on reset */
  const float* rigid_body_state; /* [N,n_body+1,13] */
  const float* contact_forces;   /* [N,n_body+1,3] */
  const float* force_sensor;     /* [N,4,6] */
  const float* torques;          /* [N,n_dof] */
  const float* actions;          /* [N,n_act] delayed action, Isaac Gym order (WG:1173) */
  float* action_history;         /* [N,action_hist_len,n_act]; zeroed on reset */
  /* per-env constants */
  const float* mass_params;      /* [N,5] */
  const float* friction;         /* [N,1] */
  const float* motor_strength;   /* [N,n_act] */
  float* env_origins;            /* [N,3] (written by the terrain curriculum) */
  const float* box_env_origins_delta_y; /* [N] */
  /* task state */
  float* goal_state;             /* [N,DWBC_GS] */
  float* derived_state;          /* [N,DWBC_DS] */
  int64_t* episode_length;       /* [N] (BT:75 dtype) */
  float* obs_history;            /* [N,history_len,num_prop] */
  float* episode_sums;           /* [N,sums_stride] */
  /* terrain (may be null when measure_heights == 0) */
  const int16_t* height_samples; /* [terrain_rows,terrain_cols] */
  float* measured_heights;       /* [N,n_height_x*n_height_y] */
  float* heights_obs;            /* optional [N,n_points]: LR:221-223 */
  int64_t* terrain_levels;       /* [N] */
  const int64_t* terrain_types;  /* [N] */
  const float* terrain_origins;  /* [max_terrain_level,terrain_n_types,3] */
  /* outputs */
  float* obs_buf;                /* [N,obs_stride] */
  int64_t obs_stride;            /* row stride in floats (num_obs, or more when writing into storage) */
  float* rew_buf;                /* [N] */
  float* arm_rew_buf;            /* [N] */
  uint8_t* reset_buf;            /* [N] torch.bool */
  uint8_t* time_out_buf;         /* [N] torch.bool */
  float* episode_stats;          /* [1+sums_stride]: #resets, then per-slot sum over reset envs (atomics;
                                    caller zeroes before the step; WG:743-750 means = sum/count/T_ep) */
  /* optional direct-to-storage transition (SURVEY 8f row f2): with store_rewards != NULL the kernel also performs
   * PPO.process_env_step's reward path (PPO:130-134) and the dones store (RS:102) of this step:
   *   store_rewards[n,:] = (rew, arm_rew) + store_gamma * store_values[n,:] * time_out[n];  store_dones[n] = reset[n]  */
  const float* store_values;     /* [N,2] values PPO.act produced for this step */
  float* store_rewards;          /* [N,2] row of RolloutStorage.rewards */
  uint8_t* store_dones;          /* [N]   row of RolloutStorage.dones (uint8, may be NULL) */
  float store_gamma;
  int32_t reserved_;
} DwbcEnvBuffers;

/* Per-step arguments: curriculum outputs (WG:678-692) and RNG source. */
typedef struct DwbcStepArgs {
  const float* rand_uniform;     /* [N,DWBC_RAND_COLS] or NULL -> Philox4x32-10(seed, step) in-kernel */
  uint64_t seed;
  uint64_t step;
  int32_t do_push;               /* common_step_counter % push_interval == 0 (WG:934) */
  float lin_vel_x[2], ang_vel_yaw[2], goal_l[2], goal_p[2], goal_y[2]; /* (lo, span=hi-lo) */
  float leg_scale[DWBC_MAX_TERMS], arm_scale[DWBC_MAX_TERMS];         /* aligned with cfg.leg_term / arm_term */
  float leg_termination_scale, arm_termination_scale;                  /* 0 when inactive */
  int32_t generic_kernel;        /* 1 = always run the warp-per-env kernel (any N / unaligned buffers), 0 = pick by shape */
  int32_t reserved_;
} DwbcStepArgs;

/* Replaces WidowGo1.post_physics_step after its four gym.refresh_* calls (WG:875-910),
 * including update_curr_ee_goal (WG:1344-1350), _post_physics_step_callback (WG:917-935),
 * check_termination (WG:937-963), compute_reward (WG:170-205), reset_idx (WG:695-754),
 * compute_observations (WG:966-1001), the obs clip of step (WG:1195-1196), and, when
 * cfg.measure_heights, LeggedRobot._get_heights (LR:793-829).  One kernel launch. */
int dwbc_post_physics_step(const DwbcEnvCfg* cfg, const DwbcEnvBuffers* buf, const DwbcStepArgs* args,
                           dwbc_stream_t stream);

/* Materialises the uniform table the in-kernel Philox stream would produce:
 * out[N,DWBC_RAND_COLS] (so table mode and Philox mode can be checked against each other). */
int dwbc_fill_uniform(float* out, int32_t num_envs, uint64_t seed, uint64_t step, dwbc_stream_t stream);

/* Pre-physics half of WidowGo1.step (WG:1162-1173): permute raisim->IG, clip, push into the
 * action-delay FIFO and emit the delayed action. policy_actions[N,n_act] (raisim order). */
int dwbc_pre_physics_actions(const float* policy_actions, const int32_t* raisim2ig, float clip_actions,
                             float* action_history, float* actions, int32_t num_envs, int32_t num_actions,
                             int32_t action_hist_len, int32_t delay_row, dwbc_stream_t stream);

/* ---------------------------------------------------------------------------------------- */
/* rsl_rl storage path                                                                       */
/* ---------------------------------------------------------------------------------------- */

/* PPO.process_env_step reward path (PPO:130-134): rewards[n,:] = (rew, arm_rew) + gamma *
 * values[n,:] * time_outs[n]; dones[n] = reset[n] (RS:102 uint8). */
int dwbc_store_rewards(const float* rew, const float* arm_rew, const float* values, const uint8_t* time_outs,
                       const uint8_t* resets, float gamma, float* rewards_out, uint8_t* dones_out, int32_t num_envs,
                       dwbc_stream_t stream);

/* RolloutStorage.compute_returns (RS:136-150): two-channel GAE backward scan over
 * rewards/values [T,N,2], dones [T,N] uint8, last_values [N,2] -> returns, advantages [T,N,2];
 * advantages are normalised jointly over all T*N*2 elements with the UNBIASED std + 1e-8.
 * stats[3] (double: n, sum, sum of squares) is device scratch the caller zeroes.  With
 * normalize == 0 the raw advantages are written and stats filled (multi-GPU: all-reduce stats,
 * then call dwbc_normalize_advantages). */
int dwbc_gae(const float* rewards, const float* values, const uint8_t* dones, const float* last_values, float* returns,
             float* advantages, double* stats, int32_t T, int32_t N, float gamma, float lam, int32_t normalize,
             dwbc_stream_t stream);
int dwbc_normalize_advantages(float* advantages, const double* stats, int64_t count, dwbc_stream_t stream);

/* ---------------------------------------------------------------------------------------- */
/* ActorCritic + PPO update                                                                  */
/* ---------------------------------------------------------------------------------------- */

#define DWBC_MAX_LAYERS 4

/* Hidden-layer activation of the ActorCritic (rsl_rl get_activation, AC): every layer of the privileged encoder, the four stages of
 * the history encoder, the actor / critic backbones and the hidden layers of the four heads.  The actor heads' last layer stays tanh,
 * the critic heads' last layer stays linear.  rsl_rl's "crelu" is a plain ReLU (DWBC_ACT_RELU). */
enum DwbcActivation {
  DWBC_ACT_ELU = 0,      /* nn.ELU() (zero: the value of a zero-filled struct) */
  DWBC_ACT_SELU = 1,     /* nn.SELU() */
  DWBC_ACT_RELU = 2,     /* nn.ReLU() */
  DWBC_ACT_LRELU = 3,    /* nn.LeakyReLU(), slope 0.01 */
  DWBC_ACT_TANH = 4,     /* nn.Tanh() */
  DWBC_ACT_SIGMOID = 5   /* nn.Sigmoid() */
};

/* Network shape (AC:86-298).  Parameters live in ONE flat fp32 buffer in
 * ActorCritic.parameters() order (std first); offsets are element offsets into it. */
typedef struct DwbcNetCfg {
  int32_t abi_version;
  int32_t num_prop, num_priv, num_hist, num_obs, n_leg, n_arm;
  int32_t n_priv_layers, priv_dims[DWBC_MAX_LAYERS];
  int32_t n_actor_layers, actor_dims[DWBC_MAX_LAYERS];
  int32_t n_critic_layers, critic_dims[DWBC_MAX_LAYERS];
  int32_t n_leg_layers, leg_dims[DWBC_MAX_LAYERS];   /* hidden dims of the leg heads (actor and critic) */
  int32_t n_arm_layers, arm_dims[DWBC_MAX_LAYERS];
  int32_t hist_proj, hist_c1, hist_k1, hist_s1, hist_c2, hist_k2, hist_s2; /* AC:49-62 (tsteps==10: 30,20,4,2,10,2,1) */
  int64_t num_params;
  int64_t off_std;
  int64_t off_priv_w[DWBC_MAX_LAYERS], off_priv_b[DWBC_MAX_LAYERS];
  int64_t off_hist_w[4], off_hist_b[4];              /* encoder.0, conv_layers.0, conv_layers.2, linear_output.0 */
  int64_t off_actor_w[DWBC_MAX_LAYERS], off_actor_b[DWBC_MAX_LAYERS];
  int64_t off_aleg_w[DWBC_MAX_LAYERS + 1], off_aleg_b[DWBC_MAX_LAYERS + 1];
  int64_t off_aarm_w[DWBC_MAX_LAYERS + 1], off_aarm_b[DWBC_MAX_LAYERS + 1];
  int64_t off_critic_w[DWBC_MAX_LAYERS], off_critic_b[DWBC_MAX_LAYERS];
  int64_t off_cleg_w[DWBC_MAX_LAYERS + 1], off_cleg_b[DWBC_MAX_LAYERS + 1];
  int64_t off_carm_w[DWBC_MAX_LAYERS + 1], off_carm_b[DWBC_MAX_LAYERS + 1];
  /* Arithmetic of the ActorCritic GEMMs, per call (no process-wide switch):
   *   0  fp32 CUDA cores (parity anchor of the tests);
   *   1  TF32 operands (10-bit mantissa, truncated), fp32 accumulation, tcgen05 tensor cores;
   *   2  "3xTF32": every operand is split into the TF32 part the tensor core reads and the exact remainder, three tensor-core
   *      products per GEMM (hi*hi + lo*hi + hi*lo), fp32 accumulation: fp32-grade results on the tensor cores. */
  int32_t precision;
  int32_t activation;            /* DwbcActivation of the hidden layers; any other value: DWBC_ERR_ARG */
} DwbcNetCfg;

/* PD torque controller of step() (WG:1262-1295 `_compute_torques`, called `decimation` times per policy step, WG:1175-1183):
 *   tau[:, j] = clip(p_j * (a_j * motor_strength_j * action_scale_j + default_j - q_j) - d_j * qdot_j, +-limit_j)   j < n_act
 *   tau[:, j] = 0                                                                                                n_act <= j < n_dof
 * `actions` are the delayed actions in Isaac Gym order (output of dwbc_pre_physics_actions).  The reference wraps column -8 of
 * the n_act-wide position tensor to (-pi, pi] (WG:1279) -- i.e. DOF n_act-8, which is not the waist; `wrap_dof` restates it as
 * written (-1: no wrap). */
typedef struct DwbcPdCfg {
  int32_t n_dof, n_act, wrap_dof;
  float p_gains[DWBC_MAX_DOF], d_gains[DWBC_MAX_DOF], action_scale[DWBC_MAX_DOF], default_dof_pos[DWBC_MAX_DOF], torque_limits[DWBC_MAX_DOF];
} DwbcPdCfg;
int dwbc_compute_torques(const DwbcPdCfg* cfg, const float* actions, const float* dof_state, const float* motor_strength,
                         float* torques, int32_t num_envs, dwbc_stream_t stream);

/* Bytes of device workspace the forward / update entry points need for `rows` rows.  The workspace must be ZERO-FILLED when it is
 * first handed to the library (its first 256 bytes hold the work-queue counters of the fused chain kernel, which every launch leaves
 * at zero again); one workspace sized for the largest `rows` may be shared by calls with smaller `rows`. */
int64_t dwbc_workspace_bytes(const DwbcNetCfg* net, int64_t rows);

/* PPO.act (PPO:115-127 = AC:337-353): obs[N,obs_stride] -> mean, sigma, actions = mean +
 * sigma*eps (eps[N,n_act] standard normal supplied by the caller), two-channel log-prob of the
 * action, critic values.  hist_encoding selects the history encoder latent (AC:207-210).
 * weights_packed: 0 = (re)build the tensor-core weight images in the workspace from `params`; 1 = reuse the images a previous
 * call left in this workspace (same net, same rows, parameters unchanged since, no other entry point run on the workspace in
 * between) -- lets a rollout pack once per iteration instead of once per step.  Ignored by the fp32 path. */
int dwbc_policy_act(const DwbcNetCfg* net, const float* params, const float* obs, int64_t obs_stride, const float* eps,
                    int32_t hist_encoding, float* actions, float* values, float* log_prob, float* mean, float* sigma,
                    int32_t rows, int32_t weights_packed, void* workspace, dwbc_stream_t stream);

/* critic only (PPO:148-150 last_values; AC:351-353) */
int dwbc_critic_values(const DwbcNetCfg* net, const float* params, const float* obs, int64_t obs_stride, float* values,
                       int32_t rows, void* workspace, dwbc_stream_t stream);

/* history-encoder latent (AC:223-225) of obs[rows, obs_stride] -> out[rows, ld_out]; ld_out = latent rounded up to 4 */
int dwbc_hist_latent(const DwbcNetCfg* net, const float* params, const float* obs, int64_t obs_stride, float* out,
                     int64_t ld_out, int32_t rows, void* workspace, dwbc_stream_t stream);

typedef struct DwbcPpoHyper {
  float clip_param, value_loss_coef, entropy_coef, priv_reg_coef, mixing_ratio; /* PPO:178-179, 301-302 */
  int32_t use_clipped_value_loss;
  float max_grad_norm, lr, beta1, beta2, adam_eps;
  float grad_scale;              /* 1/world_size applied to the (all-reduced) gradient before the clip */
  /* arm torque supervision (PPO:224-239, fixed gains PPO:318-323): weight of mean((tau_arm - target)^2) in the loss
   * (PPO:304-305 schedule, evaluated by the host); 0 or arm_coefs == NULL: branch off.  arm_coefs: device [3][n_arm] =
   * default arm p gains, d gains, default arm dof positions (PPO:307-310 set_arm_default_coeffs). */
  float torque_supervision_weight;
  const float* arm_coefs;
} DwbcPpoHyper;

/* Rollout storage views (RS:65-84), flattened [T*N, .] */
typedef struct DwbcStorage {
  const float* observations; int64_t obs_stride;
  const float* actions; const float* values; const float* returns; const float* advantages; const float* log_prob;
  /* optional: history-encoder latent of EVERY storage row [T*N, hist_latent_ld], precomputed with dwbc_hist_latent.
   * PPO.update never changes the history encoder (its output is detached, PPO:175-176, so those parameters receive no
   * gradient), hence the regulariser target of a row is the same in all epochs.  NULL: computed per mini-batch. */
  const float* hist_latent; int64_t hist_latent_ld;
  /* optional (torque supervision, RS:82-84,108-111): [T*N, n_arm] each; NULL: branch off */
  const float* target_arm_torques; const float* current_arm_dof_pos; const float* current_arm_dof_vel;
} DwbcStorage;

/* One PPO mini-batch, forward + loss + backward (PPO:166-221,244): gathers rows idx[M] from the
 * storage, writes the UNCLIPPED gradient of the mean loss into grad[num_params] (overwritten) and
 * losses_out[5] += (surrogate, value, priv_reg, entropy, arm-torque) means (device accumulators; the last one only
 * with torque supervision on). */
int dwbc_ppo_minibatch_grad(const DwbcNetCfg* net, const float* params, const DwbcStorage* st, const int64_t* idx,
                            int32_t M, const DwbcPpoHyper* hp, float* grad, float* losses_out, void* workspace,
                            dwbc_stream_t stream);

/* PPO.update_dagger mini-batch (PPO:273-283): grad of mean ||sg(z_priv) - z_hist||_2 w.r.t. the
 * history-encoder parameters only (other entries of grad are zeroed). losses_out[0] += loss. */
int dwbc_dagger_minibatch_grad(const DwbcNetCfg* net, const float* params, const DwbcStorage* st, const int64_t* idx,
                               int32_t M, float* grad, float* losses_out, void* workspace, dwbc_stream_t stream);

/* clip_grad_norm_(max_norm) + Adam step (PPO:245-246) over params[first, first+count) of the flat
 * buffers; `step` is the 1-based Adam step of this parameter group.  norm_scratch[2] is device
 * scratch.  grad_norm_out (optional, device) receives the pre-clip total norm. */
int dwbc_clip_adam_step(float* params, float* grad, float* adam_m, float* adam_v, int64_t first, int64_t count,
                        const DwbcPpoHyper* hp, int32_t step, double* norm_scratch, float* grad_norm_out,
                        dwbc_stream_t stream);

/* PPO.enforce_min_std (PPO:293-296): std = max(std, min_std). */
int dwbc_enforce_min_std(float* params, int64_t off_std, const float* min_std, int32_t n, dwbc_stream_t stream);

const char* dwbc_version(void);
/* number of kernels this library has launched in this process (host-side counter) */
uint64_t dwbc_launch_count(void);
/* sizeof(DwbcEnvCfg, DwbcEnvBuffers, DwbcStepArgs, DwbcNetCfg, DwbcPpoHyper, DwbcStorage): lets a
 * foreign-language binding verify its struct mirrors at load time. */
void dwbc_struct_sizes(int64_t out[6]);

#ifdef __cplusplus
}
#endif
#endif /* DWBC_H */
