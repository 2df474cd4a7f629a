// ActorCritic forward / PPO loss / hand-written backward, fp32 CUDA-core path (K5-K8 anchor).
//
// Layer-wise: every nn.Linear (+activation) of `rsl_rl/modules/actor_critic.py` is one launch of
// the tile GEMM in gemm_simt.cuh with the bias/activation (forward) or activation derivative
// (backward) fused into its epilogue; the mini-batch gather (RS:189-201) is fused into the
// first-layer operand loads (no gathered batch is materialised); the Conv1d history encoder
// (AC:39-84) is expressed as three more GEMMs over re-packed weights.  The PPO loss
// (PPO:199-221) and its derivative w.r.t. the network outputs is one elementwise kernel.
#include <math.h>

#include <stdlib.h>

#include "hist_fused.cuh"
#include "mlp_chain2.cuh"
#include "wgrad_group.cuh"

namespace dwbc {

// precision of the ActorCritic GEMMs of the CURRENT call (DwbcNetCfg.precision, set by every entry point):
// 0 = fp32 CUDA cores (parity anchor), 1 = TF32 tcgen05, 2 = 3xTF32 tcgen05 (error-compensated, fp32-grade)
thread_local int mlp_precision = 0;
int tc_debug = 0;

static inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

struct Bump {
  char* base;
  int64_t off;
  float* f(int64_t n) {
    float* p = base ? reinterpret_cast<float*>(base + off) : nullptr;
    off += align_up(n * (int64_t)sizeof(float), 256);
    return p;
  }
};

static inline int last(const int32_t* d, int n) { return d[n - 1]; }

// ---- workspace plan ----------------------------------------------------------------------------
struct Plan {
  // forward activations (saved for backward)
  float* priv[DWBC_MAX_LAYERS];   // priv encoder outputs; the last one is the latent z
  float* ab[DWBC_MAX_LAYERS];     // actor backbone
  float* al[DWBC_MAX_LAYERS];     // actor leg head hidden
  float* aa[DWBC_MAX_LAYERS];     // actor arm head hidden
  float* mean;                    // [rows, mean_ld] tanh outputs (leg | arm)
  float* cb[DWBC_MAX_LAYERS];
  float* cl[DWBC_MAX_LAYERS];
  float* ca[DWBC_MAX_LAYERS];
  float* value;                   // [rows, 2]
  // history encoder
  float* hproj;                   // [rows*T, 32]
  float* hc1;                     // [rows*4, 20]
  float* hc2;                     // [rows*3, 12]
  float* zh;                      // [rows, latent]
  float* hw1; float* hw2; float* hwl;      // re-packed weights
  float* wpack;                            // packed weight images of the fused chain kernels (mlp_chain2.cuh)
  int* queue;                              // work-item counters of the chain kernel (zero between launches)
  // gradients
  float* g_leg; float* g_arm; float* g_vl; float* g_va; float* g_z;   // g_vl / g_va: columns 0 / 1 of one [rows, 4] buffer
  // per-layer pre-activation gradients kept by the fused backward chain for the weight-gradient GEMMs
  float* dza_l[DWBC_MAX_LAYERS]; float* dza_a[DWBC_MAX_LAYERS]; float* dza_b[DWBC_MAX_LAYERS]; float* dzp[DWBC_MAX_LAYERS];
  float* dzc_l[DWBC_MAX_LAYERS]; float* dzc_a[DWBC_MAX_LAYERS]; float* dzc_b[DWBC_MAX_LAYERS];
  float* d0; float* d1; float* d2;         // ping-pong [rows, maxw]
  float* dz;                               // [rows, latent]
  float* dzh;                              // [rows, latent] (dagger)
  float* dh_a1; float* dh_a2;              // im2col-space grads of the conv inputs (dagger)
  float* dh_c1; float* dh_proj;
  float* dhw1; float* dhw2; float* dhwl;   // grads of the re-packed weights (dagger)
  int mean_ld, maxw, latent;
  int64_t bytes;
};

static int maxdim(const DwbcNetCfg& n) {
  int m = 32;
  auto up = [&](const int32_t* d, int k) { for (int i = 0; i < k; ++i) m = d[i] > m ? d[i] : m; };
  up(n.priv_dims, n.n_priv_layers); up(n.actor_dims, n.n_actor_layers); up(n.critic_dims, n.n_critic_layers);
  up(n.leg_dims, n.n_leg_layers); up(n.arm_dims, n.n_arm_layers);
  return (int)align_up(m, 4);
}

// activations / pre-activation gradients of 128-wide layers are kept as tile images by the tensor-core path (RowMat::image):
// whole 128-row tiles, so the buffer covers the rows rounded up to a tile
static inline bool img_dim(int d) { return d == 128; }
static inline int64_t act_floats(int64_t rows, int d) { return img_dim(d) ? align_up(rows, 128) * 128 : rows * align_up(d, 4); }
static inline RowMat act_mat(const float* p, int d) { return img_dim(d) ? rowmat_image(p) : rowmat(p, d); }

static Plan make_plan(const DwbcNetCfg& n, int64_t rows, void* ws) {
  Plan p{};
  Bump b{reinterpret_cast<char*>(ws), 0};
  p.queue = reinterpret_cast<int*>(b.f(64));      // FIRST: the same address whatever `rows` is (callers share one workspace between row counts;
                                                  // the counters must stay zero between launches, nothing else may ever be laid over them)
  p.latent = last(n.priv_dims, n.n_priv_layers);
  p.maxw = maxdim(n);
  p.mean_ld = (int)align_up(n.n_leg + n.n_arm, 4);
  for (int i = 0; i < n.n_priv_layers; ++i) p.priv[i] = b.f(rows * align_up(n.priv_dims[i], 4));
  for (int i = 0; i < n.n_actor_layers; ++i) p.ab[i] = b.f(act_floats(rows, n.actor_dims[i]));
  for (int i = 0; i < n.n_leg_layers; ++i) p.al[i] = b.f(act_floats(rows, n.leg_dims[i]));
  for (int i = 0; i < n.n_arm_layers; ++i) p.aa[i] = b.f(act_floats(rows, n.arm_dims[i]));
  p.mean = b.f(rows * p.mean_ld);
  for (int i = 0; i < n.n_critic_layers; ++i) p.cb[i] = b.f(act_floats(rows, n.critic_dims[i]));
  for (int i = 0; i < n.n_leg_layers; ++i) p.cl[i] = b.f(act_floats(rows, n.leg_dims[i]));
  for (int i = 0; i < n.n_arm_layers; ++i) p.ca[i] = b.f(act_floats(rows, n.arm_dims[i]));
  p.value = b.f(rows * 2);
  p.hproj = b.f(rows * n.num_hist * 32);
  p.hc1 = b.f(rows * 4 * 20);
  p.hc2 = b.f(rows * 3 * 12);
  p.zh = b.f(rows * align_up(p.latent, 4));
  p.hw1 = b.f(20 * 128); p.hw2 = b.f(10 * 40); p.hwl = b.f(32 * 36);
  p.wpack = b.f(C2_PACK_FLOATS);
  p.g_leg = b.f(rows * align_up(n.n_leg, 4)); p.g_arm = b.f(rows * align_up(n.n_arm, 4));
  p.g_vl = b.f(rows * 4); p.g_va = p.g_vl ? p.g_vl + 1 : nullptr; p.g_z = b.f(rows * align_up(p.latent, 4));
  for (int i = 0; i < n.n_leg_layers; ++i) { p.dza_l[i] = b.f(act_floats(rows, n.leg_dims[i])); p.dzc_l[i] = b.f(act_floats(rows, n.leg_dims[i])); }
  for (int i = 0; i < n.n_arm_layers; ++i) { p.dza_a[i] = b.f(act_floats(rows, n.arm_dims[i])); p.dzc_a[i] = b.f(act_floats(rows, n.arm_dims[i])); }
  for (int i = 0; i < n.n_actor_layers; ++i) p.dza_b[i] = b.f(act_floats(rows, n.actor_dims[i]));
  for (int i = 0; i < n.n_critic_layers; ++i) p.dzc_b[i] = b.f(act_floats(rows, n.critic_dims[i]));
  for (int i = 0; i < n.n_priv_layers; ++i) p.dzp[i] = b.f(rows * align_up(n.priv_dims[i], 4));
  p.d0 = b.f(rows * p.maxw); p.d1 = b.f(rows * p.maxw); p.d2 = b.f(rows * p.maxw);
  p.dz = b.f(rows * align_up(p.latent, 4));
  p.dzh = b.f(rows * align_up(p.latent, 4));
  p.dh_a1 = b.f(rows * 4 * 128); p.dh_a2 = b.f(rows * 3 * 40);
  p.dh_c1 = b.f(rows * 4 * 20); p.dh_proj = b.f(rows * n.num_hist * 32);
  p.dhw1 = b.f(20 * 128); p.dhw2 = b.f(10 * 40); p.dhwl = b.f(32 * 36);
  p.bytes = b.off;
  return p;
}

static int check_net(const DwbcNetCfg* n) {
  if (!n || n->abi_version != DWBC_ABI_VERSION || n->precision < 0 || n->precision > 2 || act_code(n->activation) < 0) return DWBC_ERR_ARG;
  mlp_precision = n->precision;
  if (n->n_priv_layers < 1 || n->n_priv_layers > DWBC_MAX_LAYERS || n->n_actor_layers < 1 || n->n_actor_layers > DWBC_MAX_LAYERS ||
      n->n_critic_layers < 1 || n->n_critic_layers > DWBC_MAX_LAYERS || n->n_leg_layers < 1 || n->n_leg_layers > DWBC_MAX_LAYERS ||
      n->n_arm_layers < 1 || n->n_arm_layers > DWBC_MAX_LAYERS)
    return DWBC_ERR_UNSUPPORTED;
  // history encoder: only the tsteps == 10 variant (AC:57-62) exists for widowGo1 (WGC:124)
  if (n->num_hist != 10 || n->hist_proj != 30 || n->hist_c1 != 20 || n->hist_k1 != 4 || n->hist_s1 != 2 || n->hist_c2 != 10 ||
      n->hist_k2 != 2 || n->hist_s2 != 1)
    return DWBC_ERR_UNSUPPORTED;
  if (last(n->priv_dims, n->n_priv_layers) > 32 || n->n_leg + n->n_arm > 32) return DWBC_ERR_UNSUPPORTED;
  return DWBC_OK;
}

// activation code of every hidden layer (check_net has validated it)
static inline int hid(const DwbcNetCfg& n) { return act_code(n.activation); }

// ---- history-encoder weight re-packing ---------------------------------------------------------
// conv1 [20,30,4] -> W1'[20][k*32+cin]; conv2 [10,20,2] -> W2'[10][k*20+cin]; linear [L,30] over the
// channel-major flatten (c2*3+t) -> Wl'[L][t*12+c2].  Pad entries are zero.
__global__ void hist_pack_kernel(const float* __restrict__ w1, const float* __restrict__ w2, const float* __restrict__ wl,
                                 float* __restrict__ o1, float* __restrict__ o2, float* __restrict__ ol, int latent) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 20 * 128) {
    int c1 = i / 128, r = i % 128, k = r / 32, cin = r % 32;
    o1[i] = cin < 30 ? w1[(c1 * 30 + cin) * 4 + k] : 0.0f;
  }
  if (i < 10 * 40) {
    int c2 = i / 40, r = i % 40, k = r / 20, cin = r % 20;
    o2[i] = w2[(c2 * 20 + cin) * 2 + k];
  }
  if (i < latent * 36) {
    int j = i / 36, r = i % 36, t = r / 12, c2 = r % 12;
    ol[i] = c2 < 10 ? wl[j * 30 + c2 * 3 + t] : 0.0f;
  }
}
// inverse scatter of the re-packed weight gradients into the flat gradient (reference layouts)
__global__ void hist_unpack_grad_kernel(const float* __restrict__ g1, const float* __restrict__ g2, const float* __restrict__ gl,
                                        float* __restrict__ w1, float* __restrict__ w2, float* __restrict__ wl, int latent) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 20 * 128) {
    int c1 = i / 128, r = i % 128, k = r / 32, cin = r % 32;
    if (cin < 30) w1[(c1 * 30 + cin) * 4 + k] = g1[i];
  }
  if (i < 10 * 40) {
    int c2 = i / 40, r = i % 40, k = r / 20, cin = r % 20;
    w2[(c2 * 20 + cin) * 2 + k] = g2[i];
  }
  if (i < latent * 36) {
    int j = i / 36, r = i % 36, t = r / 12, c2 = r % 12;
    if (c2 < 10) wl[j * 30 + c2 * 3 + t] = gl[i];
  }
}
// col2im of the conv input gradients (overlapping windows) fused with the activation derivative:
// dst[m][t][c] = act'(y[m][t][c]) * sum_{t'*stride + k == t} src[(m*To + t')][k*C + c]
__global__ void col2im_dact_kernel(const float* __restrict__ src, const float* __restrict__ y, float* __restrict__ dst, int64_t rows,
                                   int Tin, int C, int ldc, int To, int ksz, int stride, int act) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = rows * Tin * ldc;
  if (i >= total) return;
  int c = (int)(i % ldc);
  int t = (int)((i / ldc) % Tin);
  int64_t m = i / ((int64_t)ldc * Tin);
  float s = 0.0f;
  if (c < C) {
    for (int k = 0; k < ksz; ++k) {
      int tt = t - k;
      if (tt < 0 || tt % stride) continue;
      int to = tt / stride;
      if (to >= To) continue;
      s += src[(m * To + to) * (int64_t)(ksz * ldc) + k * ldc + c];
    }
    float yy = y[i];
    s *= act_dy(act, yy);
  }
  dst[i] = s;
}

__global__ void zero_cols_kernel(float* __restrict__ p, int64_t nrows, int ld, int c0) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int w = ld - c0;
  if (i < nrows * w) p[(i / w) * ld + c0 + (i % w)] = 0.0f;
}

// ---- forward ------------------------------------------------------------------------------------
#define TRY(x) do { int rc__ = (x); if (rc__ != DWBC_OK) return rc__; } while (0)

static int hist_forward(const DwbcNetCfg& n, const float* P, const float* obs, const int64_t* idx, int64_t obs_stride, int rows,
                        const Plan& p, cudaStream_t st) {
  const int T = n.num_hist, L = p.latent, Lld = (int)align_up(L, 4);
  hist_pack_kernel<<<(20 * 128 + 255) / 256, 256, 0, st>>>(P + n.off_hist_w[1], P + n.off_hist_w[2], P + n.off_hist_w[3], p.hw1, p.hw2,
                                                           p.hwl, L);
  dwbc_launch_counter += 3;
  // pad columns of the padded activation buffers are consumed by the next GEMM's K range
  zero_cols_kernel<<<(unsigned)(((int64_t)rows * T * 2 + 255) / 256), 256, 0, st>>>(p.hproj, (int64_t)rows * T, 32, 30);
  zero_cols_kernel<<<(unsigned)(((int64_t)rows * 3 * 2 + 255) / 256), 256, 0, st>>>(p.hc2, (int64_t)rows * 3, 12, 10);
  RowMat hist = rowmat_grouped(obs + (n.num_obs - T * n.num_prop), idx, T, obs_stride, n.num_prop);
  TRY(linear_fwd(hist, P + n.off_hist_w[0], n.num_prop, P + n.off_hist_b[0], p.hproj, 32, rows * T, 30, n.num_prop, hid(n), 0, st));  // AC:80
  RowMat a1 = rowmat_grouped(p.hproj, nullptr, 4, (int64_t)T * 32, 2 * 32);
  TRY(linear_fwd(a1, p.hw1, 128, P + n.off_hist_b[1], p.hc1, 20, rows * 4, 20, 128, hid(n), 0, st));                                  // AC:59
  RowMat a2 = rowmat_grouped(p.hc1, nullptr, 3, 80, 20);
  TRY(linear_fwd(a2, p.hw2, 40, P + n.off_hist_b[2], p.hc2, 12, rows * 3, 10, 40, hid(n), 0, st));                                     // AC:60
  TRY(linear_fwd(rowmat(p.hc2, 36), p.hwl, 36, P + n.off_hist_b[3], p.zh, Lld, rows, L, 36, hid(n), 0, st));                           // AC:72
  return DWBC_OK;
}

// history latent only (no intermediates kept): the fused exact-fp32 kernel on the tensor-core precisions (hist_fused.cuh), the layer-wise
// GEMMs on the fp32 anchor path
static int hist_latent_only(const DwbcNetCfg& n, const float* P, const float* obs, const int64_t* idx, int64_t obs_stride, int rows, const Plan& p,
                            float* out, int64_t ld_out, cudaStream_t st) {
  if (mlp_precision == 0 || (obs_stride & 3) || (reinterpret_cast<uintptr_t>(obs) & 15) || (n.num_prop & 3) || ((n.num_obs - n.num_hist * n.num_prop) & 3)) {
    Plan q = p;
    q.zh = out;
    if (ld_out != align_up(p.latent, 4)) return DWBC_ERR_ARG;
    return hist_forward(n, P, obs, idx, obs_stride, rows, q, st);
  }
  HistFusedArgs a{};
  a.wp = P + n.off_hist_w[0]; a.bp = P + n.off_hist_b[0]; a.w1 = P + n.off_hist_w[1]; a.b1 = P + n.off_hist_b[1];
  a.w2 = P + n.off_hist_w[2]; a.b2 = P + n.off_hist_b[2]; a.wl = P + n.off_hist_w[3]; a.bl = P + n.off_hist_b[3];
  a.hist = rowmat_gather(obs + (n.num_obs - n.num_hist * n.num_prop), idx, obs_stride);
  a.out = out; a.ld_out = ld_out; a.rows = rows; a.latent = p.latent;
  return launch_hist_fused(a, hid(n), st);
}

static int priv_forward(const DwbcNetCfg& n, const float* P, const float* obs, const int64_t* idx, int64_t obs_stride, int rows,
                        const Plan& p, cudaStream_t st) {
  RowMat h = rowmat_gather(obs + n.num_prop, idx, obs_stride);
  int in = n.num_priv;
  for (int l = 0; l < n.n_priv_layers; ++l) {
    int out = n.priv_dims[l], ld = (int)align_up(out, 4);
    TRY(linear_fwd(h, P + n.off_priv_w[l], in, P + n.off_priv_b[l], p.priv[l], ld, rows, out, in, hid(n), 0, st));  // AC:219-221
    h = rowmat(p.priv[l], ld);
    in = out;
  }
  return DWBC_OK;
}

static int head_forward(const float* P, RowMat h, int in, int nl, const int32_t* dims, int n_out, const int64_t* ow, const int64_t* ob,
                        float* const* acts, float* out, int64_t ldo, int hact, int last_act, int rows, cudaStream_t st) {
  for (int l = 0; l < nl; ++l) {
    TRY(linear_fwd(h, P + ow[l], in, P + ob[l], acts[l], dims[l], rows, dims[l], in, hact, 0, st));
    h = rowmat(acts[l], dims[l]);
    in = dims[l];
  }
  return linear_fwd(h, P + ow[nl], in, P + ob[nl], out, ldo, rows, n_out, in, last_act, 0, st);
}

// Actor.forward (AC:204-217); latent z must already be in `z` (row stride zld)
static int actor_forward(const DwbcNetCfg& n, const float* P, const float* obs, const int64_t* idx, int64_t obs_stride, int rows,
                         const float* z, int zld, const Plan& p, cudaStream_t st) {
  RowMat x = rowmat_gather(obs, idx, obs_stride);
  const int in0 = n.num_prop + p.latent;
  // backbone layer 0 over cat([obs_prop, z]) as two accumulating GEMMs (no concat buffer)
  int single = n.n_actor_layers;
  TRY(linear_fwd(x, P + n.off_actor_w[0], in0, P + n.off_actor_b[0], p.ab[0], n.actor_dims[0], rows, n.actor_dims[0], n.num_prop, ACT_NONE, 0, st));
  TRY(linear_fwd(rowmat(z, zld), P + n.off_actor_w[0] + n.num_prop, in0, nullptr, p.ab[0], n.actor_dims[0], rows, n.actor_dims[0], p.latent,
                 hid(n), 1, st));
  RowMat h = rowmat(p.ab[0], n.actor_dims[0]);
  int in = n.actor_dims[0];
  for (int l = 1; l < single; ++l) {
    TRY(linear_fwd(h, P + n.off_actor_w[l], in, P + n.off_actor_b[l], p.ab[l], n.actor_dims[l], rows, n.actor_dims[l], in, hid(n), 0, st));
    h = rowmat(p.ab[l], n.actor_dims[l]);
    in = n.actor_dims[l];
  }
  TRY(head_forward(P, h, in, n.n_leg_layers, n.leg_dims, n.n_leg, n.off_aleg_w, n.off_aleg_b, p.al, p.mean, p.mean_ld, hid(n), ACT_TANH, rows, st));
  TRY(head_forward(P, h, in, n.n_arm_layers, n.arm_dims, n.n_arm, n.off_aarm_w, n.off_aarm_b, p.aa, p.mean + n.n_leg, p.mean_ld, hid(n), ACT_TANH, rows, st));
  return DWBC_OK;
}

// Critic.forward (AC:280-286)
static int critic_forward(const DwbcNetCfg& n, const float* P, const float* obs, const int64_t* idx, int64_t obs_stride, int rows,
                          const Plan& p, float* value, cudaStream_t st) {
  RowMat h = rowmat_gather(obs, idx, obs_stride);
  int in = n.num_prop + n.num_priv;
  for (int l = 0; l < n.n_critic_layers; ++l) {
    TRY(linear_fwd(h, P + n.off_critic_w[l], in, P + n.off_critic_b[l], p.cb[l], n.critic_dims[l], rows, n.critic_dims[l], in, hid(n), 0, st));
    h = rowmat(p.cb[l], n.critic_dims[l]);
    in = n.critic_dims[l];
  }
  TRY(head_forward(P, h, in, n.n_leg_layers, n.leg_dims, 1, n.off_cleg_w, n.off_cleg_b, p.cl, value, 2, hid(n), ACT_NONE, rows, st));
  TRY(head_forward(P, h, in, n.n_arm_layers, n.arm_dims, 1, n.off_carm_w, n.off_carm_b, p.ca, value + 1, 2, hid(n), ACT_NONE, rows, st));
  return DWBC_OK;
}

// ---- fused forward (tensor-core paths): privileged encoder + actor and the critic as two programs of ONE launch (mlp_chain2.cuh) ----
static inline int pad8(int x) { return (x + 7) & ~7; }
constexpr int C2_COL_PRIV = 32, C2_COL_HID = 64, C2_COL_PROP = 32;     // tile columns of the encoder input / hidden layer and of obs_prop (z sits at 0)

static bool chain_usable(const DwbcNetCfg& n, const Plan& p, const float* obs, int64_t obs_stride) {
  if (mlp_precision == 0) return false;
  auto ok = [](const int32_t* d, int k) { for (int i = 0; i < k; ++i) if (d[i] > 128 || (d[i] & 3)) return false; return true; };
  if (!ok(n.priv_dims, n.n_priv_layers) || !ok(n.actor_dims, n.n_actor_layers) || !ok(n.critic_dims, n.n_critic_layers) ||
      !ok(n.leg_dims, n.n_leg_layers) || !ok(n.arm_dims, n.n_arm_layers))
    return false;
  // tile layout of the actor program: z at columns [0, 32), obs_prop at [32, 32 + num_prop), the encoder works at [32, 64) -> [64, 128) first
  if (n.n_priv_layers != 2 || n.num_priv > 32 || n.priv_dims[0] > 64 || p.latent > 32) return false;
  if ((n.num_prop & 3) || (n.num_priv & 3) || (p.latent & 3) || C2_COL_PROP + n.num_prop > 128 || n.num_prop + n.num_priv > 128) return false;
  if ((obs_stride & 3) || !c2_aligned(obs)) return false;
  if (n.n_leg > C2_GRP || n.n_arm > C2_GRP) return false;      // the epilogue hooks keep one action group in registers
  if (2 + n.n_actor_layers + n.n_leg_layers + n.n_arm_layers + 2 > C2_MAX_OPS) return false;
  if (n.n_critic_layers + n.n_leg_layers + n.n_arm_layers + 2 > C2_MAX_OPS) return false;
  return true;
}

// one head: optional trunk reload (the second head of a program), hidden layers in place, narrow last layer with its epilogue hook
static void chain_head(C2Builder& b, const float* P, const float* trunk, int trunk_ld, bool reload, int in, int nl, const int32_t* dims, int n_out,
                       const int64_t* ow, const int64_t* ob, float* const* acts, bool store, float* out, int64_t ldo, int hact, int last_act, int fin,
                       int fin_c) {
  if (reload) b.load(act_mat(trunk, trunk_ld), in, 0, pad8(in), b.pr.n_ops);
  for (int l = 0; l < nl; ++l) {
    b.fwd(P + ow[l], in, P + ob[l], dims[l], hact, 0, pad8(in), 1, C2PackSeg{0, 0, in}, C2PackSeg{0, 0, 0}, 0, store ? acts[l] : nullptr, dims[l],
          FIN_NONE, 0, store && img_dim(dims[l]));
    in = dims[l];
  }
  b.fwd(P + ow[nl], in, P + ob[nl], n_out, last_act, 0, pad8(in), 1, C2PackSeg{0, 0, in}, C2PackSeg{0, 0, 0}, -1, out, ldo, fin, fin_c);
}

// Programs of the forward pass.  z_hist == nullptr: latent from the privileged encoder (computed inside the chain); else the history
// latent [rows, zld].  `loss`: update mode (hooks FIN_REG / FIN_PPO / FIN_VALUE), else rollout mode (FIN_ACT), else none (fin_mode 0).
// With A2 / C2 (inference only: `store` off) the two heads of a network become TWO programs that each recompute the short common part
// (encoder + backbone): a 4096-row rollout then is 4 programs x 32 tiles = 128 one-tile items of at most 6 ops on 128 SMs instead of
// 2 x 32 items of 9 / 7 ops on 64 SMs -- the launch is as long as its longest item.
static int build_forward(const DwbcNetCfg& n, const float* P, const float* obs, const int64_t* idx, int64_t obs_stride, const float* z_hist, int zld,
                         const Plan& p, float* value, bool store, int fin_mode, C2Builder* A, C2Builder* C, C2Builder* A2 = nullptr,
                         C2Builder* C2 = nullptr) {
  const int Lld = (int)align_up(p.latent, 4);
  if ((A2 || C2) && store) return DWBC_ERR_ARG;
  if (A) {
    const int in0 = n.num_prop + p.latent;
    const int na = n.n_actor_layers;
    // encoder (or the history latent) + backbone; returns the backbone's width.  `keep`: the last backbone layer is stored for a second head
    auto common = [&](C2Builder& B, bool keep) {
      int first_main = 0;
      if (z_hist) {
        B.load(rowmat(z_hist, zld), p.latent, 0, 32, 0);
      } else {
        B.load(rowmat_gather(obs + n.num_prop, idx, obs_stride), n.num_priv, C2_COL_PRIV, C2_COL_PRIV + pad8(n.num_priv), 0);
        B.fwd(P + n.off_priv_w[0], n.num_priv, P + n.off_priv_b[0], n.priv_dims[0], hid(n), C2_COL_PRIV, pad8(n.num_priv), 1,      // AC:219-221
              C2PackSeg{0, 0, n.num_priv}, C2PackSeg{0, 0, 0}, C2_COL_HID, store ? p.priv[0] : nullptr, align_up(n.priv_dims[0], 4));
        B.fwd(P + n.off_priv_w[1], n.priv_dims[0], P + n.off_priv_b[1], p.latent, hid(n), C2_COL_HID, pad8(n.priv_dims[0]), 1,
              C2PackSeg{0, 0, n.priv_dims[0]}, C2PackSeg{0, 0, 0}, 0, store ? p.priv[1] : nullptr, Lld, fin_mode == 2 ? FIN_REG : FIN_NONE, 0);
        first_main = 2;
      }
      const int k0 = pad8(C2_COL_PROP + n.num_prop);
      B.load(rowmat_gather(obs, idx, obs_stride), n.num_prop, C2_COL_PROP, k0, first_main);
      // backbone layer 0 over cat([obs_prop, z]) (AC:211): z occupies tile columns [0, latent), obs_prop [32, 32 + num_prop)
      B.fwd(P + n.off_actor_w[0], in0, P + n.off_actor_b[0], n.actor_dims[0], hid(n), 0, k0, 2, C2PackSeg{0, n.num_prop, p.latent},
            C2PackSeg{C2_COL_PROP, 0, n.num_prop}, 0, (store || (keep && na == 1)) ? p.ab[0] : nullptr, n.actor_dims[0], FIN_NONE, 0,
            img_dim(n.actor_dims[0]) && (store || (keep && na == 1)));
      int in = n.actor_dims[0];
      for (int l = 1; l < na; ++l) {                                                   // AC:211-213
        const bool st = store || (keep && l == na - 1);
        B.fwd(P + n.off_actor_w[l], in, P + n.off_actor_b[l], n.actor_dims[l], hid(n), 0, pad8(in), 1, C2PackSeg{0, 0, in}, C2PackSeg{0, 0, 0}, 0,
              st ? p.ab[l] : nullptr, n.actor_dims[l], FIN_NONE, 0, img_dim(n.actor_dims[l]) && st);
        in = n.actor_dims[l];
      }
      return in;
    };
    const int fin = fin_mode == 2 ? FIN_PPO : (fin_mode == 1 ? FIN_ACT : FIN_NONE);
    float* mean = fin_mode == 0 ? p.mean : nullptr;
    const int in = common(*A, A2 == nullptr);
    chain_head(*A, P, p.ab[na - 1], in, false, in, n.n_leg_layers, n.leg_dims, n.n_leg, n.off_aleg_w, n.off_aleg_b, p.al, store, mean, p.mean_ld, hid(n), ACT_TANH, fin, 0);
    C2Builder& Barm = A2 ? *A2 : *A;
    if (A2) common(*A2, false);
    chain_head(Barm, P, p.ab[na - 1], in, A2 == nullptr, in, n.n_arm_layers, n.arm_dims, n.n_arm, n.off_aarm_w, n.off_aarm_b, p.aa, store,
               mean ? mean + n.n_leg : nullptr, p.mean_ld, hid(n), ACT_TANH, fin, 1);
    A->finish();
    if (A2) A2->finish();
    if (!A->ok || (A2 && !A2->ok)) return DWBC_ERR_UNSUPPORTED;
  }
  if (C) {
    const int nc = n.n_critic_layers;
    auto common = [&](C2Builder& B, bool keep) {
      int in = n.num_prop + n.num_priv;
      B.load(rowmat_gather(obs, idx, obs_stride), in, 0, pad8(in), 0);
      for (int l = 0; l < nc; ++l) {                                                   // AC:280-286
        const bool st = store || (keep && l == nc - 1);
        B.fwd(P + n.off_critic_w[l], in, P + n.off_critic_b[l], n.critic_dims[l], hid(n), 0, pad8(in), 1, C2PackSeg{0, 0, in}, C2PackSeg{0, 0, 0}, 0,
              st ? p.cb[l] : nullptr, n.critic_dims[l], FIN_NONE, 0, img_dim(n.critic_dims[l]) && st);
        in = n.critic_dims[l];
      }
      return in;
    };
    const int fin = fin_mode == 2 ? FIN_VALUE : FIN_NONE;
    const int in = common(*C, C2 == nullptr);
    chain_head(*C, P, p.cb[nc - 1], in, false, in, n.n_leg_layers, n.leg_dims, 1, n.off_cleg_w, n.off_cleg_b, p.cl, store, value, 2, hid(n), ACT_NONE, fin, 0);
    C2Builder& Barm = C2 ? *C2 : *C;
    if (C2) common(*C2, false);
    chain_head(Barm, P, p.cb[nc - 1], in, C2 == nullptr, in, n.n_arm_layers, n.arm_dims, 1, n.off_carm_w, n.off_carm_b, p.ca, store,
               value + 1, 2, hid(n), ACT_NONE, fin, 1);
    C->finish();
    if (C2) C2->finish();
    if (!C->ok || (C2 && !C2->ok)) return DWBC_ERR_UNSUPPORTED;
  }
  return DWBC_OK;
}

// ---- rollout sampling + log-prob (AC:326-345, PPO:119-123) -------------------------------------
constexpr float LOG_SQRT_2PI = 0.91893853320467274178f;

__global__ void act_finalize_kernel(const float* __restrict__ mean_in, int mean_ld, const float* __restrict__ std, const float* __restrict__ eps,
                                    float* __restrict__ actions, float* __restrict__ log_prob, float* __restrict__ mean_out,
                                    float* __restrict__ sigma_out, int rows, int n_leg, int n_act) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float lp[2] = {0.0f, 0.0f};
  for (int i = 0; i < n_act; ++i) {
    const float mu = mean_in[(int64_t)r * mean_ld + i], sg = std[i];
    const float a = mu + sg * eps[(int64_t)r * n_act + i];
    const float d = a - mu;
    lp[i < n_leg ? 0 : 1] += -(d * d) / (2.0f * (sg * sg)) - logf(sg) - LOG_SQRT_2PI;
    actions[(int64_t)r * n_act + i] = a;
    mean_out[(int64_t)r * n_act + i] = mu;
    sigma_out[(int64_t)r * n_act + i] = sg;
  }
  log_prob[2 * r] = lp[0];
  log_prob[2 * r + 1] = lp[1];
}

// ---- PPO loss and its derivative w.r.t. the network outputs (PPO:166-221) ----------------------
struct LossArgs {
  const float* mean; int mean_ld; const float* std; const float* value; const float* zp; int zld; const float* zh; int64_t zh_ld; int zh_by_src;
  const float* actions; const float* old_logp; const float* old_values; const float* returns; const float* adv; const int64_t* idx;
  float* g_leg; int gleg_ld; float* g_arm; int garm_ld; float* g_vl; float* g_va; int gv_ld; float* g_z;
  float* grad_std; float* losses;
  int rows, n_leg, n_act, latent;
  float clip, c_value, c_ent, c_reg, rho;
  int clipped_value;
  const float* ts_target; const float* ts_pos; const float* ts_vel; const float* ts_coef; float ts_w;      // arm torque supervision (PPO:224-239)
};

__global__ void __launch_bounds__(128) ppo_loss_kernel(const LossArgs a) {
  __shared__ float red[5][4];
  __shared__ float sred[32];
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const bool on = r < a.rows;
  const float inv2m = 1.0f / (2.0f * (float)a.rows), invm = 1.0f / (float)a.rows;
  float l_surr = 0.0f, l_val = 0.0f, l_reg = 0.0f, l_ent = 0.0f, l_ts = 0.0f;
  float gstd[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) gstd[i] = 0.0f;
  if (on) {
    const int64_t src = a.idx ? a.idx[r] : r;
    const float* mu = a.mean + (int64_t)r * a.mean_ld;
    const float* act = a.actions + src * a.n_act;
    float lp[2] = {0.0f, 0.0f}, ent[2] = {0.0f, 0.0f};
    for (int i = 0; i < a.n_act; ++i) {
      const float sg = a.std[i], d = act[i] - mu[i];
      const int c = i < a.n_leg ? 0 : 1;
      lp[c] += -(d * d) / (2.0f * (sg * sg)) - logf(sg) - LOG_SQRT_2PI;          // AC:341-345
      ent[c] += 0.5f + LOG_SQRT_2PI + logf(sg);                                  // AC:326-331 (0.5 log 2pi == log sqrt 2pi)
    }
    const float a0 = a.adv[2 * src], a1 = a.adv[2 * src + 1];
    const float mix[2] = {a0 + a.rho * a1, a1 + a.rho * a0};                       // PPO:199-201
    float glp[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const float ratio = expf(lp[c] - a.old_logp[2 * src + c]);                   // PPO:202
      const float rc = fminf(fmaxf(ratio, 1.0f - a.clip), 1.0f + a.clip);
      const float s1 = -mix[c] * ratio, s2 = -mix[c] * rc;                         // PPO:203-205
      l_surr += fmaxf(s1, s2);
      const bool inside = ratio >= 1.0f - a.clip && ratio <= 1.0f + a.clip;
      float g = 0.0f;                                                              // d max(s1,s2) / d ratio
      if (s1 > s2) g = -mix[c];
      else if (s1 == s2) g = 0.5f * -mix[c] + (inside ? 0.5f * -mix[c] : 0.0f);
      else g = inside ? -mix[c] : 0.0f;
      glp[c] = inv2m * g * ratio;
      l_ent += ent[c];
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      if (i < a.n_act) {
        const float sg = a.std[i], d = act[i] - mu[i];
        const int c = i < a.n_leg ? 0 : 1;
        float gmu = glp[c] * d / (sg * sg) * (1.0f - mu[i] * mu[i]);               // through tanh (AC:157,170)
        if (c == 1 && a.ts_target != nullptr) {
          // arm torque supervision: tau = kp (mu + q_default - q) - kd qd (PPO:318-323), loss w * mean((tau - target)^2) (PPO:236-238)
          const int n_arm = a.n_act - a.n_leg, j = i - a.n_leg;
          const float kp = a.ts_coef[j];
          const float e = kp * (mu[i] + a.ts_coef[2 * n_arm + j] - a.ts_pos[src * n_arm + j]) - a.ts_coef[n_arm + j] * a.ts_vel[src * n_arm + j] -
                          a.ts_target[src * n_arm + j];
          l_ts += e * e;
          gmu += 2.0f * a.ts_w / ((float)a.rows * (float)n_arm) * e * kp * (1.0f - mu[i] * mu[i]);
        }
        if (c == 0) a.g_leg[(int64_t)r * a.gleg_ld + i] = gmu;
        else a.g_arm[(int64_t)r * a.garm_ld + (i - a.n_leg)] = gmu;
        gstd[i] = glp[c] * ((d * d) / (sg * sg * sg) - 1.0f / sg) - a.c_ent * inv2m / sg;
      }
    }
    // value loss PPO:209-216
    float gv[2];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const float v = a.value[2 * r + c], vo = a.old_values[2 * src + c], R = a.returns[2 * src + c];
      const float l1 = (v - R) * (v - R);
      if (a.clipped_value) {
        const float dvo = v - vo;
        const float vc = vo + fminf(fmaxf(dvo, -a.clip), a.clip);
        const float l2 = (vc - R) * (vc - R);
        const bool inside = dvo >= -a.clip && dvo <= a.clip;
        l_val += fmaxf(l1, l2);
        const float g1 = 2.0f * (v - R), g2 = inside ? 2.0f * (vc - R) : 0.0f;
        gv[c] = l1 > l2 ? g1 : (l1 == l2 ? 0.5f * g1 + 0.5f * g2 : g2);
      } else {
        l_val += l1;
        gv[c] = 2.0f * (v - R);
      }
      gv[c] *= a.c_value * inv2m;
    }
    a.g_vl[(int64_t)r * a.gv_ld] = gv[0];
    a.g_va[(int64_t)r * a.gv_ld] = gv[1];
    // pad columns are read as (zero-weighted) operand columns by the tensor-core backward: keep them finite
    for (int i = 2; i < a.gv_ld; ++i) a.g_vl[(int64_t)r * a.gv_ld + i] = 0.0f;
    for (int i = a.n_leg; i < a.gleg_ld; ++i) a.g_leg[(int64_t)r * a.gleg_ld + i] = 0.0f;
    for (int i = a.n_act - a.n_leg; i < a.garm_ld; ++i) a.g_arm[(int64_t)r * a.garm_ld + i] = 0.0f;
    // privileged-latent regulariser PPO:174-177
    float nrm = 0.0f;
    const float* zhr = a.zh + (a.zh_by_src ? src : (int64_t)r) * a.zh_ld;     // precomputed per storage row, or per mini-batch row
    for (int i = 0; i < a.latent; ++i) {
      const float d = a.zp[(int64_t)r * a.zld + i] - zhr[i];
      nrm += d * d;
    }
    nrm = sqrtf(nrm);
    l_reg = nrm;
    const float s = nrm > 0.0f ? a.c_reg * invm / nrm : 0.0f;
    for (int i = 0; i < a.latent; ++i)
      a.g_z[(int64_t)r * a.zld + i] = s * (a.zp[(int64_t)r * a.zld + i] - zhr[i]);
  }
  // block reductions -> one atomic per CTA per quantity
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float v4[5] = {l_surr * inv2m, l_val * inv2m, l_reg * invm, l_ent * inv2m, l_ts * invm / (float)max(a.n_act - a.n_leg, 1)};
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    float s = warp_sum(v4[k]);
    if (lane == 0) red[k][w] = s;
  }
  if (threadIdx.x < 32) sred[threadIdx.x] = 0.0f;
  __syncthreads();
  if (threadIdx.x < (a.ts_target != nullptr ? 5 : 4)) atomicAdd(a.losses + threadIdx.x, (red[threadIdx.x][0] + red[threadIdx.x][1]) + (red[threadIdx.x][2] + red[threadIdx.x][3]));
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    if (i < a.n_act) {
      float s = warp_sum(gstd[i]);
      if (lane == 0) atomicAdd(&sred[i], s);
    }
  }
  __syncthreads();
  if (threadIdx.x < a.n_act) atomicAdd(a.grad_std + threadIdx.x, sred[threadIdx.x]);
}

// DAgger loss PPO:273-276: mean_rows || sg(zp) - zh ||_2 ; writes d/d zh_pre (the activation derivative folded in)
__global__ void __launch_bounds__(128) dagger_loss_kernel(const float* __restrict__ zp, const float* __restrict__ zh, int zld, int latent,
                                                          float* __restrict__ g, float* __restrict__ loss, int rows, int act) {
  __shared__ float red[4];
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  float l = 0.0f;
  if (r < rows) {
    float nrm = 0.0f;
    for (int i = 0; i < latent; ++i) {
      const float d = zp[(int64_t)r * zld + i] - zh[(int64_t)r * zld + i];
      nrm += d * d;
    }
    nrm = sqrtf(nrm);
    l = nrm / (float)rows;
    const float s = nrm > 0.0f ? 1.0f / ((float)rows * nrm) : 0.0f;
    for (int i = 0; i < latent; ++i) {
      const float y = zh[(int64_t)r * zld + i];
      g[(int64_t)r * zld + i] = -s * (zp[(int64_t)r * zld + i] - y) * act_dy(act, y);
    }
  }
  float s = warp_sum(l);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) atomicAdd(loss, (red[0] + red[1]) + (red[2] + red[3]));
}

// ---- backward -----------------------------------------------------------------------------------
// Backward of one head: Linear(+act) x nl, then Linear -> out.  G_out = d/d(pre-activation of the
// last layer) [rows, n_out].  Accumulates weight grads into `grad`, and adds the head's
// contribution to d(backbone output) into dtrunk (beta_trunk; act' of the trunk applied if apply_dact).
static int head_backward(const float* P, float* grad, RowMat G_out, int n_out, int nl, const int32_t* dims, const int64_t* ow,
                         const int64_t* ob, float* const* acts, RowMat trunk, int trunk_dim, float* dtrunk, int beta_trunk,
                         int apply_dact, float* dA, float* dB, int hact, int rows, cudaStream_t st) {
  RowMat G = G_out;
  int gout = n_out;
  for (int l = nl; l >= 0; --l) {
    const int in = l == 0 ? trunk_dim : dims[l - 1];
    RowMat X = l == 0 ? trunk : rowmat(acts[l - 1], dims[l - 1]);
    TRY(linear_bwd_weight(G, X, grad + ow[l], in, grad + ob[l], rows, gout, in, st));
    if (l == 0) {
      TRY(linear_bwd_data(G, P + ow[l], in, dtrunk, trunk_dim, rows, in, gout, apply_dact ? hact : ACT_NONE, trunk, beta_trunk, st));
    } else {
      float* d = (l & 1) ? dA : dB;
      TRY(linear_bwd_data(G, P + ow[l], in, d, in, rows, in, gout, hact, X, 0, st));
      G = rowmat(d, in);
      gout = in;
    }
  }
  return DWBC_OK;
}

// ---- fused backward (tensor-core paths): all data-gradient GEMMs of the actor + privileged encoder and of the critic as two
// programs of one launch (mlp_chain2.cuh, backward ops); the per-layer pre-activation gradients they leave behind feed the
// weight-gradient GEMMs (wgrad_group.cuh, MN-major operands).
struct HeadDesc { int nl; const int32_t* dims; const int64_t* ow; const int64_t* ob; float* const* acts; float* const* dz; RowMat g_out; int n_out; };

// data-gradient ops of one head, last layer first.  The head's loss gradient [rows, g_ld] is loaded into tile columns [0, g_ld) right
// before its first op; column g_col + j of that window multiplies row j of the last layer's weights.  The trunk gradient of the
// FIRST head goes to `scratch` unactivated; the second head adds it and applies the trunk's act'.
static void chain_head_bwd(C2Builder& b, const float* P, const HeadDesc& hd, const float* g, int g_ld, int g_col, int trunk_dim, const float* trunk,
                           bool second, float* scratch, float* dz_trunk, int hact) {
  b.load(rowmat(g, g_ld), g_ld, 0, pad8(g_ld), b.pr.n_ops);
  for (int l = hd.nl; l >= 0; --l) {
    const int in = l == 0 ? trunk_dim : hd.dims[l - 1];
    const int out = l == hd.nl ? hd.n_out : hd.dims[l];
    const bool narrow = l == hd.nl;
    const int kpad = narrow ? pad8(g_ld) : pad8(out);
    const C2PackSeg seg{narrow ? g_col : 0, 0, out};
    if (l > 0)
      b.bwd(P + hd.ow[l], in, in, 0, kpad, seg, hact, hd.acts[l - 1], in, nullptr, 0, 0, hd.dz[l - 1], in, img_dim(in), img_dim(in));
    else if (!second)
      b.bwd(P + hd.ow[0], in, in, 0, kpad, seg, ACT_NONE, nullptr, 0, nullptr, 0, -1, scratch, trunk_dim);
    else
      b.bwd(P + hd.ow[0], in, in, 0, kpad, seg, hact, trunk, trunk_dim, scratch, trunk_dim, 0, dz_trunk, trunk_dim, img_dim(trunk_dim), img_dim(trunk_dim));
  }
}

static void head_wgrad(WGroupBuilder& wb, float* grad, const HeadDesc& hd, RowMat trunk, int trunk_dim) {
  for (int l = hd.nl; l >= 0; --l) {
    const int in = l == 0 ? trunk_dim : hd.dims[l - 1];
    RowMat G = l == hd.nl ? hd.g_out : act_mat(hd.dz[l], hd.dims[l]);
    const int gout = l == hd.nl ? hd.n_out : hd.dims[l];
    RowMat X = l == 0 ? trunk : act_mat(hd.acts[l - 1], hd.dims[l - 1]);
    wb.add(G, X, grad + hd.ow[l], in, grad + hd.ob[l], gout, in);
  }
}

struct BwdDescs { HeadDesc cl, ca, al, aa; };
static BwdDescs bwd_descs(const DwbcNetCfg& n, const Plan& p) {
  const int gleg_ld = (int)align_up(n.n_leg, 4), garm_ld = (int)align_up(n.n_arm, 4);
  BwdDescs d;
  d.cl = HeadDesc{n.n_leg_layers, n.leg_dims, n.off_cleg_w, n.off_cleg_b, p.cl, p.dzc_l, rowmat(p.g_vl, 4), 1};
  d.ca = HeadDesc{n.n_arm_layers, n.arm_dims, n.off_carm_w, n.off_carm_b, p.ca, p.dzc_a, rowmat(p.g_va, 4), 1};
  d.al = HeadDesc{n.n_leg_layers, n.leg_dims, n.off_aleg_w, n.off_aleg_b, p.al, p.dza_l, rowmat(p.g_leg, gleg_ld), n.n_leg};
  d.aa = HeadDesc{n.n_arm_layers, n.arm_dims, n.off_aarm_w, n.off_aarm_b, p.aa, p.dza_a, rowmat(p.g_arm, garm_ld), n.n_arm};
  return d;
}

static int build_backward(const DwbcNetCfg& n, const float* P, const Plan& p, C2Builder& A, C2Builder& C) {
  const int Lld = (int)align_up(p.latent, 4);
  const int gleg_ld = (int)align_up(n.n_leg, 4), garm_ld = (int)align_up(n.n_arm, 4);
  const BwdDescs d = bwd_descs(n, p);
  // ---- critic: both value heads read their column of the [rows, 4] value-gradient buffer ----
  const int cnb = n.n_critic_layers, ctd = n.critic_dims[cnb - 1];
  chain_head_bwd(C, P, d.cl, p.g_vl, 4, 0, ctd, p.cb[cnb - 1], false, p.d1, nullptr, hid(n));
  chain_head_bwd(C, P, d.ca, p.g_vl, 4, 1, ctd, p.cb[cnb - 1], true, p.d1, p.dzc_b[cnb - 1], hid(n));
  for (int l = cnb - 1; l >= 1; --l)
    C.bwd(P + n.off_critic_w[l], n.critic_dims[l - 1], n.critic_dims[l - 1], 0, pad8(n.critic_dims[l]), C2PackSeg{0, 0, n.critic_dims[l]}, hid(n),
          p.cb[l - 1], n.critic_dims[l - 1], nullptr, 0, 0, p.dzc_b[l - 1], n.critic_dims[l - 1], img_dim(n.critic_dims[l - 1]), img_dim(n.critic_dims[l - 1]));
  C.finish();
  // ---- actor + privileged encoder ----
  const int anb = n.n_actor_layers, atd = n.actor_dims[anb - 1];
  chain_head_bwd(A, P, d.al, p.g_leg, gleg_ld, 0, atd, p.ab[anb - 1], false, p.d0, nullptr, hid(n));
  chain_head_bwd(A, P, d.aa, p.g_arm, garm_ld, 0, atd, p.ab[anb - 1], true, p.d0, p.dza_b[anb - 1], hid(n));
  for (int l = anb - 1; l >= 1; --l)
    A.bwd(P + n.off_actor_w[l], n.actor_dims[l - 1], n.actor_dims[l - 1], 0, pad8(n.actor_dims[l]), C2PackSeg{0, 0, n.actor_dims[l]}, hid(n),
          p.ab[l - 1], n.actor_dims[l - 1], nullptr, 0, 0, p.dza_b[l - 1], n.actor_dims[l - 1], img_dim(n.actor_dims[l - 1]), img_dim(n.actor_dims[l - 1]));
  const int in0 = n.num_prop + p.latent, np = n.n_priv_layers;
  float* z = p.priv[np - 1];
  // dL/dz = policy path through the latent columns of backbone layer 0 + privileged-latent regulariser (g_z), through the encoder's last activation
  A.bwd(P + n.off_actor_w[0] + n.num_prop, in0, p.latent, 0, pad8(n.actor_dims[0]), C2PackSeg{0, 0, n.actor_dims[0]}, hid(n), z, Lld, p.g_z, Lld, 0,
        p.dzp[np - 1], Lld);
  for (int l = np - 1; l >= 1; --l) {
    const int in = n.priv_dims[l - 1], ldin = (int)align_up(in, 4);
    A.bwd(P + n.off_priv_w[l], in, in, 0, pad8(n.priv_dims[l]), C2PackSeg{0, 0, n.priv_dims[l]}, hid(n), p.priv[l - 1], ldin, nullptr, 0, l - 1 > 0 ? 0 : -1,
          p.dzp[l - 1], ldin);
  }
  A.finish();
  if (!C.ok || !A.ok) return DWBC_ERR_UNSUPPORTED;
  return DWBC_OK;
}

// every layer's weight gradient of both networks in one persistent launch (wgrad_group.cuh)
static int weight_gradients(const DwbcNetCfg& n, float* grad, const DwbcStorage* s, const int64_t* idx, int rows, const Plan& p, cudaStream_t st) {
  const int Lld = (int)align_up(p.latent, 4);
  const BwdDescs d = bwd_descs(n, p);
  const int cnb = n.n_critic_layers, ctd = n.critic_dims[cnb - 1];
  const int anb = n.n_actor_layers, atd = n.actor_dims[anb - 1];
  const int in0 = n.num_prop + p.latent, np = n.n_priv_layers;
  float* z = p.priv[np - 1];
  RowMat obs_all = rowmat_gather(s->observations, idx, s->obs_stride);
  WGroupBuilder wb;
  head_wgrad(wb, grad, d.cl, act_mat(p.cb[cnb - 1], ctd), ctd);
  head_wgrad(wb, grad, d.ca, act_mat(p.cb[cnb - 1], ctd), ctd);
  for (int l = cnb - 1; l >= 0; --l) {
    const int in = l == 0 ? n.num_prop + n.num_priv : n.critic_dims[l - 1];
    wb.add(act_mat(p.dzc_b[l], n.critic_dims[l]), l == 0 ? obs_all : act_mat(p.cb[l - 1], in), grad + n.off_critic_w[l], in, grad + n.off_critic_b[l],
           n.critic_dims[l], in);
  }
  head_wgrad(wb, grad, d.al, act_mat(p.ab[anb - 1], atd), atd);
  head_wgrad(wb, grad, d.aa, act_mat(p.ab[anb - 1], atd), atd);
  for (int l = anb - 1; l >= 1; --l)
    wb.add(act_mat(p.dza_b[l], n.actor_dims[l]), act_mat(p.ab[l - 1], n.actor_dims[l - 1]), grad + n.off_actor_w[l], n.actor_dims[l - 1],
           grad + n.off_actor_b[l], n.actor_dims[l], n.actor_dims[l - 1]);
  RowMat G0 = act_mat(p.dza_b[0], n.actor_dims[0]);
  wb.add(G0, obs_all, grad + n.off_actor_w[0], in0, grad + n.off_actor_b[0], n.actor_dims[0], n.num_prop);
  wb.add(G0, rowmat(z, Lld), grad + n.off_actor_w[0] + n.num_prop, in0, nullptr, n.actor_dims[0], p.latent);
  for (int l = np - 1; l >= 0; --l) {
    const int in = l == 0 ? n.num_priv : n.priv_dims[l - 1];
    RowMat X = l == 0 ? rowmat_gather(s->observations + n.num_prop, idx, s->obs_stride) : rowmat(p.priv[l - 1], (int)align_up(in, 4));
    wb.add(rowmat(p.dzp[l], (int)align_up(n.priv_dims[l], 4)), X, grad + n.off_priv_w[l], in, grad + n.off_priv_b[l], n.priv_dims[l], in);
  }
  if (!wb.ok) return DWBC_ERR_UNSUPPORTED;
  return launch_wgrad_group(wb.g, rows, mlp_precision == 2, st);
}

}  // namespace dwbc

using namespace dwbc;

extern "C" int64_t dwbc_workspace_bytes(const DwbcNetCfg* net, int64_t rows) {
  if (check_net(net) != DWBC_OK || rows <= 0) return -1;
  return make_plan(*net, rows, nullptr).bytes;
}

// FinArgs of the rollout hooks
static FinArgs fin_rollout(const DwbcNetCfg& n, const float* P, const float* eps, float* actions, float* log_prob, float* mean, float* sigma, int rows) {
  FinArgs f{};
  f.std = P + n.off_std; f.eps = eps; f.actions = actions; f.log_prob = log_prob; f.mean_out = mean; f.sigma_out = sigma;
  f.n_leg = n.n_leg; f.n_act = n.n_leg + n.n_arm; f.rows = rows;
  return f;
}

extern "C" int dwbc_policy_act(const DwbcNetCfg* net, const float* params, const float* obs, int64_t obs_stride, const float* eps,
                               int32_t hist_encoding, float* actions, float* values, float* log_prob, float* mean, float* sigma,
                               int32_t rows, int32_t weights_packed, void* workspace, dwbc_stream_t stream) {
  TRY(check_net(net));
  if (!params || !obs || !eps || !actions || !values || !log_prob || !mean || !sigma || !workspace || rows <= 0) return DWBC_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const DwbcNetCfg& n = *net;
  Plan p = make_plan(n, rows, workspace);
  const float* z;
  int zld = (int)align_up(p.latent, 4);
  if (chain_usable(n, p, obs, obs_stride)) {
    if (hist_encoding) TRY(hist_latent_only(n, params, obs, nullptr, obs_stride, rows, p, p.zh, zld, st));
    C2PackList pl{};
    pl.out = p.wpack;
    int64_t off = 0;
    const bool x3 = mlp_precision == 2;
    C2Builder A(&pl, &off, rows, x3), C(&pl, &off, rows, x3), A2(&pl, &off, rows, x3), C2(&pl, &off, rows, x3);
    // few tiles (the rollout): one program per HEAD, so that four short programs spread over 4 x tiles SMs (build_forward)
    const bool split = 4 * ((rows + TC_M - 1) / TC_M) <= c2_sm_count();
    TRY(build_forward(n, params, obs, nullptr, obs_stride, hist_encoding ? p.zh : nullptr, zld, p, values, false, 1, &A, &C, split ? &A2 : nullptr,
                      split ? &C2 : nullptr));
    if (off > C2_PACK_FLOATS) return DWBC_ERR_UNSUPPORTED;
    if (!weights_packed) TRY(launch_pack2(pl, st));       // the images stay valid in the workspace until the parameters change
    const C2Prog* prs[4] = {&A.pr, &C.pr, &A2.pr, &C2.pr};
    return launch_chain2n(prs, split ? 4 : 2, fin_rollout(n, params, eps, actions, log_prob, mean, sigma, rows), x3, p.queue, st);
  }
  if (hist_encoding) {
    TRY(hist_forward(n, params, obs, nullptr, obs_stride, rows, p, st));
    z = p.zh;
  } else {
    TRY(priv_forward(n, params, obs, nullptr, obs_stride, rows, p, st));
    z = p.priv[n.n_priv_layers - 1];
  }
  TRY(actor_forward(n, params, obs, nullptr, obs_stride, rows, z, zld, p, st));
  TRY(critic_forward(n, params, obs, nullptr, obs_stride, rows, p, values, st));
  act_finalize_kernel<<<(rows + 127) / 128, 128, 0, st>>>(p.mean, p.mean_ld, params + n.off_std, eps, actions, log_prob, mean, sigma, rows,
                                                           n.n_leg, n.n_leg + n.n_arm);
  DWBC_LAUNCH_CHECK();
  return DWBC_OK;
}

extern "C" int dwbc_critic_values(const DwbcNetCfg* net, const float* params, const float* obs, int64_t obs_stride, float* values,
                                  int32_t rows, void* workspace, dwbc_stream_t stream) {
  TRY(check_net(net));
  if (!params || !obs || !values || !workspace || rows <= 0) return DWBC_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  Plan p = make_plan(*net, rows, workspace);
  if (chain_usable(*net, p, obs, obs_stride)) {
    C2PackList pl{};
    pl.out = p.wpack;
    int64_t off = 0;
    const bool x3 = mlp_precision == 2;
    C2Builder C(&pl, &off, rows, x3), C2(&pl, &off, rows, x3);
    const bool split = 2 * ((rows + TC_M - 1) / TC_M) <= c2_sm_count();
    TRY(build_forward(*net, params, obs, nullptr, obs_stride, nullptr, 0, p, values, false, 0, nullptr, &C, nullptr, split ? &C2 : nullptr));
    TRY(launch_pack2(pl, st));                              // (overwrites the images a previous dwbc_policy_act left behind)
    const C2Prog* prs[2] = {&C.pr, &C2.pr};
    return launch_chain2n(prs, split ? 2 : 1, FinArgs{}, x3, p.queue, st);
  }
  return critic_forward(*net, params, obs, nullptr, obs_stride, rows, p, values, st);
}

extern "C" int dwbc_hist_latent(const DwbcNetCfg* net, const float* params, const float* obs, int64_t obs_stride, float* out, int64_t ld_out,
                                int32_t rows, void* workspace, dwbc_stream_t stream) {
  TRY(check_net(net));
  if (!params || !obs || !out || !workspace || rows <= 0) return DWBC_ERR_ARG;
  Plan p = make_plan(*net, rows, workspace);
  if (ld_out != align_up(p.latent, 4)) return DWBC_ERR_ARG;
  return hist_latent_only(*net, params, obs, nullptr, obs_stride, rows, p, out, ld_out, (cudaStream_t)stream);
}

extern "C" int dwbc_ppo_minibatch_grad(const DwbcNetCfg* net, const float* params, const DwbcStorage* s, const int64_t* idx, int32_t M,
                                       const DwbcPpoHyper* hp, float* grad, float* losses_out, void* workspace, dwbc_stream_t stream) {
  TRY(check_net(net));
  if (!params || !s || !idx || !hp || !grad || !losses_out || !workspace || M <= 0) return DWBC_ERR_ARG;
  if (!s->observations || !s->actions || !s->values || !s->returns || !s->advantages || !s->log_prob) return DWBC_ERR_ARG;
  // torque supervision is on when the storage carries its three tensors (RS:82-84); then the arm coefficients are needed too
  if (s->target_arm_torques && (!s->current_arm_dof_pos || !s->current_arm_dof_vel || !hp->arm_coefs)) return DWBC_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const DwbcNetCfg& n = *net;
  const float* P = params;
  const int rows = M;
  Plan p = make_plan(n, rows, workspace);
  const int Lld = (int)align_up(p.latent, 4);
  const int gleg_ld = (int)align_up(n.n_leg, 4), garm_ld = (int)align_up(n.n_arm, 4);
  if (cudaMemsetAsync(grad, 0, sizeof(float) * n.num_params, st) != cudaSuccess) return DWBC_ERR_LAUNCH;

  // forward (the reference evaluates the actor 3x and the priv encoder 3x per mini-batch,
  // PPO:166,174,230; identical values, so each is evaluated once here)
  float* z = p.priv[n.n_priv_layers - 1];
  if (!s->hist_latent) TRY(hist_latent_only(n, P, s->observations, idx, s->obs_stride, rows, p, p.zh, Lld, st));           // PPO:175-176 (no grad)
  if (chain_usable(n, p, s->observations, s->obs_stride)) {
    // tensor-core path: forward chains with the loss in the heads' epilogues, backward chains, grouped weight gradients.  The
    // weight images of all four programs are packed by ONE launch (the parameters are constant within a mini-batch).
    C2PackList pl{};
    pl.out = p.wpack;
    int64_t off = 0;
    const bool x3 = mlp_precision == 2;
    C2Builder A(&pl, &off, rows, x3), C(&pl, &off, rows, x3), Ab(&pl, &off, rows, x3), Cb(&pl, &off, rows, x3);
    TRY(build_forward(n, P, s->observations, idx, s->obs_stride, nullptr, Lld, p, p.value, true, 2, &A, &C));
    TRY(build_backward(n, P, p, Ab, Cb));
    if (off > C2_PACK_FLOATS) return DWBC_ERR_UNSUPPORTED;
    FinArgs f{};
    f.std = P + n.off_std; f.idx = idx; f.s_actions = s->actions; f.old_logp = s->log_prob; f.old_values = s->values; f.returns = s->returns;
    f.adv = s->advantages;
    f.zh = s->hist_latent ? s->hist_latent : p.zh; f.zh_ld = s->hist_latent ? s->hist_latent_ld : Lld; f.zh_by_src = s->hist_latent ? 1 : 0;
    f.g_leg = p.g_leg; f.gleg_ld = gleg_ld; f.g_arm = p.g_arm; f.garm_ld = garm_ld; f.g_v = p.g_vl; f.gv_ld = 4; f.g_z = p.g_z; f.gz_ld = Lld;
    f.grad_std = grad + n.off_std; f.losses = losses_out;
    f.n_leg = n.n_leg; f.n_act = n.n_leg + n.n_arm; f.latent = p.latent; f.rows = rows;
    f.clip = hp->clip_param; f.c_value = hp->value_loss_coef; f.c_ent = hp->entropy_coef; f.c_reg = hp->priv_reg_coef; f.rho = hp->mixing_ratio;
    f.clipped_value = hp->use_clipped_value_loss;
    f.ts_target = s->target_arm_torques; f.ts_pos = s->current_arm_dof_pos; f.ts_vel = s->current_arm_dof_vel; f.ts_coef = hp->arm_coefs;
    f.ts_w = hp->torque_supervision_weight;
    TRY(launch_pack2(pl, st));
    TRY(launch_chain2(&A.pr, &C.pr, f, x3, p.queue, st));
    TRY(launch_chain2(&Ab.pr, &Cb.pr, FinArgs{}, x3, p.queue, st, c2_bwd_reverse != 0));
    return weight_gradients(n, grad, s, idx, rows, p, st);
  }
  TRY(priv_forward(n, P, s->observations, idx, s->obs_stride, rows, p, st));
  TRY(actor_forward(n, P, s->observations, idx, s->obs_stride, rows, z, Lld, p, st));
  TRY(critic_forward(n, P, s->observations, idx, s->obs_stride, rows, p, p.value, st));

  LossArgs a{};
  a.mean = p.mean; a.mean_ld = p.mean_ld; a.std = P + n.off_std; a.value = p.value; a.zp = z; a.zld = Lld; a.zh = s->hist_latent ? s->hist_latent : p.zh; a.zh_ld = s->hist_latent ? s->hist_latent_ld : Lld; a.zh_by_src = s->hist_latent ? 1 : 0;
  a.actions = s->actions; a.old_logp = s->log_prob; a.old_values = s->values; a.returns = s->returns; a.adv = s->advantages; a.idx = idx;
  a.g_leg = p.g_leg; a.gleg_ld = gleg_ld; a.g_arm = p.g_arm; a.garm_ld = garm_ld; a.g_vl = p.g_vl; a.g_va = p.g_va; a.gv_ld = 4; a.g_z = p.g_z;
  a.grad_std = grad + n.off_std; a.losses = losses_out;
  a.rows = rows; a.n_leg = n.n_leg; a.n_act = n.n_leg + n.n_arm; a.latent = p.latent;
  a.clip = hp->clip_param; a.c_value = hp->value_loss_coef; a.c_ent = hp->entropy_coef; a.c_reg = hp->priv_reg_coef; a.rho = hp->mixing_ratio;
  a.clipped_value = hp->use_clipped_value_loss;
  a.ts_target = s->target_arm_torques; a.ts_pos = s->current_arm_dof_pos; a.ts_vel = s->current_arm_dof_vel; a.ts_coef = hp->arm_coefs;
  a.ts_w = hp->torque_supervision_weight;
  ppo_loss_kernel<<<(rows + 127) / 128, 128, 0, st>>>(a);
  DWBC_LAUNCH_CHECK();

  // ---- critic backward ----
  {
    const int nb = n.n_critic_layers, tdim = n.critic_dims[nb - 1];
    RowMat trunk = rowmat(p.cb[nb - 1], tdim);
    TRY(head_backward(P, grad, rowmat(p.g_vl, 4), 1, n.n_leg_layers, n.leg_dims, n.off_cleg_w, n.off_cleg_b, p.cl, trunk, tdim, p.d2, 0, 0,
                      p.d0, p.d1, hid(n), rows, st));
    TRY(head_backward(P, grad, rowmat(p.g_va, 4), 1, n.n_arm_layers, n.arm_dims, n.off_carm_w, n.off_carm_b, p.ca, trunk, tdim, p.d2, 1, 1,
                      p.d0, p.d1, hid(n), rows, st));
    RowMat G = rowmat(p.d2, tdim);
    int gout = tdim;
    for (int l = nb - 1; l >= 0; --l) {
      const int in = l == 0 ? n.num_prop + n.num_priv : n.critic_dims[l - 1];
      RowMat X = l == 0 ? rowmat_gather(s->observations, idx, s->obs_stride) : rowmat(p.cb[l - 1], in);
      TRY(linear_bwd_weight(G, X, grad + n.off_critic_w[l], in, grad + n.off_critic_b[l], rows, gout, in, st));
      if (l > 0) {
        float* d = (l & 1) ? p.d0 : p.d1;
        TRY(linear_bwd_data(G, P + n.off_critic_w[l], in, d, in, rows, in, gout, hid(n), X, 0, st));
        G = rowmat(d, in);
        gout = in;
      }
    }
  }
  // ---- actor backward ----
  {
    const int nb = n.n_actor_layers, tdim = n.actor_dims[nb - 1];
    RowMat trunk = rowmat(p.ab[nb - 1], tdim);
    TRY(head_backward(P, grad, rowmat(p.g_leg, gleg_ld), n.n_leg, n.n_leg_layers, n.leg_dims, n.off_aleg_w, n.off_aleg_b, p.al, trunk, tdim,
                      p.d2, 0, 0, p.d0, p.d1, hid(n), rows, st));
    TRY(head_backward(P, grad, rowmat(p.g_arm, garm_ld), n.n_arm, n.n_arm_layers, n.arm_dims, n.off_aarm_w, n.off_aarm_b, p.aa, trunk, tdim,
                      p.d2, 1, 1, p.d0, p.d1, hid(n), rows, st));
    RowMat G = rowmat(p.d2, tdim);
    int gout = tdim;
    for (int l = nb - 1; l >= 1; --l) {
      const int in = n.actor_dims[l - 1];
      RowMat X = rowmat(p.ab[l - 1], in);
      TRY(linear_bwd_weight(G, X, grad + n.off_actor_w[l], in, grad + n.off_actor_b[l], rows, gout, in, st));
      float* d = (l & 1) ? p.d0 : p.d1;
      TRY(linear_bwd_data(G, P + n.off_actor_w[l], in, d, in, rows, in, gout, hid(n), X, 0, st));
      G = rowmat(d, in);
      gout = in;
    }
    // backbone layer 0: input = cat([obs_prop, z])
    const int in0 = n.num_prop + p.latent;
    TRY(linear_bwd_weight(G, rowmat_gather(s->observations, idx, s->obs_stride), grad + n.off_actor_w[0], in0, grad + n.off_actor_b[0], rows,
                          gout, n.num_prop, st));
    TRY(linear_bwd_weight(G, rowmat(z, Lld), grad + n.off_actor_w[0] + n.num_prop, in0, nullptr, rows, gout, p.latent, st));
    // dL/dz = (policy path) + (priv-reg path, already in g_z); then through the activation of the encoder's last layer
    TRY(linear_bwd_data(G, P + n.off_actor_w[0] + n.num_prop, in0, p.g_z, Lld, rows, p.latent, gout, hid(n), rowmat(z, Lld), 1, st));
    RowMat Gp = rowmat(p.g_z, Lld);
    int gp = p.latent;
    for (int l = n.n_priv_layers - 1; l >= 0; --l) {
      const int in = l == 0 ? n.num_priv : n.priv_dims[l - 1];
      const int ldin = (int)align_up(in, 4);
      RowMat X = l == 0 ? rowmat_gather(s->observations + n.num_prop, idx, s->obs_stride) : rowmat(p.priv[l - 1], ldin);
      TRY(linear_bwd_weight(Gp, X, grad + n.off_priv_w[l], in, grad + n.off_priv_b[l], rows, gp, in, st));
      if (l > 0) {
        float* d = (l & 1) ? p.d0 : p.d1;
        TRY(linear_bwd_data(Gp, P + n.off_priv_w[l], in, d, ldin, rows, in, gp, hid(n), X, 0, st));
        Gp = rowmat(d, ldin);
        gp = in;
      }
    }
  }
  return DWBC_OK;
}

extern "C" int dwbc_dagger_minibatch_grad(const DwbcNetCfg* net, const float* params, const DwbcStorage* s, const int64_t* idx, int32_t M,
                                          float* grad, float* losses_out, void* workspace, dwbc_stream_t stream) {
  TRY(check_net(net));
  if (!params || !s || !s->observations || !idx || !grad || !losses_out || !workspace || M <= 0) return DWBC_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const DwbcNetCfg& n = *net;
  const float* P = params;
  const int rows = M, T = n.num_hist;
  Plan p = make_plan(n, rows, workspace);
  const int L = p.latent, Lld = (int)align_up(L, 4);
  if (cudaMemsetAsync(grad, 0, sizeof(float) * n.num_params, st) != cudaSuccess) return DWBC_ERR_LAUNCH;
  if (cudaMemsetAsync(p.dhw1, 0, sizeof(float) * (20 * 128), st) != cudaSuccess) return DWBC_ERR_LAUNCH;
  if (cudaMemsetAsync(p.dhw2, 0, sizeof(float) * (10 * 40), st) != cudaSuccess) return DWBC_ERR_LAUNCH;
  if (cudaMemsetAsync(p.dhwl, 0, sizeof(float) * (32 * 36), st) != cudaSuccess) return DWBC_ERR_LAUNCH;
  TRY(priv_forward(n, P, s->observations, idx, s->obs_stride, rows, p, st));             // PPO:273-274 (no grad)
  TRY(hist_forward(n, P, s->observations, idx, s->obs_stride, rows, p, st));             // PPO:275
  dagger_loss_kernel<<<(rows + 127) / 128, 128, 0, st>>>(p.priv[n.n_priv_layers - 1], p.zh, Lld, L, p.dzh, losses_out, rows, hid(n));
  DWBC_LAUNCH_CHECK();
  // linear_output: zh = act(flat . Wl'^T + b)
  RowMat G4 = rowmat(p.dzh, Lld);
  TRY(linear_bwd_weight(G4, rowmat(p.hc2, 36), p.dhwl, 36, grad + n.off_hist_b[3], rows, L, 36, st));
  TRY(linear_bwd_data(G4, p.hwl, 36, p.d0, 36, rows, 36, L, hid(n), rowmat(p.hc2, 36), 0, st));    // d(conv2 pre-act) as [rows*3, 12]
  // conv2
  RowMat G3 = rowmat(p.d0, 12);
  TRY(linear_bwd_weight(G3, rowmat_grouped(p.hc1, nullptr, 3, 80, 20), p.dhw2, 40, grad + n.off_hist_b[2], rows * 3, 10, 40, st));
  TRY(linear_bwd_data(G3, p.hw2, 40, p.dh_a2, 40, rows * 3, 40, 10, ACT_NONE, RowMat{}, 0, st));
  {
    int64_t tot = (int64_t)rows * 4 * 20;
    col2im_dact_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(p.dh_a2, p.hc1, p.dh_c1, rows, 4, 20, 20, 3, 2, 1, hid(n));
    DWBC_LAUNCH_CHECK();
  }
  // conv1
  RowMat G2 = rowmat(p.dh_c1, 20);
  TRY(linear_bwd_weight(G2, rowmat_grouped(p.hproj, nullptr, 4, (int64_t)T * 32, 64), p.dhw1, 128, grad + n.off_hist_b[1], rows * 4, 20, 128, st));
  TRY(linear_bwd_data(G2, p.hw1, 128, p.dh_a1, 128, rows * 4, 128, 20, ACT_NONE, RowMat{}, 0, st));
  {
    int64_t tot = (int64_t)rows * T * 32;
    col2im_dact_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(p.dh_a1, p.hproj, p.dh_proj, rows, T, 30, 32, 4, 4, 2, hid(n));
    DWBC_LAUNCH_CHECK();
  }
  // projection
  RowMat G1 = rowmat(p.dh_proj, 32);
  RowMat hist = rowmat_grouped(s->observations + (n.num_obs - T * n.num_prop), idx, T, s->obs_stride, n.num_prop);
  TRY(linear_bwd_weight(G1, hist, grad + n.off_hist_w[0], n.num_prop, grad + n.off_hist_b[0], rows * T, 30, n.num_prop, st));
  hist_unpack_grad_kernel<<<(20 * 128 + 255) / 256, 256, 0, st>>>(p.dhw1, p.dhw2, p.dhwl, grad + n.off_hist_w[1], grad + n.off_hist_w[2],
                                                                   grad + n.off_hist_w[3], L);
  DWBC_LAUNCH_CHECK();
  return DWBC_OK;
}

// Debug / test entry: one GEMM of the selected implementation on plain row-major device matrices.
//   mode 0: Y[M,N] = act(X[M,K] W[N,K]^T + b)      mode 1: dX[M,N] = G[M,K] W[K,N]      mode 2: dW[M,N] += G[K,M]^T X[K,N], db += colsum(G)
extern "C" int dwbc_debug_gemm(int mode, int tc, const float* A, int64_t lda, const float* Bm, int64_t ldb, float* C, int64_t ldc,
                               const float* bias, float* dbias, int M, int N, int K, int act, dwbc_stream_t stream) {
  if (act < 0 || act >= ACT_COUNT) return DWBC_ERR_ARG;
  const int saved = mlp_precision;
  mlp_precision = tc;
  int rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == 0) rc = linear_fwd(rowmat(A, lda), Bm, ldb, bias, C, ldc, M, N, K, act, 0, st);
  else if (mode == 1) rc = linear_bwd_data(rowmat(A, lda), Bm, ldb, C, ldc, M, N, K, ACT_NONE, RowMat{}, 0, st);
  else rc = linear_bwd_weight(rowmat(A, lda), rowmat(Bm, ldb), C, ldc, dbias, K, M, N, st);
  mlp_precision = saved;
  return rc;
}

// tuning aid (tools/update_timing.py): time ratio of a one-tile chain item to half a two-tile item in the work-item planner; <= 0 switches
// the one-tile tail items off
extern "C" int dwbc_debug_set_chain_single_penalty(double v) {
  c2_single_penalty = v;
  return DWBC_OK;
}
// The chain PROGRAMS a call would launch, described without launching anything (host code only, no GPU; every pointer is formed from the
// fake bases below and never dereferenced).  what: 0 = dwbc_policy_act, 1 = dwbc_critic_values, 2 = forward + loss of dwbc_ppo_minibatch_grad,
// 3 = its backward launch.  out = [nprog, pack items, then per program: n_ops, n_loads, then per op: N, kpad, act, fin, fin_c, out_col0,
// has_global_output, output_is_tile_image].  Returns the number of ints written, or a negative error code (DWBC_ERR_UNSUPPORTED: the
// configuration does not run on the fused chains).  tests/test_host_cpu.py pins the program structure with it.
extern "C" int dwbc_debug_describe_chain(const DwbcNetCfg* net, int32_t rows, int what, int hist_encoding, int sms, int32_t* out, int32_t out_len) {
  TRY(check_net(net));
  if (rows <= 0 || what < 0 || what > 3 || sms <= 0 || !out) return DWBC_ERR_ARG;
  const DwbcNetCfg& n = *net;
  float* const ws = reinterpret_cast<float*>(uintptr_t(1) << 40);
  const float* const P = reinterpret_cast<const float*>(uintptr_t(2) << 40);
  const float* const obs = reinterpret_cast<const float*>(uintptr_t(3) << 40);
  const int64_t* const idx = what >= 2 ? reinterpret_cast<const int64_t*>(uintptr_t(4) << 40) : nullptr;
  Plan p = make_plan(n, rows, ws);
  if (!chain_usable(n, p, obs, n.num_obs)) return DWBC_ERR_UNSUPPORTED;
  C2PackList pl{};
  pl.out = p.wpack;
  int64_t off = 0;
  const bool x3 = mlp_precision == 2;
  C2Builder A(&pl, &off, rows, x3), C(&pl, &off, rows, x3), A2(&pl, &off, rows, x3), C2(&pl, &off, rows, x3);
  const C2Prog* prs[4] = {nullptr, nullptr, nullptr, nullptr};
  int nprog = 0;
  const int tiles = (rows + TC_M - 1) / TC_M, zld = (int)align_up(p.latent, 4);
  if (what == 0) {
    const bool split = 4 * tiles <= sms;
    TRY(build_forward(n, P, obs, nullptr, n.num_obs, hist_encoding ? p.zh : nullptr, zld, p, p.value, false, 1, &A, &C, split ? &A2 : nullptr, split ? &C2 : nullptr));
    prs[0] = &A.pr; prs[1] = &C.pr; prs[2] = &A2.pr; prs[3] = &C2.pr;
    nprog = split ? 4 : 2;
  } else if (what == 1) {
    const bool split = 2 * tiles <= sms;
    TRY(build_forward(n, P, obs, nullptr, n.num_obs, nullptr, 0, p, p.value, false, 0, nullptr, &C, nullptr, split ? &C2 : nullptr));
    prs[0] = &C.pr; prs[1] = &C2.pr;
    nprog = split ? 2 : 1;
  } else {
    C2Builder Ab(&pl, &off, rows, x3), Cb(&pl, &off, rows, x3);
    TRY(build_forward(n, P, obs, idx, n.num_obs, nullptr, zld, p, p.value, true, 2, &A, &C));
    TRY(build_backward(n, P, p, Ab, Cb));
    static C2Prog keep[2];                 // (the builders of this branch go out of scope)
    keep[0] = what == 2 ? A.pr : Ab.pr; keep[1] = what == 2 ? C.pr : Cb.pr;
    prs[0] = &keep[0]; prs[1] = &keep[1];
    nprog = 2;
  }
  if (off > C2_PACK_FLOATS) return DWBC_ERR_UNSUPPORTED;
  int k = 0;
  auto put = [&](int v) { if (k < out_len) out[k] = v; ++k; };
  put(nprog); put(pl.n);
  for (int q = 0; q < nprog; ++q) {
    const C2Prog& pr = *prs[q];
    put(pr.n_ops); put(pr.n_loads);
    for (int i = 0; i < pr.n_ops; ++i) {
      const C2Op& o = pr.op[i];
      put(o.N); put(o.kpad); put(o.act); put(o.fin); put(o.fin_c); put(o.out_col0); put(o.y != nullptr); put(o.y_img);
    }
  }
  return k <= out_len ? k : DWBC_ERR_ARG;
}

// The work-item planner of launch_chain2n on its own (host code only, no GPU): for `tiles` row tiles x `nprog` programs of per-two-tile-item
// costs cost[nprog] on `sms` persistent CTAs, the number of two-tile (np2) and one-tile (ns1) items per program it would launch and the
// simulated makespans with (span) and without (span0) one-tile items.  tests/test_host_cpu.py checks coverage and the decision.
extern "C" int dwbc_debug_chain_plan(int tiles, int nprog, const double* cost, int sms, int* np2, int* ns1, double* span, double* span0) {
  if (tiles <= 0 || nprog < 1 || nprog > C2_MAX_PROGS || !cost || sms <= 0 || !np2 || !ns1) return DWBC_ERR_ARG;
  if (tiles * nprog <= sms) { *np2 = 0; *ns1 = tiles; }
  else { *ns1 = c2_pick_singles(tiles, nprog, cost, sms); *np2 = (tiles - *ns1 + 1) / 2; }
  if (span) *span = c2_makespan(tiles, nprog, cost, sms, *np2 ? *ns1 : 0);
  if (span0) *span0 = c2_makespan(tiles, nprog, cost, sms, 0);
  return DWBC_OK;
}
// tuning aid: deal of the grouped weight-gradient work items (1 = sorted + boustrophedon, 0 = round-robin in construction order)
extern "C" int dwbc_debug_set_wgrad_snake(int on) {
  wg_snake = on ? 1 : 0;
  return DWBC_OK;
}
extern "C" int dwbc_debug_set_chain_bwd_reverse(int on) {
  c2_bwd_reverse = on ? 1 : 0;
  return DWBC_OK;
}
extern "C" int dwbc_debug_set_wgrad_reverse(int on) {
  wg_reverse = on ? 1 : 0;
  return DWBC_OK;
}
extern "C" int dwbc_debug_set_wgrad_items(int per_cta) {
  if (per_cta < 1 || per_cta > 64) return DWBC_ERR_ARG;
  wg_items_per_cta = per_cta;
  return DWBC_OK;
}
// tuning aid: force the number of one-tile items per program of the large chain launches (-1: planner)
extern "C" int dwbc_debug_set_chain_singles(int n) {
  c2_force_singles = n;
  return DWBC_OK;
}
extern "C" int dwbc_debug_set_tc_cycle_buffer(unsigned long long* dev_ptr) {
  return cudaMemcpyToSymbol(g_tc_cycles, &dev_ptr, sizeof(dev_ptr)) == cudaSuccess ? DWBC_OK : DWBC_ERR_LAUNCH;
}
extern "C" int dwbc_debug_set_wg_cycle_buffer(unsigned long long* dev_ptr) {
  return cudaMemcpyToSymbol(g_wg_cycles, &dev_ptr, sizeof(dev_ptr)) == cudaSuccess ? DWBC_OK : DWBC_ERR_LAUNCH;
}
