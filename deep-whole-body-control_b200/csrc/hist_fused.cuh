// History encoder (StateHistoryEncoder, AC:39-84: Linear 76->30 + act per time step, Conv1d(30->20, k=4, s=2) + act, Conv1d(20->10, k=2, s=1) + act,
// Flatten, Linear 30->latent + act; act = the network's hidden activation, ELU in the shipped config) as ONE exact-fp32 kernel for the inference uses: the regulariser target of PPO.update (PPO:175-176, no
// gradient), rollouts with hist_encoding (AC:207-210) and act_inference.  The layer-wise path needs four GEMM launches plus packing / padding
// kernels and moves the [rows x 10 x 32] projection through HBM; here a thread owns a row, streams its 10 x 76 history once (the only HBM
// traffic: 3 040 B per row), and keeps every intermediate in registers:
//   * weights sit in shared memory transposed to [input][output], so one 16-byte broadcast load feeds four FMAs of four outputs;
//   * the strided convolution is accumulated as the time steps arrive: step t feeds tap t - 2p of the (at most two) open output positions
//     p = t/2 and p - 1, so no window of projected steps is kept and every register array is indexed with compile-time constants;
//   * the second convolution and the output layer consume a finished conv-1 position immediately.
// 34 200 FMA per row on the fp32 pipe (the 3xTF32 mode uses it too: exact fp32, no tensor-core split needed for 4 % of the flops).
#pragma once
#include "gemm_simt.cuh"

namespace dwbc {

constexpr int HF_THREADS = 128;
// shared-memory image (floats): Wp[76][32] bp[32] | W1[4*30][20] b1[20] | W2[2*20][12] b2[12] | Wl[3*10][32] bl[32]
constexpr int HF_WP = 0, HF_BP = 76 * 32, HF_W1 = HF_BP + 32, HF_B1 = HF_W1 + 120 * 20, HF_W2 = HF_B1 + 20, HF_B2 = HF_W2 + 40 * 12, HF_WL = HF_B2 + 12,
              HF_BL = HF_WL + 30 * 32, HF_FLOATS = HF_BL + 32;

struct HistFusedArgs {
  const float* wp; const float* bp;     // encoder.0          [30][76], [30]
  const float* w1; const float* b1;     // conv_layers.0      [20][30][4], [20]
  const float* w2; const float* b2;     // conv_layers.2      [10][20][2], [10]
  const float* wl; const float* bl;     // linear_output.0    [latent][30] over the channel-major flatten (c2*3 + t), [latent]
  RowMat hist;                          // row r -> first float of its [10][76] history block
  float* out; int64_t ld_out;           // [rows, ld_out]; columns [latent, ld_out) are zero-filled
  int rows, latent;
};

// the hidden activation, precise expf / tanhf: this is the exact path.  One kernel per activation (kAct is a compile-time constant,
// so the ELU instance is the plain ELU line)
template <int kAct>
__device__ __forceinline__ float hf_act(float x) { return kAct == ACT_ELU ? (x > 0.0f ? x : expf(x) - 1.0f) : act_f(kAct, x); }

template <int kAct>
__global__ void __launch_bounds__(HF_THREADS) hist_fused_kernel(const HistFusedArgs a) {
  __shared__ __align__(16) float w[HF_FLOATS];
  // ---- weights -> shared memory, transposed to [input][output] (pads zero) ----
  for (int i = threadIdx.x; i < HF_FLOATS; i += HF_THREADS) {
    float v = 0.0f;
    if (i < HF_BP) { const int in = i >> 5, o = i & 31; if (o < 30) v = a.wp[o * 76 + in]; }
    else if (i < HF_W1) { const int o = i - HF_BP; if (o < 30) v = a.bp[o]; }
    else if (i < HF_B1) { const int j = i - HF_W1, row = j / 20, o = j - row * 20, k = row / 30, c = row - k * 30; v = a.w1[(o * 30 + c) * 4 + k]; }
    else if (i < HF_W2) v = a.b1[i - HF_B1];
    else if (i < HF_B2) { const int j = i - HF_W2, row = j / 12, o = j - row * 12, k = row / 20, c = row - k * 20; if (o < 10) v = a.w2[(o * 20 + c) * 2 + k]; }
    else if (i < HF_WL) { const int o = i - HF_B2; if (o < 10) v = a.b2[o]; }
    else if (i < HF_BL) { const int j = i - HF_WL, row = j >> 5, o = j & 31, t = row / 10, c = row - t * 10; if (o < a.latent) v = a.wl[o * 30 + c * 3 + t]; }
    else { const int o = i - HF_BL; if (o < a.latent) v = a.bl[o]; }
    w[i] = v;
  }
  __syncthreads();
  const int r = blockIdx.x * HF_THREADS + threadIdx.x;
  if (r >= a.rows) return;
  const float* hp = a.hist.row(r);
  float c1a[20], c1b[20], c1prev[20], z[32];
#pragma unroll
  for (int o = 0; o < 20; ++o) { c1a[o] = 0.0f; c1b[o] = w[HF_B1 + o]; c1prev[o] = 0.0f; }
#pragma unroll
  for (int o = 0; o < 32; ++o) z[o] = w[HF_BL + o];
  float4 xnext = __ldg(reinterpret_cast<const float4*>(hp));
#pragma unroll 1
  for (int t = 0; t < 10; ++t) {
    // ---- projection of step t: h = act(Wp x + bp) ----
    float h[32];
#pragma unroll
    for (int o = 0; o < 32; ++o) h[o] = w[HF_BP + o];
    // (the whole [10][76] block of a row is contiguous: the next 16 bytes -- of this step or the first of the next one -- are requested
    // before the 128 FMAs of the current four inputs, so a thread always has one load in flight instead of waiting for each in turn)
    const float4* x4p = reinterpret_cast<const float4*>(hp + t * 76);
#pragma unroll 1
    for (int i4 = 0; i4 < 19; ++i4) {
      const float4 x4 = xnext;
      if (t * 19 + i4 + 1 < 190) xnext = __ldg(x4p + i4 + 1);
      const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float4* wr = reinterpret_cast<const float4*>(w + HF_WP + (4 * i4 + e) * 32);
#pragma unroll
        for (int o4 = 0; o4 < 8; ++o4) {
          const float4 w4 = wr[o4];
          h[4 * o4] = fmaf(w4.x, xs[e], h[4 * o4]); h[4 * o4 + 1] = fmaf(w4.y, xs[e], h[4 * o4 + 1]);
          h[4 * o4 + 2] = fmaf(w4.z, xs[e], h[4 * o4 + 2]); h[4 * o4 + 3] = fmaf(w4.w, xs[e], h[4 * o4 + 3]);
        }
      }
    }
#pragma unroll
    for (int o = 0; o < 30; ++o) h[o] = hf_act<kAct>(h[o]);
    // ---- conv 1: step t is tap (t & 1) + 2 of position p - 1 and tap t & 1 of position p = t / 2 ----
    const int kb = t & 1, ka = kb + 2;
    if (t >= 2) {
      const float* wk = w + HF_W1 + ka * 30 * 20;
#pragma unroll
      for (int c = 0; c < 30; ++c) {
        const float4* wr = reinterpret_cast<const float4*>(wk + c * 20);
#pragma unroll
        for (int o4 = 0; o4 < 5; ++o4) {
          const float4 w4 = wr[o4];
          c1a[4 * o4] = fmaf(w4.x, h[c], c1a[4 * o4]); c1a[4 * o4 + 1] = fmaf(w4.y, h[c], c1a[4 * o4 + 1]);
          c1a[4 * o4 + 2] = fmaf(w4.z, h[c], c1a[4 * o4 + 2]); c1a[4 * o4 + 3] = fmaf(w4.w, h[c], c1a[4 * o4 + 3]);
        }
      }
    }
    if (t <= 7) {
      const float* wk = w + HF_W1 + kb * 30 * 20;
#pragma unroll
      for (int c = 0; c < 30; ++c) {
        const float4* wr = reinterpret_cast<const float4*>(wk + c * 20);
#pragma unroll
        for (int o4 = 0; o4 < 5; ++o4) {
          const float4 w4 = wr[o4];
          c1b[4 * o4] = fmaf(w4.x, h[c], c1b[4 * o4]); c1b[4 * o4 + 1] = fmaf(w4.y, h[c], c1b[4 * o4 + 1]);
          c1b[4 * o4 + 2] = fmaf(w4.z, h[c], c1b[4 * o4 + 2]); c1b[4 * o4 + 3] = fmaf(w4.w, h[c], c1b[4 * o4 + 3]);
        }
      }
    }
    if (t & 1) {
      if (t >= 3) {
        // position q = (t - 3) / 2 of conv 1 is complete
        const int q = (t - 3) >> 1;
#pragma unroll
        for (int o = 0; o < 20; ++o) c1a[o] = hf_act<kAct>(c1a[o]);
        if (q >= 1) {
          // conv 2 position q - 1 = taps (c1[q-1], c1[q]); then its share of the output layer
          float c2[12];
#pragma unroll
          for (int o = 0; o < 12; ++o) c2[o] = w[HF_B2 + o];
#pragma unroll
          for (int c = 0; c < 20; ++c) {
            const float4* w0 = reinterpret_cast<const float4*>(w + HF_W2 + c * 12);
            const float4* w1 = reinterpret_cast<const float4*>(w + HF_W2 + (20 + c) * 12);
#pragma unroll
            for (int o4 = 0; o4 < 3; ++o4) {
              const float4 u = w0[o4], v = w1[o4];
              c2[4 * o4] = fmaf(v.x, c1a[c], fmaf(u.x, c1prev[c], c2[4 * o4])); c2[4 * o4 + 1] = fmaf(v.y, c1a[c], fmaf(u.y, c1prev[c], c2[4 * o4 + 1]));
              c2[4 * o4 + 2] = fmaf(v.z, c1a[c], fmaf(u.z, c1prev[c], c2[4 * o4 + 2])); c2[4 * o4 + 3] = fmaf(v.w, c1a[c], fmaf(u.w, c1prev[c], c2[4 * o4 + 3]));
            }
          }
          const float* wl = w + HF_WL + (q - 1) * 10 * 32;
#pragma unroll
          for (int c = 0; c < 10; ++c) {
            const float cv = hf_act<kAct>(c2[c]);
            const float4* wr = reinterpret_cast<const float4*>(wl + c * 32);
#pragma unroll
            for (int o4 = 0; o4 < 8; ++o4) {
              const float4 w4 = wr[o4];
              z[4 * o4] = fmaf(w4.x, cv, z[4 * o4]); z[4 * o4 + 1] = fmaf(w4.y, cv, z[4 * o4 + 1]);
              z[4 * o4 + 2] = fmaf(w4.z, cv, z[4 * o4 + 2]); z[4 * o4 + 3] = fmaf(w4.w, cv, z[4 * o4 + 3]);
            }
          }
        }
#pragma unroll
        for (int o = 0; o < 20; ++o) c1prev[o] = c1a[o];
      }
#pragma unroll
      for (int o = 0; o < 20; ++o) { c1a[o] = c1b[o]; c1b[o] = w[HF_B1 + o]; }
    }
  }
  float* orow = a.out + (int64_t)r * a.ld_out;
#pragma unroll
  for (int o = 0; o < 32; ++o)
    if (o < a.ld_out) orow[o] = o < a.latent ? hf_act<kAct>(z[o]) : 0.0f;
}

// latent <= 32, ld_out <= 32, history rows 16-byte aligned
inline int launch_hist_fused(const HistFusedArgs& a, int act, cudaStream_t st) {
  if (a.rows <= 0 || a.latent > 32 || a.ld_out > 32 || a.ld_out < a.latent) return DWBC_ERR_UNSUPPORTED;
  const unsigned grid = (a.rows + HF_THREADS - 1) / HF_THREADS;
  switch (act) {
    case ACT_ELU: hist_fused_kernel<ACT_ELU><<<grid, HF_THREADS, 0, st>>>(a); break;
    case ACT_SELU: hist_fused_kernel<ACT_SELU><<<grid, HF_THREADS, 0, st>>>(a); break;
    case ACT_RELU: hist_fused_kernel<ACT_RELU><<<grid, HF_THREADS, 0, st>>>(a); break;
    case ACT_LRELU: hist_fused_kernel<ACT_LRELU><<<grid, HF_THREADS, 0, st>>>(a); break;
    case ACT_TANH: hist_fused_kernel<ACT_TANH><<<grid, HF_THREADS, 0, st>>>(a); break;
    case ACT_SIGMOID: hist_fused_kernel<ACT_SIGMOID><<<grid, HF_THREADS, 0, st>>>(a); break;
    default: return DWBC_ERR_ARG;
  }
  ++dwbc_launch_counter;
  return cudaGetLastError() == cudaSuccess ? DWBC_OK : DWBC_ERR_LAUNCH;
}

}  // namespace dwbc
