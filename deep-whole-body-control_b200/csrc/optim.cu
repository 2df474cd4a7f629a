// clip_grad_norm_ + torch.optim.Adam step (PPO:245-246) on the flat parameter buffer (K9), and
// PPO.enforce_min_std (PPO:293-296).  HBM-bound: 7 floats per parameter (28 B) -> 4.7 MB.
#include <math.h>

#include "common.cuh"

namespace dwbc {

__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, int64_t n, float scale, double* __restrict__ out) {
  __shared__ double red[8];
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = g[i] * scale;
    s += (double)v * (double)v;
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[i];
    atomicAdd(out, t);
  }
}

struct AdamArgs {
  float* p; float* g; float* m; float* v;
  int64_t n;
  float scale, max_norm, beta1, beta2, eps, step_size, bc2_sqrt;
  const double* sumsq;
  float* norm_out;
};

__global__ void __launch_bounds__(256) clip_adam_kernel(const AdamArgs a) {
  const float total = (float)sqrt(*a.sumsq);                        // clip_grad_norm_: ||g||_2 over all tensors
  const float coef = fminf(a.max_norm / (total + 1e-6f), 1.0f);
  if (a.norm_out && blockIdx.x == 0 && threadIdx.x == 0) *a.norm_out = total;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (int64_t)gridDim.x * blockDim.x) {
    const float g = (a.g[i] * a.scale) * coef;
    const float m = a.m[i] * a.beta1 + g * (1.0f - a.beta1);
    const float v = a.v[i] * a.beta2 + (g * g) * (1.0f - a.beta2);
    const float denom = sqrtf(v) / a.bc2_sqrt + a.eps;
    a.g[i] = g;  // leave the clipped gradient behind (what .grad holds after PPO:245)
    a.m[i] = m;
    a.v[i] = v;
    a.p[i] = a.p[i] - a.step_size * (m / denom);
  }
}

__global__ void min_std_kernel(float* __restrict__ std, const float* __restrict__ min_std, int n) {
  int i = threadIdx.x;
  if (i < n) std[i] = fmaxf(std[i], min_std[i]);
}

}  // namespace dwbc

using namespace dwbc;

extern "C" int dwbc_clip_adam_step(float* params, float* grad, float* adam_m, float* adam_v, int64_t first, int64_t count,
                                   const DwbcPpoHyper* hp, int32_t step, double* norm_scratch, float* grad_norm_out,
                                   dwbc_stream_t stream) {
  if (!params || !grad || !adam_m || !adam_v || !hp || !norm_scratch || count <= 0 || first < 0 || step < 1) return DWBC_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(norm_scratch, 0, sizeof(double), st) != cudaSuccess) return DWBC_ERR_LAUNCH;
  const float scale = hp->grad_scale == 0.0f ? 1.0f : hp->grad_scale;
  int grid = (int)((count + 1023) / 1024);
  if (grid > 592) grid = 592;
  if (grid < 1) grid = 1;
  sumsq_kernel<<<grid, 256, 0, st>>>(grad + first, count, scale, norm_scratch);
  DWBC_LAUNCH_CHECK();
  const double bc1 = 1.0 - pow((double)hp->beta1, (double)step), bc2 = 1.0 - pow((double)hp->beta2, (double)step);
  AdamArgs a{params + first, grad + first, adam_m + first, adam_v + first, count, scale, hp->max_grad_norm, hp->beta1, hp->beta2,
             hp->adam_eps, (float)((double)hp->lr / bc1), (float)sqrt(bc2), norm_scratch, grad_norm_out};
  clip_adam_kernel<<<grid, 256, 0, st>>>(a);
  DWBC_LAUNCH_CHECK();
  return DWBC_OK;
}

extern "C" int dwbc_enforce_min_std(float* params, int64_t off_std, const float* min_std, int32_t n, dwbc_stream_t stream) {
  if (!params || !min_std || n <= 0 || n > 1024) return DWBC_ERR_ARG;
  min_std_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(params + off_std, min_std, n);
  DWBC_LAUNCH_CHECK();
  return DWBC_OK;
}

unsigned long long dwbc_launch_counter = 0;
extern "C" uint64_t dwbc_launch_count(void) { return dwbc_launch_counter; }

extern "C" const char* dwbc_version(void) { return "dwbc-b200 0.1 (sm_100a, abi 4)"; }

extern "C" void dwbc_struct_sizes(int64_t out[6]) {
  out[0] = sizeof(DwbcEnvCfg); out[1] = sizeof(DwbcEnvBuffers); out[2] = sizeof(DwbcStepArgs);
  out[3] = sizeof(DwbcNetCfg); out[4] = sizeof(DwbcPpoHyper); out[5] = sizeof(DwbcStorage);
}
