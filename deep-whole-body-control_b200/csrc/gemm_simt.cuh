// fp32 CUDA-core GEMM building block of the ActorCritic path ("precision = fp32" mode; the
// parity anchor for the tensor-core kernels).  One 64x64x16 tile kernel, three operand modes:
//
//   FWD      Y[m,n]  = act( beta*Y + sum_k X[m,k] * W[n,k] + b[n] )            (nn.Linear fwd)
//   BWD_DATA dX[m,n] = ( beta*dX + sum_k G[m,k] * W[k,n] ) * act'(Xact[m,n])   (dgrad, fused act')
//   BWD_WGT  dW[m,n] += sum_k G[k,m] * X[k,n];  db[m] += sum_k G[k,m]          (wgrad, split-K + atomics)
//
// Matrices that are indexed by a *row* (activations, the rollout storage) are described by a
// RowMat, which can gather rows through an index vector (mini-batch gather, RS:189-201, without
// materialising the batch) and can address `rpg` sub-rows per gathered row (the 10x76 history
// block inside an 860-float observation, AC:223-225).
#pragma once
#include "common.cuh"

namespace dwbc {

// activation codes of the layer ops (GemmArgs.act, C2Op.act): the heads' outputs use NONE / TANH, every hidden layer the network's
// DwbcNetCfg.activation (act_code)
enum { ACT_NONE = 0, ACT_ELU = 1, ACT_TANH = 2, ACT_SELU = 3, ACT_RELU = 4, ACT_LRELU = 5, ACT_SIGMOID = 6, ACT_COUNT = 7 };
constexpr float SELU_SCALE = 1.0507009873554805f, SELU_ALPHA = 1.6732632423543772f, LRELU_SLOPE = 0.01f;
// DwbcActivation (ABI) -> activation code; -1: unknown
inline int act_code(int32_t abi_act) {
  switch (abi_act) {
    case DWBC_ACT_ELU: return ACT_ELU;
    case DWBC_ACT_SELU: return ACT_SELU;
    case DWBC_ACT_RELU: return ACT_RELU;
    case DWBC_ACT_LRELU: return ACT_LRELU;
    case DWBC_ACT_TANH: return ACT_TANH;
    case DWBC_ACT_SIGMOID: return ACT_SIGMOID;
    default: return -1;
  }
}

struct RowMat {
  const float* p;       // base (already offset to the first column)
  const int64_t* idx;   // optional gather index over groups
  int rpg;              // rows per group (1 = plain); 0 = "tile image" (below)
  int64_t stride_g;     // floats between groups
  int64_t ld;           // floats between sub-rows of a group
  // rpg == 0: the matrix [rows x 128] is stored as the fused chain kernels keep it in shared memory, one 64 KB image per 128-row tile
  // (mlp_chain2.cuh: element (r, k) of a tile at float ((r/8)*32 + k/4)*32 + (r%8)*4 + k%4), so that a tile leaves / enters the SM as
  // ONE bulk copy.  row() then returns the address of column 0 of the row; 16-byte piece c of the row sits 32*c floats further on.
  __device__ __forceinline__ bool image() const { return rpg == 0; }
  __device__ __forceinline__ const float* row(int64_t r) const {
    if (rpg == 0) return p + (r >> 7) * 16384 + ((r & 127) >> 3) * 1024 + (r & 7) * 4;
    if (rpg == 1) return p + (idx ? idx[r] : r) * stride_g;
    int64_t g = r / rpg, s = r - g * rpg;
    return p + (idx ? idx[g] : g) * stride_g + s * ld;
  }
};
inline RowMat rowmat(const float* p, int64_t ld) { return RowMat{p, nullptr, 1, ld, ld}; }
inline RowMat rowmat_image(const float* p) { return RowMat{p, nullptr, 0, 128, 128}; }
inline RowMat rowmat_gather(const float* p, const int64_t* idx, int64_t stride) { return RowMat{p, idx, 1, stride, stride}; }
inline RowMat rowmat_grouped(const float* p, const int64_t* idx, int rpg, int64_t stride_g, int64_t ld) {
  return RowMat{p, idx, rpg, stride_g, ld};
}

__device__ __forceinline__ float elu_f(float x) { return x > 0.0f ? x : expf(x) - 1.0f; }
// exact fp32 forms (precise expf / tanhf) of every activation, the derivative written in terms of the OUTPUT y = f(x)
__device__ __forceinline__ float act_f(int act, float x) {
  switch (act) {
    case ACT_ELU: return elu_f(x);
    case ACT_TANH: return tanhf(x);
    case ACT_SELU: return x > 0.0f ? SELU_SCALE * x : (SELU_SCALE * SELU_ALPHA) * (expf(x) - 1.0f);
    case ACT_RELU: return fmaxf(x, 0.0f);
    case ACT_LRELU: return x > 0.0f ? x : x * LRELU_SLOPE;
    case ACT_SIGMOID: return 1.0f / (1.0f + expf(-x));
    default: return x;
  }
}
__device__ __forceinline__ float act_dy(int act, float y) {
  switch (act) {
    case ACT_ELU: return y > 0.0f ? 1.0f : y + 1.0f;
    case ACT_TANH: return 1.0f - y * y;
    case ACT_SELU: return y > 0.0f ? SELU_SCALE : y + SELU_SCALE * SELU_ALPHA;
    case ACT_RELU: return y > 0.0f ? 1.0f : 0.0f;
    case ACT_LRELU: return y > 0.0f ? 1.0f : LRELU_SLOPE;
    case ACT_SIGMOID: return y * (1.0f - y);
    default: return 1.0f;
  }
}

constexpr int GT_M = 64, GT_N = 64, GT_K = 16, GT_PAD = 4, GT_THREADS = 256;

enum { GEMM_FWD = 0, GEMM_BWD_DATA = 1, GEMM_BWD_WGT = 2 };

struct GemmArgs {
  RowMat A;             // FWD: X (rows m);  BWD_DATA: G (rows m);  BWD_WGT: G (rows k)
  RowMat B;             // FWD: W (rows n, ld=ldw);  BWD_DATA: W (rows k);  BWD_WGT: X (rows k)
  float* C;             // output, row-major
  int64_t ldc;
  const float* bias;    // FWD only (may be null)
  float* dbias;         // BWD_WGT only (may be null)
  RowMat Xact;          // BWD_DATA: activation OUTPUT whose derivative multiplies dX
  int act;              // FWD: activation;  BWD_DATA: activation whose derivative is applied (ACT_NONE = none)
  int beta;             // 0/1: accumulate onto C (FWD, BWD_DATA)
  int M, N, K;          // C is M x N, reduction length K
  int k_chunk;          // BWD_WGT: reduction rows per CTA (split-K)
};

// tile loaders: S is [GT_K][GT_M + GT_PAD]
// (a) rows of the RowMat run along the tile's M/N axis, columns along K  -> transposed store
template <bool kVec>
__device__ __forceinline__ void load_rows_as_mn(float (*S)[GT_M + GT_PAD], const RowMat& R, int row0, int nrows, int col0, int ncols) {
  const int t = threadIdx.x, r = t >> 2, c = (t & 3) * 4;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (row0 + r < nrows) {
    const float* src = R.row(row0 + r) + col0 + c;
    if (kVec && col0 + c + 3 < ncols) {
      float4 q = *reinterpret_cast<const float4*>(src);
      v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (col0 + c + i < ncols) v[i] = src[i];
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) S[c + i][r] = v[i];
}
// (b) rows of the RowMat run along K, columns along the tile's M/N axis  -> direct store
template <bool kVec>
__device__ __forceinline__ void load_rows_as_k(float (*S)[GT_M + GT_PAD], const RowMat& R, int row0, int nrows, int col0, int ncols) {
  const int t = threadIdx.x, r = t >> 4, c = (t & 15) * 4;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (row0 + r < nrows) {
    const float* src = R.row(row0 + r) + col0 + c;
    if (kVec && col0 + c + 3 < ncols) {
      float4 q = *reinterpret_cast<const float4*>(src);
      v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (col0 + c + i < ncols) v[i] = src[i];
    }
  }
  *reinterpret_cast<float4*>(&S[r][c]) = make_float4(v[0], v[1], v[2], v[3]);
}

template <int kMode, bool kVecA, bool kVecB>
__global__ void __launch_bounds__(GT_THREADS) gemm_tile_kernel(const GemmArgs g) {
  __shared__ __align__(16) float As[2][GT_K][GT_M + GT_PAD];
  __shared__ __align__(16) float Bs[2][GT_K][GT_N + GT_PAD];
  const int m0 = blockIdx.x * GT_M, n0 = blockIdx.y * GT_N;
  int k_begin = 0, k_end = g.K;
  if (kMode == GEMM_BWD_WGT) {
    k_begin = blockIdx.z * g.k_chunk;
    k_end = min(g.K, k_begin + g.k_chunk);
    if (k_begin >= k_end) return;
  }
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

  auto load = [&](int buf, int k0) {
    if (kMode == GEMM_FWD) {
      load_rows_as_mn<kVecA>(As[buf], g.A, m0, g.M, k0, k_end);
      load_rows_as_mn<kVecB>(Bs[buf], g.B, n0, g.N, k0, k_end);
    } else if (kMode == GEMM_BWD_DATA) {
      load_rows_as_mn<kVecA>(As[buf], g.A, m0, g.M, k0, k_end);
      load_rows_as_k<kVecB>(Bs[buf], g.B, k0, k_end, n0, g.N);
    } else {
      load_rows_as_k<kVecA>(As[buf], g.A, k0, k_end, m0, g.M);
      load_rows_as_k<kVecB>(Bs[buf], g.B, k0, k_end, n0, g.N);
    }
  };

  int buf = 0;
  load(0, k_begin);
  __syncthreads();
  for (int k0 = k_begin; k0 < k_end; k0 += GT_K) {
    if (k0 + GT_K < k_end) load(buf ^ 1, k0 + GT_K);
#pragma unroll
    for (int k = 0; k < GT_K; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
    buf ^= 1;
  }

  // ---- epilogue ----
  if (kMode == GEMM_BWD_WGT) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      if (m >= g.M) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        if (n < g.N) atomicAdd(g.C + (int64_t)m * g.ldc + n, acc[i][j]);
      }
    }
    if (g.dbias && blockIdx.y == 0) {
      // column sums of G over this CTA's row chunk: thread t < 64 sums column m0+t
      __shared__ float part[4][GT_M];
      const int col = threadIdx.x & 63, q = threadIdx.x >> 6;
      float s = 0.0f;
      if (m0 + col < g.M)
        for (int k = k_begin + q; k < k_end; k += 4) s += g.A.row(k)[m0 + col];
      part[q][col] = s;
      __syncthreads();
      if (q == 0 && m0 + col < g.M) atomicAdd(g.dbias + m0 + col, (part[0][col] + part[1][col]) + (part[2][col] + part[3][col]));
    }
    return;
  } else {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
    float* crow = g.C + (int64_t)m * g.ldc;
    const float* xrow = (kMode == GEMM_BWD_DATA && g.act != ACT_NONE) ? g.Xact.row(m) : nullptr;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      float v = acc[i][j];
      if (g.beta) v += crow[n];
      if (kMode == GEMM_FWD) {
        if (g.bias) v += g.bias[n];
        if (g.act == ACT_ELU) v = elu_f(v);
        else if (g.act == ACT_TANH) v = tanhf(v);
        else if (g.act != ACT_NONE) v = act_f(g.act, v);
      } else if (xrow) {
        const float y = xrow[n];
        if (g.act == ACT_ELU) v *= (y > 0.0f ? 1.0f : y + 1.0f);
        else if (g.act == ACT_TANH) v *= (1.0f - y * y);
        else v *= act_dy(g.act, y);
      }
      crow[n] = v;
    }
  }
  }
}

inline bool rowmat_vec_ok(const RowMat& r) {
  return ((reinterpret_cast<uintptr_t>(r.p) & 15) == 0) && (r.stride_g % 4 == 0) && (r.ld % 4 == 0);
}

template <int kMode>
inline int launch_gemm(const GemmArgs& g, cudaStream_t st) {
  if (g.M <= 0 || g.N <= 0 || g.K <= 0) return DWBC_ERR_ARG;
  dim3 grid((g.M + GT_M - 1) / GT_M, (g.N + GT_N - 1) / GT_N, 1);
  if (kMode == GEMM_BWD_WGT) grid.z = (g.K + g.k_chunk - 1) / g.k_chunk;
  const bool va = rowmat_vec_ok(g.A), vb = rowmat_vec_ok(g.B);
  if (va && vb) gemm_tile_kernel<kMode, true, true><<<grid, GT_THREADS, 0, st>>>(g);
  else if (va) gemm_tile_kernel<kMode, true, false><<<grid, GT_THREADS, 0, st>>>(g);
  else if (vb) gemm_tile_kernel<kMode, false, true><<<grid, GT_THREADS, 0, st>>>(g);
  else gemm_tile_kernel<kMode, false, false><<<grid, GT_THREADS, 0, st>>>(g);
  ++dwbc_launch_counter;
  return cudaGetLastError() == cudaSuccess ? DWBC_OK : DWBC_ERR_LAUNCH;
}

}  // namespace dwbc
