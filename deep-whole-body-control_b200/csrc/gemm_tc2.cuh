// Warp-specialised, mbarrier-pipelined tcgen05 GEMM (TF32 in, FP32 accumulate in TMEM) -- the layer-wise tensor-core
// path (history encoder, DAgger update, network shapes the fused chains do not cover).  The three phases of a tile overlap:
//
//   warps 0-3  PRODUCERS : gather + pad the A operand of tile i+1 into shared-memory stage (i+1)%S while ...
//   warp  4    MMA       : ... one thread issues the tcgen05.mma chain of tile i into TMEM accumulator i%2,
//                          tcgen05.commit -> "stage free" and "accumulator full" mbarriers, while ...
//   warps 5-8  EPILOGUE  : ... drain accumulator (i-1)%2 with tcgen05.ld, fuse bias / ELU / tanh / act', store.
//
//   FWD / BWD_DATA: CTA = persistent over 128-row tiles; weights (<= 64 KB) resident in smem; 2 A stages of 64 KB.
//   BWD_WGT      : CTA = one slab of rows; 3 stages of {G^T chunk, X^T chunk} (64 rows each, 32 KB + 32 KB);
//                  one accumulator over the whole slab; split-K partials reduced with global atomics.
//
// The gather index of a tile is prefetched to shared memory first so every operand load is a single round trip,
// and each producer thread keeps 8 independent 16-byte loads in flight.
#pragma once
#include "tc_common.cuh"

namespace dwbc {

constexpr int T2_PROD = 128, T2_EPI = 128;
constexpr int T2_THREADS = T2_PROD + 32 + T2_EPI;   // 288
constexpr int T2_WCH = 64;                          // rows per weight-gradient chunk
constexpr int T2_LDS = TC_MAXN + 4;                 // padded row stride (floats) of the epilogue staging tile: conflict-free float4 rows

__device__ __forceinline__ void t2_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem_u32(bar)) : "memory");
}
// tanh for the TF32 path: 1 - 2/(e^{2x}+1) with ex2.approx / rcp.approx (a few ulp; saturates correctly at +-inf). Short enough that an
// if-converted activation select costs nothing for the ELU layers (precise tanhf is ~60 predicated instructions per element).
__device__ __forceinline__ float t2_tanh(float x) { return 1.0f - __fdividef(2.0f, __expf(2.0f * x) + 1.0f); }
// the other hidden activations on the TF32 paths (ex2.approx / rcp.approx like t2_tanh; ELU and tanh keep their own lines)
__device__ __forceinline__ float t2_act(int act, float x) {
  switch (act) {
    case ACT_SELU: return x > 0.0f ? SELU_SCALE * x : (SELU_SCALE * SELU_ALPHA) * (__expf(x) - 1.0f);
    case ACT_RELU: return fmaxf(x, 0.0f);
    case ACT_LRELU: return x > 0.0f ? x : x * LRELU_SLOPE;
    case ACT_SIGMOID: return __fdividef(1.0f, 1.0f + __expf(-x));
    default: return act_f(act, x);
  }
}
// named barriers are the warp-aligned form: reconverge the warp first (a lane may still be behind a single-lane mbarrier arrive)
__device__ __forceinline__ void t2_pbar() { __syncwarp(); asm volatile("bar.sync 2, %0;" ::"n"(T2_PROD) : "memory"); }   // producers only
__device__ __forceinline__ void t2_ebar() { __syncwarp(); asm volatile("bar.sync 3, %0;" ::"n"(T2_EPI) : "memory"); }    // epilogue only

// profiling aid: clock64 stamps of CTA events, [grid][64] (set with dwbc_debug_set_tc_cycle_buffer)
__device__ unsigned long long* g_tc_cycles = nullptr;
#define T2_STAMP(slot) do { if (g_tc_cycles && (slot) < 64) g_tc_cycles[blockIdx.x * 64 + (slot)] = clock64(); } while (0)

struct T2Shared {
  uint64_t full[3], empty[3], tfull[2], tempty[2];
  uint32_t tmem_base;
  int64_t rowoff[128];     // gathered row offsets (floats) of the tile being filled
  float dbias[128];
};

// K-major fill by the 128 producer threads, rows addressed through a row-offset table in shared memory
__device__ __forceinline__ void t2_fill_rows(float* smem, const float* base, const int64_t* rowoff, int nrows, int rows_pad, int kvalid, int kpad,
                                             bool vec, int ptid) {
  const int chunks = kpad >> 2, total = rows_pad * chunks;
  for (int b0 = ptid; b0 < total; b0 += 8 * T2_PROD) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = b0 + u * T2_PROD;
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < total) {
        const int r8 = i & 7, c = (i >> 3) % chunks, g = (i >> 3) / chunks;
        const int r = g * 8 + r8;
        if (r < nrows) {
          const float* src = base + rowoff[r] + 4 * c;
          if (vec && 4 * c + 3 < kvalid) v[u] = ldg_stream(reinterpret_cast<const float4*>(src));
          else {
            if (4 * c + 0 < kvalid) v[u].x = src[0];
            if (4 * c + 1 < kvalid) v[u].y = src[1];
            if (4 * c + 2 < kvalid) v[u].z = src[2];
            if (4 * c + 3 < kvalid) v[u].w = src[3];
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = b0 + u * T2_PROD;
      if (i < total) *reinterpret_cast<float4*>(smem + (size_t)i * 4) = v[u];
    }
  }
}
// same fill with cp.async (LDGSTS, 16 B, zero-fill): no register staging, so a producer warp keeps its whole share
// of the tile (64 KB per CTA) in flight.  Requires 16-byte aligned rows and kvalid % 4 == 0.
__device__ __forceinline__ void t2_fill_rows_async(float* smem, const float* base, const int64_t* rowoff, int nrows, int rows_pad, int kvalid,
                                                   int kpad, int ptid) {
  const int chunks = kpad >> 2, total = rows_pad * chunks;
  const uint32_t s0 = tc_smem_u32(smem);
  const int r8 = ptid & 7;                       // T2_PROD % 8 == 0: a thread always serves the same row-in-group
  int c = ptid >> 3, g = 0;                      // (i >> 3) = c + g * chunks, advanced incrementally (no divisions)
  while (c >= chunks) { c -= chunks; ++g; }
#pragma unroll 4
  for (int i = ptid; i < total; i += T2_PROD) {
    const int r = g * 8 + r8;
    const float* src = base;
    int nb = 0;
    if (r < nrows && 4 * c < kvalid) { src = base + rowoff[r] + 4 * c; nb = 16; }
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s0 + (uint32_t)i * 16), "l"(src), "r"(nb) : "memory");
    c += T2_PROD >> 3;
    while (c >= chunks) { c -= chunks; ++g; }
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
}
// transposing K-major fill (source indexed [k][mn]); optional column sums of the source into dsum (smem atomics)
__device__ __forceinline__ void t2_fill_T(float* smem, const float* base, const int64_t* rowoff, int nk, int kpad, int mnvalid, int mnpad,
                                          bool vec, int ptid, float* dsum) {
  const int chunks = mnpad >> 2, kq = kpad >> 2, cg = (chunks + 3) >> 2, total = (kpad >> 3) * cg * 32;
  for (int b0 = ptid; b0 < total; b0 += 8 * T2_PROD) {
    float4 v[8];
    int cc[8], kk[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = b0 + u * T2_PROD;
      const int k8 = i & 7, c4 = (i >> 3) & 3, rest = i >> 5;
      const int c = (rest % cg) * 4 + c4, k = (rest / cg) * 8 + k8;
      cc[u] = (i < total && c < chunks) ? c : -1;
      kk[u] = k;
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (cc[u] >= 0 && k < nk) {
        const float* src = base + rowoff[k] + 4 * c;
        if (vec && 4 * c + 3 < mnvalid) v[u] = ldg_stream(reinterpret_cast<const float4*>(src));
        else {
          if (4 * c + 0 < mnvalid) v[u].x = src[0];
          if (4 * c + 1 < mnvalid) v[u].y = src[1];
          if (4 * c + 2 < mnvalid) v[u].z = src[2];
          if (4 * c + 3 < mnvalid) v[u].w = src[3];
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (cc[u] < 0) continue;
      const float vv[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
      const int k = kk[u];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int mn = 4 * cc[u] + j;
        smem[((size_t)((mn >> 3) * kq + (k >> 2)) * 8 + (mn & 7)) * 4 + (k & 3)] = vv[j];
        if (dsum && mn < mnvalid) atomicAdd(dsum + mn, vv[j]);
      }
    }
  }
}

template <int kMode>
__global__ void __launch_bounds__(T2_THREADS, 1) gemm_tc2_kernel(const GemmArgs g, const int items, const int vecA, const int vecB) {
  extern __shared__ __align__(1024) float t2_smem[];
  __shared__ T2Shared sh;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int NST = kMode == GEMM_BWD_WGT ? 3 : 2;

  if (tid == 0) {
    for (int i = 0; i < 3; ++i) {
      tc_mbar_init(&sh.full[i], kMode == GEMM_BWD_WGT ? T2_PROD + T2_EPI : T2_PROD);
      // weight-gradient mode: a stage is released by the MMA commit plus, when a bias gradient is wanted, one lane of each of the 4 epilogue warps
      tc_mbar_init(&sh.empty[i], kMode == GEMM_BWD_WGT ? (g.dbias != nullptr ? 5 : 1) : T2_EPI);
    }
    for (int i = 0; i < 2; ++i) { tc_mbar_init(&sh.tfull[i], 1); tc_mbar_init(&sh.tempty[i], T2_EPI); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) tc_tmem_alloc(&sh.tmem_base, 256);
  if (tid < 128) sh.dbias[tid] = 0.0f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sh.tmem_base;
  if (tid == 0) T2_STAMP(0);
  const int my_items = blockIdx.x < items ? (items - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (kMode != GEMM_BWD_WGT) {
    const int N = g.N, K = g.K;
    const int npad = (N + 15) & ~15, kpad = (K + 7) & ~7;
    float* sB = t2_smem;
    float* sA[2] = {t2_smem + TC_MAXN * TC_MAXK, t2_smem + TC_MAXN * TC_MAXK + TC_M * T2_LDS};   // stages double as epilogue staging [128][132]
    if (warp < 4) {
      // ===================== PRODUCERS =====================
      const int ptid = tid;
      // weight operand once (rows of B are plain: no gather)
      if (kMode == GEMM_FWD) {
        for (int r = ptid; r < 128; r += T2_PROD) sh.rowoff[r] = g.B.row(r < N ? r : 0) - g.B.p;
        t2_pbar();
        if ((vecB & 1) && (K & 3) == 0) t2_fill_rows_async(sB, g.B.p, sh.rowoff, N, npad, K, kpad, ptid);
        else t2_fill_rows(sB, g.B.p, sh.rowoff, N, npad, K, kpad, vecB & 1, ptid);
        if (ptid == 0) T2_STAMP(1);
      } else {
        for (int r = ptid; r < 128; r += T2_PROD) sh.rowoff[r] = g.B.row(r < K ? r : 0) - g.B.p;
        t2_pbar();
        t2_fill_T(sB, g.B.p, sh.rowoff, K, kpad, N, npad, vecB & 1, ptid, nullptr);
      }
      for (int j = 0; j < my_items; ++j) {
        const int it = blockIdx.x + j * gridDim.x, s = j & 1;
        const int64_t m0 = (int64_t)it * TC_M;
        const int rows = (int)min((int64_t)TC_M, (int64_t)g.M - m0);
        t2_pbar();                                        // previous tile's reads of rowoff are done
        if (ptid < TC_M) sh.rowoff[ptid] = ptid < rows ? (g.A.row(m0 + ptid) - g.A.p) : 0;
        tc_mbar_wait(&sh.empty[s], ((j >> 1) & 1) ^ 1);   // stage free (MMA of tile j-2 retired)
        t2_pbar();
        if (!(vecA & 2)) {
          if ((vecA & 1) && (K & 3) == 0) t2_fill_rows_async(sA[s], g.A.p, sh.rowoff, rows, TC_M, K, kpad, ptid);
          else t2_fill_rows(sA[s], g.A.p, sh.rowoff, rows, TC_M, K, kpad, vecA & 1, ptid);
        }
        tc_fence_async_smem();
        t2_arrive(&sh.full[s]);
        if (ptid == 0) T2_STAMP(2 + j);
      }
    } else if (warp == 4) {
      // ===================== MMA ISSUER =====================
      if (lane == 0) {
        const uint32_t idesc = tc_idesc(npad, false, false);
        const uint32_t b0 = tc_smem_u32(sB);
        for (int j = 0; j < my_items; ++j) {
          const int s = j & 1, t = j & 1;
          tc_mbar_wait(&sh.full[s], (j >> 1) & 1);
          tc_mbar_wait(&sh.tempty[t], ((j >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t a0 = tc_smem_u32(sA[s]);
          for (int kk = 0; kk < kpad; kk += 8) {
            const uint64_t ad = tc_desc(a0 + (kk >> 2) * 128, 128, (kpad >> 2) * 128);
            const uint64_t bd = tc_desc(b0 + (kk >> 2) * 128, 128, (kpad >> 2) * 128);
            tc_mma_tf32(tmem + t * 128, ad, bd, idesc, kk > 0 ? 1u : 0u);
          }
          tc_commit(&sh.tfull[t]);      // (the A stage is released by the epilogue, which reuses it as its staging tile)
          T2_STAMP(8 + j);
        }
      }
    } else {
      // ===================== EPILOGUE =====================
      // phase A: TMEM -> registers -> padded staging tile in the (now consumed) A stage;  phase B: warp per row,
      // lane per 4 columns: fully coalesced 512-byte row stores with bias / activation / act' fused.
      const int ew = warp - 5;                       // 0..3
      const int q = warp & 3;                        // TMEM lane quarter this warp may access
      const int rloc = q * 32 + lane;
      const int n4 = 4 * lane;
      float bias4[4] = {0.f, 0.f, 0.f, 0.f};
      if (kMode == GEMM_FWD && g.bias)
        for (int qq = 0; qq < 4; ++qq) if (n4 + qq < N) bias4[qq] = __ldg(g.bias + n4 + qq);
      const bool c_al = ((g.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0);
      for (int j = 0; j < my_items; ++j) {
        const int it = blockIdx.x + j * gridDim.x, t = j & 1, s = j & 1;
        const int64_t m0 = (int64_t)it * TC_M;
        const int rows = (int)min((int64_t)TC_M, (int64_t)g.M - m0);
        float* stg = sA[s];
        tc_mbar_wait(&sh.tfull[t], (j >> 1) & 1);
        tc_fence_after();
        if (tid == 160) T2_STAMP(16 + 4 * j);
        for (int c0 = 0; c0 < npad; c0 += 32) {
          float v[32];
          tc_ld32(tmem + t * 128 + ((uint32_t)(q * 32) << 16) + c0, v);
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4)
            *reinterpret_cast<float4*>(stg + (size_t)rloc * T2_LDS + c0 + 4 * j4) = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
        }
        tc_fence_before();
        t2_arrive(&sh.tempty[t]);                    // accumulator drained: the MMA warp may start tile j+2
        t2_ebar();
        if (tid == 160) T2_STAMP(17 + 4 * j);
        if (!(vecB & 2) && n4 < N) {
          const bool full = n4 + 3 < N;
          for (int r0 = ew; r0 < rows; r0 += 16) {          // 4 independent rows per iteration (ILP over the dependent exp / store chains)
            float x[4][4], y[4][4];
            bool ok[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int r = r0 + 4 * u;
              ok[u] = r < rows;
              const float4 a = ok[u] ? *reinterpret_cast<const float4*>(stg + (size_t)r * T2_LDS + n4) : make_float4(0.f, 0.f, 0.f, 0.f);
              x[u][0] = a.x; x[u][1] = a.y; x[u][2] = a.z; x[u][3] = a.w;
              y[u][0] = y[u][1] = y[u][2] = y[u][3] = 0.f;
              if (!ok[u]) continue;
              const int64_t m = m0 + r;
              if (g.beta) {
                const float* crow = g.C + m * g.ldc + n4;
                if (full && c_al) { const float4 o = *reinterpret_cast<const float4*>(crow); x[u][0] += o.x; x[u][1] += o.y; x[u][2] += o.z; x[u][3] += o.w; }
                else for (int qq = 0; qq < 4; ++qq) if (n4 + qq < N) x[u][qq] += crow[qq];
              }
              if (kMode == GEMM_BWD_DATA && g.act != ACT_NONE) {
                const float* xr = g.Xact.row(m) + n4;
                if (full && ((reinterpret_cast<uintptr_t>(xr) & 15) == 0)) { const float4 o = *reinterpret_cast<const float4*>(xr); y[u][0] = o.x; y[u][1] = o.y; y[u][2] = o.z; y[u][3] = o.w; }
                else for (int qq = 0; qq < 4; ++qq) if (n4 + qq < N) y[u][qq] = xr[qq];
              }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
#pragma unroll
              for (int qq = 0; qq < 4; ++qq) {
                float tt = x[u][qq];
                if (kMode == GEMM_FWD) {
                  tt += bias4[qq];
                  if (vecB & 8) { }
                  else if (g.act == ACT_ELU) tt = tt > 0.0f ? tt : __expf(tt) - 1.0f;   // ex2.approx: 2 ulp, far below the TF32 input rounding
                  else if (g.act == ACT_TANH) tt = t2_tanh(tt);
                  else if (g.act != ACT_NONE) tt = t2_act(g.act, tt);
                } else if (g.act == ACT_ELU) tt *= (y[u][qq] > 0.0f ? 1.0f : y[u][qq] + 1.0f);
                else if (g.act == ACT_TANH) tt *= (1.0f - y[u][qq] * y[u][qq]);
                else if (g.act != ACT_NONE) tt *= act_dy(g.act, y[u][qq]);
                x[u][qq] = tt;
              }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              if (!ok[u] || (vecB & 4)) continue;
              float* crow = g.C + (m0 + r0 + 4 * u) * g.ldc + n4;
              if (full && c_al) *reinterpret_cast<float4*>(crow) = make_float4(x[u][0], x[u][1], x[u][2], x[u][3]);
              else for (int qq = 0; qq < 4; ++qq) if (n4 + qq < N) crow[qq] = x[u][qq];
            }
          }
        }
        t2_ebar();
        if (tid == 160) T2_STAMP(18 + 4 * j);
        t2_arrive(&sh.empty[s]);                     // staging (= A stage s) free for the producers
      }
    }
  } else {
    // ---------------- weight gradient ---------------------------------------------------------------------------------
    // D[out x in] += G^T X over this CTA's slab of rows, 64 rows per chunk.  The contraction index is the ROW of the
    // row-major sources, i.e. both operands are "MN-major".  For 32-bit operands tcgen05 supports exactly one MN-major
    // shared-memory layout, SWIZZLE_128B_BASE32B (layout type 1; verified on B200 with tools/probes/mn_probe.cu; the
    // no-swizzle MN-major form silently yields zeros for kind::tf32):
    //   atom = 4 rows (k) x 32 features (128 B per row), 32-byte chunk c of row r stored at chunk c ^ (r & 3);
    //   feature-atom stride (LBO) 512 B, row-atom stride (SBO) 4 x 512 B.
    // A 16-byte piece of a source row stays a 16-byte piece, so the producers cp.async rows straight from global
    // memory into the operand tiles: no transposition pass.
    //   warps 0-3 : cp.async producers (3 stages of {G tile, X tile}, 32 KB each);
    //   warp  4   : 8 tcgen05.mma (K = 8 rows each) per chunk into one TMEM accumulator;
    //   warps 5-8 : bias gradient (column sums of the G tile, conflict-free LDS), then the split-K epilogue (atomics).
    const int Mo = g.M, Ni = g.N;
    const int nipad = (Ni + 15) & ~15;
    constexpr int TILE = T2_WCH * 128;                // floats per operand tile: 64 rows x 128 features
    const int64_t k_begin = (int64_t)blockIdx.x * g.k_chunk;      // one slab per CTA (grid == items)
    const int64_t k_end = min((int64_t)g.K, k_begin + g.k_chunk);
    const int nch = (int)((k_end - k_begin + T2_WCH - 1) / T2_WCH);
    // all eight non-MMA warps issue the operand copies (the copy issue rate of four warps was the bottleneck); the four
    // epilogue warps additionally sum the bias gradient of the PREVIOUS chunk after issuing the current one.
    auto fill_chunk = [&](int c, int pt) {
      const bool fastA = (vecA & 1) && (Mo & 3) == 0, fastB = (vecB & 1) && (Ni & 3) == 0;
      const int s = c % 3;
      const int64_t k0 = k_begin + (int64_t)c * T2_WCH;
      const int nk = (int)min((int64_t)T2_WCH, k_end - k0);
      asm volatile("bar.sync 4, 256;" ::: "memory");      // row-offset table of the previous chunk no longer read
      if (pt < T2_WCH) sh.rowoff[pt] = pt < nk ? (g.A.row(k0 + pt) - g.A.p) : 0;
      else if (pt < 2 * T2_WCH) sh.rowoff[pt] = (pt - T2_WCH) < nk ? (g.B.row(k0 + pt - T2_WCH) - g.B.p) : 0;
      tc_mbar_wait(&sh.empty[s], ((c / 3) & 1) ^ 1);
      asm volatile("bar.sync 4, 256;" ::: "memory");
      for (int op = 0; op < 2; ++op) {
        float* dst = t2_smem + (2 * s + op) * TILE;
        const float* base = op == 0 ? g.A.p : g.B.p;
        const int64_t* ro = sh.rowoff + 64 * op;
        const int ncol = op == 0 ? Mo : Ni;
        if (op == 0 ? fastA : fastB) {
          const int cpr = ncol >> 2;                          // 16-byte pieces per row
          const uint32_t d0 = tc_smem_u32(dst);
          const bool pow2 = (cpr & (cpr - 1)) == 0;
          const int sh2 = 31 - __clz(cpr);
          for (int i = pt; i < T2_WCH * cpr; i += 256) {
            const int k = pow2 ? (i >> sh2) : i / cpr, cc = i - k * cpr;          // row, piece
            const float* src = k < nk ? base + ro[k] + 4 * cc : base;
            const uint32_t off = (uint32_t)((cc >> 3) * 512 + (k >> 2) * 2048 + (k & 3) * 128 + ((((cc >> 1) & 3) ^ (k & 3)) << 5) + ((cc & 1) << 4));
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d0 + off), "l"(src), "r"(k < nk ? 16 : 0) : "memory");
          }
        } else {
          for (int i = pt; i < T2_WCH * ncol; i += 256) {
            const int k = i / ncol, f = i - k * ncol;
            const int off = ((f >> 5) * 512 + (k >> 2) * 2048 + (k & 3) * 128 + (((((f & 31) >> 3)) ^ (k & 3)) << 5) + ((f & 7) << 2)) >> 2;
            dst[off] = k < nk ? base[ro[k] + f] : 0.0f;
          }
        }
      }
      // asynchronous arrival: the stage is signalled when this thread's copies have landed, the thread moves on
      asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(tc_smem_u32(&sh.full[s])) : "memory");
    };
    if (warp < 4) {
      for (int c = 0; c < nch; ++c) {
        fill_chunk(c, tid);
        if (tid == 0) T2_STAMP(1 + c);
      }
    } else if (warp == 4) {
      if (lane == 0) {
        const uint32_t idesc = tc_idesc(nipad, true, true);
        for (int c = 0; c < nch; ++c) {
          const int s = c % 3;
          tc_mbar_wait(&sh.full[s], (c / 3) & 1);
          tc_fence_async_smem();          // generic-proxy writes of the producers (made visible by the barrier) -> async proxy reads of the MMA
          tc_fence_after();
          const uint32_t a0 = tc_smem_u32(t2_smem + (2 * s) * TILE), b0 = a0 + TILE * 4;
          for (int kk = 0; kk < T2_WCH; kk += 8) {
            const uint64_t ad = tc_desc(a0 + (kk >> 2) * 2048, 512, 2048) | ((uint64_t)1 << 61);
            const uint64_t bd = tc_desc(b0 + (kk >> 2) * 2048, 512, 2048) | ((uint64_t)1 << 61);
            tc_mma_tf32(tmem, ad, bd, idesc, (c > 0 || kk > 0) ? 1u : 0u);
          }
          tc_commit(&sh.empty[s]);
          T2_STAMP(16 + c);
        }
        tc_commit(&sh.tfull[0]);
      }
    } else {
      const int et = tid - (T2_PROD + 32);             // 0..127: output feature whose bias gradient / accumulator row this thread owns
      const int q = warp & 3;
      float bsum = 0.0f;
      const int fo = (et >> 5) * 128 + (et & 7);       // float offset of feature et inside row 0 of its atom (before the chunk swizzle)
      const int c32 = (et & 31) >> 3;
      auto bias_chunk = [&](int c) {
        const int s = c % 3;
        tc_mbar_wait(&sh.full[s], (c / 3) & 1);
        const float* gt = t2_smem + (2 * s) * TILE;
        if (et < Mo) {
#pragma unroll 8
          for (int k = 0; k < T2_WCH; ++k) bsum += gt[fo + (k >> 2) * 512 + (k & 3) * 32 + ((c32 ^ (k & 3)) << 3)];
        }
        __syncwarp();
        if (lane == 0) t2_arrive(&sh.empty[s]);
      };
      for (int c = 0; c < nch; ++c) {
        fill_chunk(c, T2_PROD + et);
        if (g.dbias != nullptr && c > 0) bias_chunk(c - 1);
      }
      if (g.dbias != nullptr && nch > 0) bias_chunk(nch - 1);
      if (nch > 0) {
        if (et == 0) T2_STAMP(32);
        if (g.dbias && et < Mo) atomicAdd(g.dbias + et, bsum);
        const int o = q * 32 + lane;
        tc_mbar_wait(&sh.tfull[0], 0);
        tc_fence_after();
        if (et == 0) T2_STAMP(33);
        t2_ebar();                                      // every epilogue warp is done reading G tiles (bias gradient) before the stages are reused
        // all MMAs have completed: the operand stages are free and become the staging tile [128][132], so that the split-K
        // reduction goes out as row-contiguous vector reductions (one 512-byte row per warp instruction) instead of 32 lines per instruction
        float* stg = t2_smem;
        for (int c0 = 0; c0 < nipad; c0 += 32) {
          float v[32];
          tc_ld32(tmem + ((uint32_t)(q * 32) << 16) + c0, v);
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4)
            *reinterpret_cast<float4*>(stg + (size_t)o * T2_LDS + c0 + 4 * j4) = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
        }
        __syncwarp();                                   // warp q wrote rows q*32 .. q*32+31 and reduces exactly those rows
        const bool v4 = (g.ldc & 3) == 0 && (Ni & 3) == 0 && (reinterpret_cast<uintptr_t>(g.C) & 15) == 0;
        for (int r = q * 32; r < min(q * 32 + 32, Mo); ++r) {
          float* crow = g.C + (int64_t)r * g.ldc;
          if (v4) {
            if (4 * lane < Ni) {
              const float4 a = *reinterpret_cast<const float4*>(stg + (size_t)r * T2_LDS + 4 * lane);
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(crow + 4 * lane), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w) : "memory");
            }
          } else {
            for (int n = lane; n < Ni; n += 32) atomicAdd(crow + n, stg[(size_t)r * T2_LDS + n]);
          }
        }
        tc_fence_before();
        if (et == 0) T2_STAMP(34);
      }
    }
  }
  __syncthreads();
  if (warp == 4) tc_tmem_dealloc(tmem, 256);
}

extern int tc_debug;   // profiling switches: 2 = skip A fills, 4 = skip epilogue global traffic (results invalid)

template <int kMode>
inline int launch_gemm_tc2(const GemmArgs& g_in, cudaStream_t st) {
  GemmArgs g = g_in;
  if (g.M <= 0 || g.N <= 0 || g.K <= 0) return DWBC_ERR_ARG;
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  int items, grid;
  if (kMode == GEMM_BWD_WGT) {
    int64_t chunk = (g.K + sms - 1) / sms;
    chunk = (chunk + T2_WCH - 1) / T2_WCH * T2_WCH;
    if (chunk < T2_WCH) chunk = T2_WCH;
    g.k_chunk = (int)chunk;
    items = (int)((g.K + chunk - 1) / chunk);
    grid = items;
  } else {
    items = (g.M + TC_M - 1) / TC_M;
    grid = items < sms ? items : sms;
  }
  const size_t smem = (size_t)(TC_MAXN * TC_MAXK + 2 * TC_M * T2_LDS) * sizeof(float);   // 196 KB: {B, A0, A1 (padded)} or 3 x {G^T, X^T} chunks
  static bool attr[3] = {false, false, false};
  if (!attr[kMode]) {
    if (cudaFuncSetAttribute(gemm_tc2_kernel<kMode>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return DWBC_ERR_LAUNCH;
    attr[kMode] = true;
  }
  gemm_tc2_kernel<kMode><<<grid, T2_THREADS, smem, st>>>(g, items, (rowmat_vec_ok(g.A) ? 1 : 0) | (tc_debug & 2), (rowmat_vec_ok(g.B) ? 1 : 0) | ((tc_debug & 4) >> 1) | ((tc_debug & 24) >> 1));
  ++dwbc_launch_counter;
  return cudaGetLastError() == cudaSuccess ? DWBC_OK : DWBC_ERR_LAUNCH;
}

// precision of the ActorCritic GEMMs of the current call (defined in mlp.cu): 0 = fp32 CUDA cores (parity anchor), 1 = TF32 tcgen05,
// 2 = 3xTF32: the fused chain / grouped weight-gradient kernels compensate the truncation; these layer-wise GEMMs (history encoder,
// DAgger) then run on the exact fp32 kernels
extern thread_local int mlp_precision;

template <int kMode>
inline int dispatch_gemm(const GemmArgs& g, cudaStream_t st) {
  if (mlp_precision == 1 && tc_shape_ok(kMode, g)) return launch_gemm_tc2<kMode>(g, st);
  return launch_gemm<kMode>(g, st);
}

// Y = act(beta*Y + X W^T + b)
inline int linear_fwd(RowMat X, const float* W, int64_t ldw, const float* b, float* Y, int64_t ldy, int M, int N, int K,
                      int act, int beta, cudaStream_t st) {
  GemmArgs g{};
  g.A = X; g.B = rowmat(W, ldw); g.C = Y; g.ldc = ldy; g.bias = b; g.act = act; g.beta = beta; g.M = M; g.N = N; g.K = K;
  return dispatch_gemm<GEMM_FWD>(g, st);
}
// dX[M x Nin] = (beta*dX + G[M x Nout] W[Nout x Nin]) * act'(Xact)
inline int linear_bwd_data(RowMat G, const float* W, int64_t ldw, float* dX, int64_t lddx, int M, int Nin, int Nout,
                           int act, RowMat Xact, int beta, cudaStream_t st) {
  GemmArgs g{};
  g.A = G; g.B = rowmat(W, ldw); g.C = dX; g.ldc = lddx; g.act = act; g.Xact = Xact; g.beta = beta; g.M = M; g.N = Nin; g.K = Nout;
  return dispatch_gemm<GEMM_BWD_DATA>(g, st);
}
// dW[Nout x Nin] += G^T X ; db += colsum(G)   (over `rows` rows)
inline int linear_bwd_weight(RowMat G, RowMat X, float* dW, int64_t lddw, float* db, int rows, int Nout, int Nin, cudaStream_t st) {
  GemmArgs g{};
  g.A = G; g.B = X; g.C = dW; g.ldc = lddw; g.dbias = db; g.M = Nout; g.N = Nin; g.K = rows;
  int tiles = ((Nout + GT_M - 1) / GT_M) * ((Nin + GT_N - 1) / GT_N);
  int splits = (592 + tiles - 1) / tiles;                 // ~4 CTAs per SM over the whole grid
  int chunk = (rows + splits - 1) / splits;
  chunk = ((chunk + GT_K - 1) / GT_K) * GT_K;
  if (chunk < 64) chunk = 64;
  g.k_chunk = chunk;
  return dispatch_gemm<GEMM_BWD_WGT>(g, st);
}

}  // namespace dwbc
