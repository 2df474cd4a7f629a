// Fused layer chains of the ActorCritic (AC:86-353) on the tcgen05 tensor cores, second generation.
//
// What changed against the first chain kernel (round 1: one 128-row tile per CTA, strict MMA -> epilogue -> MMA):
//   * TWO row tiles in flight per CTA (slots X and Y).  Each slot owns ONE operand tile in shared memory that every op
//     updates in place, one accumulator in TMEM and (error-compensated mode) one TMEM region for the low parts of its
//     operand.  The MMA thread issues  X.op_n, Y.op_n, X.op_n+1, ...  and the sixteen epilogue warps drain X.op_n while the
//     tensor core works on Y.op_n: the serial chain of one tile is hidden behind the other tile.
//   * Both slots run the same program, so one weight image per op serves two tiles (half the L2 traffic per tile).
//   * The trunk a second head needs is re-read from the activation buffer the backward pass needs anyway (L2 hit) instead
//     of occupying a second shared-memory tile -- that is what makes room for the second slot.
//   * "3xTF32" (precision 2): x = hi + lo with hi = the 19 leading bits the tensor core reads (kind::tf32 TRUNCATES the
//     13 low mantissa bits of a 32-bit operand -- measured, tools/probes/ts_probe.cu) and lo = x - hi (exact in fp32).
//     D = A_hi W_hi + A_lo W_hi + A_hi W_lo: the first and third products read the fp32 tile / the raw and the "lo" weight
//     image from shared memory, the second reads A_lo from TMEM (tcgen05.mma with the A operand in tensor memory), written
//     there by the epilogue that produced A.  The dropped A_lo W_lo term is 2^-22 relative: fp32-grade results.
//   * The heads' epilogues finish the job (north_star: "log-prob, ratio/clip/min and entropy fused into the epilogue"):
//     rollout: action sampling + two-channel Gaussian log-prob (AC:326-345); update: PPO surrogate / clipped value loss /
//     entropy / privileged-latent regulariser and their gradients w.r.t. the network outputs (PPO:166-221).
//   * Work items (program, tile pair) are handed out through an atomic queue (longest program first).
//
// Tile geometry (unchanged): [128 rows x 128 k] fp32, element (r, k) at float ((r/8)*32 + k/4)*32 + (r%8)*4 + k%4
// (8-row x 16-byte core matrices, LBO = 128 B, SBO = 4096 B).  TMEM: slot s owns columns [256 s, 256 s + 256):
// accumulator D at +0 (lane = row, column = output feature), A_lo at +128 (lane = row, column = k).
#pragma once
#include <stdlib.h>

#include <algorithm>
#include <functional>
#include <vector>

#include "gemm_tc2.cuh"

namespace dwbc {

constexpr int C2_MAX_OPS = 12, C2_MAX_LOADS = 6, C2_MAX_PACK = 36, C2_MAX_PROGS = 4;   // pack items of one launch: forward + backward programs of both networks
constexpr int C2_TILE = 128 * 128;                       // floats per operand tile
constexpr int C2_WORKERS = 8;                            // epilogue / load warps: lane quarter = warp % 4, column group = warp / 4
constexpr int C2_H = C2_WORKERS / 4;                     // column groups: a warp takes the 32-column chunks ci with ci % C2_H == its group
constexpr int C2_CPW = 4 / C2_H;                         // chunks per warp and op (N <= 128).  Eight warps (+ the MMA warp) leave 224 registers per
                                                         // thread: two chunks of accumulator, activation and low-part values stay in registers (with
                                                         // sixteen warps the 96-register cap spilled ~1 KB per thread and the epilogue ran from local memory)
constexpr int C2_THREADS = 32 * (C2_WORKERS + 1);        // + the MMA warp (warp 16)
constexpr int C2_NW = 32 * C2_WORKERS;                   // 512 worker threads
constexpr int C2_SMEM_FLOATS = 3 * C2_TILE + 2 * 128;    // tile X, tile Y, weight image, two bias slots

enum { FIN_NONE = 0, FIN_ACT = 1, FIN_PPO = 2, FIN_VALUE = 3, FIN_REG = 4 };

struct C2Load {
  RowMat src;        // rows of the source (already offset to the first column)
  int ncols;         // columns copied (multiple of 4)
  int col0;          // destination column (multiple of 4)
  int zero_to;       // columns [col0 + ncols, zero_to) are zero-filled (K padding of the consuming op)
  int before_op;     // issued once the ops < before_op of the slot have retired (0: with the item)
  int img;           // 1: src.p is a tile-image buffer (RowMat::image): the whole 128 x 128 tile arrives as ONE bulk copy (ncols = 128, col0 = 0)
};
struct C2Op {
  const float* wp;       // packed image: canonical K-major [npad x kpad] weights, then [npad] bias
  const float* wp_lo;    // 3xTF32: image of the low parts (no bias); null otherwise
  float* y;              // global output (nullable), row-major
  int64_t ldy;
  int a_col0, kpad;      // first column of the A window inside the tile (multiple of 4), padded reduction length (multiple of 8)
  int N, npad;           // outputs (npad: multiple of 16)
  int act;               // forward: activation; backward: activation whose derivative multiplies
  int out_col0;          // column of the tile the result is written to (multiple of 32), -1: none
  int copy_after;        // 1: the global copy is taken from the tile after the slot has been handed back to the MMA thread
  int mode;              // 0 forward (bias + act), 1 backward ((+ add) * act'(xact))
  const float* xact; int64_t ldx;     // backward: activation OUTPUT [M x ldx] whose derivative multiplies; null: none
  const float* add; int64_t ldadd;    // backward: optional addend [M x ldadd]
  int fin, fin_c;        // epilogue hook of a head's last op and its channel (0 leg, 1 arm)
  int y_img;             // 1: y is a tile-image buffer: the MMA warp sends the finished tile there with one bulk copy (no thread stores)
  int x_img;             // 1: xact is a tile-image buffer
};
struct alignas(16) C2Prog {
  int M, n_loads, n_ops, pad_;
  C2Load ld[C2_MAX_LOADS];
  C2Op op[C2_MAX_OPS];
};
static_assert(sizeof(C2Prog) % 16 == 0, "copied to shared memory in 16-byte pieces");

// everything the epilogue hooks need (AC:326-345, PPO:166-221)
struct FinArgs {
  const float* std;                                          // [n_act]
  // FIN_ACT (rollout): a = mu + std * eps
  const float* eps; float* actions; float* log_prob; float* mean_out; float* sigma_out;
  // FIN_PPO / FIN_VALUE / FIN_REG (update)
  const int64_t* idx;                                        // mini-batch gather index (storage row of mini-batch row r)
  const float* s_actions; const float* old_logp; const float* old_values; const float* returns; const float* adv;
  const float* zh; int64_t zh_ld; int zh_by_src;
  float* g_leg; int gleg_ld; float* g_arm; int garm_ld; float* g_v; int gv_ld; float* g_z; int gz_ld;
  float* grad_std; float* losses;
  int n_leg, n_act, latent, rows;
  float clip, c_value, c_ent, c_reg, rho;
  int clipped_value;
  // arm torque supervision (PPO:224-239, fixed gains PPO:318-323); ts_target == nullptr: off.  Rows of [T*N, n_arm] storage tensors,
  // ts_coef = [3][n_arm] default p gains, d gains, default dof positions; ts_w = schedule weight (PPO:304-305); losses[4] += mean loss
  const float* ts_target; const float* ts_pos; const float* ts_vel; const float* ts_coef;
  float ts_w;
};

struct C2Launch {
  int nprog, x3;             // programs (1 or 2), error-compensated mode
  // work items of ONE program: np2 two-tile items over the tiles [0, 2 np2), then ns1 one-tile items over the rest.  All two-tile items (of
  // every program, longest program first) are queued in front of all one-tile items: the tail of a launch is filled with half-size items
  // (launch_chain2 picks ns1 by simulating the queue on the SM count)
  int np2, ns1;
  int rev;                   // tiles are taken from the last one downwards
  int* queue;                // [2] device counters (next item, finished CTAs), zero between launches
  C2Prog p[C2_MAX_PROGS];
  FinArgs fin;
};

// ---- weight packing ---------------------------------------------------------------------------------------------------
// image(n, k) of an op: up to two column segments of the source map into the K window of the tile,
//   transpose = 0: image(n, k) = w[n * ldw + ksrc]     (forward: W [N x K])
//   transpose = 1: image(n, k) = w[ksrc * ldw + n]     (backward: W [Kout x Nin], D = dZ W)
// for k = kdst + j, ksrc = ksrc0 + j, j < len; zero elsewhere and for n >= N.  With `lo` the image of w - trunc_tf32(w) is written too.
struct C2PackSeg { int kdst, ksrc, len; };
struct C2PackItem { const float* w; int64_t ldw; const float* bias; int N, npad, kpad, transpose, nseg; C2PackSeg seg[2]; int64_t dst, dst_lo; };
struct C2PackList { int n; float* out; C2PackItem it[C2_MAX_PACK]; };

__global__ void pack_weights2_kernel(const __grid_constant__ C2PackList pl) {
  const C2PackItem& it = pl.it[blockIdx.y];
  const int wn = it.npad * it.kpad, total = wn + it.npad;
  float* dst = pl.out + it.dst;
  float* dlo = it.dst_lo >= 0 ? pl.out + it.dst_lo : nullptr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    if (i < wn) {
      const int n = i / it.kpad, k = i - n * it.kpad;
      float v = 0.0f;
      if (n < it.N) {
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          if (s < it.nseg) {
            const int j = k - it.seg[s].kdst;
            if (j >= 0 && j < it.seg[s].len) {
              const int ks = it.seg[s].ksrc + j;
              v = it.transpose ? it.w[(int64_t)ks * it.ldw + n] : it.w[(int64_t)n * it.ldw + ks];
            }
          }
        }
      }
      const size_t o = ((size_t)((n >> 3) * (it.kpad >> 2) + (k >> 2)) * 8 + (n & 7)) * 4 + (k & 3);
      dst[o] = v;
      if (dlo) dlo[o] = tf32_lo(v);
    } else {
      const int n = i - wn;
      dst[i] = (it.bias && n < it.N) ? it.bias[n] : 0.0f;
    }
  }
}

// ---- device helpers ---------------------------------------------------------------------------------------------------
struct C2Shared {
  uint64_t w_full, w_free, ready[2], mma_done[2], ld_bar;
  uint32_t tmem_base;
  int item;
};

__device__ __forceinline__ void c2_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void c2_bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tc_smem_u32(dst_smem)), "l"(src),
               "r"(bytes), "r"(tc_smem_u32(bar))
               : "memory");
}
// shared -> global bulk copy of this thread's bulk group (the tile images of the activations)
__device__ __forceinline__ void c2_bulk_s2g(void* dst, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(tc_smem_u32(src_smem)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void c2_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }   // sources may be overwritten
__device__ __forceinline__ void c2_bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }         // writes complete
// tcgen05.mma with the A operand in tensor memory (lane = row, one 32-bit column per k)
__device__ __forceinline__ void c2_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 32 columns: registers -> tensor memory (thread = lane = row)
__device__ __forceinline__ void c2_st32(uint32_t taddr, const float* v) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
      "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]),
      "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
// elect.sync: true in exactly one lane of the (converged) warp
__device__ __forceinline__ bool c2_elect() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// tcgen05.ld of 32 lanes x 32 columns without the wait (tc_ld32 waits right away)
__device__ __forceinline__ void c2_ld32_nowait(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void c2_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void c2_wbar() { __syncwarp(); asm volatile("bar.sync 1, %0;" ::"n"(C2_NW) : "memory"); }     // the worker warps
// hand-over of a worker warp: all its lanes have written (and fenced), ONE lane arrives (512 single-thread arrivals on one mbarrier
// serialise to ~2 k cycles per op; 16 do not)
__device__ __forceinline__ void c2_warp_arrive(uint64_t* bar, int lane) {
  __syncwarp();
  if (lane == 0) t2_arrive(bar);
}

constexpr float C2_LOG_SQRT_2PI = 0.91893853320467274178f;

// ---- packed fp32 pairs ---------------------------------------------------------------------------------------------------
// sm_100 issues add / sub / mul / fma on TWO fp32 values per lane as one instruction (PTX .f32x2 on a 64-bit register -> FADD2 / FMUL2 /
// FFMA2).  The epilogues are bound by their instruction stream (ncu: 30 warp instructions per output element, 0.16 IPC per scheduler with two
// worker warps each, tensor pipe 12 % active), so the element-wise fp32 arithmetic runs on pairs; max / min / ex2 / and have no paired form.
// Packing two registers that tcgen05.ld, a 16-byte load or an earlier paired instruction delivered side by side costs no instruction.
__device__ __forceinline__ uint64_t c2_pk(float a, float b) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void c2_upk(uint64_t p, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(p)); }
__device__ __forceinline__ uint64_t c2_add2(uint64_t a, uint64_t b) { uint64_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t c2_sub2(uint64_t a, uint64_t b) { uint64_t r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t c2_mul2(uint64_t a, uint64_t b) { uint64_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ uint64_t c2_fma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
// 2^x, flush-to-zero form: ONE MUFU.EX2.  (__expf = ex2.approx.f32 of x * log2 e WITHOUT .ftz, which ptxas wraps in a range test and two
// scaling multiplies per element for results in the denormal range -- irrelevant for e^x - 1.)
__device__ __forceinline__ float c2_ex2(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
constexpr float C2_LOG2E = 1.4426950408889634f;
// low parts x - trunc_tf32(x) of a pair
__device__ __forceinline__ uint64_t c2_lo2(uint64_t p) { return c2_sub2(p, p & 0xFFFFE000FFFFE000ull); }
// low parts of a 32-column chunk, in place
__device__ __forceinline__ void c2_lo_chunk(float* v) {
#pragma unroll
  for (int jj = 0; jj < 32; jj += 2) c2_upk(c2_lo2(c2_pk(v[jj], v[jj + 1])), v[jj], v[jj + 1]);
}

// kAct == ACT_RELU stands for ReLU and leaky ReLU (negative-side `slope`)
template <int kAct, bool kFull>
__device__ __forceinline__ void c2_bias_act(float* v, const float* bias, int nvalid, float slope = 0.0f) {
  const uint64_t l2e = c2_pk(C2_LOG2E, C2_LOG2E), m1 = c2_pk(-1.0f, -1.0f);
#pragma unroll
  for (int j4 = 0; j4 < 8; ++j4) {
    const float4 b4 = *reinterpret_cast<const float4*>(bias + 4 * j4);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int jj = 4 * j4 + 2 * h;
      float x0, x1;
      c2_upk(c2_add2(c2_pk(v[jj], v[jj + 1]), h ? c2_pk(b4.z, b4.w) : c2_pk(b4.x, b4.y)), x0, x1);
      if (kAct == ACT_ELU) {        // ELU without a select: max(x,0) + (e^{min(x,0)} - 1); 5 instructions per element (9 as scalar code with __expf)
        float e0, e1;
        c2_upk(c2_mul2(c2_pk(fminf(x0, 0.0f), fminf(x1, 0.0f)), l2e), e0, e1);
        c2_upk(c2_add2(c2_add2(c2_pk(c2_ex2(e0), c2_ex2(e1)), m1), c2_pk(fmaxf(x0, 0.0f), fmaxf(x1, 0.0f))), x0, x1);
      }
      if (kAct == ACT_SELU) {       // lambda max(x,0) + lambda alpha (e^{min(x,0)} - 1): the ELU line with two scales
        float e0, e1;
        c2_upk(c2_mul2(c2_pk(fminf(x0, 0.0f), fminf(x1, 0.0f)), l2e), e0, e1);
        c2_upk(c2_fma2(c2_add2(c2_pk(c2_ex2(e0), c2_ex2(e1)), m1), c2_pk(SELU_SCALE * SELU_ALPHA, SELU_SCALE * SELU_ALPHA),
                       c2_mul2(c2_pk(fmaxf(x0, 0.0f), fmaxf(x1, 0.0f)), c2_pk(SELU_SCALE, SELU_SCALE))), x0, x1);
      }
      if (kAct == ACT_RELU) {       // ReLU and leaky ReLU: max(x,0) + slope min(x,0), slope = 0 / 0.01 (exact: one rounding)
        c2_upk(c2_fma2(c2_pk(fminf(x0, 0.0f), fminf(x1, 0.0f)), c2_pk(slope, slope), c2_pk(fmaxf(x0, 0.0f), fmaxf(x1, 0.0f))), x0, x1);
      }
      if (kAct == ACT_TANH) { x0 = t2_tanh(x0); x1 = t2_tanh(x1); }
      if (kAct == ACT_SIGMOID) { x0 = __fdividef(1.0f, 1.0f + c2_ex2(-C2_LOG2E * x0)); x1 = __fdividef(1.0f, 1.0f + c2_ex2(-C2_LOG2E * x1)); }
      v[jj] = (kFull || jj < nvalid) ? x0 : 0.0f;
      v[jj + 1] = (kFull || jj + 1 < nvalid) ? x1 : 0.0f;
    }
  }
}
__device__ __forceinline__ void c2_bias_act_any(float* v, const float* bias, int act, int nvalid) {
  const float slope = act == ACT_LRELU ? LRELU_SLOPE : 0.0f;
  if (nvalid >= 32) {
    if (act == ACT_ELU) c2_bias_act<ACT_ELU, true>(v, bias, 32);
    else if (act == ACT_TANH) c2_bias_act<ACT_TANH, true>(v, bias, 32);
    else if (act == ACT_SELU) c2_bias_act<ACT_SELU, true>(v, bias, 32);
    else if (act == ACT_RELU || act == ACT_LRELU) c2_bias_act<ACT_RELU, true>(v, bias, 32, slope);
    else if (act == ACT_SIGMOID) c2_bias_act<ACT_SIGMOID, true>(v, bias, 32);
    else c2_bias_act<ACT_NONE, true>(v, bias, 32);
  } else {
    if (act == ACT_ELU) c2_bias_act<ACT_ELU, false>(v, bias, nvalid);
    else if (act == ACT_TANH) c2_bias_act<ACT_TANH, false>(v, bias, nvalid);
    else if (act == ACT_SELU) c2_bias_act<ACT_SELU, false>(v, bias, nvalid);
    else if (act == ACT_RELU || act == ACT_LRELU) c2_bias_act<ACT_RELU, false>(v, bias, nvalid, slope);
    else if (act == ACT_SIGMOID) c2_bias_act<ACT_SIGMOID, false>(v, bias, nvalid);
    else c2_bias_act<ACT_NONE, false>(v, bias, nvalid);
  }
}

// ---- epilogue hooks: one thread per row, v[0 .. N) = the head's outputs of that row ---------------------------------------
// Both action-group hooks first pull everything they need into registers with independent (8-byte vector) loads, then compute, then
// store: written element by element the compiler had to order every load after the previous store (possible aliasing), i.e. a dozen
// dependent global round trips per row.  A group has at most 16 actions (host check), rows of the [.., n_act] tensors are 8-byte aligned
// at both group offsets when n_act and n_leg are even (host check; else the scalar path).
constexpr int C2_GRP = 16;
__device__ __forceinline__ void c2_ld_group(const float* p, int cnt, bool vec2, float* out) {
  if (vec2) {
#pragma unroll
    for (int i = 0; i < C2_GRP; i += 2)
      if (i < cnt) { const float2 t = *reinterpret_cast<const float2*>(p + i); out[i] = t.x; out[i + 1] = t.y; }
  } else {
#pragma unroll
    for (int i = 0; i < C2_GRP; ++i)
      if (i < cnt) out[i] = p[i];
  }
}
__device__ __forceinline__ void c2_st_group(float* p, int cnt, bool vec2, const float* v) {
  if (vec2) {
#pragma unroll
    for (int i = 0; i < C2_GRP; i += 2)
      if (i < cnt) *reinterpret_cast<float2*>(p + i) = make_float2(v[i], v[i + 1]);
  } else {
#pragma unroll
    for (int i = 0; i < C2_GRP; ++i)
      if (i < cnt) p[i] = v[i];
  }
}
// FIN_ACT (PPO:119-123, AC:326-345): group c = 0 legs (columns [0, n_leg)), 1 arm ([n_leg, n_act))
__device__ __forceinline__ void c2_fin_act(const FinArgs& f, int c, int64_t m, bool on, const float* v) {
  if (!on) return;
  const int off = c == 0 ? 0 : f.n_leg, cnt = c == 0 ? f.n_leg : f.n_act - f.n_leg;
  const bool vec2 = ((f.n_act | f.n_leg) & 1) == 0;
  float sg[C2_GRP], ep[C2_GRP], ac[C2_GRP], mu[C2_GRP];
  c2_ld_group(f.std + off, cnt, vec2, sg);
  c2_ld_group(f.eps + m * f.n_act + off, cnt, vec2, ep);
  float lp = 0.0f;
#pragma unroll
  for (int i = 0; i < C2_GRP; ++i) {            // compile-time indices keep the arrays in registers
    if (i < cnt) {
      mu[i] = v[i];
      ac[i] = mu[i] + sg[i] * ep[i];
      const float d = ac[i] - mu[i];
      lp += -(d * d) / (2.0f * (sg[i] * sg[i])) - logf(sg[i]) - C2_LOG_SQRT_2PI;
    }
  }
  c2_st_group(f.actions + m * f.n_act + off, cnt, vec2, ac);
  c2_st_group(f.mean_out + m * f.n_act + off, cnt, vec2, mu);
  c2_st_group(f.sigma_out + m * f.n_act + off, cnt, vec2, sg);
  f.log_prob[2 * m + c] = lp;
}
// Arm torque supervision (PPO:224-239, off in the shipped config WGC:173) of arm joint i: tau = kp (mu + q_default - q) - kd qd (fixed gains,
// PPO:318-323) on act_inference(obs)[:, -n_arm:] (PPO:230: the arm means this hook holds), loss = w * mean((tau - target)^2) (PPO:236-238).
// Returns (squared error, d loss / d pre-tanh output).  Deliberately NOT inlined and scalar-only (no array leaves the caller's registers): the
// optional branch must not cost the hot epilogue anything.
__device__ __noinline__ float2 c2_fin_torque(const FinArgs& f, int64_t src, int cnt, int i, float mu) {
  const float kp = f.ts_coef[i];
  const float e = kp * (mu + f.ts_coef[2 * cnt + i] - f.ts_pos[src * cnt + i]) - f.ts_coef[cnt + i] * f.ts_vel[src * cnt + i] - f.ts_target[src * cnt + i];
  return make_float2(e * e, 2.0f * f.ts_w / ((float)f.rows * (float)cnt) * e * kp * (1.0f - mu * mu));
}
// FIN_PPO (AC:341-345, PPO:199-205): log-prob of the stored action, ratio, mixed advantage, clipped surrogate, entropy and
// the gradients w.r.t. the mean (through the tanh, AC:157,170) and std of this group
__device__ __forceinline__ void c2_fin_ppo(const FinArgs& f, int c, int64_t m, bool on, const float* v, int lane) {
  const int off = c == 0 ? 0 : f.n_leg, cnt = c == 0 ? f.n_leg : f.n_act - f.n_leg;
  const bool vec2 = ((f.n_act | f.n_leg) & 1) == 0;
  const float inv2m = 1.0f / (2.0f * (float)f.rows);
  float l_surr = 0.0f, l_ent = 0.0f, glp = 0.0f, l_ts = 0.0f;
  float sg[C2_GRP], act[C2_GRP], gm[C2_GRP];
  c2_ld_group(f.std + off, cnt, vec2, sg);
  if (on) {
    const int64_t src = f.idx ? f.idx[m] : m;
    c2_ld_group(f.s_actions + src * f.n_act + off, cnt, vec2, act);
    const float2 adv = *reinterpret_cast<const float2*>(f.adv + 2 * src);
    const float old_lp = f.old_logp[2 * src + c];
    float lp = 0.0f;
#pragma unroll
    for (int i = 0; i < C2_GRP; ++i) {
      if (i < cnt) {
        const float d = act[i] - v[i];
        const float ls = logf(sg[i]);
        lp += -(d * d) / (2.0f * (sg[i] * sg[i])) - ls - C2_LOG_SQRT_2PI;
        l_ent += 0.5f + C2_LOG_SQRT_2PI + ls;
      }
    }
    const float mix = c == 0 ? adv.x + f.rho * adv.y : adv.y + f.rho * adv.x;      // PPO:199-201
    const float ratio = expf(lp - old_lp);                                           // PPO:202
    const float rc = fminf(fmaxf(ratio, 1.0f - f.clip), 1.0f + f.clip);
    const float s1 = -mix * ratio, s2 = -mix * rc;                                   // PPO:203-205
    l_surr = fmaxf(s1, s2);
    const bool inside = ratio >= 1.0f - f.clip && ratio <= 1.0f + f.clip;
    float g;
    if (s1 > s2) g = -mix;
    else if (s1 == s2) g = 0.5f * -mix + (inside ? 0.5f * -mix : 0.0f);
    else g = inside ? -mix : 0.0f;
    glp = inv2m * g * ratio;
    const int gld = c == 0 ? f.gleg_ld : f.garm_ld;
#pragma unroll
    for (int i = 0; i < C2_GRP; ++i) {
      gm[i] = 0.0f;
      if (i < cnt) {
        const float d = act[i] - v[i];
        gm[i] = glp * d / (sg[i] * sg[i]) * (1.0f - v[i] * v[i]);
      }
    }
    if (c == 1 && f.ts_target != nullptr) {
#pragma unroll
      for (int i = 0; i < C2_GRP; ++i)
        if (i < cnt) { const float2 t = c2_fin_torque(f, src, cnt, i, v[i]); l_ts += t.x; gm[i] += t.y; }
    }
    float* grow = c == 0 ? f.g_leg + m * f.gleg_ld : f.g_arm + m * f.garm_ld;
    if ((gld & 3) == 0) {
#pragma unroll
      for (int i = 0; i < C2_GRP; i += 4)
        if (i < gld) *reinterpret_cast<float4*>(grow + i) = make_float4(gm[i], gm[i + 1], gm[i + 2], gm[i + 3]);
    } else {
#pragma unroll
      for (int i = 0; i < C2_GRP; ++i)
        if (i < gld) grow[i] = gm[i];
    }
  }
#pragma unroll
  for (int i = 0; i < C2_GRP; ++i) {           // gradient of std: one atomic per warp and column
    if (i < cnt) {                             // (warp-uniform)
      float gs = 0.0f;
      if (on) {
        const float d = act[i] - v[i];
        gs = glp * ((d * d) / (sg[i] * sg[i] * sg[i]) - 1.0f / sg[i]) - f.c_ent * inv2m / sg[i];
      }
      gs = warp_sum(gs);
      if (lane == 0) atomicAdd(f.grad_std + off + i, gs);
    }
  }
  const float ss = warp_sum(l_surr * inv2m), se = warp_sum(l_ent * inv2m);
  if (lane == 0) { atomicAdd(f.losses + 0, ss); atomicAdd(f.losses + 1 + 2, se); }
  if (c == 1 && f.ts_target != nullptr) {          // (warp-uniform)
    const float st = warp_sum(l_ts / ((float)f.rows * (float)cnt));
    if (lane == 0) atomicAdd(f.losses + 4, st);
  }
}
// FIN_VALUE (PPO:209-216), channel c
__device__ __forceinline__ void c2_fin_value(const FinArgs& f, int c, int64_t m, bool on, float val, int lane) {
  const float inv2m = 1.0f / (2.0f * (float)f.rows);
  float l_val = 0.0f;
  if (on) {
    const int64_t src = f.idx ? f.idx[m] : m;
    const float vo = f.old_values[2 * src + c], R = f.returns[2 * src + c];
    const float l1 = (val - R) * (val - R);
    float gv;
    if (f.clipped_value) {
      const float dvo = val - vo;
      const float vc = vo + fminf(fmaxf(dvo, -f.clip), f.clip);
      const float l2 = (vc - R) * (vc - R);
      const bool inside = dvo >= -f.clip && dvo <= f.clip;
      l_val = fmaxf(l1, l2);
      const float g1 = 2.0f * (val - R), g2 = inside ? 2.0f * (vc - R) : 0.0f;
      gv = l1 > l2 ? g1 : (l1 == l2 ? 0.5f * g1 + 0.5f * g2 : g2);
    } else {
      l_val = l1;
      gv = 2.0f * (val - R);
    }
    f.g_v[m * f.gv_ld + c] = gv * f.c_value * inv2m;
    if (c == 0) for (int i = 2; i < f.gv_ld; ++i) f.g_v[m * f.gv_ld + i] = 0.0f;     // pad columns are operand columns of the backward pass
  }
  const float s = warp_sum(l_val * inv2m);
  if (lane == 0) atomicAdd(f.losses + 1, s);
}
// FIN_REG (PPO:174-177): || z_priv - sg(z_hist) ||_2 per row, mean over rows
__device__ __forceinline__ void c2_fin_reg(const FinArgs& f, int64_t m, bool on, const float* v, int lane) {
  const float invm = 1.0f / (float)f.rows;
  float nrm = 0.0f;
  if (on) {
    const int64_t src = f.idx ? f.idx[m] : m;
    const float* zhr = f.zh + (f.zh_by_src ? src : m) * f.zh_ld;
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (i < f.latent) { const float d = v[i] - zhr[i]; nrm += d * d; }
    nrm = sqrtf(nrm);
    const float s = nrm > 0.0f ? f.c_reg * invm / nrm : 0.0f;
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (i < f.gz_ld) f.g_z[m * f.gz_ld + i] = i < f.latent ? s * (v[i] - zhr[i]) : 0.0f;
  }
  const float s = warp_sum(nrm * invm);
  if (lane == 0) atomicAdd(f.losses + 2, s);
}

// ---- the kernel -------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(C2_THREADS, 1) chain2_kernel(const __grid_constant__ C2Launch L, const int tiles) {
  extern __shared__ __align__(1024) float c2_smem[];
  __shared__ C2Shared sh;
  __shared__ __align__(16) C2Prog sprog;
  int cur_prog = -1;
  float* tile[2] = {c2_smem, c2_smem + C2_TILE};
  float* wbuf = c2_smem + 2 * C2_TILE;
  float* bias_s = c2_smem + 3 * C2_TILE;                 // two slots of 128 (parity of the CTA-wide op counter)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    tc_mbar_init(&sh.w_full, 1);
    tc_mbar_init(&sh.w_free, 1);
    tc_mbar_init(&sh.ld_bar, 1);
    for (int s = 0; s < 2; ++s) { tc_mbar_init(&sh.ready[s], C2_WORKERS); tc_mbar_init(&sh.mma_done[s], 1); }   // one arrival per worker WARP
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == C2_WORKERS) tc_tmem_alloc(&sh.tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sh.tmem_base;
  const int n_pair_items = L.np2 * L.nprog;
  const int items = n_pair_items + L.ns1 * L.nprog;
  const bool x3 = L.x3 != 0;

  // running counters, identical in every thread: ops of all items so far (bias slot parity) and ops per slot (phase of that
  // slot's ready / mma_done barriers: a slot without a tile in some item does not advance)
  uint32_t nop = 0, cnt[2] = {0, 0}, rcnt[2] = {0, 0}, nld = 0;   // rcnt: phases of ready[] (one per op + one after the last op of an item); nld: ld_bar
  uint32_t nw = 0, nf = 0;          // weight images fetched (phase of w_full) / released (phase of w_free): used by the MMA thread only
  if (tid == 0) T2_STAMP(62);       // profiling aid (tools/chain_profile.py): clock64 stamps of the CTA's FIRST item, 6 per op

  for (;;) {
    // ---- next work item ----
    __syncthreads();                                     // everybody is done with the previous item (sh.item may be overwritten)
    if (tid == 0) sh.item = atomicAdd(L.queue, 1);
    __syncthreads();
    const int item = sh.item;
    if (item >= items) break;
    int pi, t0, nslots;                                  // program (0 = the longer one, first), first tile, tiles of this item
    {
      const bool two = item < n_pair_items;
      const int k = two ? item : item - n_pair_items, per = two ? L.np2 : L.ns1;
      pi = k / per;
      t0 = two ? 2 * (k - pi * per) : 2 * L.np2 + (k - pi * per);
      nslots = min(two ? 2 : 1, tiles - t0);
      asm volatile("" : "+r"(nslots));                   // opaque: one body for both item sizes (the compiler cloned the whole item loop otherwise)
    }
    // slot s works on tile tb + s * td: upwards from t0, or (L.rev: the backward launch) downwards from the last tile -- the forward launch
    // that produced the activation images this one reads walked upwards, so its most recent output, still in L2, belongs to the last tiles
    const int tb = L.rev ? tiles - 1 - t0 : t0, td = L.rev ? -1 : 1;
    // the item's program goes to shared memory: read through the kernel parameter, every field access with a run-time op index is an
    // indexed constant-bank load (LDC c[0x0][R + off]) -- a long-scoreboard stall in front of most addresses and predicates of the epilogue
    if (pi != cur_prog) {
      const int4* src = reinterpret_cast<const int4*>(&L.p[pi]);
      int4* dst = reinterpret_cast<int4*>(&sprog);
      for (int k = tid; k < (int)(sizeof(C2Prog) / 16); k += C2_THREADS) dst[k] = src[k];
      cur_prog = pi;
      __syncthreads();
    }
    const C2Prog& pr = sprog;
    const int nops = pr.n_ops;

    if (warp == C2_WORKERS) {
      // ===================== weight copies + MMA issue =====================
      // The WHOLE warp runs this control flow (converged, every value warp-uniform); only the instructions that must be issued once sit
      // under elect.sync.  Issued from inside `if (lane == 0)` the compiler could not prove the descriptors uniform and wrapped every
      // tcgen05.mma in an elect / 7 x R2UR.BROADCAST / branch loop: ~300 cycles per MMA, i.e. the MMA thread, not the tensor core or the
      // epilogue, set the pace of the whole kernel.
      const uint32_t b0 = tc_smem_u32(wbuf);
      // one tile in this item (small batches: the rollout's act(); the half-size items at the tail of a large launch): slot Y's tile is
      // unused, so in 3xTF32 mode the low-part image of an op is fetched into it TOGETHER with the raw image instead of after the first
      // two products (no serial second fetch per op)
      const bool lo_side = x3 && nslots == 1;
      const uint32_t b0_lo = lo_side ? tc_smem_u32(tile[1]) : b0;
      auto fetch = [&](const float* img, uint32_t wbytes, uint32_t bbytes, uint32_t slot, const float* img_lo = nullptr) {
        if (c2_elect()) {
          c2_expect_tx(&sh.w_full, wbytes + bbytes + (img_lo ? wbytes : 0u));
          c2_bulk_g2s(wbuf, img, wbytes, &sh.w_full);
          if (bbytes) c2_bulk_g2s(bias_s + slot * 128, img + (wbytes >> 2), bbytes, &sh.w_full);
          if (img_lo) c2_bulk_g2s(tile[1], img_lo, wbytes, &sh.w_full);
        }
        __syncwarp();
      };
      uint32_t n = nop;
      {
        const C2Op& o0 = pr.op[0];
        fetch(o0.wp, (uint32_t)(o0.npad * o0.kpad) * 4u, (uint32_t)o0.npad * 4u, n & 1, lo_side ? o0.wp_lo : nullptr);
      }
      for (int i = 0; i < nops; ++i, ++n) {
        const C2Op& o = pr.op[i];
        const uint32_t idesc = tc_idesc(o.npad, false, false);
        const uint32_t wsbo = (uint32_t)(o.kpad >> 2) * 128u;
        const int nk = o.kpad >> 3;
        tc_mbar_wait(&sh.w_full, nw & 1); ++nw;
        if (lane == 0 && nop == 0 && i < 10) T2_STAMP(6 * i + 0);
        // the previous op left a finished tile behind: if its output is a tile image it goes out now, as one 64 KB bulk copy issued right
        // before the MMAs that read the same tile; its shared-memory reads must have completed before the epilogue of THIS op may overwrite
        // the tile, i.e. before mma_done is signalled
        const bool st_prev = i > 0 && pr.op[i - 1].y_img != 0;
        bool reload_next = false;                      // an image written earlier is re-read before the next op: those writes must have landed
        for (int l = 0; l < pr.n_loads; ++l) reload_next |= pr.ld[l].before_op == i + 1 && pr.ld[l].img != 0;
        for (int s = 0; s < nslots; ++s) {
          tc_mbar_wait(&sh.ready[s], (rcnt[s] + i) & 1);   // loads landed / previous epilogue done: operand tile written, accumulator drained
          if (lane == 0 && nop == 0 && i < 10) T2_STAMP(6 * i + 1 + s);
          tc_fence_async_smem();                       // generic-proxy tile writes -> async-proxy MMA / bulk-copy reads
          tc_fence_after();
          const uint32_t a0 = tc_smem_u32(tile[s]) + (uint32_t)(o.a_col0 >> 2) * 128u;
          const uint32_t dt = tmem + s * 256;
          if (c2_elect()) {
            if (st_prev) c2_bulk_s2g(pr.op[i - 1].y + (size_t)(tb + s * td) * C2_TILE, tile[s], C2_TILE * 4);
            // one K step (8 columns = two 16-byte pieces) advances both start addresses by 256 bytes: +16 in the descriptors' address field
            uint64_t ad = tc_desc(a0, 128, 4096), bd = tc_desc(b0, 128, wsbo);
            tc_mma_tf32(dt, ad, bd, idesc, 0u);
#pragma unroll 4
            for (int k = 1; k < nk; ++k) { ad += 16; bd += 16; tc_mma_tf32(dt, ad, bd, idesc, 1u); }
            if (x3) {
              bd = tc_desc(b0, 128, wsbo);
              uint32_t at = dt + 128 + o.a_col0;
#pragma unroll 4
              for (int k = 0; k < nk; ++k, at += 8, bd += 16) c2_mma_ts(dt, at, bd, idesc, 1u);
              if (lo_side) {                               // third product right away: the low-part image is already there
                ad = tc_desc(a0, 128, 4096); bd = tc_desc(b0_lo, 128, wsbo);
#pragma unroll 4
                for (int k = 0; k < nk; ++k, ad += 16, bd += 16) tc_mma_tf32(dt, ad, bd, idesc, 1u);
                if (reload_next) c2_bulk_wait_all(); else if (st_prev) c2_bulk_wait_read();
                tc_commit(&sh.mma_done[s]);
              }
            } else {
              if (reload_next) c2_bulk_wait_all(); else if (st_prev) c2_bulk_wait_read();
              tc_commit(&sh.mma_done[s]);
            }
          }
          __syncwarp();
        }
        if (c2_elect()) tc_commit(&sh.w_free);
        __syncwarp();
        tc_mbar_wait(&sh.w_free, nf & 1); ++nf;        // every MMA reading the image has retired: the buffer may be refilled
        if (lane == 0 && nop == 0 && i < 10) T2_STAMP(6 * i + 3);
        if (x3 && !lo_side) {
          fetch(o.wp_lo, (uint32_t)(o.npad * o.kpad) * 4u, 0u, 0);
          tc_mbar_wait(&sh.w_full, nw & 1); ++nw;
          for (int s = 0; s < nslots; ++s) {
            const uint32_t a0 = tc_smem_u32(tile[s]) + (uint32_t)(o.a_col0 >> 2) * 128u;
            const uint32_t dt = tmem + s * 256;
            if (c2_elect()) {
              uint64_t ad = tc_desc(a0, 128, 4096), bd = tc_desc(b0, 128, wsbo);
#pragma unroll 4
              for (int k = 0; k < nk; ++k, ad += 16, bd += 16) tc_mma_tf32(dt, ad, bd, idesc, 1u);
              if (reload_next) c2_bulk_wait_all(); else if (st_prev) c2_bulk_wait_read();
              tc_commit(&sh.mma_done[s]);
            }
            __syncwarp();
          }
          if (c2_elect()) tc_commit(&sh.w_free);
          __syncwarp();
          tc_mbar_wait(&sh.w_free, nf & 1); ++nf;
        }
        if (i + 1 < nops) {
          const C2Op& o1 = pr.op[i + 1];
          fetch(o1.wp, (uint32_t)(o1.npad * o1.kpad) * 4u, (uint32_t)o1.npad * 4u, (n + 1) & 1, lo_side ? o1.wp_lo : nullptr);
        }
      }
      // the last op's tiles: every slot is handed back once more; an image output leaves now, and the tiles may be reloaded (next item)
      // only after the copies have read them
      for (int s = 0; s < nslots; ++s) {
        tc_mbar_wait(&sh.ready[s], (rcnt[s] + nops) & 1);
        tc_fence_async_smem();
        if (c2_elect()) {
          if (pr.op[nops - 1].y_img) c2_bulk_s2g(pr.op[nops - 1].y + (size_t)(tb + s * td) * C2_TILE, tile[s], C2_TILE * 4);
          if (s + 1 == nslots) c2_bulk_wait_read();
        }
        __syncwarp();
      }
    } else {
      // ===================== loads + epilogues (sixteen warps) =====================
      const int q = warp & 3, h = warp >> 2;               // TMEM lane quarter, column group (32-column chunks ci with ci % 4 == h)
      const int r = q * 32 + lane;                         // tile row of this thread in the epilogue
      constexpr int LRW = 128 / C2_WORKERS, LPS = 32 / LRW;     // load role: rows per warp, piece stride
      const int lrow = warp * LRW + (lane % LRW), lpc = lane / LRW;   // fixed row, 16-byte pieces lpc, lpc + LPS, ...

      // cp.async of one load into the tile of slot s (no waiting); rows beyond the matrix are zero-filled
      auto issue_load = [&](const C2Load& ld, int s, int64_t m0, int rows) {
        float* tl = tile[s];
        const int c40 = ld.col0 >> 2, cpr = ld.ncols >> 2;
        const int z0 = (ld.col0 + ld.ncols) >> 2, z1 = ld.zero_to >> 2;
        float* rowbase = tl + ((size_t)(lrow >> 3) * 32) * 32 + (lrow & 7) * 4;
        for (int cz = z0 + lpc; cz < z1; cz += LPS) *reinterpret_cast<float4*>(rowbase + (size_t)cz * 32) = make_float4(0.f, 0.f, 0.f, 0.f);
        const bool on = lrow < rows;
        const float* src = on ? ld.src.row(m0 + lrow) : ld.src.p;
        const uint32_t d0 = tc_smem_u32(rowbase);
        for (int cc = lpc; cc < cpr; cc += LPS)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d0 + (uint32_t)(c40 + cc) * 128u), "l"(src + 4 * cc), "r"(on ? 16 : 0)
                       : "memory");
      };
      // 3xTF32: low parts of tile columns [c_lo, c_hi) (whole 32-column chunks) -> A_lo of slot s
      auto split_cols = [&](int s, int c_lo, int c_hi) {
        const float* trow = tile[s] + ((size_t)(r >> 3) * 32) * 32 + (r & 7) * 4;
        for (int ci = (c_lo >> 5) + h; ci * 32 < c_hi; ci += C2_H) {
          float v[32];
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 t = *reinterpret_cast<const float4*>(trow + (size_t)(ci * 8 + j4) * 32);
            c2_upk(c2_lo2(c2_pk(t.x, t.y)), v[4 * j4], v[4 * j4 + 1]);
            c2_upk(c2_lo2(c2_pk(t.z, t.w)), v[4 * j4 + 2], v[4 * j4 + 3]);
          }
          c2_st32(tmem + s * 256 + 128 + ((uint32_t)(q * 32) << 16) + ci * 32, v);
        }
        c2_wait_st();
      };
      // loads of the slot that precede op `before`: issue, wait, (split), hand over
      auto do_loads = [&](int before, bool sync_first) {
        bool any = false;
        for (int l = 0; l < pr.n_loads; ++l) any |= pr.ld[l].before_op == before;
        if (!any) return false;
        if (sync_first) c2_wbar();                       // every worker has finished writing / copying the tiles the loads overwrite
        int nimg = 0;
        for (int s = 0; s < nslots; ++s) {
          const int64_t m0 = (int64_t)(tb + s * td) * TC_M;
          const int rows = (int)min((int64_t)TC_M, (int64_t)pr.M - m0);
          for (int l = 0; l < pr.n_loads; ++l) {
            if (pr.ld[l].before_op != before) continue;
            if (pr.ld[l].img) ++nimg; else issue_load(pr.ld[l], s, m0, rows);
          }
        }
        if (nimg) {                                      // tile images come back as one bulk copy each (warp-uniform count)
          if (tid == 0) {
            c2_expect_tx(&sh.ld_bar, (uint32_t)nimg * C2_TILE * 4u);
            for (int s = 0; s < nslots; ++s)
              for (int l = 0; l < pr.n_loads; ++l)
                if (pr.ld[l].before_op == before && pr.ld[l].img) c2_bulk_g2s(tile[s], pr.ld[l].src.p + (size_t)(tb + s * td) * C2_TILE, C2_TILE * 4, &sh.ld_bar);
          }
          tc_mbar_wait(&sh.ld_bar, nld & 1);
          ++nld;
        }
        asm volatile("cp.async.wait_all;" ::: "memory");
        if (x3) {
          c2_wbar();                                     // the pieces were copied by other threads than the ones that split them
          for (int s = 0; s < nslots; ++s)
            for (int l = 0; l < pr.n_loads; ++l)
              if (pr.ld[l].before_op == before) split_cols(s, pr.ld[l].col0, pr.ld[l].zero_to);
        }
        return true;
      };

      uint32_t n = nop;
      // ---- item start: the rows a LATER gather of this item will read are pulled into L2 now (its latency is exposed otherwise: the tile
      // columns it fills are still in use), then both slots' initial loads ----
      for (int l = 0; l < pr.n_loads; ++l) {
        const C2Load& ld = pr.ld[l];
        if (ld.before_op == 0 || ld.img) continue;
        for (int s = 0; s < nslots; ++s) {
          const int64_t m0 = (int64_t)(tb + s * td) * TC_M;
          if (m0 + lrow >= pr.M) continue;
          const float* src = ld.src.row(m0 + lrow);
          for (int b = lpc * 32; b < ld.ncols; b += LPS * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + b));
        }
      }
      do_loads(0, false);
      tc_fence_before();
      tc_fence_async_smem();
      for (int s = 0; s < nslots; ++s) c2_warp_arrive(&sh.ready[s], lane);

      for (int i = 0; i < nops; ++i, ++n) {
        const C2Op& o = pr.op[i];
        bool pending = false;                              // loads that precede op i+1 cover both slots and follow the last slot's epilogue
        for (int l = 0; l < pr.n_loads; ++l) pending |= pr.ld[l].before_op == i + 1;
        for (int s = 0; s < nslots; ++s) {
          const int64_t m0 = (int64_t)(tb + s * td) * TC_M;
          const int rows = (int)min((int64_t)TC_M, (int64_t)pr.M - m0);
          const bool on = r < rows;
          // backward: the activation chunks whose derivative multiplies, fetched while the MMAs run
          float x[C2_CPW][32];
          const bool use_x = o.mode == 1 && o.xact != nullptr;
          if (use_x) {
#pragma unroll
            for (int u = 0; u < C2_CPW; ++u) {
              const int c0 = 32 * (h + u * C2_H);
              // row-major: 32 consecutive floats of the row; tile image: eight 16-byte pieces 128 bytes apart (eight rows share each line)
              const float* xr = o.x_img ? o.xact + (size_t)(tb + s * td) * C2_TILE + ((size_t)((r >> 3) * 32 + (c0 >> 2)) * 8 + (r & 7)) * 4
                                        : o.xact + (m0 + r) * o.ldx + c0;
              const int xst = o.x_img ? 32 : 4;
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4) {
                float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                if (on && c0 + 4 * j4 < o.N) t = *reinterpret_cast<const float4*>(xr + xst * j4);
                x[u][4 * j4] = t.x; x[u][4 * j4 + 1] = t.y; x[u][4 * j4 + 2] = t.z; x[u][4 * j4 + 3] = t.w;
              }
            }
          }
          tc_mbar_wait(&sh.mma_done[s], (cnt[s] + i) & 1);
          tc_fence_after();
          if (tid == 0 && s == 0 && nop == 0 && i < 10) T2_STAMP(6 * i + 4);
#pragma unroll
          for (int u = 0; u < C2_CPW; ++u) {
            const int c0 = 32 * (h + u * C2_H);            // this warp's u-th chunk
            if (c0 >= o.npad) continue;
            float v[32];
            tc_ld32(tmem + s * 256 + ((uint32_t)(q * 32) << 16) + c0, v);
            if (o.mode == 0) {
              c2_bias_act_any(v, bias_s + (n & 1) * 128 + c0, o.act, o.N - c0);
            } else {
              if (o.add != nullptr && on) {
                const float* ar = o.add + (m0 + r) * o.ldadd + c0;
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                  if (c0 + 4 * j4 < o.N) {
                    const float4 t = *reinterpret_cast<const float4*>(ar + 4 * j4);
                    c2_upk(c2_add2(c2_pk(v[4 * j4], v[4 * j4 + 1]), c2_pk(t.x, t.y)), v[4 * j4], v[4 * j4 + 1]);
                    c2_upk(c2_add2(c2_pk(v[4 * j4 + 2], v[4 * j4 + 3]), c2_pk(t.z, t.w)), v[4 * j4 + 2], v[4 * j4 + 3]);
                  }
                }
              }
              if (use_x) {                                   // activation derivatives from the layer's OUTPUTS
                if (o.act == ACT_TANH) {
#pragma unroll
                  for (int jj = 0; jj < 32; ++jj) v[jj] *= 1.0f - x[u][jj] * x[u][jj];
                } else if (o.act == ACT_ELU) {               // ELU'(y) = y > 0 ? 1 : y + 1 = min(y + 1, 1), on pairs
                  const uint64_t one2 = c2_pk(1.0f, 1.0f);
#pragma unroll
                  for (int jj = 0; jj < 32; jj += 2) {
                    float d0, d1;
                    c2_upk(c2_add2(c2_pk(x[u][jj], x[u][jj + 1]), one2), d0, d1);
                    c2_upk(c2_mul2(c2_pk(v[jj], v[jj + 1]), c2_pk(fminf(d0, 1.0f), fminf(d1, 1.0f))), v[jj], v[jj + 1]);
                  }
                } else if (o.act == ACT_SIGMOID) {           // y (1 - y)
#pragma unroll
                  for (int jj = 0; jj < 32; ++jj) v[jj] *= x[u][jj] * (1.0f - x[u][jj]);
                } else {                                     // SELU / ReLU / leaky ReLU: y > 0 ? p : q y + r
                  const bool selu = o.act == ACT_SELU;
                  const float p = selu ? SELU_SCALE : 1.0f, qq = selu ? 1.0f : 0.0f,
                              rr = selu ? SELU_SCALE * SELU_ALPHA : (o.act == ACT_LRELU ? LRELU_SLOPE : 0.0f);
#pragma unroll
                  for (int jj = 0; jj < 32; ++jj) v[jj] *= x[u][jj] > 0.0f ? p : fmaf(qq, x[u][jj], rr);
                }
              }
              if (o.N - c0 < 32) {                           // ragged last chunk: the pad columns are operand columns of the next op
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) v[jj] = c0 + jj < o.N ? v[jj] : 0.0f;
              }
            }
            if (o.out_col0 >= 0) {
              float* otile = tile[s] + ((size_t)((r >> 3) * 32 + ((o.out_col0 + c0) >> 2)) * 8 + (r & 7)) * 4;
#pragma unroll
              for (int j4 = 0; j4 < 8; ++j4)
                *reinterpret_cast<float4*>(otile + (size_t)j4 * 32) = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
            }
            if (o.fin != FIN_NONE && c0 == 0) {
              if (o.fin == FIN_ACT) c2_fin_act(L.fin, o.fin_c, m0 + r, on, v);
              else if (o.fin == FIN_PPO) c2_fin_ppo(L.fin, o.fin_c, m0 + r, on, v, lane);
              else if (o.fin == FIN_VALUE) c2_fin_value(L.fin, o.fin_c, m0 + r, on, v[0], lane);
              else c2_fin_reg(L.fin, m0 + r, on, v, lane);
            }
            if (o.y != nullptr && !o.copy_after && !o.y_img && on) {       // straight from the registers: 128 contiguous bytes per thread
              float* yr = o.y + (m0 + r) * o.ldy + c0;
              if ((o.ldy & 3) == 0 && (o.N & 3) == 0) {
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4)
                  if (c0 + 4 * j4 < o.N) *reinterpret_cast<float4*>(yr + 4 * j4) = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
              } else {
#pragma unroll
                for (int jj = 0; jj < 32; ++jj)
                  if (c0 + jj < o.N) yr[jj] = v[jj];
              }
            }
            if (x3 && o.out_col0 >= 0) {                       // low parts last, in place: v is dead afterwards
              c2_lo_chunk(v);
              c2_st32(tmem + s * 256 + 128 + ((uint32_t)(q * 32) << 16) + o.out_col0 + c0, v);
            }
          }
          if (x3 && o.out_col0 >= 0) c2_wait_st();
          tc_fence_before();                               // tcgen05.ld / st of this op precede the hand-over
          if (!pending || i + 1 == nops) {              // (after the last op too: the MMA warp sends image outputs off and frees the tiles)
            tc_fence_async_smem();
            c2_warp_arrive(&sh.ready[s], lane);
          } else if (s + 1 == nslots) {
            do_loads(i + 1, true);
            tc_fence_before();
            tc_fence_async_smem();
            for (int s2 = 0; s2 < nslots; ++s2) c2_warp_arrive(&sh.ready[s2], lane);
          }
          if (tid == 0 && s + 1 == nslots && nop == 0 && i < 10) T2_STAMP(6 * i + 5);
          if (o.y != nullptr && o.copy_after && !o.y_img) {
            // global copy of the chunks this warp just wrote, out of the tile: 8 rows x 64 contiguous bytes per instruction
            __syncwarp();
            const int r8 = lane & 7, pp = lane >> 3;
            const float* tl = tile[s];
#pragma unroll
            for (int u = 0; u < C2_CPW; ++u) {
              const int c0 = 32 * (h + u * C2_H);
              if (c0 >= o.N) continue;
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                const int rr = q * 32 + g * 8 + r8;
                if (rr >= rows) continue;
                const float* trow = tl + ((size_t)((rr >> 3) * 32 + ((o.out_col0 + c0) >> 2)) * 8 + r8) * 4;
                float* yr = o.y + (m0 + rr) * o.ldy + c0;
#pragma unroll
                for (int p0 = 0; p0 < 8; p0 += 4) {
                  const int piece = p0 + pp;
                  if (c0 + 4 * piece < o.N) *reinterpret_cast<float4*>(yr + 4 * piece) = *reinterpret_cast<const float4*>(trow + (size_t)piece * 32);
                }
              }
            }
          }
        }
      }
    }
    nop += nops;
    for (int s = 0; s < nslots; ++s) { cnt[s] += nops; rcnt[s] += nops + 1; }
  }
  if (warp == C2_WORKERS && c2_elect()) c2_bulk_wait_all();      // the image stores of this CTA have landed
  tc_fence_before();
  __syncthreads();
  if (tid == 0) T2_STAMP(63);
  if (warp == C2_WORKERS) tc_tmem_dealloc(tmem, 512);
  if (tid == 0) {                        // the last CTA re-arms the queue for the next launch
    __threadfence();
    if (atomicAdd(L.queue + 1, 1) == (int)gridDim.x - 1) { L.queue[0] = 0; L.queue[1] = 0; __threadfence(); }
  }
}


// ---- host side ------------------------------------------------------------------------------------------------------
inline bool c2_aligned(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
constexpr int64_t C2_PACK_FLOATS = (int64_t)2 * C2_MAX_PACK * (C2_TILE + 256);      // raw + low images of every item

inline int launch_pack2(const C2PackList& pl, cudaStream_t st) {
  if (pl.n <= 0) return DWBC_OK;
  pack_weights2_kernel<<<dim3(8, pl.n), 256, 0, st>>>(pl);
  ++dwbc_launch_counter;
  return cudaGetLastError() == cudaSuccess ? DWBC_OK : DWBC_ERR_LAUNCH;
}

// Keeps the pack list and the program in step.  `off` is the running float offset into the packed-weight buffer.
struct C2Builder {
  C2Prog pr{};
  C2PackList* pl;
  int64_t* off;
  bool x3, ok = true;
  C2Builder(C2PackList* pl_, int64_t* off_, int M, bool x3_) : pl(pl_), off(off_), x3(x3_) { pr.M = M; }
  void load(RowMat src, int ncols, int col0, int zero_to, int before_op) {
    if (src.rpg == 0) {                 // tile image: the whole tile, one bulk copy
      if (pr.n_loads >= C2_MAX_LOADS || ncols != 128 || col0 != 0 || zero_to != 128 || !c2_aligned(src.p)) { ok = false; return; }
      pr.ld[pr.n_loads++] = C2Load{src, ncols, col0, zero_to, before_op, 1};
      return;
    }
    if (pr.n_loads >= C2_MAX_LOADS || (ncols & 3) || (col0 & 3) || (zero_to & 3) || zero_to < col0 + ncols || zero_to > 128 || !c2_aligned(src.p) ||
        (src.stride_g & 3) || (src.ld & 3) || src.rpg != 1) { ok = false; return; }
    pr.ld[pr.n_loads++] = C2Load{src, ncols, col0, zero_to, before_op, 0};
  }
  C2Op* push(const float* W, int64_t ldw, const float* bias, int N, int kpad, int transpose, int nseg, C2PackSeg s0, C2PackSeg s1) {
    const int npad = (N + 15) & ~15;
    if (pr.n_ops >= C2_MAX_OPS || pl->n >= C2_MAX_PACK || N <= 0 || N > 128 || kpad <= 0 || kpad > 128 || (kpad & 7)) { ok = false; return nullptr; }
    C2PackItem& it = pl->it[pl->n++];
    it = C2PackItem{W, ldw, bias, N, npad, kpad, transpose, nseg, {s0, s1}, *off, -1};
    C2Op& o = pr.op[pr.n_ops++];
    o = C2Op{};
    o.wp = pl->out ? pl->out + *off : nullptr;
    *off = (*off + (int64_t)npad * kpad + npad + 63) & ~(int64_t)63;       // 256-byte aligned images (bulk copies need 16)
    if (x3) {
      it.dst_lo = *off;
      o.wp_lo = pl->out ? pl->out + *off : nullptr;
      *off = (*off + (int64_t)npad * kpad + 63) & ~(int64_t)63;
    }
    o.kpad = kpad; o.N = N; o.npad = npad;
    return &o;
  }
  // y = act(A[:, a_col0 : a_col0 + kpad] W'^T + b): W [N x ldw]; tile column a_col0 + seg.kdst + j multiplies W[:, seg.ksrc + j]
  // y_img: y is a tile-image buffer (only for full-width outputs written at tile column 0)
  void fwd(const float* W, int64_t ldw, const float* bias, int N, int act, int a_col0, int kpad, int nseg, C2PackSeg s0, C2PackSeg s1, int out_col0,
           float* y, int64_t ldy, int fin = FIN_NONE, int fin_c = 0, bool y_img = false) {
    if (y_img && (N != 128 || out_col0 != 0 || !y || !c2_aligned(y))) { ok = false; return; }
    if ((a_col0 & 3) || a_col0 + kpad > 128 || (out_col0 >= 0 && ((out_col0 & 31) || out_col0 + ((N + 31) & ~31) > 128)) || (fin != FIN_NONE && N > 32)) { ok = false; return; }
    C2Op* o = push(W, ldw, bias, N, kpad, 0, nseg, s0, s1);
    if (!o) return;
    o->y = y; o->ldy = ldy; o->a_col0 = a_col0; o->act = act; o->out_col0 = out_col0; o->mode = 0; o->fin = fin; o->fin_c = fin_c;
    o->y_img = y_img ? 1 : 0;
  }
  // dX[:, :Nin] = (dZ[:, a_col0 : a_col0 + kpad] W' (+ add)) (*) act'(xact): W [Kout x ldw] (row = output feature);
  // tile column a_col0 + seg.kdst + j multiplies row seg.ksrc + j of W
  void bwd(const float* W, int64_t ldw, int Nin, int a_col0, int kpad, C2PackSeg seg, int act, const float* xact, int64_t ldx, const float* add,
           int64_t ldadd, int out_col0, float* y, int64_t ldy, bool x_img = false, bool y_img = false) {
    if ((y_img && (Nin != 128 || out_col0 != 0 || !y)) || (x_img && Nin != 128)) { ok = false; return; }
    if ((a_col0 & 3) || a_col0 + kpad > 128 || (Nin & 3) || (xact && ((ldx & 3) || !c2_aligned(xact))) || (add && ((ldadd & 3) || !c2_aligned(add))) ||
        (out_col0 >= 0 && (out_col0 & 31))) { ok = false; return; }
    C2Op* o = push(W, ldw, nullptr, Nin, kpad, 1, 1, seg, C2PackSeg{0, 0, 0});
    if (!o) return;
    o->y = y; o->ldy = ldy; o->a_col0 = a_col0; o->act = act; o->out_col0 = out_col0; o->mode = 1;
    o->xact = act == ACT_NONE ? nullptr : xact; o->ldx = ldx; o->add = add; o->ldadd = ldadd;
    o->x_img = x_img ? 1 : 0; o->y_img = y_img ? 1 : 0;
  }
  // global copies may be taken from the tile after the hand-over only if nothing overwrites those tile columns before the
  // same warp's next epilogue: same column mapping in the next op (out_col0 0 or none) and no load in between
  void finish() {
    for (int i = 0; i < pr.n_ops; ++i) {
      C2Op& o = pr.op[i];
      bool load_next = false;
      for (int l = 0; l < pr.n_loads; ++l) load_next |= pr.ld[l].before_op == i + 1;
      const bool next_ok = i + 1 == pr.n_ops || pr.op[i + 1].out_col0 <= 0;
      o.copy_after = (o.y && !o.y_img && o.out_col0 == 0 && !load_next && next_ok && (o.ldy & 3) == 0 && (o.N & 3) == 0 && c2_aligned(o.y)) ? 1 : 0;
      if (o.y && (o.ldy & 3) == 0 && (o.N & 3) == 0 && !c2_aligned(o.y)) ok = false;   // vector stores need 16-byte aligned rows
      // an image written by op i is sent off while op i+1 runs and must have landed before it is re-read: not by a load in front of op i+1
      if (o.y_img)
        for (int l = 0; l < pr.n_loads; ++l)
          if (pr.ld[l].img && pr.ld[l].src.p == o.y && pr.ld[l].before_op <= i + 1) ok = false;
    }
  }
};

// pr1 may be null.  The longer program goes first in the queue.
// ---- how many tiles of a large launch run as one-tile items ---------------------------------------------------------------------------
// A launch of T tiles x P programs on S persistent CTAs: with two-tile items only, the last wave is badly quantised (320 tiles x 2 programs on
// 148 SMs: 12 CTAs get a second long item while 136 wait for a short one, then 24 short items are left for a wave of their own: the
// makespan is 3.2 short items for 2.4 of work per CTA).  One-tile items are half the work at a worse rate (no second slot to hide the MMA
// and the weight fetch behind: factor c2_single_penalty, measured), but they fill the tail.  The number of them is chosen by simulating the
// queue (greedy: a CTA that becomes free takes the next item) with a per-op cost model of the epilogue-bound kernel; the choice depends
// only on (tiles, programs), so it is cached.
inline double c2_single_penalty = 1.35;                  // time of a one-tile item / half the time of a two-tile item; <= 0: no one-tile items
inline double c2_prog_cost(const C2Prog& pr) {
  double c = 0.0;
  for (int i = 0; i < pr.n_ops; ++i) c += 0.3 + (double)pr.op[i].npad / 128.0;       // fixed hand-over + epilogue work ~ output chunks
  return c + 0.3 * pr.n_loads;
}
inline double c2_makespan(int tiles, int nprog, const double* cost, int sms, int ns1) {
  std::vector<double> heap(sms, 0.0);                    // min-heap of the CTAs' free times
  auto take = [&](double c) {
    std::pop_heap(heap.begin(), heap.end(), std::greater<double>());
    heap.back() += c;
    std::push_heap(heap.begin(), heap.end(), std::greater<double>());
  };
  const int np2 = (tiles - ns1 + 1) / 2;
  const double pen = c2_single_penalty > 0.0 ? c2_single_penalty : 1.35;
  for (int p = 0; p < nprog; ++p)
    for (int j = 0; j < np2; ++j) take(2 * j + 1 < tiles - ns1 ? cost[p] : 0.5 * pen * cost[p]);   // (an odd last pair holds one tile)
  for (int p = 0; p < nprog; ++p)
    for (int j = 0; j < ns1; ++j) take(0.5 * pen * cost[p]);
  return *std::max_element(heap.begin(), heap.end());
}
inline int c2_force_singles = -1;                         // tuning aid: >= 0 overrides the planner (rounded so that whole pairs stay in front)
inline int c2_pick_singles(int tiles, int nprog, const double* cost, int sms) {
  if (c2_force_singles >= 0) {
    int s1 = c2_force_singles < tiles ? c2_force_singles : tiles;
    if (s1 > 0 && ((tiles - s1) & 1)) s1 += s1 < tiles ? 1 : -1;
    return s1;
  }
  if (c2_single_penalty <= 0.0) return 0;
  struct Key { int tiles, nprog, sms; double c0, c1, pen; int ns1; };       // (c1: the sum of the other programs' costs)
  static thread_local Key cache[8];
  static thread_local int ncache = 0;
  double rest = 0.0;
  for (int k = 1; k < nprog; ++k) rest += cost[k] * (1.0 + 1e-3 * k);
  for (int i = 0; i < ncache; ++i) {
    const Key& k = cache[i];
    if (k.tiles == tiles && k.nprog == nprog && k.sms == sms && k.c0 == cost[0] && k.c1 == rest && k.pen == c2_single_penalty) return k.ns1;
  }
  int best = 0;
  double best_t = c2_makespan(tiles, nprog, cost, sms, 0);
  for (int s1 = 2 - (tiles & 1); s1 <= tiles && s1 <= 2 * sms; s1 += 2) {      // (tiles - s1) even: whole pairs in front
    const double t = c2_makespan(tiles, nprog, cost, sms, s1);
    if (t < best_t * (1.0 - 1e-9)) { best_t = t; best = s1; }
  }
  Key& k = cache[ncache < 8 ? ncache++ : 7];
  k = Key{tiles, nprog, sms, cost[0], rest, c2_single_penalty, best};
  return best;
}

inline int c2_sm_count() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  return sms;
}

inline int c2_bwd_reverse = 1;                            // tuning aid (dwbc_debug_set_chain_bwd_reverse): the backward launch walks the tiles downwards
inline int launch_chain2n(const C2Prog* const* prs, int nprog, const FinArgs& fin, bool x3, int* queue, cudaStream_t st, bool rev = false);
inline int launch_chain2(const C2Prog* pr0, const C2Prog* pr1, const FinArgs& fin, bool x3, int* queue, cudaStream_t st, bool rev = false) {
  const C2Prog* prs[2] = {pr0, pr1};
  return launch_chain2n(prs, pr1 ? 2 : 1, fin, x3, queue, st, rev);
}
// up to C2_MAX_PROGS programs over the same rows in one launch; queued longest program first
inline int launch_chain2n(const C2Prog* const* prs, int nprog, const FinArgs& fin, bool x3, int* queue, cudaStream_t st, bool rev) {
  if (nprog < 1 || nprog > C2_MAX_PROGS) return DWBC_ERR_ARG;
  C2Launch L{};
  L.rev = rev ? 1 : 0;
  L.nprog = nprog;
  L.x3 = x3 ? 1 : 0;
  L.queue = queue;
  L.fin = fin;
  int order[C2_MAX_PROGS];
  for (int k = 0; k < nprog; ++k) order[k] = k;
  std::stable_sort(order, order + nprog, [&](int a, int b) { return prs[a]->n_ops > prs[b]->n_ops; });
  for (int k = 0; k < nprog; ++k) L.p[k] = *prs[order[k]];
  for (int k = 0; k < L.nprog; ++k) {
    const C2Prog& pr = L.p[k];
    if (pr.M <= 0 || pr.M != L.p[0].M || pr.n_ops <= 0 || pr.n_ops > C2_MAX_OPS || pr.n_loads < 0 || pr.n_loads > C2_MAX_LOADS) return DWBC_ERR_ARG;
  }
  if (!queue) return DWBC_ERR_ARG;
#ifdef DWBC_C2_DROP_STORES      // timing experiments only (results invalid): no global activation stores
  for (int k = 0; k < L.nprog; ++k)
    for (int i = 0; i < L.p[k].n_ops; ++i) L.p[k].op[i].y = nullptr;
#endif
  const int sms = c2_sm_count();
  const int tiles = (L.p[0].M + TC_M - 1) / TC_M;
  if (tiles * L.nprog <= sms) {                            // small batches (rollout): one tile per item, spread over more SMs
    L.np2 = 0;
    L.ns1 = tiles;
  } else {
    double cost[C2_MAX_PROGS] = {};
    for (int k = 0; k < L.nprog; ++k) cost[k] = c2_prog_cost(L.p[k]);
    L.ns1 = c2_pick_singles(tiles, L.nprog, cost, sms);
    L.np2 = (tiles - L.ns1 + 1) / 2;
  }
  const int items = (L.np2 + L.ns1) * L.nprog;
  const int grid = items < sms ? items : sms;
  const size_t smem = (size_t)C2_SMEM_FLOATS * sizeof(float);
  static bool attr = false;
  if (!attr) {
    if (cudaFuncSetAttribute(chain2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return DWBC_ERR_LAUNCH;
    attr = true;
  }
  chain2_kernel<<<grid, C2_THREADS, smem, st>>>(L, tiles);
  ++dwbc_launch_counter;
  return cudaGetLastError() == cudaSuccess ? DWBC_OK : DWBC_ERR_LAUNCH;
}

}  // namespace dwbc
