/* Profiling / tuning entry points of libdwbc.so.  NOT part of the drop-in boundary (include/dwbc.h): nothing in the product path calls
 * them; tools/ and tests/test_gpu_gemm.py do.  Declared here so that every exported symbol of the library has a header. */
#ifndef DWBC_DEBUG_H
#define DWBC_DEBUG_H
#include "dwbc.h"
#ifdef __cplusplus
extern "C" {
#endif

/* One GEMM of the selected implementation (tc: 0 = fp32 CUDA cores, 1 = TF32 tcgen05) on plain row-major device matrices.
 *   mode 0: Y[M,N] = act(X[M,K] W[N,K]^T + b)   mode 1: dX[M,N] = G[M,K] W[K,N]   mode 2: dW[M,N] += G[K,M]^T X[K,N], db += colsum(G)
 * act (mode 0): the library's internal activation codes, 0 none, 1 ELU, 2 tanh, 3 SELU, 4 ReLU, 5 leaky ReLU, 6 sigmoid; others DWBC_ERR_ARG */
int dwbc_debug_gemm(int mode, int tc, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                    const float* bias, float* dbias, int M, int N, int K, int act, dwbc_stream_t stream);

/* clock64 stamp buffers (device memory, NULL switches the stamps off): tcgen05 GEMM / chain kernels (64 slots per CTA), grouped
 * weight-gradient kernel, post-physics kernel */
int dwbc_debug_set_tc_cycle_buffer(unsigned long long* dev_ptr);
int dwbc_debug_set_wg_cycle_buffer(unsigned long long* dev_ptr);
int dwbc_debug_set_cycle_buffer(unsigned long long* dev_ptr);

/* Work-item planner of the fused chain kernel (mlp_chain2.cuh): assumed time ratio of a one-tile item to half a two-tile item
 * (<= 0: no one-tile items at the tail of a large launch), and a forced number of one-tile items per program (-1: planner decides) */
int dwbc_debug_set_chain_single_penalty(double ratio);
int dwbc_debug_set_chain_singles(int n);
/* The chain programs a call would launch, described without launching (host code, no GPU).  what: 0 = dwbc_policy_act, 1 = dwbc_critic_values,
 * 2 / 3 = forward + loss / backward launch of dwbc_ppo_minibatch_grad.  out = [nprog, pack items, per program: n_ops, n_loads, per op: N, kpad,
 * act, fin, fin_c, out_col0, has_global_output, output_is_tile_image]; returns the number of ints written or a negative DWBC_ERR_*. */
int dwbc_debug_describe_chain(const DwbcNetCfg* net, int32_t rows, int what, int hist_encoding, int sms, int32_t* out, int32_t out_len);
/* the planner on its own (host code, no GPU): items per program and simulated makespans with / without one-tile items */
int dwbc_debug_chain_plan(int tiles, int nprog, const double* cost, int sms, int* np2, int* ns1, double* span, double* span0);

/* Deal of the grouped weight-gradient work items (wgrad_group.cuh): 0 = round-robin in construction order (default), 1 = GEMMs
 * sorted by operand width, items dealt boustrophedon (measured slower: all CTAs reduce into the same dW at the same time) */
int dwbc_debug_set_wgrad_snake(int on);
/* tile order of the backward chain launch: 1 = from the last tile downwards (default), 0 = upwards */
int dwbc_debug_set_chain_bwd_reverse(int on);
/* slab order of the grouped weight-gradient launch: 1 = from the last rows downwards (default: the rows the backward chain touched last
 * are still in L2), 0 = upwards */
int dwbc_debug_set_wgrad_reverse(int on);
/* work items per CTA the slab length of the grouped weight-gradient launch aims at (default 4) */
int dwbc_debug_set_wgrad_items(int per_cta);

#ifdef __cplusplus
}
#endif
#endif
