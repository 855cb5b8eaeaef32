// Internal interface of the tcgen05 GEMM engine (tc_gemm.cu) for the other translation units of libgnf_sm100.
#pragma once
#include "common.cuh"

#ifndef GNF_EMU
namespace gnf {

enum { TCG_EPI_BIAS_ACT = 0, TCG_EPI_MASK = 1, TCG_EPI_ATOMIC = 2 };
enum { TCG_SRC_K = 0, TCG_SRC_MN = 1 };  // global memory contiguous along the reduction index / along the row index

struct TcGemmParams {
  // C[m, n] = sum_k A(m, k) * B(n, k);  A: Mrows x Kred,  B: Ncols x Kred
  const float* A; long long lda; int a_src;    // TCG_SRC_K: A(m,k) = A[m*lda + k];  TCG_SRC_MN: A(m,k) = A[k*lda + m]
  const float* B; long long ldb; int b_src;    // same convention with n in place of m
  const float* B_lo;                           // 3xTF32 only, nullable: B is already rn_tf32(b) and B_lo = rn_tf32(b - B) (same layout):
                                               // both are TMA-loaded and the stagers skip the B split (weights: split once per call)
  int M, N, K;
  int BN, stages, passes, splits, k_per_split;
  int fold, acc_stride;                        // k-chunks per in-core accumulation group; TMEM columns between accumulator regions
  int epi;
  float* C; long long ldc;
  const float* bias; int bias_ld, bias_period, relu;   // TCG_EPI_BIAS_ACT
  const float* act; long long ldact;                    // TCG_EPI_MASK: keep dX where act > 0 ...
  const uint32_t* mask_bits; long long mask_ld;         // ... or where bit n of row m is set ([M][mask_ld] words; wins over act)
  uint32_t* bits_out; long long bits_ld;                // TCG_EPI_BIAS_ACT: also emit the bit mask (Y > 0), same layout
  float* rowsum;                                        // engine v2 wgrad only, nullable: rowsum[m] += sum_k A(m, k) (= the bias gradient, atomics)
  const float* rowterm; long long rt_ld; int rt_group;  // TCG_EPI_BIAS_ACT, nullable: C[m, n] also adds rowterm[(m / rt_group) * rt_ld + n]
                                                        // (the context term of a conditional DAG flow's layer 1: one row per sample)
  int use_tma, c_vec, act_vec, bias_vec, rt_vec;                  // set by launch_tc_gemm
  long long* trace;                                     // measurement: SM-clock stamps of CTA 0 (gnf_tc_gemm_set_trace)
};

// Enqueue C = A * B^T (+ epilogue) on the persistent warp-specialised tcgen05 kernel.  BN / stages / splits are chosen here.
int launch_tc_gemm(TcGemmParams p, cudaStream_t s);

}  // namespace gnf
#endif
