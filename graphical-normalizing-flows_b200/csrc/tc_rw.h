// Internal interface of the resident weight-gradient tcgen05 kernel (tc_rw_wgrad.cu) for the other translation units.
#pragma once
#include "common.cuh"

#ifndef GNF_EMU
namespace gnf {

// dW[N x K] = dY^T X over Q rows (N, K <= 160; X a dense [Q][pad32(K)] plane), partial tiles in `partial`
// (rw_wgrad_partial_floats(K) floats), summed by a second kernel.
bool rw_wgrad_supported(int N, int K);
size_t rw_wgrad_partial_floats(int K);
// dY given as a masked rank-one product instead of a plane: dY[q][n] = g[q] w[n] if bit (n % 32) of bits[q * bits_ld + n / 32] else 0
// (the top of the UMNN backward: delta_L = (g_q w_L) o relu'(a_L))
struct RwRankOne { const float* g; const float* w; const uint32_t* bits; int bits_ld; };
int launch_rw_wgrad(const float* dY, long long lddy, const float* X, long long ldx, float* dW, long long lddw, int Q, int N, int K, int passes,
                    float* partial, cudaStream_t s, const Branches* br = nullptr, int side = 0, const RwRankOne* rank_one = nullptr);

}  // namespace gnf
#endif
