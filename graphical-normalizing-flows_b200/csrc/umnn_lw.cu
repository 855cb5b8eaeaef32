// K3 (layer-wise): MonotonicNormalizer — the Clenshaw-Curtis UMNN integral as per-layer passes over all node-rows,
// with the hidden-layer GEMMs on the tcgen05 engine (tc_gemm.cu; 3xTF32 = fp32-equivalent, or single-pass TF32).
// (MonotonicNormalizer.forward / IntegrandNet, models/Normalizers/MonotonicNormalizer.py:12-66; UMNN==1.0
//  NeuralIntegral / ParallelNeuralIntegral forward + backward, SURVEY.md App. B.)
//
// The fused FFMA kernels of umnn.cu keep a 64-row tile on chip through every layer but are bound by the fp32 CUDA-core
// pipe.  Here every layer is one pass over ALL node-rows q = r*nodes + k (r = (sample, dim) row, k = quadrature node):
//   layer 0        a1[q] = relu(t_q * W0[:,0] + P[r]),  P = h W0[:,1:]^T + b0 computed ONCE per row r (the conditioning
//                  half of the first Linear is identical for all nodes of a row: 1/(S+1) of the reference's work)
//   layers 1..L-1  a_{l+1} = relu(a_l W_l^T + b_l)                       tensor-core GEMM, bias+ReLU epilogue
//   output         y = a_L . w_L + b_L, f = ELU(y)+1.05, CC-weighted sums -> z, jac, logdet
// and the backward mirrors it (out_bwd -> [wgrad, dgrad+ReLU-mask] per hidden layer -> layer-0 reductions).  Hidden
// activations live in HBM between passes ([L][Q][NP] fp32): 180 GB of HBM3e at ~7 TB/s buys tensor-core GEMMs for the
// 2*Q*I^2 layers, which are >95 % of the FLOPs.  In training one extra node-row per r (k = S+1, t = x, quadrature weight
// 0) carries the plain chain rule of the jac output, exactly like the fused backward.
#include "common.cuh"
#include "tc_gemm.h"
#include "tc_rw.h"
#include "tc_umnn3.h"

namespace gnf {

constexpr int kLwRL = 8;  // row lanes per block in the reduction kernels: blockDim = (NP/4) * kLwRL
constexpr int kOutBwdU = 3;  // node-rows in flight per thread in lw_out_bwd_kernel: 59 registers -> 3 blocks of 320 threads per SM, ~46 KB in flight

struct LwGeom {
  int R, d, E, S, nodes, NP, L;
  long long Q;  // R * nodes
};

__device__ __forceinline__ float lw_node_abscissa(float xv, const float* __restrict__ ccn, int kn, int S) {
  return (kn <= S) ? (xv * (__ldg(ccn + kn) + 1.f)) / 2.f : xv;
}

// Zero-padded copy of a hidden weight matrix: Wp[n][k], ld = NP (16-byte vector loads for both GEMM orientations).
__global__ void lw_pad_weight_kernel(const float* __restrict__ W, int N, int K, float* __restrict__ Wp, int NP, int rows) {
  const int total = rows * NP;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int n = i / NP, k = i % NP;
    Wp[i] = (n < N && k < K) ? W[(size_t)n * K + k] : 0.f;
  }
}

// a1[q][c] = relu(t_q * W0[c][0] + P[r][c]) for c < N1, 0 in the padding columns.  bits (nullable): ReLU mask of a1, one bit per
// element, [Q][NP/32] words (8 consecutive lanes own one word: nibbles combined by shuffles).
// Block = (NP/4) column quads x kLwRL row lanes: a thread's column quad is fixed, rows advance by a grid stride (the first
// version decoded a flat 64-bit element index with two 64-bit divisions per float4: 43 us for an 89 MB plane).
__global__ void lw_layer1_fwd_kernel(const float* __restrict__ x, const float* __restrict__ ccn, const float* __restrict__ P,
                                     const float* __restrict__ W0, int ldw0, int N1, float* __restrict__ a1,
                                     uint32_t* __restrict__ bits, LwGeom g) {
  const int C4 = g.NP / 4;                               // multiple of 8: 8 consecutive lanes cover one 32-column word of one row
  const int c4 = threadIdx.x % C4, rl = threadIdx.x / C4, c = 4 * c4;
  float w[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) w[e] = (c + e < N1) ? __ldg(W0 + (size_t)(c + e) * ldw0) : 0.f;
  const int Q = (int)g.Q;
  for (int q0 = blockIdx.x * kLwRL; q0 < Q; q0 += gridDim.x * kLwRL) {   // uniform trip count per block: the shuffles below are warp-wide
    const int q = q0 + rl;
    const bool valid = q < Q;
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) {
      const int r = q / g.nodes, kn = q - r * g.nodes;
      const float t = lw_node_abscissa(__ldg(x + r), ccn, kn, g.S);
      const float4 pv = __ldg(reinterpret_cast<const float4*>(P + (size_t)r * g.NP + c));
      o.x = (c + 0 < N1) ? fmaxf(fmaf(t, w[0], pv.x), 0.f) : 0.f;
      o.y = (c + 1 < N1) ? fmaxf(fmaf(t, w[1], pv.y), 0.f) : 0.f;
      o.z = (c + 2 < N1) ? fmaxf(fmaf(t, w[2], pv.z), 0.f) : 0.f;
      o.w = (c + 3 < N1) ? fmaxf(fmaf(t, w[3], pv.w), 0.f) : 0.f;
      *reinterpret_cast<float4*>(a1 + (size_t)q * g.NP + c) = o;
    }
    if (bits) {
      uint32_t wv = ((o.x > 0.f ? 1u : 0u) | (o.y > 0.f ? 2u : 0u) | (o.z > 0.f ? 4u : 0u) | (o.w > 0.f ? 8u : 0u)) << (4 * (threadIdx.x & 7));
      wv |= __shfl_xor_sync(0xffffffffu, wv, 1);
      wv |= __shfl_xor_sync(0xffffffffu, wv, 2);
      wv |= __shfl_xor_sync(0xffffffffu, wv, 4);
      if (valid && (threadIdx.x & 7) == 0) bits[(size_t)q * (g.NP / 32) + (c >> 5)] = wv;
    }
  }
}

// One warp per row r; 8 lanes per node-row (4 node-rows in flight per warp), float4 loads, shuffle reductions.
// J = NP / 32 float4 per lane and node-row (compile time: the first version kept 8 x 4 weight registers and 8 guarded
// loads for any width -- 104 registers, 21 % occupancy, 61 us for an 89 MB plane).
template <int J>
__global__ void __launch_bounds__(256, 4) lw_out_fwd_kernel(const float* __restrict__ aL, const float* __restrict__ wl, const float* __restrict__ bl,
                                                             int NL, const float* __restrict__ x, const float* __restrict__ h,
                                                             const float* __restrict__ ccw, float* __restrict__ z, float* __restrict__ zrev,
                                                             float* __restrict__ jac, float* __restrict__ logdet, float* __restrict__ ysave,
                                                             LwGeom g) {
  const int lane = threadIdx.x & 31, grp = lane >> 3, sub = lane & 7;
  float4 w[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int c = (j * 8 + sub) * 4;
    w[j].x = (c + 0 < NL) ? __ldg(wl + c + 0) : 0.f;
    w[j].y = (c + 1 < NL) ? __ldg(wl + c + 1) : 0.f;
    w[j].z = (c + 2 < NL) ? __ldg(wl + c + 2) : 0.f;
    w[j].w = (c + 3 < NL) ? __ldg(wl + c + 3) : 0.f;
  }
  const float blast = __ldg(bl);
  const int wpb = blockDim.x >> 5;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < g.R; r += gridDim.x * wpb) {
    const float xv = __ldg(x + r);
    float s = 0.f;
    for (int kn0 = 0; kn0 < g.nodes; kn0 += 4) {
      const int kn = kn0 + grp;
      const bool valid = kn < g.nodes;
      const long long q = (long long)r * g.nodes + kn;
      float4 v[J];
      if (valid) {
        const float4* row = reinterpret_cast<const float4*>(aL + (size_t)q * g.NP) + sub;
#pragma unroll
        for (int j = 0; j < J; ++j) v[j] = __ldg(row + 8 * j);
      } else {
#pragma unroll
        for (int j = 0; j < J; ++j) v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      // the FFMA engine leaves the padding columns of a plane unwritten: select, do not multiply by a zero weight
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < J; ++j) {
        const int c = (j * 8 + sub) * 4;
        if (c + 0 < NL) acc = fmaf(v[j].x, w[j].x, acc);
        if (c + 1 < NL) acc = fmaf(v[j].y, w[j].y, acc);
        if (c + 2 < NL) acc = fmaf(v[j].z, w[j].z, acc);
        if (c + 3 < NL) acc = fmaf(v[j].w, w[j].w, acc);
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      if (valid && sub == 0) {
        const float y = acc + blast;
        const float f = (y > 0.f ? y : expm1f(y)) + 1.05f;
        if (ysave) ysave[q] = y;
        if (kn <= g.S) s = fmaf(__ldg(ccw + kn), f, s);
        if (kn == 0) {
          jac[r] = f;
          if (logdet) atomicAdd(logdet + r / g.d, logf(f));
        }
      }
    }
    s += __shfl_xor_sync(0xffffffffu, s, 8);
    s += __shfl_xor_sync(0xffffffffu, s, 16);
    if (lane == 0) {
      const float zv = s * xv / 2.f + __ldg(h + (size_t)r * g.E);
      z[r] = zv;
      if (zrev) { const int b = r / g.d, i = r % g.d; zrev[(size_t)b * g.d + (g.d - 1 - i)] = zv; }
    }
  }
}

__device__ __forceinline__ float lw_gz_total(const float* __restrict__ gz, const float* __restrict__ gzrev, int r, int d) {
  float v = gz ? __ldg(gz + r) : 0.f;
  if (gzrev) { const int b = r / d, i = r % d; v += __ldg(gzrev + (size_t)b * d + (d - 1 - i)); }
  return v;
}

// Cotangent of the pre-ELU output per node-row, last-layer gradients and delta_L = (gy w_L) o relu'(a_L):
//   dW_L[c] += sum_q gy_q a_L[q][c];  db_L += sum_q gy_q;  db_{L-1}[c] += sum_q delta_L[q][c].
// Block = (NP/4) column lanes x kLwRL row lanes; per-thread column partials, one shared-memory reduction per block.
__global__ void lw_out_bwd_kernel(const float* __restrict__ aL, const float* __restrict__ ysave, const float* __restrict__ wl, int NL,
                                  const float* __restrict__ x, const float* __restrict__ ccw, const float* __restrict__ jac,
                                  const float* __restrict__ gz, const float* __restrict__ gzrev, const float* __restrict__ gjac,
                                  const float* __restrict__ glogdet, float* __restrict__ dL, float* __restrict__ gq_out, float* __restrict__ dWl,
                                  float* __restrict__ dbl, float* __restrict__ dbprev, LwGeom g) {
  GNF_SMEM(float, red);                       // [kLwRL][NP] + [kLwRL]
  const int C4 = g.NP / 4;
  const int c4 = threadIdx.x % C4, rl = threadIdx.x / C4, c = 4 * c4;
  float w[4], sW[4] = {0.f, 0.f, 0.f, 0.f}, sB[4] = {0.f, 0.f, 0.f, 0.f}, sy = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) w[e] = (c + e < NL) ? __ldg(wl + c + e) : 0.f;
  // Q < 2^31 (lw_plan): 32-bit indices; (r, kn) of a thread's node-row advance incrementally -- a 64-bit q / nodes per row
  // is a function call (CALL.REL) -- and kOutBwdU node-rows are in flight per thread
  const int Q = (int)g.Q;
  const int per = (Q + gridDim.x - 1) / gridDim.x;
  const int q0 = blockIdx.x * per;
  const int q1 = (q0 + per < Q) ? q0 + per : Q;
  int q = q0 + rl;
  int r = q / g.nodes, kn = q - r * g.nodes;
  const int dr = kLwRL / g.nodes, dk = kLwRL - dr * g.nodes;     // q += kLwRL  ==  (r, kn) += (dr, dk) with one carry
  for (; q < q1; q += kOutBwdU * kLwRL) {
    int rr[kOutBwdU], kk[kOutBwdU];
    float4 av[kOutBwdU];
    float ys[kOutBwdU];
    bool ok[kOutBwdU];
#pragma unroll
    for (int u = 0; u < kOutBwdU; ++u) {
      rr[u] = r; kk[u] = kn;
      ok[u] = q + u * kLwRL < q1;
      const int qq = ok[u] ? q + u * kLwRL : q;             // clamped address, masked at use
      av[u] = __ldg(reinterpret_cast<const float4*>(aL + (size_t)qq * g.NP + c));
      ys[u] = __ldg(ysave + qq);
      r += dr; kn += dk;
      if (kn >= g.nodes) { kn -= g.nodes; ++r; }
    }
#pragma unroll
    for (int u = 0; u < kOutBwdU; ++u) {
      if (!ok[u]) continue;
      const int ru = rr[u];
      float gq;
      if (kk[u] <= g.S) {
        gq = (lw_gz_total(gz, gzrev, ru, g.d) * __ldg(x + ru) / 2.f) * __ldg(ccw + kk[u]);
      } else {
        gq = gjac ? __ldg(gjac + ru) : 0.f;
        if (glogdet) gq += __ldg(glogdet + ru / g.d) / __ldg(jac + ru);
      }
      const float y = ys[u];
      gq *= (y > 0.f) ? 1.f : expf(y);
      const float a[4] = {c + 0 < NL ? av[u].x : 0.f, c + 1 < NL ? av[u].y : 0.f, c + 2 < NL ? av[u].z : 0.f, c + 3 < NL ? av[u].w : 0.f};
      float o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        sW[e] = fmaf(gq, a[e], sW[e]);
        o[e] = a[e] > 0.f ? gq * w[e] : 0.f;
        sB[e] += o[e];
      }
      // gq_out: the caller's weight-gradient kernel rebuilds delta_L = (g_q w_L) o relu'(a_L) from g_q and the saved ReLU bit mask --
      // one float per node-row leaves instead of a [Q][NP] plane (89 MB at cfg4, written here and read back there)
      if (gq_out) { if (c4 == 0) gq_out[q + u * kLwRL] = gq; }
      else *reinterpret_cast<float4*>(dL + (size_t)(q + u * kLwRL) * g.NP + c) = make_float4(o[0], o[1], o[2], o[3]);
      if (c4 == 0) sy += gq;
    }
  }
  float* ry = red + kLwRL * g.NP;
  for (int pass = 0; pass < 2; ++pass) {
    const float* src = pass == 0 ? sW : sB;
#pragma unroll
    for (int e = 0; e < 4; ++e) red[rl * g.NP + c + e] = src[e];
    if (pass == 0 && c4 == 0) ry[rl] = sy;
    __syncthreads();
    if (rl == 0) {
      float* dst = pass == 0 ? dWl : dbprev;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (c + e < NL) {
          float s = 0.f;
          for (int k = 0; k < kLwRL; ++k) s += red[k * g.NP + c + e];
          atomicAdd(dst + c + e, s);
        }
      }
      if (pass == 0 && c4 == 0) {
        float s = 0.f;
        for (int k = 0; k < kLwRL; ++k) s += ry[k];
        atomicAdd(dbl, s);
      }
    }
    __syncthreads();
  }
}

// First-layer reductions over delta_1 [Q][NP]:
//   D[r][c]     = sum_k delta_1[(r,k)][c]                   (-> dh = D W0[:,1:], dW0[:,1:] = D^T h, db0 = colsum D)
//   dW0[c][0]  += sum_q delta_1[q][c] * t_q
//   dx[r]       = delta_1[(r,S+1)] . W0[:,0]  +  jac[r] * gz[r]         (chain rule of the jac output + Leibniz rule)
// Block = (NP/4) column quads x kLwRL row lanes; a row lane owns WHOLE rows r (all nodes of the row, four 16-byte loads in
// flight per thread), so D[r] leaves from registers and the only block-wide exchange per batch of kLwRL rows is the dx dot
// product (one __syncthreads per batch, double-buffered partials).  (The first version split the nodes of ONE row over the row
// lanes: <= 3 loads per thread between two block barriers per row -- latency-bound at 1.3 TB/s, 67 us for an 89 MB plane.)
__global__ void lw_layer1_bwd_kernel(const float* __restrict__ d1, const float* __restrict__ x, const float* __restrict__ ccn,
                                     const float* __restrict__ W0, int ldw0, int N1, const float* __restrict__ jac,
                                     const float* __restrict__ gz, const float* __restrict__ gzrev, float* __restrict__ D,
                                     float* __restrict__ dW0, float* __restrict__ db0, float* __restrict__ dx, LwGeom g) {
  GNF_SMEM(float, red);                       // [kLwRL][NP]; the loop uses its first 2*kLwRL*(NP/4) floats for the dx partials
  const int C4 = g.NP / 4;
  const int c4 = threadIdx.x % C4, rl = threadIdx.x / C4, c = 4 * c4;
  float w[4], sT[4] = {0.f, 0.f, 0.f, 0.f}, sD[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int e = 0; e < 4; ++e) w[e] = (c + e < N1) ? __ldg(W0 + (size_t)(c + e) * ldw0) : 0.f;
  const bool m0 = c + 0 < N1, m1 = c + 1 < N1, m2 = c + 2 < N1, m3 = c + 3 < N1;
  const int per = ((g.R + gridDim.x - 1) / gridDim.x + kLwRL - 1) / kLwRL * kLwRL;    // whole batches of kLwRL rows per block
  const int r0 = blockIdx.x * per, r1 = (r0 + per < g.R) ? r0 + per : g.R;
  int it = 0;
  for (int rb = r0; rb < r1; rb += kLwRL, ++it) {          // uniform trip count per block
    const int r = rb + rl;
    const bool valid = r < r1;
    float dot = 0.f;
    if (valid) {
      const float xv = __ldg(x + r);
      const float* row = d1 + (size_t)r * g.nodes * g.NP + c;
      float Dp[4] = {0.f, 0.f, 0.f, 0.f};
      for (int kn0 = 0; kn0 < g.nodes; kn0 += 4) {
        float4 dv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {                      // unconditional loads from clamped addresses, masked at use
          const int kn = (kn0 + u < g.nodes) ? kn0 + u : g.nodes - 1;
          dv[u] = __ldg(reinterpret_cast<const float4*>(row + (size_t)kn * g.NP));
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int kn = kn0 + u;
          if (kn < g.nodes) {
            const float t = lw_node_abscissa(xv, ccn, kn, g.S);
            const float v[4] = {m0 ? dv[u].x : 0.f, m1 ? dv[u].y : 0.f, m2 ? dv[u].z : 0.f, m3 ? dv[u].w : 0.f};
#pragma unroll
            for (int e = 0; e < 4; ++e) { Dp[e] += v[e]; sT[e] = fmaf(v[e], t, sT[e]); }
            if (kn == g.S + 1) dot = (v[0] * w[0] + v[1] * w[1]) + (v[2] * w[2] + v[3] * w[3]);
          }
        }
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) sD[e] += Dp[e];
      *reinterpret_cast<float4*>(D + (size_t)r * g.NP + c) = make_float4(Dp[0], Dp[1], Dp[2], Dp[3]);
    }
    float* part = red + (it & 1) * (kLwRL * C4);
    part[rl * C4 + c4] = dot;
    __syncthreads();
    if (valid && c4 == 0) {
      float s = 0.f;
      for (int k = 0; k < C4; ++k) s += part[rl * C4 + k];
      dx[r] = s + __ldg(jac + r) * lw_gz_total(gz, gzrev, r, g.d);
    }
  }
  for (int pass = 0; pass < 2; ++pass) {
    __syncthreads();
    const float* src = pass == 0 ? sT : sD;
#pragma unroll
    for (int e = 0; e < 4; ++e) red[rl * g.NP + c + e] = src[e];
    __syncthreads();
    if (rl == 0) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (c + e < N1) {
          float s = 0.f;
          for (int k = 0; k < kLwRL; ++k) s += red[k * g.NP + c + e];
          if (pass == 0) atomicAdd(dW0 + (size_t)(c + e) * ldw0, s);
          else atomicAdd(db0 + c + e, s);
        }
      }
    }
  }
}

// z = integral + h[..., 0]: the first conditioning feature also receives gz directly.
__global__ void lw_finish_dh_kernel(float* __restrict__ dh, int E, const float* __restrict__ gz, const float* __restrict__ gzrev, int R, int d) {
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < R; r += gridDim.x * blockDim.x) dh[(size_t)r * E] += lw_gz_total(gz, gzrev, r, d);
}

static int g_lw_use_rw_wgrad = 1;   // measurement switch (gnf_umnn_lw_set_rw bit 1): 0 = wgrad on the generic tensor-core engine
static int g_lw_use_rw = 1;   // measurement switch (gnf_umnn_lw_set_rw): 0 = hidden GEMMs on the generic tensor-core engine

struct LwPlan {
  int L, NP, E, nodes;
  int rw;          // hidden layers fit the resident-weight tensor-core kernel (tc_rw.cu)
  long long Q;
  size_t off_P, off_Wp[GNF_MAX_LAYERS], off_dA, off_dB, off_D, off_part, total;  // workspace offsets in floats
};

static int lw_plan(const gnf_mlp_t* net, int R, int S, int train, int backward, LwPlan* pl) {
  if (!net || net->n_layers < 2 || net->n_layers > GNF_MAX_LAYERS) return fail(GNF_ERR_UNSUPPORTED, "umnn (layer-wise): integrand needs 2..%d linear layers", GNF_MAX_LAYERS);
  if (net->dims[net->n_layers] != 1) return fail(GNF_ERR_UNSUPPORTED, "umnn (layer-wise): integrand output size must be 1");
  if (net->dims[0] < 2) return fail(GNF_ERR_UNSUPPORTED, "umnn (layer-wise): needs at least one conditioning feature");
  if (R < 0 || S < 1) return fail(GNF_ERR_INVALID, "umnn (layer-wise): bad R / S");
  const int L = net->n_layers - 1;
  int maxh = 0;
  for (int l = 1; l <= L; ++l) maxh = net->dims[l] > maxh ? net->dims[l] : maxh;
  if (maxh < 1 || maxh > 256) return fail(GNF_ERR_UNSUPPORTED, "umnn (layer-wise): hidden widths must be in 1..256 (got %d)", maxh);
  pl->L = L;
  pl->NP = (maxh + 31) / 32 * 32;
  pl->E = net->dims[0] - 1;
  pl->nodes = S + 1 + (train ? 1 : 0);
  pl->Q = (long long)R * pl->nodes;
  if (pl->Q > 0x7fffffffLL) return fail(GNF_ERR_UNSUPPORTED, "umnn (layer-wise): %lld node-rows exceed the GEMM engine's row index range", pl->Q);
  size_t off = 0;
  const size_t plane = (size_t)pl->Q * pl->NP;
  pl->off_P = off; off += (size_t)R * pl->NP;            // forward: P;  backward: D (same shape)
  pl->off_D = pl->off_P;
#ifdef GNF_EMU
  pl->rw = 0;
#else
  pl->rw = 1;                                              // every hidden layer, both directions (dgrad swaps N and K)
  for (int l = 1; l < L; ++l)
    if (!rw_supported(net->dims[l + 1], net->dims[l]) || !rw_supported(net->dims[l], net->dims[l + 1])) pl->rw = 0;
#endif
  // per hidden layer: the zero-padded weight copy (generic engines) or the hi/lo TF32 images + bias (resident-weight kernel)
  for (int l = 1; l < L; ++l) { pl->off_Wp[l] = off; off += (size_t)2 * pl->NP * pl->NP + pl->NP; }
  pl->off_dA = pl->off_dB = 0;
  pl->off_part = 0;
  if (backward) {
    pl->off_dA = off; off += plane;
    pl->off_dB = off; off += plane;
#ifndef GNF_EMU
    if (pl->rw) { pl->off_part = off; off += rw_wgrad_partial_floats(pl->NP); }   // per-CTA partial tiles of the wgrad kernel
#endif
  }
  pl->total = off;
  return 0;
}

static inline int lw_blocks(long long work_items, int per_block, int max_per_sm) {
  long long b = (work_items + per_block - 1) / per_block;
  const long long cap = (long long)kNumSMs * max_per_sm;
  if (b > cap) b = cap;
  return b < 1 ? 1 : (int)b;
}

// Y = act(X W^T + b) / dX = (dY W) o relu'(act) / dW = dY^T X through the selected GEMM engine.
// passes: 0 = strict FFMA tile GEMM, 1 = TF32, 3 = 3xTF32 (tcgen05).
static int lw_fwd_gemm(const float* X, int ldx, const float* W, int ldw, const float* bias, float* Y, int ldy, int M, int N, int K,
                       int relu, uint32_t* bits_out, int bits_ld, int passes, int rw_np, cudaStream_t s) {
  if (passes == 0) return gnf_linear_fwd(X, ldx, W, ldw, bias, 1, Y, ldy, M, N, K, relu, (gnf_stream_t)s);
#ifdef GNF_EMU
  return fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (rw_np) {                                           // W = packed hi/lo images + bias (rw_pack_image)
    RwGemmParams r = {};
    r.A = X; r.lda = ldx; r.C = Y; r.ldc = ldy; r.image = W;
    r.M = M; r.NP = rw_np; r.KP = (K + 7) / 8 * 8; r.passes = passes; r.epi = RW_EPI_BIAS_ACT; r.relu = relu;
    r.bits_out = bits_out; r.bits_ld = bits_ld;
    if (int e = launch_rw_gemm(r, s)) return e;
    return check_launch("gnf_umnn_fwd_lw (resident-weight GEMM)");
  }
  TcGemmParams p = {};
  p.A = X; p.lda = ldx; p.a_src = TCG_SRC_K;
  p.B = W; p.ldb = ldw; p.b_src = TCG_SRC_K;
  p.M = M; p.N = N; p.K = K; p.passes = passes;
  p.epi = TCG_EPI_BIAS_ACT; p.C = Y; p.ldc = ldy; p.bias = bias; p.bias_ld = N; p.bias_period = 1; p.relu = relu;
  p.bits_out = bits_out; p.bits_ld = bits_ld;
  if (int e = launch_tc_gemm(p, s)) return e;
  return check_launch("gnf_umnn_fwd_lw (GEMM)");
#endif
}
static int lw_dgrad_gemm(const float* dY, int lddy, const float* W, int ldw, const float* act, int ldact, const uint32_t* mask_bits,
                         int mask_ld, float* dX, int lddx, int M, int N, int K, int passes, int rw_np, cudaStream_t s) {
  if (passes == 0) return gnf_linear_dgrad(dY, lddy, W, ldw, act, ldact, dX, lddx, M, N, K, (gnf_stream_t)s);
#ifdef GNF_EMU
  return fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (rw_np) {                                           // W = packed hi/lo images of the TRANSPOSED weights
    RwGemmParams r = {};
    r.A = dY; r.lda = lddy; r.C = dX; r.ldc = lddx; r.image = W;
    r.M = M; r.NP = rw_np; r.KP = (N + 7) / 8 * 8; r.passes = passes; r.epi = RW_EPI_MASK;   // reduction over the out-features
    r.mask_bits = mask_bits; r.mask_ld = mask_ld; r.act = act; r.ldact = ldact;
    if (int e = launch_rw_gemm(r, s)) return e;
    return check_launch("gnf_umnn_bwd_lw (resident-weight GEMM)");
  }
  TcGemmParams p = {};
  p.A = dY; p.lda = lddy; p.a_src = TCG_SRC_K;
  p.B = W; p.ldb = ldw; p.b_src = TCG_SRC_MN;
  p.M = M; p.N = K; p.K = N; p.passes = passes;
  p.epi = TCG_EPI_MASK; p.C = dX; p.ldc = lddx; p.act = act; p.ldact = ldact; p.mask_bits = mask_bits; p.mask_ld = mask_ld;
  if (int e = launch_tc_gemm(p, s)) return e;
  return check_launch("gnf_umnn_bwd_lw (GEMM)");
#endif
}
static int lw_wgrad_gemm(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, int M, int N, int K, int passes,
                         float* rw_partial, cudaStream_t s) {
  if (passes == 0) return gnf_linear_wgrad(dY, lddy, X, ldx, dW, lddw, M, N, K, (gnf_stream_t)s);
#ifndef GNF_EMU
  if (rw_partial) {                                      // lane = output row: dY^T goes to TMEM untransposed (tc_rw_wgrad.cu)
    if (int e = launch_rw_wgrad(dY, lddy, X, ldx, dW, lddw, M, N, K, passes, rw_partial, s)) return e;
    return check_launch("gnf_umnn_bwd_lw (resident wgrad)");
  }
#endif
  return gnf_linear_wgrad_tc(dY, lddy, X, ldx, dW, lddw, M, N, K, passes, (gnf_stream_t)s);
}

// Per-call weight staging of the hidden layers: hi/lo TF32 images for the resident-weight kernel (transposed for the
// dgrad direction), else zero-padded copies for the generic engines.
static void lw_pad_weights(const gnf_mlp_t* net, const LwPlan& pl, float* ws, int use_rw, int transpose, cudaStream_t s) {
  for (int l = 1; l < pl.L; ++l) {
#ifndef GNF_EMU
    if (use_rw) {
      if (transpose) rw_pack_image(net->W[l], net->dims[l], net->dims[l], net->dims[l + 1], 1, nullptr, ws + pl.off_Wp[l], pl.NP, (net->dims[l + 1] + 7) / 8 * 8, s);
      else rw_pack_image(net->W[l], net->dims[l], net->dims[l + 1], net->dims[l], 0, net->b[l], ws + pl.off_Wp[l], pl.NP, (net->dims[l] + 7) / 8 * 8, s);
      continue;
    }
#endif
    GNF_LAUNCH(lw_pad_weight_kernel, lw_blocks((long long)pl.NP * pl.NP, 256, 2), 256, 0, s, net->W[l], net->dims[l + 1], net->dims[l],
               ws + pl.off_Wp[l], pl.NP, pl.NP);
  }
}

}  // namespace gnf

using namespace gnf;

extern "C" {

#ifdef GNF_DEVTOOLS
int gnf_umnn_lw_set_rw(int enable) {
  g_lw_use_rw = (enable & 1) != 0;
  g_lw_use_rw_wgrad = (enable & 1) != 0 && (enable & 2) == 0;      // 1: everything resident; 3: forward/dgrad only; 0: generic engine
  return 0;
}
#endif

size_t gnf_umnn_lw_saved_floats(const gnf_mlp_t* net, int R, int S, int train) {
  LwPlan pl;
  if (lw_plan(net, R, S, train, 0, &pl)) return 0;
  // L activation planes [Q][NP], y [Q], and (training) the ReLU bit masks of a_1..a_{L-1}: [Q][NP/32] words each
  return (size_t)pl.L * pl.Q * pl.NP + (size_t)pl.Q + (train ? (size_t)(pl.L - 1) * pl.Q * (pl.NP / 32) : 0);
}

size_t gnf_umnn_lw_workspace_bytes(const gnf_mlp_t* net, int R, int S, int backward) {
  LwPlan pl;
  if (lw_plan(net, R, S, 1, backward, &pl)) return 0;
  return (pl.total + 4) * sizeof(float);
}

int gnf_umnn_fwd_lw(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn, float* z,
                    float* zrev, float* jac, float* logdet, float* saved, int train, int passes, int R, int d, void* work,
                    size_t work_bytes, gnf_stream_t stream) {
  if (!x || !h || !net || !ccw || !ccn || !z || !jac || !saved || R < 0 || d <= 0 || S < 1 || (R % d) != 0) return fail(GNF_ERR_INVALID, "gnf_umnn_fwd_lw: bad arguments");
  if (passes != 0 && passes != 1 && passes != 3) return fail(GNF_ERR_INVALID, "gnf_umnn_fwd_lw: passes must be 0 (FFMA), 1 (TF32) or 3 (3xTF32)");
  LwPlan pl;
  if (int e = lw_plan(net, R, S, train, 0, &pl)) return e;
  if (!work || work_bytes < pl.total * sizeof(float)) return fail(GNF_ERR_WORKSPACE, "gnf_umnn_fwd_lw: workspace too small (%zu < %zu)", work_bytes, pl.total * sizeof(float));
  cudaStream_t s = (cudaStream_t)stream;
  if (R == 0) return 0;
  float* ws = (float*)work;
  const int NP = pl.NP, L = pl.L, E = pl.E;
  const size_t plane = (size_t)pl.Q * NP;
  LwGeom g;
  g.R = R; g.d = d; g.E = E; g.S = S; g.nodes = pl.nodes; g.NP = NP; g.L = L; g.Q = pl.Q;
  if (logdet) cudaMemsetAsync(logdet, 0, (size_t)(R / d) * sizeof(float), s);
  // P = h W0[:,1:]^T + b0  (once per row r; strict fp32 on the FFMA engine: R x N1 x E is tiny)
  float* P = ws + pl.off_P;
  if (int e = gnf_linear_fwd(h, E, net->W[0] + 1, 1 + E, net->b[0], 1, P, NP, R, net->dims[1], E, 0, stream)) return e;
  const int use_rw = (pl.rw && passes != 0 && g_lw_use_rw) ? 1 : 0;
  lw_pad_weights(net, pl, ws, use_rw, 0, s);
  // ReLU bit masks of a_1 .. a_{L-1} (what the backward's dgrad epilogues consume), kept only when training on the tensor cores
  const int WB = NP / 32;
  const size_t bplane = (size_t)pl.Q * WB;
  uint32_t* bits = (train && passes != 0 && L > 1) ? reinterpret_cast<uint32_t*>(saved + (size_t)L * plane + pl.Q) : nullptr;
  GNF_LAUNCH(lw_layer1_fwd_kernel, lw_blocks(pl.Q, kLwRL * 4, 6), (NP / 4) * kLwRL, 0, s, x, ccn, P, net->W[0], 1 + E,
             net->dims[1], saved, bits, g);
  for (int l = 1; l < L; ++l) {
    uint32_t* bo = (bits && l + 1 < L) ? bits + (size_t)l * bplane : nullptr;     // mask of a_{l+1}
    if (int e = lw_fwd_gemm(saved + (size_t)(l - 1) * plane, NP, ws + pl.off_Wp[l], NP, net->b[l], saved + (size_t)l * plane, NP,
                            (int)pl.Q, net->dims[l + 1], net->dims[l], 1, bo, WB, passes, use_rw ? NP : 0, s)) return e;
  }
  float* ysave = saved + (size_t)L * plane;
  {
    const float* aLp = saved + (size_t)(L - 1) * plane;
    const int nb = lw_blocks(R, 8, 8);
#define LW_OUT_FWD(J) case J: GNF_LAUNCH(lw_out_fwd_kernel<J>, nb, 256, 0, s, aLp, net->W[L], net->b[L], net->dims[L], x, h, ccw, z, zrev, jac, logdet, ysave, g); break;
    switch (NP / 32) { LW_OUT_FWD(1) LW_OUT_FWD(2) LW_OUT_FWD(3) LW_OUT_FWD(4) LW_OUT_FWD(5) LW_OUT_FWD(6) LW_OUT_FWD(7) default: LW_OUT_FWD(8) }
#undef LW_OUT_FWD
  }
  return check_launch("gnf_umnn_fwd_lw");
}

int gnf_umnn_bwd_lw(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn, const float* jac,
                    const float* gz, const float* gzrev, const float* gjac, const float* glogdet, const float* saved, float* dx,
                    float* dh, const gnf_mlp_grad_t* grads, int passes, int R, int d, void* work, size_t work_bytes,
                    gnf_stream_t stream) {
  if (!x || !h || !net || !ccw || !ccn || !jac || !saved || !dx || !dh || !grads || R < 0 || d <= 0 || S < 1 || (R % d) != 0) return fail(GNF_ERR_INVALID, "gnf_umnn_bwd_lw: bad arguments");
  if (passes != 0 && passes != 1 && passes != 3) return fail(GNF_ERR_INVALID, "gnf_umnn_bwd_lw: passes must be 0 (FFMA), 1 (TF32) or 3 (3xTF32)");
  LwPlan pl;
  if (int e = lw_plan(net, R, S, 1, 1, &pl)) return e;
  if (!work || work_bytes < pl.total * sizeof(float)) return fail(GNF_ERR_WORKSPACE, "gnf_umnn_bwd_lw: workspace too small (%zu < %zu)", work_bytes, pl.total * sizeof(float));
  cudaStream_t s = (cudaStream_t)stream;
  const int NP = pl.NP, L = pl.L, E = pl.E;
  for (int l = 0; l < net->n_layers; ++l) {
    if (!grads->dW[l] || !grads->db[l]) return fail(GNF_ERR_INVALID, "gnf_umnn_bwd_lw: gradient pointer %d is NULL", l);
    cudaMemsetAsync(grads->dW[l], 0, (size_t)net->dims[l] * net->dims[l + 1] * sizeof(float), s);
    cudaMemsetAsync(grads->db[l], 0, (size_t)net->dims[l + 1] * sizeof(float), s);
  }
  if (R == 0) return check_launch("gnf_umnn_bwd_lw");
  float* ws = (float*)work;
  const size_t plane = (size_t)pl.Q * NP;
  LwGeom g;
  g.R = R; g.d = d; g.E = E; g.S = S; g.nodes = pl.nodes; g.NP = NP; g.L = L; g.Q = pl.Q;
  const int use_rw = (pl.rw && passes != 0 && g_lw_use_rw) ? 1 : 0;
  lw_pad_weights(net, pl, ws, use_rw, 1, s);
  float* dcur = ws + pl.off_dA;
  float* dnxt = ws + pl.off_dB;
  const int red_threads = (NP / 4) * kLwRL;
  const size_t red_smem = ((size_t)kLwRL * NP + kLwRL + 4) * sizeof(float);
  const float* ysave = saved + (size_t)L * plane;
  // output layer: delta_L, dW_L, db_L, db_{L-1}
  // one resident wave: at 64 registers per thread an SM holds 65536 / (64 * threads) blocks (3 at NP = 160; the grid of 4 per
  // SM ran as 1.33 waves)
  const int out_bwd_per_sm = 65536 / (64 * red_threads) < 1 ? 1 : (65536 / (64 * red_threads) > 4 ? 4 : 65536 / (64 * red_threads));
  GNF_LAUNCH(lw_out_bwd_kernel, lw_blocks(pl.Q, 64, out_bwd_per_sm), red_threads, red_smem, s, saved + (size_t)(L - 1) * plane, ysave, net->W[L],
             net->dims[L], x, ccw, jac, gz, gzrev, gjac, glogdet, dcur, (float*)nullptr, grads->dW[L], grads->db[L], grads->db[L - 1], g);
  // hidden layers, top down: dW_l = delta_{l+1}^T a_l;  delta_l = (delta_{l+1} W_l) o relu'(a_l);  db_{l-1} = colsum delta_l
  for (int l = L - 1; l >= 1; --l) {
    const float* a_l = saved + (size_t)(l - 1) * plane;
    if (int e = lw_wgrad_gemm(dcur, NP, a_l, NP, grads->dW[l], net->dims[l], (int)pl.Q, net->dims[l + 1], net->dims[l], passes,
                              (use_rw && g_lw_use_rw_wgrad) ? ws + pl.off_part : nullptr, s)) return e;
    const uint32_t* mb = passes != 0 ? reinterpret_cast<const uint32_t*>(saved + (size_t)L * plane + pl.Q) + (size_t)(l - 1) * pl.Q * (NP / 32) : nullptr;
    if (int e = lw_dgrad_gemm(dcur, NP, ws + pl.off_Wp[l], NP, a_l, NP, mb, NP / 32, dnxt, NP, (int)pl.Q, net->dims[l + 1], net->dims[l], passes, use_rw ? NP : 0, s)) return e;
    if (l > 1) {
      if (int e = gnf_colsum(dnxt, NP, grads->db[l - 1], (int)pl.Q, net->dims[l], 1, stream)) return e;
    }
    float* t = dcur; dcur = dnxt; dnxt = t;
  }
  // first layer
  float* D = ws + pl.off_D;
  // db0 = colsum(D) comes out of the reduction kernel below (for L == 1 the output pass has already put colsum(delta_1) there)
  cudaMemsetAsync(grads->db[0], 0, (size_t)net->dims[1] * sizeof(float), s);
  GNF_LAUNCH(lw_layer1_bwd_kernel, lw_blocks(R, kLwRL, 6), red_threads, red_smem, s, dcur, x, ccn, net->W[0], 1 + E, net->dims[1], jac, gz,
             gzrev, D, grads->dW[0], grads->db[0], dx, g);
  if (int e = gnf_linear_wgrad(D, NP, h, E, grads->dW[0] + 1, 1 + E, R, net->dims[1], E, stream)) return e;
  if (int e = gnf_linear_dgrad(D, NP, net->W[0] + 1, 1 + E, nullptr, 0, dh, E, R, net->dims[1], E, stream)) return e;
  GNF_LAUNCH(lw_finish_dh_kernel, lw_blocks(R, 256, 4), 256, 0, s, dh, E, gz, gzrev, R, d);
  return check_launch("gnf_umnn_bwd_lw");
}


/* Fused-chain flavour of gnf_umnn_bwd_lw (same cotangents, outputs and gradient conventions; 3xTF32): the output pass
 * (lw_out_bwd_kernel: delta_L, dW_L, db_L, db_{L-1}), then ONE tensor-core kernel for the whole dgrad chain delta_L -> delta_1
 * with the column sums and the first-layer reductions taken on chip (tc_umnn3.cu), then the weight-gradient GEMMs over the delta /
 * activation planes (tc_rw_wgrad.cu) and the small per-row GEMMs of the first layer.  `saved` must come from gnf_umnn_fwd_tc3
 * (it also holds the ReLU mask of the last hidden activation). */
size_t gnf_umnn_bwd_tc3_workspace_bytes(const gnf_mlp_t* net, int R, int S) {
#ifdef GNF_EMU
  (void)net; (void)R; (void)S;
  gnf::set_error("tensor-core kernels have no host-simulator flavour");
  return 0;
#else
  LwPlan pl;
  if (lw_plan(net, R, S, 1, 1, &pl)) return 0;
  const size_t img = u3_bwd_image_floats(net);
  if (img == 0) return 0;
  if (!pl.rw) { set_error("umnn tc3 backward: the hidden layers do not fit the resident weight-gradient kernel"); return 0; }
  const size_t plane = (size_t)pl.Q * pl.NP;
  return ((size_t)R * pl.NP + (size_t)(pl.L - 1) * plane + 2 * (rw_wgrad_partial_floats(pl.NP) + 4) + img + 8) * sizeof(float);
#endif
}

int gnf_umnn_bwd_tc3(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn, const float* jac,
                     const float* gz, const float* gzrev, const float* gjac, const float* glogdet, const float* saved, float* dx,
                     float* dh, const gnf_mlp_grad_t* grads, int R, int d, void* work, size_t work_bytes, gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!x || !h || !net || !ccw || !ccn || !jac || !saved || !dx || !dh || !grads || R < 0 || d <= 0 || S < 1 || (R % d) != 0) return fail(GNF_ERR_INVALID, "gnf_umnn_bwd_tc3: bad arguments");
  LwPlan pl;
  if (int e = lw_plan(net, R, S, 1, 1, &pl)) return e;
  const size_t need = gnf_umnn_bwd_tc3_workspace_bytes(net, R, S);
  if (need == 0) return GNF_ERR_UNSUPPORTED;
  if (!work || work_bytes < need) return fail(GNF_ERR_WORKSPACE, "gnf_umnn_bwd_tc3: workspace too small (%zu < %zu)", work_bytes, need);
  if ((reinterpret_cast<uintptr_t>(work) & 15) != 0) return fail(GNF_ERR_INVALID, "gnf_umnn_bwd_tc3: workspace must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  const int NP = pl.NP, L = pl.L, E = pl.E;
  ZeroList zl;
  for (int l = 0; l < net->n_layers; ++l) {
    if (!grads->dW[l] || !grads->db[l]) return fail(GNF_ERR_INVALID, "gnf_umnn_bwd_tc3: gradient pointer %d is NULL", l);
    zl.add(grads->dW[l], (size_t)net->dims[l] * net->dims[l + 1]);
    zl.add(grads->db[l], (size_t)net->dims[l + 1]);
  }
  if (R == 0) { zero_many(zl, s); return check_launch("gnf_umnn_bwd_tc3"); }
  float* ws = (float*)work;
  const size_t plane = (size_t)pl.Q * NP;
  float* D = ws;
  float* dplanes = ws + (((size_t)R * NP + 3) / 4) * 4;            // plane 0: delta_L, planes 1..L-2: delta_{L-1} .. delta_2
  float* part = dplanes + (size_t)(L - 1) * plane;
  const size_t part_floats = ((rw_wgrad_partial_floats(NP) + 3) / 4) * 4;     // two buffers: the reduction of one layer overlaps the next layer's kernel
  float* image = part + 2 * part_floats;
  LwGeom g;
  g.R = R; g.d = d; g.E = E; g.S = S; g.nodes = pl.nodes; g.NP = NP; g.L = L; g.Q = pl.Q;
  const int red_threads = (NP / 4) * kLwRL;
  const size_t red_smem = ((size_t)kLwRL * NP + kLwRL + 4) * sizeof(float);
  const float* ysave = saved + (size_t)L * plane;
  zl.add(D, (size_t)R * NP);
  zl.add(dx, (size_t)R);
  const Branches& br = branches();
  cudaStream_t pack_stream = br.ok ? br.begin(s, 0) : nullptr;     // the chain's weight images: next to the zero-fill and the output pass
  zero_many(zl, s);                    // every gradient tensor, D and dx: one launch (GNF_MAX_LAYERS = 8: at most 18 entries)
  // output layer: g_q per node-row (the weight-gradient kernel of W_{L-1} rebuilds delta_L from it and the saved ReLU mask of a_L: no
  // delta_L plane), dW_L, db_L, db_{L-1}.  g_q lives in the first Q floats of what used to be that plane.
  float* gq = dplanes;
  const uint32_t* bits_top = reinterpret_cast<const uint32_t*>(saved + (size_t)L * plane + pl.Q) + (size_t)(L - 1) * pl.Q * (NP / 32);
  const int out_bwd_per_sm = 65536 / (64 * red_threads) < 1 ? 1 : (65536 / (64 * red_threads) > 4 ? 4 : 65536 / (64 * red_threads));
  GNF_LAUNCH(lw_out_bwd_kernel, lw_blocks(pl.Q, 64, out_bwd_per_sm), red_threads, red_smem, s, saved + (size_t)(L - 1) * plane, ysave, net->W[L],
             net->dims[L], x, ccw, jac, gz, gzrev, gjac, glogdet, dplanes, gq, grads->dW[L], grads->db[L], grads->db[L - 1], g);
  // the dgrad chain on the tensor cores: delta_{L-1} .. delta_2 planes, hidden db, dW0[:,0], D, dx
  if (int e = launch_u3_bwd_chain(x, net, S, ccw, ccn, jac, gz, gzrev, gjac, glogdet, saved, image, dplanes + plane, D, dx, grads, R, d, s, &br, 0, pack_stream)) return e;
  // Branch 0 (small per-row kernels, a fraction of the SMs each; they fill in around the persistent kernels of the main branch):
  // the first layer -- db0 = colsum(D), dW0[:,1:] = D^T h, dh = D W0[:,1:] (+ gz on the first conditioning feature)
  {
    cudaStream_t s0 = br.begin(s, 0);
    gnf_stream_t st0 = (gnf_stream_t)s0;
    if (int e = gnf_colsum(D, NP, grads->db[0], R, net->dims[1], 1, st0)) return e;
    if (int e = gnf_linear_wgrad(D, NP, h, E, grads->dW[0] + 1, 1 + E, R, net->dims[1], E, st0)) return e;
    if (int e = gnf_linear_dgrad(D, NP, net->W[0] + 1, 1 + E, nullptr, 0, dh, E, R, net->dims[1], E, st0)) return e;
    GNF_LAUNCH(lw_finish_dh_kernel, lw_blocks(R, 256, 4), 256, 0, s0, dh, E, gz, gzrev, R, d);
  }
  // Main branch: weight gradients of the hidden GEMM layers, dW_l = delta_{l+1}^T a_l; the second stage (sum of the per-CTA partial
  // tiles) of each layer is branch 1 and overlaps the next layer's kernel
  int k = 0;
  for (int l = L - 1; l >= 1; --l, ++k) {
    const float* dnext = dplanes + (size_t)(L - 1 - l) * plane;    // delta_{l+1}
    const float* a_l = saved + (size_t)(l - 1) * plane;
    if (k >= 2) br.end(s, 1);                                      // the partial buffer about to be reused has been summed
    const RwRankOne top = {gq, net->W[L], bits_top, NP / 32};
    if (int e = launch_rw_wgrad(dnext, NP, a_l, NP, grads->dW[l], net->dims[l], (int)pl.Q, net->dims[l + 1], net->dims[l], 3,
                                part + (size_t)(k & 1) * part_floats, s, &br, 1, l == L - 1 ? &top : nullptr)) return e;
  }
  br.end(s, 1);
  br.end(s, 0);
  return check_launch("gnf_umnn_bwd_tc3");
#endif
}

/* Floats of the saved-activation buffer written by gnf_umnn_fwd_tc3 in training: gnf_umnn_lw_saved_floats(net, R, S, 1) plus
 * the ReLU bit mask of the last hidden activation ([Q][NP/32] words), which the fused backward chain starts from. */
size_t gnf_umnn_tc3_saved_floats(const gnf_mlp_t* net, int R, int S) {
  LwPlan pl;
  if (lw_plan(net, R, S, 1, 0, &pl)) return 0;
  return gnf_umnn_lw_saved_floats(net, R, S, 1) + (size_t)pl.Q * (pl.NP / 32);
}

}  // extern "C"
