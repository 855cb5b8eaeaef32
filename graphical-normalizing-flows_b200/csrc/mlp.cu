// Conditioner MLP engine: Linear(+ReLU) forward / dgrad / wgrad on the fp32 FFMA tile GEMM, the
// DAGConditioner's first layer with the masked embedding generated inside the operand loader, and
// the small pack / reduce helpers around them.  See include/gnf.h for the reference lines each
// entry point replaces.
#include "gemm.cuh"
#include "thin.cuh"

namespace gnf {

// ------------------------------------------------------------------------------------------------
// DAG gate: e[b,i,j] and its partial derivatives  (DAGConditioner.py:94-153)
// ------------------------------------------------------------------------------------------------
struct GateCtx {
  const float* x;   // [B,d]
  const float* P;   // [d,d] importance table
  const float* n1;  // replayed noise (nullable)
  const float* n2;
  uint64_t seed, offset;
  const uint64_t* offset_dev;  // optional device-side addend to `offset`
  float T;
  int mode, d;
};

__device__ __forceinline__ void gate_noise(const GateCtx& g, size_t idx, float& a, float& b) {
  if (g.n1) {
    a = __ldg(g.n1 + idx);
    b = g.n2 ? __ldg(g.n2 + idx) : 0.f;
    return;
  }
  const uint4 r = Philox::gen(g.seed, (uint64_t)idx, g.offset + (g.offset_dev ? *g.offset_dev : 0ull));
  if (g.mode == GNF_GATE_GUMBEL) {
    a = Philox::u01(r.x);
    b = Philox::u01(r.y);
  } else {  // standard normal by Box-Muller
    const float u = Philox::u01(r.x), v = Philox::u01(r.y);
    a = sqrtf(-2.f * logf(u)) * cosf(6.283185307179586f * v);
    b = 0.f;
  }
}

// The heavy part of the stochastic gate is NOT inlined: the tile GEMM evaluates the gate once per element of its fully
// unrolled register tiles (32-64 call sites per kernel); inlined, Philox + six transcendentals per site made the layer-1
// kernels 0.2-0.4 MB of code and ncu showed 23-53 % of their warp samples stalled on instruction fetch (stall_no_inst).
// Everything goes in and out by value (registers): an out-of-line gate_e taking the context by reference and returning
// through pointers cost 20 % at d = 784, where the gate math is the whole kernel.
//   returns (G, dG/dp) of the relaxed Bernoulli gate, DAGConditioner.stochastic_gate (DAGConditioner.py:94-103)
__device__ __forceinline__ float2 gumbel_gate_math_inl(float p, float na, float nb, float T) {
  const float eps = 1e-6f;
  const float g1 = -logf(-logf(na)), g2 = -logf(-logf(nb));
  const float z1 = expf((logf(p + eps) + g1) / T);
  const float z2 = expf((logf(1.f - p + eps) + g2) / T);
  const float G = z1 / (z1 + z2);
  return make_float2(G, (G * (1.f - G) / T) * (1.f / (p + eps) + 1.f / (1.f - p + eps)));
}
// same with the uniforms drawn in place (training path: no replayed noise)
__device__ __forceinline__ float2 gumbel_gate_philox_inl(float p, float T, uint64_t seed, uint64_t idx, uint64_t offset) {
  const uint4 r = Philox::gen(seed, idx, offset);
  return gumbel_gate_math_inl(p, Philox::u01(r.x), Philox::u01(r.y), T);
}
__device__ GNF_NOINLINE float2 gumbel_gate_math(float p, float na, float nb, float T) { return gumbel_gate_math_inl(p, na, nb, T); }
__device__ GNF_NOINLINE float2 gumbel_gate_philox(float p, float T, uint64_t seed, uint64_t idx, uint64_t offset) {
  return gumbel_gate_philox_inl(p, T, seed, idx, offset);
}

// standard normal by Box-Muller (DAGConditioner.noiser_gate, DAGConditioner.py:114-116), out of line for the same reason
__device__ GNF_NOINLINE float normal_philox(uint64_t seed, uint64_t idx, uint64_t offset) {
  const uint4 r = Philox::gen(seed, idx, offset);
  const float u = Philox::u01(r.x), v = Philox::u01(r.y);
  return sqrtf(-2.f * logf(u)) * cosf(6.283185307179586f * v);
}

// kInl: inline the Gumbel math after all -- for wide flows (d >= 256: d^2 gate evaluations per sample) the gate math IS the
// kernel and the call overhead costs 10-15 % (cfg5, d = 784), while the short-K kernels of narrow flows are fetch-bound.
template <bool kGrad, bool kInl>
__device__ __forceinline__ float gate_e(const GateCtx& g, int b, int i, int j, float* de_dx, float* de_dP) {
  const float p = __ldg(g.P + (size_t)i * g.d + j);
  const float xv = __ldg(g.x + (size_t)b * g.d + j);
  if (g.mode == GNF_GATE_TABLE) {
    if (kGrad) { *de_dx = p; *de_dP = xv; }
    return xv * p;
  }
  const size_t idx = ((size_t)b * g.d + i) * g.d + j;
  if (g.mode == GNF_GATE_GUMBEL) {
    float2 G;
    const uint64_t off = g.offset + (g.offset_dev ? *g.offset_dev : 0ull);
    if (g.n1) G = kInl ? gumbel_gate_math_inl(p, __ldg(g.n1 + idx), __ldg(g.n2 + idx), g.T) : gumbel_gate_math(p, __ldg(g.n1 + idx), __ldg(g.n2 + idx), g.T);
    else G = kInl ? gumbel_gate_philox_inl(p, g.T, g.seed, (uint64_t)idx, off) : gumbel_gate_philox(p, g.T, g.seed, (uint64_t)idx, off);
    if (kGrad) {
      *de_dx = G.x;
      *de_dP = xv * G.y;
    }
    return xv * G.x;
  }
  // noiser gate: e = P*(x + n*sqrt((1-P)^2))
  const float na = g.n1 ? __ldg(g.n1 + idx) : normal_philox(g.seed, (uint64_t)idx, g.offset + (g.offset_dev ? *g.offset_dev : 0ull));
  const float a = fabsf(1.f - p);
  if (kGrad) {
    const float sgn = (1.f - p) > 0.f ? 1.f : ((1.f - p) < 0.f ? -1.f : 0.f);
    *de_dx = p;
    *de_dP = xv + na * a - p * na * sgn;
  }
  return p * (xv + na * a);
}

constexpr int kGateInlineMinD = 256;

template <bool kInl>
struct LoadDagA {  // A(m,k) = e[b,i,j], m = b*d+i, k = j
  static constexpr bool kContigK = true;
  GateCtx g;
  __device__ __forceinline__ float operator()(int m, int k) const { return gate_e<false, kInl>(g, m / g.d, m % g.d, k, nullptr, nullptr); }
};
template <bool kInl>
struct LoadDagB {  // B(k,n) = e[m=k, j=n]
  static constexpr bool kContigK = false;
  GateCtx g;
  __device__ __forceinline__ float operator()(int k, int n) const { return gate_e<false, kInl>(g, k / g.d, k % g.d, n, nullptr, nullptr); }
};
template <bool kInl>
struct EpiDagDgrad {  // ebar[m,j] -> dx[b,j] += ebar*de/dx ; dP[i,j] += ebar*de/dP
  GateCtx g;
  float* dx;
  float* dP;
  __device__ __forceinline__ void operator()(int m, int n, const float* v, int nv) const {
    const int b = m / g.d, i = m % g.d;
    for (int jj = 0; jj < nv; ++jj) {
      float ddx, ddp;
      gate_e<true, kInl>(g, b, i, n + jj, &ddx, &ddp);
      atomicAdd(dx + (size_t)b * g.d + n + jj, v[jj] * ddx);
      atomicAdd(dP + (size_t)i * g.d + n + jj, v[jj] * ddp);
    }
  }
};

// ------------------------------------------------------------------------------------------------
// Layer 1 of narrow DAG flows (d <= 64): gate tile resident in shared memory
// ------------------------------------------------------------------------------------------------
// The functor loaders above evaluate the gate wherever the tile GEMM asks for an operand element: once per (row block, N tile) in
// the forward (630 outputs = 5 N tiles), once per (N tile, row block) in the wgrad and once per split-K slice in the dgrad's
// epilogue -- 5-6 evaluations of ~300 instructions (Philox4x32-10 + six logf/expf + divisions) per gate.  ncu on cfg4
// (profiles/r01zt_ncu_dag_l1.txt): 36-40 M warp instructions per kernel against 7.8 M FFMA, issue slots 59-63 % busy: the gate
// math, not the contraction, was the kernel.  With K = d <= 64 the whole e tile of a row block ([rows, d]) fits in shared memory:
// these kernels evaluate every gate exactly ONCE per direction and loop over the layer width around the resident tile.
constexpr int kDagMaxD = 64;
constexpr int kDagKP = 64;                       // padded K / j extent of the resident tile

// All three prefetch the next operand tile into registers (batched, unconditional loads from clamped addresses) while the
// current one is being consumed: the first version loaded tile by tile between two barriers and was slower than the redundant
// kernels (latency-bound at ~1.3 CTAs per SM: 81 / 76 / 91 us vs 73 / 62 / 75 us).

// Forward: Y[m, :] = act(e[m, :] W1[:, :d]^T + T[m % period, :]).  CTA = 32 rows, 256 threads; both operands k-contiguous in
// shared memory (Es[m][k], Ws[n][k], row stride 68 floats): a thread owns 4 rows (its warp's) x 4 columns {lane + 32 c} and
// reads float4 along k -- every 16-byte shared-memory access (quarter-warp phases) and every store is conflict-free, and the
// global stores of a warp are 128 contiguous bytes per row.  Loops over the N tiles of 128.  grid = ceil(M / 32).
constexpr int kDagFwdBM = 32, kDagFwdBN = 128, kDagFwdThreads = 256;
constexpr int kDagLDK = kDagKP + 4;
constexpr int kDagFwdWPer = kDagFwdBN * kDagKP / kDagFwdThreads;       // 32 prefetch registers
constexpr size_t kDagFwdSmem = (size_t)(kDagFwdBM + kDagFwdBN) * kDagLDK * sizeof(float);

// Training with a stochastic gate (round 2): the forward also leaves e, de/dx and de/dP as [M][kDagKP] planes (3 x 1.6 MB at cfg4)
// and the two backward kernels read them instead of drawing and evaluating every gate again -- the gate math (Philox4x32-10 + six
// transcendentals + divisions, ~300 instructions) was most of each of the three kernels (see above), now it runs once per step.
struct GatePlanes { float* E; float* DX; float* DP; };

template <bool kSave>
__global__ void __launch_bounds__(kDagFwdThreads, 2) dag_l1_fwd_kernel(GateCtx g, GatePlanes sv, const float* __restrict__ W1, int ldw, const float* __restrict__ T,
                                                                    int bias_ld, int period, int relu, float* __restrict__ Y, int ldy, int M, int N) {
  GNF_SMEM(float, smem);
  float* Es = smem;                              // [BM][LDK]   Es[m][j]
  float* Ws = smem + kDagFwdBM * kDagLDK;        // [BN][LDK]   Ws[n][k]
  const int t = threadIdx.x, m0 = blockIdx.x * kDagFwdBM, d = g.d;
  float rw[kDagFwdWPer];
  auto prefetch = [&](int n0) {
#pragma unroll
    for (int e = 0; e < kDagFwdWPer; ++e) {
      const int idx = t + e * kDagFwdThreads, k = idx % kDagKP, nn = idx / kDagKP;
      const bool ok = k < d && n0 + nn < N;
      const float v = __ldg(W1 + (size_t)(ok ? n0 + nn : 0) * ldw + (ok ? k : 0));
      rw[e] = ok ? v : 0.f;
    }
  };
  prefetch(0);
  // a gate is a ~1.5 k-clock dependent chain (Philox rounds, logf(-logf), divisions, expf) and the SM holds ~10 warps here:
  // inlined and unrolled by four so that four independent chains are in flight per thread (this loop is rolled, unlike the
  // register-tile loaders above: the code stays small)
#pragma unroll 4
  for (int idx = t; idx < kDagFwdBM * kDagKP; idx += kDagFwdThreads) {
    const int j = idx % kDagKP, mm = idx / kDagKP, m = m0 + mm;
    float v = 0.f;
    if (kSave) {
      float ddx = 0.f, ddp = 0.f;
      if (m < M && j < d) v = gate_e<true, true>(g, m / d, m % d, j, &ddx, &ddp);
      if (m < M) {
        sv.E[(size_t)m * kDagKP + j] = v;
        sv.DX[(size_t)m * kDagKP + j] = ddx;
        sv.DP[(size_t)m * kDagKP + j] = ddp;
      }
    } else if (m < M && j < d) v = gate_e<false, true>(g, m / d, m % d, j, nullptr, nullptr);
    Es[mm * kDagLDK + j] = v;
  }
  const int tx = t % 32, ty = t / 32;            // lane = column residue, warp = group of 4 rows
  const float* brow[4];                          // bias-table row of each of the thread's rows (clamped for rows >= M)
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = (m0 + ty * 4 + i < M) ? m0 + ty * 4 + i : M - 1;
    brow[i] = T + (size_t)(period > 1 ? (m % period) : 0) * bias_ld;
  }
  for (int n0 = 0; n0 < N; n0 += kDagFwdBN) {
#pragma unroll
    for (int e = 0; e < kDagFwdWPer; ++e) {
      const int idx = t + e * kDagFwdThreads;
      Ws[(idx / kDagKP) * kDagLDK + idx % kDagKP] = rw[e];
    }
    __syncthreads();
    if (n0 + kDagFwdBN < N) prefetch(n0 + kDagFwdBN);
    // the accumulators start from the bias table: these 16 loads are in flight during the k loop (added in the epilogue, each
    // was a full L2 round trip in front of its store: half of the kernel's warp samples, profiles/r01zx_ncu_dag_l1_fwd.txt)
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int n = n0 + tx + 32 * c;
        acc[i][c] = T ? __ldg(brow[i] + (n < N ? n : N - 1)) : 0.f;
      }
#pragma unroll 2
    for (int k = 0; k < kDagKP; k += 4) {
      float4 a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(&Es[(ty * 4 + i) * kDagLDK + k]);
#pragma unroll
      for (int c = 0; c < 4; ++c) b[c] = *reinterpret_cast<const float4*>(&Ws[(tx + 32 * c) * kDagLDK + k]);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          acc[i][c] = fmaf(a[i].x, b[c].x, acc[i][c]);
          acc[i][c] = fmaf(a[i].y, b[c].y, acc[i][c]);
          acc[i][c] = fmaf(a[i].z, b[c].z, acc[i][c]);
          acc[i][c] = fmaf(a[i].w, b[c].w, acc[i][c]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      if (m >= M) continue;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int n = n0 + tx + 32 * c;
        if (n < N) Y[(size_t)m * ldy + n] = relu ? fmaxf(acc[i][c], 0.f) : acc[i][c];
      }
    }
    __syncthreads();                             // Ws is overwritten by the next N tile
  }
}

// Weight gradient: dW1[n, j] += sum_{m in the CTA's 64 rows} dY[m, n] e[m, j].  CTA = 64 rows of the reduction, 256 threads
// (thread tile 8 n x 4 j, outer-product form: both operands are stored as they arrive, [m][n] and [m][j]), loops over the N tiles
// of 128 and adds its partial tiles with atomics.  grid = ceil(M / 64).
constexpr int kDagWgBK = 64, kDagWgBN = 128, kDagWgThreads = 256;
constexpr int kDagWgLDN = kDagWgBN + 4;
constexpr int kDagWgPer = kDagWgBK * kDagWgBN / kDagWgThreads;         // 32 prefetch registers
constexpr size_t kDagWgSmem = (size_t)kDagWgBK * (kDagLDK + kDagWgLDN) * sizeof(float);

template <bool kSaved>     // kSaved: e comes from the forward's plane (g.x = the plane, [M][kDagKP])
__global__ void __launch_bounds__(kDagWgThreads, 2) dag_l1_wgrad_kernel(GateCtx g, const float* __restrict__ dY, int lddy, EpiAtomicAdd epi, int M, int N) {
  GNF_SMEM(float, smem);
  float* Em = smem;                              // [BK][LDK]   Em[m][j]
  float* Ds = smem + kDagWgBK * kDagLDK;         // [BK][LDN]   Ds[m][n]
  const int t = threadIdx.x, m0 = blockIdx.x * kDagWgBK, d = g.d;
  const int rows = (M - m0 < kDagWgBK) ? M - m0 : kDagWgBK;
  float rd[kDagWgPer];
  auto prefetch = [&](int n0) {
#pragma unroll
    for (int e = 0; e < kDagWgPer; ++e) {
      const int idx = t + e * kDagWgThreads, nn = idx % kDagWgBN, mm = idx / kDagWgBN;
      const bool ok = mm < rows && n0 + nn < N;
      const float v = __ldg(dY + (size_t)(m0 + (ok ? mm : 0)) * lddy + (ok ? n0 + nn : 0));
      rd[e] = ok ? v : 0.f;
    }
  };
  // every CTA adds into the same dW1 tiles: start at a different N tile per CTA so that the atomics of concurrently running
  // CTAs do not pile up on the same addresses
  const int ntiles = (N + kDagWgBN - 1) / kDagWgBN, first = blockIdx.x % ntiles;
  prefetch(first * kDagWgBN);
#pragma unroll 4
  for (int idx = t; idx < kDagWgBK * kDagKP; idx += kDagWgThreads) {   // four independent gate chains in flight (see the forward)
    const int j = idx % kDagKP, mm = idx / kDagKP, m = m0 + mm;
    float v = 0.f;
    if (kSaved) { if (m < M) v = __ldg(g.x + (size_t)m * kDagKP + j); }
    else if (m < M && j < d) v = gate_e<false, true>(g, m / d, m % d, j, nullptr, nullptr);
    Em[mm * kDagLDK + j] = v;
  }
  const int tx = t % 16, ty = t / 16;            // 16 j quads x 16 groups of 8 output rows n
  for (int it = 0; it < ntiles; ++it) {
    const int n0 = ((first + it) % ntiles) * kDagWgBN;
#pragma unroll
    for (int e = 0; e < kDagWgPer; ++e) {
      const int idx = t + e * kDagWgThreads;
      Ds[(idx / kDagWgBN) * kDagWgLDN + idx % kDagWgBN] = rd[e];
    }
    __syncthreads();
    if (it + 1 < ntiles) prefetch(((first + it + 1) % ntiles) * kDagWgBN);
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[i][c] = 0.f;
#pragma unroll 4
    for (int mm = 0; mm < kDagWgBK; ++mm) {       // rows >= `rows` of both tiles are zero
      const float4 a0 = *reinterpret_cast<const float4*>(&Ds[mm * kDagWgLDN + ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&Ds[mm * kDagWgLDN + ty * 8 + 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Em[mm * kDagLDK + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[i][c] = fmaf(a[i], b[c], acc[i][c]);
    }
    const int j = tx * 4;
    if (j < d) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int n = n0 + ty * 8 + i;
        if (n < N) epi(n, j, acc[i], (d - j < 4) ? d - j : 4);
      }
    }
    __syncthreads();
  }
}

// Input gradient: ebar[m, j] = sum_n dY[m, n] W1[n, j] over the WHOLE layer width in one CTA (no split-K: the gate derivatives of
// the epilogue are evaluated once), then dx[b, j] += ebar de/dx, dP[i, j] += ebar de/dP.  CTA = 32 rows, 128 threads (thread tile
// 4 rows x 4 j), k-chunks of 32 (As[m][k] as it arrives, Bs[k][j] as it arrives; four k per step).  grid = ceil(M / 32).
constexpr int kDagDgBM = 32, kDagDgBK = 32, kDagDgThreads = 128;
constexpr int kDagDgLDA = kDagDgBK + 4;
constexpr int kDagDgAPer = kDagDgBM * kDagDgBK / kDagDgThreads, kDagDgBPer = kDagDgBK * kDagKP / kDagDgThreads;   // 8 + 16
constexpr size_t kDagDgSmem = (size_t)(kDagDgBM * kDagDgLDA + kDagDgBK * kDagLDK) * sizeof(float);

template <bool kSaved>     // kSaved: de/dx and de/dP come from the forward's planes (g.x = DX, g.P = DP, both [M][kDagKP])
__global__ void __launch_bounds__(kDagDgThreads, 4) dag_l1_dgrad_kernel(GateCtx g, const float* __restrict__ dY, int lddy, const float* __restrict__ W1, int ldw,
                                                                     float* __restrict__ dx, float* __restrict__ dP, int M, int N) {
  GNF_SMEM(float, smem);
  float* As = smem;                              // [BM][LDA]   As[m][k] = dY[m0 + m, n0 + k]
  float* Bs = smem + kDagDgBM * kDagDgLDA;       // [BK][LDK]   Bs[k][j] = W1[n0 + k, j]
  const int t = threadIdx.x, m0 = blockIdx.x * kDagDgBM, d = g.d;
  const int tx = t % 16, ty = t / 16;            // 16 j quads x 8 groups of 4 rows
  float ra[kDagDgAPer], rb[kDagDgBPer];
  auto prefetch = [&](int n0) {
#pragma unroll
    for (int e = 0; e < kDagDgAPer; ++e) {
      const int idx = t + e * kDagDgThreads, kk = idx % kDagDgBK, mm = idx / kDagDgBK;
      const bool ok = m0 + mm < M && n0 + kk < N;
      const float v = __ldg(dY + (size_t)(ok ? m0 + mm : 0) * lddy + (ok ? n0 + kk : 0));
      ra[e] = ok ? v : 0.f;
    }
#pragma unroll
    for (int e = 0; e < kDagDgBPer; ++e) {
      const int idx = t + e * kDagDgThreads, j = idx % kDagKP, kk = idx / kDagKP;
      const bool ok = j < d && n0 + kk < N;
      const float v = __ldg(W1 + (size_t)(ok ? n0 + kk : 0) * ldw + (ok ? j : 0));
      rb[e] = ok ? v : 0.f;
    }
  };
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[i][c] = 0.f;
  prefetch(0);
  for (int n0 = 0; n0 < N; n0 += kDagDgBK) {
#pragma unroll
    for (int e = 0; e < kDagDgAPer; ++e) {
      const int idx = t + e * kDagDgThreads;
      As[(idx / kDagDgBK) * kDagDgLDA + idx % kDagDgBK] = ra[e];
    }
#pragma unroll
    for (int e = 0; e < kDagDgBPer; ++e) {
      const int idx = t + e * kDagDgThreads;
      Bs[(idx / kDagKP) * kDagLDK + idx % kDagKP] = rb[e];
    }
    __syncthreads();
    if (n0 + kDagDgBK < N) prefetch(n0 + kDagDgBK);
#pragma unroll 2
    for (int kk = 0; kk < kDagDgBK; kk += 4) {
      float4 a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(&As[(ty * 4 + i) * kDagDgLDA + kk]);
#pragma unroll
      for (int u = 0; u < 4; ++u) b[u] = *reinterpret_cast<const float4*>(&Bs[(kk + u) * kDagLDK + tx * 4]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[i][0] = fmaf(a[i].x, b[0].x, acc[i][0]); acc[i][1] = fmaf(a[i].x, b[0].y, acc[i][1]);
        acc[i][2] = fmaf(a[i].x, b[0].z, acc[i][2]); acc[i][3] = fmaf(a[i].x, b[0].w, acc[i][3]);
        acc[i][0] = fmaf(a[i].y, b[1].x, acc[i][0]); acc[i][1] = fmaf(a[i].y, b[1].y, acc[i][1]);
        acc[i][2] = fmaf(a[i].y, b[1].z, acc[i][2]); acc[i][3] = fmaf(a[i].y, b[1].w, acc[i][3]);
        acc[i][0] = fmaf(a[i].z, b[2].x, acc[i][0]); acc[i][1] = fmaf(a[i].z, b[2].y, acc[i][1]);
        acc[i][2] = fmaf(a[i].z, b[2].z, acc[i][2]); acc[i][3] = fmaf(a[i].z, b[2].w, acc[i][3]);
        acc[i][0] = fmaf(a[i].w, b[3].x, acc[i][0]); acc[i][1] = fmaf(a[i].w, b[3].y, acc[i][1]);
        acc[i][2] = fmaf(a[i].w, b[3].z, acc[i][2]); acc[i][3] = fmaf(a[i].w, b[3].w, acc[i][3]);
      }
    }
    __syncthreads();
  }
  // epilogue: the four gates of a row are evaluated together (inlined: independent chains in flight), then their atomics
  const int j = tx * 4;
  if (j < d) {
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {                // rolled: four inlined gates per trip, not sixteen (instruction fetch)
      const int m = m0 + ty * 4 + i;
      if (m >= M) continue;
      const int b = m / d, iv = m % d;
      float av[4], ddx[4], ddp[4];
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) av[jj] = i == 0 ? acc[0][jj] : (i == 1 ? acc[1][jj] : (i == 2 ? acc[2][jj] : acc[3][jj]));
      if (kSaved) {
        const float4 vx = __ldg(reinterpret_cast<const float4*>(g.x + (size_t)m * kDagKP + j));
        const float4 vp = __ldg(reinterpret_cast<const float4*>(g.P + (size_t)m * kDagKP + j));
        ddx[0] = vx.x; ddx[1] = vx.y; ddx[2] = vx.z; ddx[3] = vx.w;
        ddp[0] = vp.x; ddp[1] = vp.y; ddp[2] = vp.z; ddp[3] = vp.w;
      } else {
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          ddx[jj] = ddp[jj] = 0.f;
          if (j + jj < d) gate_e<true, true>(g, b, iv, j + jj, &ddx[jj], &ddp[jj]);
        }
      }
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        if (j + jj < d) {
          atomicAdd(dx + (size_t)b * d + j + jj, av[jj] * ddx[jj]);
          atomicAdd(dP + (size_t)iv * d + j + jj, av[jj] * ddp[jj]);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Layer 1 of wide DAG flows (d > 64) for the tensor-core GEMM engine: the masked embedding as a plane
// ------------------------------------------------------------------------------------------------
// At d = 784 (cfg5) layer 1 is three 126-GFLOP GEMMs whose operand e[b,i,j] = x[b,j] G[b,i,j] costs a Philox draw, four
// logarithms and two exponentials per element.  The functor-loader kernels above run them on the FP32 pipe and re-evaluate the
// gate once per N tile / split-K slice: 9.4 + 15.1 + 5.6 ms per step.  With 180 GB of HBM the other trade is better: write
// e ONCE as a [B*d, ld] plane (246 MB at cfg5 -- 40 us of HBM time, every gate evaluated once), run forward / wgrad / dgrad on
// the tcgen05 engine (3xTF32) against it, and fold the gate derivatives into one reduction pass over the [B*d, d] cotangent
// plane the dgrad GEMM leaves.  Same Philox counters (idx = (b d + i) d + j) as the other kernels: the draws are identical.

// E[m, j] = e[b,i,j], m = b d + i; padding columns [d, ld) = 0.  One CTA per row m.  kGrad (training): the gate's partial
// derivatives de/dx and de/dP go to two more planes of the same shape, so that the backward reduction is a pure streaming pass
// (the Philox + Gumbel math of 61 M gates is 0.7 ms at cfg5; reading two planes back is 0.08 ms of HBM time).
template <bool kGrad>
__global__ void __launch_bounds__(256) dag_embed_fwd_kernel(GateCtx g, float* __restrict__ E, float* __restrict__ DX, float* __restrict__ DP, int lde) {
  const int m = blockIdx.x, b = m / g.d, i = m - b * g.d;
  const size_t row = (size_t)m * lde;
  for (int j4 = threadIdx.x * 4; j4 < lde; j4 += blockDim.x * 4) {
    float v[4], dx[4], dp[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      dx[k] = dp[k] = 0.f;
      v[k] = (j4 + k < g.d) ? gate_e<kGrad, true>(g, b, i, j4 + k, &dx[k], &dp[k]) : 0.f;
    }
    *reinterpret_cast<float4*>(E + row + j4) = make_float4(v[0], v[1], v[2], v[3]);
    if (kGrad) {
      *reinterpret_cast<float4*>(DX + row + j4) = make_float4(dx[0], dx[1], dx[2], dx[3]);
      *reinterpret_cast<float4*>(DP + row + j4) = make_float4(dp[0], dp[1], dp[2], dp[3]);
    }
  }
}

// dx[b,j] += sum_i dE[(b,i),j] de/dx(b,i,j)  (atomic over the i tiles);  dP[i,j] = sum_b dE[(b,i),j] de/dP(b,i,j)  (owned).
// CTA = 128 columns j x 8 rows i (two thread rows of four i each), loops over the batch.  grid = (ceil(d/128), ceil(d/8)).
constexpr int kEmbBwdI = 4;
// ... the same reduction from the derivative planes the training forward kept (no gate math: HBM-bound, three planes in).
// CTA = 256 columns (64 threads x float4) x 8 rows i (four thread rows of two i each); two batch entries in flight per thread.
constexpr int kEmbSavedI = 2;
__global__ void __launch_bounds__(256) dag_embed_bwd_saved_kernel(const float* __restrict__ dE, const float* __restrict__ DX,
                                                                  const float* __restrict__ DP, int lde, float* __restrict__ dx,
                                                                  float* __restrict__ dP, int B, int d) {
  const int j = blockIdx.x * 256 + (threadIdx.x & 63) * 4;
  const int i0 = blockIdx.y * (4 * kEmbSavedI) + (threadIdx.x >> 6) * kEmbSavedI;
  if (j >= d || i0 >= d) return;                             // lde % 4 == 0 and the padding columns of the planes are zero: float4 is safe
  const int ni = (d - i0 < kEmbSavedI) ? d - i0 : kEmbSavedI;
  float4 acc[kEmbSavedI];
#pragma unroll
  for (int k = 0; k < kEmbSavedI; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  auto fma4 = [](float4& a, const float4& v, const float4& w) {
    a.x = fmaf(v.x, w.x, a.x); a.y = fmaf(v.y, w.y, a.y); a.z = fmaf(v.z, w.z, a.z); a.w = fmaf(v.w, w.w, a.w);
  };
#pragma unroll 2
  for (int b = 0; b < B; ++b) {
    float4 dxs = make_float4(0.f, 0.f, 0.f, 0.f);
    const size_t base = ((size_t)b * d + i0) * lde + j;
#pragma unroll
    for (int k = 0; k < kEmbSavedI; ++k) {
      if (k < ni) {
        const size_t o = base + (size_t)k * lde;
        const float4 v = __ldg(reinterpret_cast<const float4*>(dE + o));
        fma4(dxs, v, __ldg(reinterpret_cast<const float4*>(DX + o)));
        fma4(acc[k], v, __ldg(reinterpret_cast<const float4*>(DP + o)));
      }
    }
    float* dst = dx + (size_t)b * d + j;
    atomicAdd(dst, dxs.x);
    if (j + 1 < d) atomicAdd(dst + 1, dxs.y);
    if (j + 2 < d) atomicAdd(dst + 2, dxs.z);
    if (j + 3 < d) atomicAdd(dst + 3, dxs.w);
  }
#pragma unroll
  for (int k = 0; k < kEmbSavedI; ++k)
    if (k < ni) {
      float* dst = dP + (size_t)(i0 + k) * d + j;
      dst[0] = acc[k].x;
      if (j + 1 < d) dst[1] = acc[k].y;
      if (j + 2 < d) dst[2] = acc[k].z;
      if (j + 3 < d) dst[3] = acc[k].w;
    }
}

__global__ void __launch_bounds__(256) dag_embed_bwd_kernel(GateCtx g, const float* __restrict__ dE, int lde, float* __restrict__ dx,
                                                            float* __restrict__ dP, int B) {
  const int j = blockIdx.x * 128 + (threadIdx.x & 127);
  const int i0 = blockIdx.y * (2 * kEmbBwdI) + (threadIdx.x >> 7) * kEmbBwdI;
  if (j >= g.d || i0 >= g.d) return;
  float acc[kEmbBwdI];
#pragma unroll
  for (int k = 0; k < kEmbBwdI; ++k) acc[k] = 0.f;
  for (int b = 0; b < B; ++b) {
    float dxs = 0.f;
#pragma unroll
    for (int k = 0; k < kEmbBwdI; ++k) {
      const int i = i0 + k;
      if (i < g.d) {
        const float v = __ldg(dE + ((size_t)b * g.d + i) * lde + j);
        float ddx, ddp;
        gate_e<true, true>(g, b, i, j, &ddx, &ddp);
        dxs = fmaf(v, ddx, dxs);
        acc[k] = fmaf(v, ddp, acc[k]);
      }
    }
    atomicAdd(dx + (size_t)b * g.d + j, dxs);
  }
#pragma unroll
  for (int k = 0; k < kEmbBwdI; ++k)
    if (i0 + k < g.d) dP[(size_t)(i0 + k) * g.d + j] = acc[k];
}

// ------------------------------------------------------------------------------------------------
// Skinny layers: launchers of thin.cuh (return false when the shape does not fit: the tile GEMM takes over)
// ------------------------------------------------------------------------------------------------
static int g_thin = 1;                     // measurement switch (gnf_linear_set_thin, dev build)
constexpr int kThinMinRows = 512;

static bool thin_launch_red(const float* in, int ldin, const float* Wp, long long s_t, long long s_w, const float* bias, int relu, const float* act,
                            int ldact, float* out, int ldout, int M, int T, int Wd, cudaStream_t s) {
  const size_t smem = thin_red_smem(T, Wd);
  if (T > kThinT || smem > 200 * 1024) return false;
#ifndef GNF_EMU
  cudaFuncSetAttribute(thin_red_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
  // every CTA loads the weight image before it can start: no more CTAs than one resident wave (each warp streams its share of the rows)
  const long long warps = ((long long)M + kThinRows - 1) / kThinRows;
  long long grid = (warps + kThinThreads / 32 - 1) / (kThinThreads / 32);
  const int per_sm = thin_per_sm(smem, 4);
  if (grid > (long long)per_sm * kNumSMs) grid = (long long)per_sm * kNumSMs;
  GNF_LAUNCH(thin_red_kernel, (int)grid, kThinThreads, smem, s, in, ldin, Wp, s_t, s_w, bias, relu, act, ldact, out, ldout, M, T, Wd);
  return true;
}

static int g_dag_l1_resident = 1;   // measurement switch (gnf_dag_l1_set_resident): 0 = functor-loader tile GEMM for every d

static int make_gate(GateCtx* out, const float* x, const float* P, const gnf_gate_t* gate, int d) {
  if (!gate) return fail(GNF_ERR_INVALID, "gate descriptor is NULL");
  if (gate->mode < GNF_GATE_TABLE || gate->mode > GNF_GATE_NOISER) return fail(GNF_ERR_UNSUPPORTED, "unknown gate mode %d", gate->mode);
  if (gate->mode == GNF_GATE_GUMBEL && !(gate->temperature > 0.f)) return fail(GNF_ERR_INVALID, "gumble_T must be > 0");
  if (gate->mode == GNF_GATE_GUMBEL && ((gate->noise1 == nullptr) != (gate->noise2 == nullptr)))
    return fail(GNF_ERR_INVALID, "Gumbel replay needs both noise tensors");
  out->x = x; out->P = P; out->n1 = gate->noise1; out->n2 = gate->noise2;
  out->seed = gate->seed; out->offset = gate->offset; out->offset_dev = gate->offset_dev;
  out->T = gate->temperature; out->mode = gate->mode; out->d = d;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Small kernels
// ------------------------------------------------------------------------------------------------
__global__ void zero2d_kernel(float* p, int ld, int rows, int cols) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    p[(i / cols) * ld + (i % cols)] = 0.f;
}
static void zero2d(float* p, int ld, int rows, int cols, cudaStream_t s) {
  if (rows <= 0 || cols <= 0) return;
  if (ld == cols) { cudaMemsetAsync(p, 0, (size_t)rows * cols * sizeof(float), s); return; }
  const size_t n = (size_t)rows * cols;
  int blocks = (int)((n + 255) / 256);
  if (blocks > 4 * kNumSMs) blocks = 4 * kNumSMs;
  GNF_LAUNCH(zero2d_kernel, blocks, 256, 0, s, p, ld, rows, cols);
}

// out[c] += sum_{q in chunk} Y[q*rowstride + c]  for the [Q, C] view (C = period*ldy)
__global__ void colsum_kernel(const float* __restrict__ Y, float* __restrict__ out, int Q, int C, int ldy, int N, size_t rowstride, int q_per) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int q0 = blockIdx.y * q_per;
  const int q1 = (q0 + q_per < Q) ? q0 + q_per : Q;
  if (c < C && (c % ldy) < N) {
    // eight independent row loads in flight per thread (one per iteration left a few KB in flight per SM: 26 us for an 89 MB plane)
    float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float* src = Y + c;
    int q = q0;
    for (; q + 7 < q1; q += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldg(src + (size_t)(q + u) * rowstride);
#pragma unroll
      for (int u = 0; u < 8; ++u) s[u] += v[u];
    }
    for (; q < q1; ++q) s[0] += __ldg(src + (size_t)q * rowstride);
    atomicAdd(out + (size_t)(c / ldy) * N + (c % ldy), ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7])));
  }
}

__global__ void pack_rows_kernel(const float* __restrict__ W, const float* __restrict__ mask, const int32_t* __restrict__ perm, float* __restrict__ out, int R, int K) {
  const size_t n = (size_t)R * K;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / K, k = i % K;
    const size_t src = (size_t)(perm ? perm[r] : (int)r) * K + k;
    out[i] = mask ? W[src] * mask[src] : W[src];
  }
}
__global__ void unpack_rows_kernel(const float* __restrict__ dWp, const float* __restrict__ mask, const int32_t* __restrict__ perm, float* __restrict__ dW, int R, int K) {
  const size_t n = (size_t)R * K;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t r = i / K, k = i % K;
    const size_t dst = (size_t)(perm ? perm[r] : (int)r) * K + k;
    dW[dst] = mask ? dWp[i] * mask[dst] : dWp[i];
  }
}
__global__ void unpack_vec_kernel(const float* __restrict__ src, const int32_t* __restrict__ perm, float* __restrict__ dst, int R) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < R; i += gridDim.x * blockDim.x) dst[perm ? perm[i] : i] = src[i];
}

__global__ void dag_importance_kernel(const float* __restrict__ A, int n, int imp, float h, float* __restrict__ P, float* __restrict__ dPdA) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float a = A[i];
    float p, dp;
    if (imp == GNF_IMP_RAW) {
      p = a; dp = 1.f;
    } else if (imp == GNF_IMP_HARD_SQ) {
      const float a2 = a * a;
      const float keep = (a2 > h) ? 1.f : 0.f;
      p = a2 * keep; dp = 2.f * a * keep;
    } else {
      const float s = 1.f / (1.f + expf(-2.f * (a * a)));   // sigmoid(2 A^2)
      p = 2.f * (s - .5f);
      dp = 8.f * a * s * (1.f - s);
      if (imp == GNF_IMP_HARD_SOFT) {
        const float keep = (p > h) ? 1.f : 0.f;
        p *= keep; dp *= keep;
      }
    }
    P[i] = p;
    if (dPdA) dPdA[i] = dp;
  }
}

__global__ void dag_bias_table_kernel(const float* __restrict__ W1, int ldw, const float* __restrict__ b1, float* __restrict__ T, int ldt, int d, int N, int hot) {
  const int rows = hot ? d : 1;
  const size_t n = (size_t)rows * ldt;          // padding columns [N, ldt) = 0
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / ldt), c = (int)(idx % ldt);
    T[idx] = c < N ? (hot ? W1[(size_t)c * ldw + d + i] : 0.f) + (b1 ? b1[c] : 0.f) : 0.f;
  }
}
__global__ void dag_bias_table_bwd_kernel(const float* __restrict__ dT, float* __restrict__ dW1, int ldw, float* __restrict__ db1, int d, int N, int hot) {
  const int rows = hot ? d : 1;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < N; c += gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int i = 0; i < rows; ++i) {
      const float v = dT[(size_t)i * N + c];
      s += v;
      if (hot) dW1[(size_t)c * ldw + d + i] = v;
    }
    if (db1) db1[c] = s;
  }
}
__global__ void dag_finish_dA_kernel(const float* __restrict__ dP, const float* __restrict__ dPdA, float* __restrict__ dA, int n, int accumulate) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float v = dP[i] * dPdA[i];
    dA[i] = accumulate ? dA[i] + v : v;
  }
}
__global__ void dag_dump_noise_kernel(GateCtx g, float* n1, float* n2, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float a, b;
    gate_noise(g, i, a, b);
    n1[i] = a;
    if (n2) n2[i] = b;
  }
}

static inline int ew_blocks(size_t n) {
  size_t b = (n + 255) / 256;
  if (b > (size_t)8 * kNumSMs) b = (size_t)8 * kNumSMs;
  return b < 1 ? 1 : (int)b;
}
}  // namespace gnf

using namespace gnf;

extern "C" {

int gnf_linear_fwd(const float* X, int ldx, const float* W, int ldw, const float* bias, int bias_period, float* Y,
                   int ldy, int M, int N, int K, int relu, gnf_stream_t stream) {
  if (!X || !W || !Y || M < 0 || N <= 0 || K <= 0 || ldx < K || ldw < K || ldy < N) return fail(GNF_ERR_INVALID, "gnf_linear_fwd: bad arguments");
  if (M == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (g_thin && bias_period <= 1 && M >= kThinMinRows) {
    // a reduction of a few terms (thin.cuh): Y[m, n] = sum_k X[m, k] W[n, k]
    if (K <= kThinT && N <= kThinMaxWide && thin_launch_red(X, ldx, W, 1, ldw, bias, relu, nullptr, 0, Y, ldy, M, K, N, s)) return check_launch("gnf_linear_fwd");
  }
  LoadRowMajorA al{X, ldx};
  LoadWeightT bl{W, ldw};
  EpiBiasAct epi{Y, ldy, bias, N, bias_period < 1 ? 1 : bias_period, relu};
  launch_gemm_auto(al, bl, epi, M, N, K, false, s);
  return check_launch("gnf_linear_fwd");
}

// Skinny output layer with a long reduction (cfg4: 6300 x 30 <- 630): 50 row tiles cannot fill the chip and one CTA per tile is a chain
// of ten global round trips (35 us).  Split-K over kSkSplits slices into partial tiles + a fixed-order sum with bias / ReLU.
constexpr int kSkSplits = 6, kSkLD = 32;
static int sk_splits(int K) { return K / kSkSplits >= 64 ? kSkSplits : (K >= 128 ? K / 64 : 1); }

__global__ void __launch_bounds__(256) splitk_sum_kernel(const float* __restrict__ P, size_t split_stride, int splits, const float* __restrict__ bias,
                                                         int relu, float* __restrict__ Y, int ldy, int M, int N) {
  const size_t total = (size_t)M * kSkLD;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int n = (int)(idx % kSkLD);
    const size_t m = idx / kSkLD;
    if (n >= N) continue;
    float v = bias ? __ldg(bias + n) : 0.f;
    for (int z = 0; z < splits; ++z) v += __ldg(P + (size_t)z * split_stride + idx);
    Y[m * ldy + n] = relu ? fmaxf(v, 0.f) : v;
  }
}

size_t gnf_linear_fwd_splitk_workspace_bytes(int M, int N, int K) {
  if (M < 1024 || N > kSkLD || sk_splits(K) < 2) return 0;
  return (size_t)sk_splits(K) * M * kSkLD * sizeof(float);
}

int gnf_linear_fwd_splitk(const float* X, int ldx, const float* W, int ldw, const float* bias, float* Y, int ldy, int M, int N, int K, int relu,
                          void* work, size_t work_bytes, gnf_stream_t stream) {
  if (!X || !W || !Y || M < 0 || N <= 0 || K <= 0 || ldx < K || ldw < K || ldy < N) return fail(GNF_ERR_INVALID, "gnf_linear_fwd_splitk: bad arguments");
  const size_t need = gnf_linear_fwd_splitk_workspace_bytes(M, N, K);
  if (need == 0) return fail(GNF_ERR_UNSUPPORTED, "gnf_linear_fwd_splitk: N <= 32, M >= 1024, K >= 128 only (else gnf_linear_fwd)");
  if (!work || work_bytes < need) return fail(GNF_ERR_WORKSPACE, "gnf_linear_fwd_splitk: workspace too small (%zu < %zu)", work_bytes, need);
  cudaStream_t s = (cudaStream_t)stream;
  const int splits = sk_splits(K);
  const size_t stride = (size_t)M * kSkLD;
  LoadRowMajorA al{X, ldx};
  LoadWeightT bl{W, ldw};
  EpiStoreSplit epi{(float*)work, kSkLD, stride};
  launch_gemm<TileSkinny>(al, bl, epi, M, N, K, splits, s);
  // launch_gemm rounds the slice to whole k tiles: the number of slices it really made
  const int ktiles = ceil_div(K, TileSkinny::BK), per = ceil_div(ktiles, splits) * TileSkinny::BK, made = ceil_div(K, per);
  GNF_LAUNCH(splitk_sum_kernel, ew_blocks(stride), 256, 0, s, (const float*)work, stride, made, bias, relu, Y, ldy, M, N);
  return check_launch("gnf_linear_fwd_splitk");
}

int gnf_linear_dgrad(const float* dY, int lddy, const float* W, int ldw, const float* act, int ldact, float* dX,
                     int lddx, int M, int N, int K, gnf_stream_t stream) {
  if (!dY || !W || !dX || M < 0 || N <= 0 || K <= 0 || lddy < N || ldw < K || lddx < K) return fail(GNF_ERR_INVALID, "gnf_linear_dgrad: bad arguments");
  if (M == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (g_thin && M >= kThinMinRows) {
    // a reduction of a few terms (thin.cuh): dX[m, k] = sum_n dY[m, n] W[n, k]
    if (N <= kThinT && K <= kThinMaxWide && thin_launch_red(dY, lddy, W, ldw, 1, nullptr, 0, act, ldact, dX, lddx, M, N, K, s)) return check_launch("gnf_linear_dgrad");
  }
  LoadRowMajorA al{dY, lddy};        // A(m, n) reduction over n
  LoadRowMajorB bl{W, ldw};          // B(n, k) = W[n, k]
  EpiMaskStore epi{dX, lddx, act, ldact};
  launch_gemm_auto(al, bl, epi, M, K, N, false, s);
  return check_launch("gnf_linear_dgrad");
}

int gnf_linear_wgrad(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, int M, int N, int K,
                     gnf_stream_t stream) {
  if (!dY || !X || !dW || M < 0 || N <= 0 || K <= 0 || lddy < N || ldx < K || lddw < K) return fail(GNF_ERR_INVALID, "gnf_linear_wgrad: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  zero2d(dW, lddw, N, K, s);
  if (M == 0) return check_launch("gnf_linear_wgrad");
  LoadColMajorA al{dY, lddy};        // A(n, m) = dY[m, n]
  LoadRowMajorB bl{X, ldx};          // B(m, k) = X[m, k]
  EpiAtomicAdd epi{dW, lddw};
  launch_gemm_auto(al, bl, epi, N, K, M, true, s);
  return check_launch("gnf_linear_wgrad");
}

int gnf_colsum(const float* Y, int ldy, float* out, int M, int N, int period, gnf_stream_t stream) {
  if (!Y || !out || M < 0 || N <= 0 || period < 1 || ldy < N || (M % period) != 0) return fail(GNF_ERR_INVALID, "gnf_colsum: bad arguments (M must be a multiple of period)");
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(out, 0, (size_t)period * N * sizeof(float), s);
  if (M == 0) return check_launch("gnf_colsum");
  const int Q = M / period, C = period * ldy;
  const int cblocks = ceil_div(C, 256);
  int qsplit = ceil_div(8 * kNumSMs, cblocks);
  if (qsplit > ceil_div(Q, 8)) qsplit = ceil_div(Q, 8);
  if (qsplit < 1) qsplit = 1;
  const int q_per = ceil_div(Q, qsplit);
  GNF_LAUNCH(colsum_kernel, dim3(cblocks, ceil_div(Q, q_per)), 256, 0, s, Y, out, Q, C, ldy, N, (size_t)period * ldy, q_per);
  return check_launch("gnf_colsum");
}

int gnf_pack_rows(const float* W, const float* mask, const int32_t* perm, float* out, int R, int K, gnf_stream_t stream) {
  if (!W || !out || R <= 0 || K <= 0) return fail(GNF_ERR_INVALID, "gnf_pack_rows: bad arguments");
  GNF_LAUNCH(pack_rows_kernel, ew_blocks((size_t)R * K), 256, 0, (cudaStream_t)stream, W, mask, perm, out, R, K);
  return check_launch("gnf_pack_rows");
}
int gnf_unpack_rows(const float* dWp, const float* mask, const int32_t* perm, float* dW, int R, int N, int K, gnf_stream_t stream) {
  if (!dWp || !dW || R <= 0 || K <= 0 || N < R) return fail(GNF_ERR_INVALID, "gnf_unpack_rows: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(dW, 0, (size_t)N * K * sizeof(float), s);
  GNF_LAUNCH(unpack_rows_kernel, ew_blocks((size_t)R * K), 256, 0, s, dWp, mask, perm, dW, R, K);
  return check_launch("gnf_unpack_rows");
}
int gnf_unpack_vec(const float* src, const int32_t* perm, float* dst, int R, int N, gnf_stream_t stream) {
  if (!src || !dst || R <= 0 || N < R) return fail(GNF_ERR_INVALID, "gnf_unpack_vec: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(dst, 0, (size_t)N * sizeof(float), s);
  GNF_LAUNCH(unpack_vec_kernel, ew_blocks((size_t)R), 256, 0, s, src, perm, dst, R);
  return check_launch("gnf_unpack_vec");
}

int gnf_dag_importance(const float* A, int d, int imp, float h_thresh, float* P, float* dPdA, gnf_stream_t stream) {
  if (!A || !P || d <= 0 || imp < GNF_IMP_RAW || imp > GNF_IMP_HARD_SQ) return fail(GNF_ERR_INVALID, "gnf_dag_importance: bad arguments");
  GNF_LAUNCH(dag_importance_kernel, ew_blocks((size_t)d * d), 256, 0, (cudaStream_t)stream, A, d * d, imp, h_thresh, P, dPdA);
  return check_launch("gnf_dag_importance");
}
int gnf_dag_bias_table(const float* W1, int ldw, const float* b1, float* T, int d, int N, int hot, gnf_stream_t stream) {
  if (!W1 || !T || d <= 0 || N <= 0 || ldw < (hot ? 2 * d : d)) return fail(GNF_ERR_INVALID, "gnf_dag_bias_table: bad arguments");
  GNF_LAUNCH(dag_bias_table_kernel, ew_blocks((size_t)(hot ? d : 1) * N), 256, 0, (cudaStream_t)stream, W1, ldw, b1, T, N, d, N, hot);
  return check_launch("gnf_dag_bias_table");
}
int gnf_dag_bias_table_ld(const float* W1, int ldw, const float* b1, float* T, int ldt, int d, int N, int hot, gnf_stream_t stream) {
  if (!W1 || !T || d <= 0 || N <= 0 || ldt < N || ldw < (hot ? 2 * d : d)) return fail(GNF_ERR_INVALID, "gnf_dag_bias_table_ld: bad arguments");
  GNF_LAUNCH(dag_bias_table_kernel, ew_blocks((size_t)(hot ? d : 1) * ldt), 256, 0, (cudaStream_t)stream, W1, ldw, b1, T, ldt, d, N, hot);
  return check_launch("gnf_dag_bias_table_ld");
}
int gnf_dag_bias_table_bwd(const float* dT, float* dW1, int ldw, float* db1, int d, int N, int hot, gnf_stream_t stream) {
  if (!dT || (hot && !dW1) || d <= 0 || N <= 0) return fail(GNF_ERR_INVALID, "gnf_dag_bias_table_bwd: bad arguments");
  GNF_LAUNCH(dag_bias_table_bwd_kernel, ew_blocks((size_t)N), 256, 0, (cudaStream_t)stream, dT, dW1, ldw, db1, d, N, hot);
  return check_launch("gnf_dag_bias_table_bwd");
}

int gnf_dag_l1_fwd(const float* x, const float* P, const gnf_gate_t* gate, const float* W1, int ldw, const float* T,
                   int bias_period, float* Y, int ldy, int B, int d, int N, int relu, gnf_stream_t stream) {
  if (!x || !P || !W1 || !Y || B < 0 || d <= 0 || N <= 0 || ldw < d || ldy < N) return fail(GNF_ERR_INVALID, "gnf_dag_l1_fwd: bad arguments");
  GateCtx g;
  if (int e = make_gate(&g, x, P, gate, d)) return e;
  if (B == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  LoadWeightT bl{W1, ldw};
  EpiBiasAct epi{Y, ldy, T, N, bias_period < 1 ? 1 : bias_period, relu};
  const int M = B * d;
  if (d <= kDagMaxD && g_dag_l1_resident) {
    GNF_LAUNCH(dag_l1_fwd_kernel<false>, ceil_div(M, kDagFwdBM), kDagFwdThreads, kDagFwdSmem, s, g, GatePlanes{nullptr, nullptr, nullptr}, W1, ldw, T, N,
               bias_period < 1 ? 1 : bias_period, relu, Y, ldy, M, N);
    return check_launch("gnf_dag_l1_fwd");
  }
  if (d >= kGateInlineMinD) launch_gemm_auto(LoadDagA<true>{g}, bl, epi, M, N, d, false, s);
  else launch_gemm_auto(LoadDagA<false>{g}, bl, epi, M, N, d, false, s);
  return check_launch("gnf_dag_l1_fwd");
}

int gnf_dag_l1_wgrad(const float* dY, int lddy, const float* x, const float* P, const gnf_gate_t* gate, float* dW1,
                     int ldw, int B, int d, int N, gnf_stream_t stream) {
  if (!dY || !x || !P || !dW1 || B < 0 || d <= 0 || N <= 0 || ldw < d || lddy < N) return fail(GNF_ERR_INVALID, "gnf_dag_l1_wgrad: bad arguments");
  GateCtx g;
  if (int e = make_gate(&g, x, P, gate, d)) return e;
  cudaStream_t s = (cudaStream_t)stream;
  zero2d(dW1, ldw, N, d, s);
  if (B == 0) return check_launch("gnf_dag_l1_wgrad");
  const int M = B * d;
  LoadColMajorA al{dY, lddy};   // A(n, m) = dY[m, n]
  EpiAtomicAdd epi{dW1, ldw};
  if (d <= kDagMaxD && g_dag_l1_resident) {
#ifndef GNF_EMU
    cudaFuncSetAttribute(dag_l1_wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDagWgSmem);   // per device: set per launch
#endif
    GNF_LAUNCH(dag_l1_wgrad_kernel<false>, ceil_div(M, kDagWgBK), kDagWgThreads, kDagWgSmem, s, g, dY, lddy, epi, M, N);
    return check_launch("gnf_dag_l1_wgrad");
  }
  if (d >= kGateInlineMinD) launch_gemm_auto(al, LoadDagB<true>{g}, epi, N, d, M, true, s);    // B(m, j) = e[m, j]
  else launch_gemm_auto(al, LoadDagB<false>{g}, epi, N, d, M, true, s);
  return check_launch("gnf_dag_l1_wgrad");
}

int gnf_dag_l1_dgrad(const float* dY, int lddy, const float* W1, int ldw, const float* x, const float* P,
                     const gnf_gate_t* gate, float* dx, float* dP, int B, int d, int N, gnf_stream_t stream) {
  if (!dY || !W1 || !x || !P || !dx || !dP || B < 0 || d <= 0 || N <= 0 || ldw < d || lddy < N) return fail(GNF_ERR_INVALID, "gnf_dag_l1_dgrad: bad arguments");
  GateCtx g;
  if (int e = make_gate(&g, x, P, gate, d)) return e;
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(dx, 0, (size_t)B * d * sizeof(float), s);
  cudaMemsetAsync(dP, 0, (size_t)d * d * sizeof(float), s);
  if (B == 0) return check_launch("gnf_dag_l1_dgrad");
  const int M = B * d;
  LoadRowMajorA al{dY, lddy};   // A(m, n)
  LoadRowMajorB bl{W1, ldw};    // B(n, j) = W1[n, j]
  if (d <= kDagMaxD && g_dag_l1_resident) {
    GNF_LAUNCH(dag_l1_dgrad_kernel<false>, ceil_div(M, kDagDgBM), kDagDgThreads, kDagDgSmem, s, g, dY, lddy, W1, ldw, dx, dP, M, N);
    return check_launch("gnf_dag_l1_dgrad");
  }
  // wide flows: N = d gives few tile columns: split the reduction over the layer width.  The epilogue is
  // linear in the accumulator and already reduces with atomics, so partial sums need no second pass.
  if (d >= kGateInlineMinD) launch_gemm_auto(al, bl, EpiDagDgrad<true>{g, dx, dP}, M, d, N, true, s);
  else launch_gemm_auto(al, bl, EpiDagDgrad<false>{g, dx, dP}, M, d, N, true, s);
  return check_launch("gnf_dag_l1_dgrad");
}

// The three planes alone (layer 1's forward GEMM then runs on the tensor-core engine against E): one gate per thread, grid-stride.
__global__ void __launch_bounds__(256) dag_gate_planes_kernel(GateCtx g, GatePlanes sv, int M) {
  const int d = g.d;
  const size_t total = (size_t)M * kDagKP;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(idx % kDagKP), m = (int)(idx / kDagKP);
    float v = 0.f, ddx = 0.f, ddp = 0.f;
    if (j < d) v = gate_e<true, true>(g, m / d, m % d, j, &ddx, &ddp);
    sv.E[idx] = v;
    sv.DX[idx] = ddx;
    sv.DP[idx] = ddp;
  }
}

// dx[b, j] = sum_i dE[(b,i), j] DX[(b,i), j]  (owned by the CTA of batch entry b),  dP[i, j] += sum_b dE[(b,i), j] DP[(b,i), j]  (atomics;
// every CTA sums kNarrowRedB batch entries in registers first).  Planes [B d][64]; thread = (j quad, i residue mod 16).  grid = ceil(B / kNarrowRedB).
constexpr int kNarrowRedB = 2;
__global__ void __launch_bounds__(256) dag_l1_reduce_narrow_kernel(const float* __restrict__ dE, const float* __restrict__ DX, const float* __restrict__ DP,
                                                                   float* __restrict__ dx, float* __restrict__ dP, int B, int d) {
  GNF_SMEM(float, red);                           // [16 i residues][64 j]
  const int jq = threadIdx.x & 15, ig = threadIdx.x >> 4, j = jq * 4;
  const int b0 = blockIdx.x * kNarrowRedB;
  float4 accp[4];                                 // dP partial sums of rows i = ig + 16 r (d <= 64: r < 4)
#pragma unroll
  for (int r = 0; r < 4; ++r) accp[r] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int bb = 0; bb < kNarrowRedB; ++bb) {
    const int b = b0 + bb;
    float4 sx = make_float4(0.f, 0.f, 0.f, 0.f);
    if (b < B) {
      float4 e[4], vx[4], vp[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {               // unconditional loads from clamped rows, masked at use
        const int i = ig + 16 * r, ic = i < d ? i : d - 1;
        const size_t o = ((size_t)b * d + ic) * kDagKP + j;
        e[r] = __ldg(reinterpret_cast<const float4*>(dE + o));
        vx[r] = __ldg(reinterpret_cast<const float4*>(DX + o));
        vp[r] = __ldg(reinterpret_cast<const float4*>(DP + o));
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        if (ig + 16 * r < d) {
          sx.x = fmaf(e[r].x, vx[r].x, sx.x); sx.y = fmaf(e[r].y, vx[r].y, sx.y); sx.z = fmaf(e[r].z, vx[r].z, sx.z); sx.w = fmaf(e[r].w, vx[r].w, sx.w);
          accp[r].x = fmaf(e[r].x, vp[r].x, accp[r].x); accp[r].y = fmaf(e[r].y, vp[r].y, accp[r].y);
          accp[r].z = fmaf(e[r].z, vp[r].z, accp[r].z); accp[r].w = fmaf(e[r].w, vp[r].w, accp[r].w);
        }
      }
    }
    *reinterpret_cast<float4*>(red + ig * kDagKP + j) = sx;
    __syncthreads();
    if (threadIdx.x < kDagKP && b < B && (int)threadIdx.x < d) {
      float t = 0.f;
#pragma unroll
      for (int g = 0; g < 16; ++g) t += red[g * kDagKP + threadIdx.x];
      dx[(size_t)b * d + threadIdx.x] = t;
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i = ig + 16 * r;
    if (i < d) {
      float* dst = dP + (size_t)i * d + j;
      if (j < d) atomicAdd(dst, accp[r].x);
      if (j + 1 < d) atomicAdd(dst + 1, accp[r].y);
      if (j + 2 < d) atomicAdd(dst + 2, accp[r].z);
      if (j + 3 < d) atomicAdd(dst + 3, accp[r].w);
    }
  }
}

// Narrow flows (d <= GNF_DAG_L1_MAX_D), training: the forward keeps the gate planes, the backward kernels read them
int gnf_dag_l1_fwd_save(const float* x, const float* P, const gnf_gate_t* gate, const float* W1, int ldw, const float* T, int bias_period,
                        float* Y, int ldy, float* E, float* DX, float* DP, int B, int d, int N, int relu, gnf_stream_t stream) {
  if (!x || !P || !W1 || !Y || !E || !DX || !DP || B < 0 || d <= 0 || N <= 0 || ldw < d || ldy < N) return fail(GNF_ERR_INVALID, "gnf_dag_l1_fwd_save: bad arguments");
  if (d > kDagMaxD) return fail(GNF_ERR_UNSUPPORTED, "gnf_dag_l1_fwd_save: d <= 64 only (wide flows: gnf_dag_embed_fwd + the GEMM engine)");
  if (((reinterpret_cast<uintptr_t>(DX) | reinterpret_cast<uintptr_t>(DP)) & 15) != 0) return fail(GNF_ERR_INVALID, "gnf_dag_l1_fwd_save: planes must be 16-byte aligned");
  GateCtx g;
  if (int e = make_gate(&g, x, P, gate, d)) return e;
  if (B == 0) return 0;
  const int M = B * d;
  GNF_LAUNCH(dag_l1_fwd_kernel<true>, ceil_div(M, kDagFwdBM), kDagFwdThreads, kDagFwdSmem, (cudaStream_t)stream, g, GatePlanes{E, DX, DP}, W1, ldw, T, N,
             bias_period < 1 ? 1 : bias_period, relu, Y, ldy, M, N);
  return check_launch("gnf_dag_l1_fwd_save");
}

int gnf_dag_gate_planes(const float* x, const float* P, const gnf_gate_t* gate, float* E, float* DX, float* DP, int B, int d, gnf_stream_t stream) {
  if (!x || !P || !E || !DX || !DP || B < 0 || d <= 0 || d > kDagMaxD) return fail(GNF_ERR_INVALID, "gnf_dag_gate_planes: bad arguments (d <= 64)");
  GateCtx g;
  if (int e = make_gate(&g, x, P, gate, d)) return e;
  if (B == 0) return 0;
  const int M = B * d;
  GNF_LAUNCH(dag_gate_planes_kernel, ew_blocks((size_t)M * kDagKP), 256, 0, (cudaStream_t)stream, g, GatePlanes{E, DX, DP}, M);
  return check_launch("gnf_dag_gate_planes");
}

int gnf_dag_l1_wgrad_saved(const float* dY, int lddy, const float* E, float* dW1, int ldw, int B, int d, int N, gnf_stream_t stream) {
  if (!dY || !E || !dW1 || B < 0 || d <= 0 || d > kDagMaxD || N <= 0 || ldw < d || lddy < N) return fail(GNF_ERR_INVALID, "gnf_dag_l1_wgrad_saved: bad arguments (d <= 64)");
  cudaStream_t s = (cudaStream_t)stream;
  zero2d(dW1, ldw, N, d, s);
  if (B == 0) return check_launch("gnf_dag_l1_wgrad_saved");
  GateCtx g = {};
  g.x = E; g.d = d;
  const int M = B * d;
#ifndef GNF_EMU
  cudaFuncSetAttribute(dag_l1_wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDagWgSmem);
#endif
  GNF_LAUNCH(dag_l1_wgrad_kernel<true>, ceil_div(M, kDagWgBK), kDagWgThreads, kDagWgSmem, s, g, dY, lddy, EpiAtomicAdd{dW1, ldw}, M, N);
  return check_launch("gnf_dag_l1_wgrad_saved");
}

int gnf_dag_l1_dgrad_saved(const float* dY, int lddy, const float* W1, int ldw, const float* DX, const float* DP, float* dx, float* dP,
                           int B, int d, int N, gnf_stream_t stream) {
  if (!dY || !W1 || !DX || !DP || !dx || !dP || B < 0 || d <= 0 || d > kDagMaxD || N <= 0 || ldw < d || lddy < N ||
      ((reinterpret_cast<uintptr_t>(DX) | reinterpret_cast<uintptr_t>(DP)) & 15) != 0)
    return fail(GNF_ERR_INVALID, "gnf_dag_l1_dgrad_saved: bad arguments (d <= 64, 16-byte aligned planes)");
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(dx, 0, (size_t)B * d * sizeof(float), s);
  cudaMemsetAsync(dP, 0, (size_t)d * d * sizeof(float), s);
  if (B == 0) return check_launch("gnf_dag_l1_dgrad_saved");
  GateCtx g = {};
  g.x = DX; g.P = DP; g.d = d;
  const int M = B * d;
  GNF_LAUNCH(dag_l1_dgrad_kernel<true>, ceil_div(M, kDagDgBM), kDagDgThreads, kDagDgSmem, s, g, dY, lddy, W1, ldw, dx, dP, M, N);
  return check_launch("gnf_dag_l1_dgrad_saved");
}

int gnf_dag_l1_reduce_saved(const float* dE, const float* DX, const float* DP, float* dx, float* dP, int B, int d, gnf_stream_t stream) {
  if (!dE || !DX || !DP || !dx || !dP || B < 0 || d <= 0 || d > kDagMaxD ||
      ((reinterpret_cast<uintptr_t>(dE) | reinterpret_cast<uintptr_t>(DX) | reinterpret_cast<uintptr_t>(DP)) & 15) != 0)
    return fail(GNF_ERR_INVALID, "gnf_dag_l1_reduce_saved: bad arguments (d <= 64, 16-byte aligned [B d, 64] planes)");
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(dP, 0, (size_t)d * d * sizeof(float), s);
  if (B == 0) return check_launch("gnf_dag_l1_reduce_saved");
  GNF_LAUNCH(dag_l1_reduce_narrow_kernel, ceil_div(B, kNarrowRedB), 256, 16 * kDagKP * sizeof(float), s, dE, DX, DP, dx, dP, B, d);
  return check_launch("gnf_dag_l1_reduce_saved");
}

int gnf_dag_embed_fwd(const float* x, const float* P, const gnf_gate_t* gate, float* E, float* DX, float* DP, int lde, int B, int d,
                      gnf_stream_t stream) {
  if (!x || !P || !E || B < 0 || d <= 0 || lde < d || (lde % 4) != 0 || (reinterpret_cast<uintptr_t>(E) & 15) != 0 || ((DX == nullptr) != (DP == nullptr)) ||
      (reinterpret_cast<uintptr_t>(DX) & 15) != 0 || (reinterpret_cast<uintptr_t>(DP) & 15) != 0)
    return fail(GNF_ERR_INVALID, "gnf_dag_embed_fwd: bad arguments (plane rows must be 16-byte aligned: lde %% 4 == 0; DX and DP go together)");
  GateCtx g;
  if (int e = make_gate(&g, x, P, gate, d)) return e;
  if (B == 0) return 0;
  if (DX) GNF_LAUNCH(dag_embed_fwd_kernel<true>, B * d, 256, 0, (cudaStream_t)stream, g, E, DX, DP, lde);
  else GNF_LAUNCH(dag_embed_fwd_kernel<false>, B * d, 256, 0, (cudaStream_t)stream, g, E, DX, DP, lde);
  return check_launch("gnf_dag_embed_fwd");
}

int gnf_dag_embed_bwd(const float* dE, int lde, const float* x, const float* P, const gnf_gate_t* gate, const float* DX, const float* DP,
                      float* dx, float* dP, int B, int d, gnf_stream_t stream) {
  if (!dE || !dx || !dP || B < 0 || d <= 0 || lde < d || ((DX == nullptr) != (DP == nullptr)) || (!DX && (!x || !P)))
    return fail(GNF_ERR_INVALID, "gnf_dag_embed_bwd: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemsetAsync(dx, 0, (size_t)B * d * sizeof(float), s);
  if (B == 0) {
    cudaMemsetAsync(dP, 0, (size_t)d * d * sizeof(float), s);
    return check_launch("gnf_dag_embed_bwd");
  }
  const dim3 grid(ceil_div(d, 128), ceil_div(d, 2 * kEmbBwdI));
  if (DX) {
    if ((lde % 4) != 0 || ((reinterpret_cast<uintptr_t>(dE) | reinterpret_cast<uintptr_t>(DX) | reinterpret_cast<uintptr_t>(DP)) & 15) != 0)
      return fail(GNF_ERR_INVALID, "gnf_dag_embed_bwd: the planes must have 16-byte aligned rows (lde %% 4 == 0)");
    GNF_LAUNCH(dag_embed_bwd_saved_kernel, dim3(ceil_div(d, 256), ceil_div(d, 4 * kEmbSavedI)), 256, 0, s, dE, DX, DP, lde, dx, dP, B, d);
  } else {
    GateCtx g;
    if (int e = make_gate(&g, x, P, gate, d)) return e;
    GNF_LAUNCH(dag_embed_bwd_kernel, grid, 256, 0, s, g, dE, lde, dx, dP, B);
  }
  return check_launch("gnf_dag_embed_bwd");
}

#ifdef GNF_DEVTOOLS
int gnf_linear_set_thin(int enable) {
  g_thin = enable != 0;
  return 0;
}
#endif

#ifdef GNF_DEVTOOLS
int gnf_dag_l1_set_resident(int enable) {
  g_dag_l1_resident = enable != 0;
  return 0;
}
#endif

int gnf_dag_finish_dA(const float* dP, const float* dPdA, float* dA, int d, int accumulate, gnf_stream_t stream) {
  if (!dP || !dPdA || !dA || d <= 0) return fail(GNF_ERR_INVALID, "gnf_dag_finish_dA: bad arguments");
  GNF_LAUNCH(dag_finish_dA_kernel, ew_blocks((size_t)d * d), 256, 0, (cudaStream_t)stream, dP, dPdA, dA, d * d, accumulate);
  return check_launch("gnf_dag_finish_dA");
}

int gnf_dag_dump_noise(const gnf_gate_t* gate, float* n1, float* n2, int B, int d, gnf_stream_t stream) {
  if (!gate || !n1 || B <= 0 || d <= 0) return fail(GNF_ERR_INVALID, "gnf_dag_dump_noise: bad arguments");
  GateCtx g;
  gnf_gate_t tmp = *gate;
  tmp.noise1 = tmp.noise2 = nullptr;
  if (int e = make_gate(&g, nullptr, nullptr, &tmp, d)) return e;
  const size_t n = (size_t)B * d * d;
  GNF_LAUNCH(dag_dump_noise_kernel, ew_blocks(n), 256, 0, (cudaStream_t)stream, g, n1, n2, n);
  return check_launch("gnf_dag_dump_noise");
}

}  // extern "C"
