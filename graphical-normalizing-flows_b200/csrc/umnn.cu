// K3: MonotonicNormalizer — fused Clenshaw-Curtis UMNN integral, forward and recompute backward.
// (MonotonicNormalizer.forward / IntegrandNet, models/Normalizers/MonotonicNormalizer.py:12-66;
//  UMNN==1.0 NeuralIntegral / ParallelNeuralIntegral, SURVEY.md App. B.)
//
// Strict-fp32 FFMA version.  A "node-row" is one evaluation of the integrand network
// f([X, h_r]) for one (sample, dim) row r and one quadrature node k.  Node-rows are flattened
// (q = r*(S+1)+k) and processed in tiles of 64; a tile's activations live in shared memory from
// the first layer to the CC-weighted reduction, so neither the [B(S+1), d*E] expansion of h nor any
// [B(S+1)d, I] activation of the reference ever reaches HBM.  Weights are streamed from L2 in
// 16-row K-panels with cp.async double buffering.
//
// Thread layout of a 64 x NP tile (NP = 16*TN = padded hidden width), 256 threads:
//   ty = tid/16 -> rows 4ty..4ty+3,  tx = tid%16 -> cols tx + 16j (j < TN);  acc[4][TN] registers.
// Activations are stored k-major, act[col][row] with row stride LDR = 68 floats, so the GEMM's
// A-operand read is one broadcast float4 per k and the epilogue store is a float4 per column.
#include "common.cuh"

namespace gnf {

constexpr int kTileM = 64;
constexpr int kLDR = kTileM + 4;
constexpr int kKC = 16;  // weight panel depth
constexpr int kUThreads = 256;

struct UmnnPacked {
  // device pointers into the workspace (all zero padded)
  const float* Wt[GNF_MAX_LAYERS];    // [KP_l][NP]   Wt[k][n] = W[n][k]          (hidden-output layers)
  const float* Wn[GNF_MAX_LAYERS];    // [NP][KPo_l]  Wn[n][k] = W[n][k]          (for dgrad)
  const float* bias[GNF_MAX_LAYERS];  // [NP]
  const float* wlast;                 // [NP]
  int kpad[GNF_MAX_LAYERS];           // round_up(dims[l], 16): number of K rows actually streamed
  int kb0;                            // backward input-tile rows: 32*ceil(dims[0]/32); Wn[0] is stored as
                                      // kb0/32 column blocks [blk][NP][32]
  int dims[GNF_MAX_LAYERS + 1];
  int L;                              // number of hidden layers (= n_layers - 1)
  float blast;                        // unused on device (bias of last layer read from pointer)
  const float* blast_ptr;
};

struct PackPlan {
  size_t off_Wt[GNF_MAX_LAYERS], off_Wn[GNF_MAX_LAYERS], off_bias[GNF_MAX_LAYERS], off_wlast, total;
  int NP, KP0, KB0;
};

__host__ __device__ static inline int round16(int v) { return (v + 15) / 16 * 16; }

static int make_plan(const gnf_mlp_t* net, PackPlan* pl, int* TN_out) {
  if (!net || net->n_layers < 2 || net->n_layers > GNF_MAX_LAYERS) return fail(GNF_ERR_UNSUPPORTED, "umnn: integrand needs 2..%d linear layers", GNF_MAX_LAYERS);
  if (net->dims[net->n_layers] != 1) return fail(GNF_ERR_UNSUPPORTED, "umnn: integrand output size must be 1");
  const int L = net->n_layers - 1;
  int maxh = 0;
  for (int l = 1; l <= L; ++l) maxh = net->dims[l] > maxh ? net->dims[l] : maxh;
  if (net->dims[0] < 1 || net->dims[0] > 256 || maxh < 1 || maxh > 256) return fail(GNF_ERR_UNSUPPORTED, "umnn: layer widths must be in 1..256 (got in=%d, hidden max=%d)", net->dims[0], maxh);
  const int want = ceil_div(maxh, 16);
  const int opts[6] = {2, 4, 7, 10, 13, 16};
  int TN = 16;
  for (int i = 0; i < 6; ++i) if (opts[i] >= want) { TN = opts[i]; break; }
  const int NP = 16 * TN;
  const int KP0 = round16(net->dims[0]);
  const int KB0 = (net->dims[0] + 31) / 32 * 32;
  if (KP0 > NP) return fail(GNF_ERR_UNSUPPORTED, "umnn: 1+cond_size (%d) wider than padded hidden width (%d)", net->dims[0], NP);
  size_t off = 0;
  for (int l = 0; l < L; ++l) {
    const int KP = (l == 0) ? KP0 : NP;
    pl->off_Wt[l] = off; off += (size_t)KP * NP;
    pl->off_Wn[l] = off; off += (size_t)NP * ((l == 0) ? KB0 : NP);
    pl->off_bias[l] = off; off += NP;
  }
  pl->off_wlast = off; off += NP;
  pl->total = off;
  pl->NP = NP; pl->KP0 = KP0; pl->KB0 = KB0;
  *TN_out = TN;
  return 0;
}

struct PackArgs {
  const float* W[GNF_MAX_LAYERS];
  const float* b[GNF_MAX_LAYERS];
  size_t off_Wt[GNF_MAX_LAYERS], off_Wn[GNF_MAX_LAYERS], off_bias[GNF_MAX_LAYERS], off_wlast;
  int dims[GNF_MAX_LAYERS + 1];
  int L, NP, KP0, KB0;
};

__global__ void umnn_pack_kernel(PackArgs a, float* __restrict__ ws, size_t total) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    float v = 0.f;
    if (i >= a.off_wlast) {
      const int k = (int)(i - a.off_wlast);
      if (k < a.dims[a.L]) v = a.W[a.L][k];
    } else {
      int l = 0;
      while (l + 1 < a.L && i >= a.off_Wt[l + 1]) ++l;
      const int KP = (l == 0) ? a.KP0 : a.NP;
      const int K = a.dims[l], N = a.dims[l + 1];
      if (i >= a.off_bias[l]) {
        const int n = (int)(i - a.off_bias[l]);
        if (n < N) v = a.b[l][n];
      } else if (i >= a.off_Wn[l]) {
        const size_t e = i - a.off_Wn[l];
        int n, k;
        if (l == 0) {  // column-blocked [blk][NP][32]
          const int blk = (int)(e / ((size_t)a.NP * 32));
          n = (int)((e / 32) % a.NP);
          k = blk * 32 + (int)(e % 32);
        } else {
          n = (int)(e / KP); k = (int)(e % KP);
        }
        if (n < N && k < K) v = a.W[l][(size_t)n * K + k];
      } else {
        const size_t e = i - a.off_Wt[l];
        const int k = (int)(e / a.NP), n = (int)(e % a.NP);
        if (n < N && k < K) v = a.W[l][(size_t)n * K + k];
      }
    }
    ws[i] = v;
  }
}

static void fill_packed(const gnf_mlp_t* net, const PackPlan& pl, float* ws, UmnnPacked* pk) {
  const int L = net->n_layers - 1;
  pk->L = L;
  for (int l = 0; l <= net->n_layers; ++l) pk->dims[l] = net->dims[l];
  for (int l = 0; l < L; ++l) {
    pk->Wt[l] = ws + pl.off_Wt[l];
    pk->Wn[l] = ws + pl.off_Wn[l];
    pk->bias[l] = ws + pl.off_bias[l];
    pk->kpad[l] = round16(net->dims[l]);
  }
  pk->kb0 = pl.KB0;
  pk->wlast = ws + pl.off_wlast;
  pk->blast_ptr = net->b[L];
  pk->blast = 0.f;
}

static void launch_pack(const gnf_mlp_t* net, const PackPlan& pl, float* ws, cudaStream_t s) {
  PackArgs a;
  const int L = net->n_layers - 1;
  for (int l = 0; l < GNF_MAX_LAYERS; ++l) { a.W[l] = nullptr; a.b[l] = nullptr; a.off_Wt[l] = a.off_Wn[l] = a.off_bias[l] = 0; }
  for (int l = 0; l <= L; ++l) { a.W[l] = net->W[l]; a.b[l] = net->b[l]; }
  for (int l = 0; l < L; ++l) { a.off_Wt[l] = pl.off_Wt[l]; a.off_Wn[l] = pl.off_Wn[l]; a.off_bias[l] = pl.off_bias[l]; }
  a.off_wlast = pl.off_wlast;
  for (int l = 0; l <= net->n_layers; ++l) a.dims[l] = net->dims[l];
  a.L = L; a.NP = pl.NP; a.KP0 = pl.KP0; a.KB0 = pl.KB0;
  int blocks = (int)((pl.total + 255) / 256);
  if (blocks > 2 * kNumSMs) blocks = 2 * kNumSMs;
  GNF_LAUNCH(umnn_pack_kernel, blocks, 256, 0, s, a, ws, pl.total);
}

// ------------------------------------------------------------------------------------------------
// 64 x (16*TN) tile GEMM: acc = act_in^T-tile (k-major in smem) x W panels streamed from global.
//   act_in : smem [K][kLDR];  Wg: global [npanels*16][16*TN] (zero padded);  wp: smem [2][16][16*TN]
// ------------------------------------------------------------------------------------------------
template <int TN>
__device__ __forceinline__ void tile_gemm(float (&acc)[4][TN], const float* __restrict__ act_in, const float* __restrict__ Wg, int npanels, float* __restrict__ wp) {
  constexpr int NPo = 16 * TN;
  constexpr int PANEL_F4 = kKC * NPo / 4;
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
  auto issue = [&](int pi) {
    const float4* src = reinterpret_cast<const float4*>(Wg + (size_t)pi * kKC * NPo);
    float4* dst = reinterpret_cast<float4*>(wp + (pi & 1) * kKC * NPo);
    for (int i = t; i < PANEL_F4; i += kUThreads) cp_async16(dst + i, src + i);
    cp_async_commit();
  };
  issue(0);
  for (int pi = 0; pi < npanels; ++pi) {
    if (pi + 1 < npanels) { issue(pi + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    const float* w = wp + (pi & 1) * kKC * NPo + tx;
    const float* a = act_in + (size_t)(pi * kKC) * kLDR + 4 * ty;
#pragma unroll
    for (int kk = 0; kk < kKC; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(a + kk * kLDR);
#pragma unroll
      for (int j = 0; j < TN; ++j) {
        const float b = w[kk * NPo + 16 * j];
        acc[0][j] = fmaf(av.x, b, acc[0][j]);
        acc[1][j] = fmaf(av.y, b, acc[1][j]);
        acc[2][j] = fmaf(av.z, b, acc[2][j]);
        acc[3][j] = fmaf(av.w, b, acc[3][j]);
      }
    }
    __syncthreads();
  }
}

// Epilogue: out[col][row] = relu(acc + bias[col])  (k-major store, float4 over the thread's 4 rows).
// gsave (nullable): also keep the activations in global memory, row-major [tile row][gsave_ld], for a backward that
// loads them instead of recomputing the forward (rows >= rows_valid are not written).
template <int TN>
__device__ __forceinline__ void store_bias_relu(const float (&acc)[4][TN], const float* __restrict__ bias, float* __restrict__ act_out,
                                                float* __restrict__ gsave = nullptr, int gsave_ld = 0, int rows_valid = 0) {
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
#pragma unroll
  for (int j = 0; j < TN; ++j) {
    const int col = tx + 16 * j;
    const float b = __ldg(bias + col);
    float4 o;
    o.x = fmaxf(acc[0][j] + b, 0.f);
    o.y = fmaxf(acc[1][j] + b, 0.f);
    o.z = fmaxf(acc[2][j] + b, 0.f);
    o.w = fmaxf(acc[3][j] + b, 0.f);
    *reinterpret_cast<float4*>(act_out + (size_t)col * kLDR + 4 * ty) = o;
    if (gsave) {
      float* gp = gsave + (size_t)(4 * ty) * gsave_ld + col;
      if (4 * ty + 0 < rows_valid) gp[0] = o.x;
      if (4 * ty + 1 < rows_valid) gp[(size_t)gsave_ld] = o.y;
      if (4 * ty + 2 < rows_valid) gp[(size_t)2 * gsave_ld] = o.z;
      if (4 * ty + 3 < rows_valid) gp[(size_t)3 * gsave_ld] = o.w;
    }
  }
}

// y[row] = sum_k act[k][row]*wlast[k] + blast  -> yout[row]   (red: smem [4][64] scratch)
__device__ __forceinline__ void last_layer(const float* __restrict__ act, const float* __restrict__ wlast, float blast, int NP, float* __restrict__ red, float* __restrict__ yout) {
  const int t = threadIdx.x, row = t & 63, part = t >> 6;
  float s = 0.f;
  for (int k = part; k < NP; k += 4) s = fmaf(act[(size_t)k * kLDR + row], __ldg(wlast + k), s);
  red[part * 64 + row] = s;
  __syncthreads();
  if (t < 64) yout[t] = ((red[t] + red[64 + t]) + (red[128 + t] + red[192 + t])) + blast;
  __syncthreads();
}

static size_t fwd_smem_bytes_for(int NP) { return ((size_t)2 * NP * kLDR + 2 * kKC * NP + 256 + 64) * sizeof(float); }

struct UmnnFwdParams {
  const float* x; const float* h; const float* ccw; const float* ccn;
  float* z; float* zrev; float* jac; float* logdet;
  float* saved;   // nullable: [Q][L*NP] hidden activations kept for the backward
  int R, d, E, S;
  long long Q;  // R*(S+1)
  UmnnPacked pk;
};

template <int TN>
__global__ void __launch_bounds__(kUThreads) umnn_fwd_kernel(UmnnFwdParams p) {
  constexpr int NP = 16 * TN;
  GNF_SMEM(float, smem);
  float* act0 = smem;                       // [NP][kLDR]
  float* act1 = act0 + NP * kLDR;           // [NP][kLDR]
  float* wp = act1 + NP * kLDR;             // [2][16][NP]
  float* red = wp + 2 * kKC * NP;           // [256]
  float* yout = red + 256;                  // [64]
  const int t = threadIdx.x;
  const int nodes = p.S + 1;
  const int KP0 = p.pk.kpad[0];
  const long long ntiles = (p.Q + kTileM - 1) / kTileM;
  const float blast = __ldg(p.pk.blast_ptr);

  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long q0 = tile * kTileM;
    // ---- input tile [KP0][64]: k=0 -> node abscissa, k=1..E -> h[r, k-1]
    for (int idx = t; idx < KP0 * kTileM; idx += kUThreads) {
      const int row = idx & 63, k = idx >> 6;
      const long long q = q0 + row;
      float v = 0.f;
      if (q < p.Q && k <= p.E) {
        const int r = (int)(q / nodes), kn = (int)(q % nodes);
        if (k == 0) v = (__ldg(p.x + r) * (__ldg(p.ccn + kn) + 1.f)) / 2.f;
        else v = __ldg(p.h + (size_t)r * p.E + (k - 1));
      }
      act0[(size_t)k * kLDR + row] = v;
    }
    __syncthreads();
    float* cur = act0;
    float* nxt = act1;
    float acc[4][TN];
    for (int l = 0; l < p.pk.L; ++l) {
      tile_gemm<TN>(acc, cur, p.pk.Wt[l], p.pk.kpad[l] / kKC, wp);
      if (p.saved) {
        const long long left = p.Q - q0;
        store_bias_relu<TN>(acc, p.pk.bias[l], nxt, p.saved + (size_t)q0 * (p.pk.L * NP) + (size_t)l * NP, p.pk.L * NP,
                            left < kTileM ? (int)left : kTileM);
      } else {
        store_bias_relu<TN>(acc, p.pk.bias[l], nxt);
      }
      float* tmp = cur; cur = nxt; nxt = tmp;
      __syncthreads();
    }
    last_layer(cur, p.pk.wlast, blast, NP, red, yout);
    // ---- integrand value, CC-weighted segment sums
    if (t < 64) {
      const float y = yout[t];
      const float f = (y > 0.f ? y : expm1f(y)) + 1.05f;
      const long long q = q0 + t;
      float wv = 0.f;
      if (q < p.Q) {
        const int kn = (int)(q % nodes);
        wv = __ldg(p.ccw + kn) * f;
        if (kn == 0) {
          const int r = (int)(q / nodes);
          p.jac[r] = f;
          if (p.logdet) atomicAdd(p.logdet + r / p.d, logf(f));
        }
      }
      red[t] = wv;
    }
    __syncthreads();
    if (t < 64) {
      const long long q = q0 + t;
      if (q < p.Q) {
        const int r = (int)(q / nodes), kn = (int)(q % nodes);
        if (kn == 0 || t == 0) {
          float s = 0.f;
          int rem = nodes - kn;               // node-rows of r from here on
          if (rem > 64 - t) rem = 64 - t;
          for (int i = 0; i < rem; ++i) s += red[t + i];
          const float xv = __ldg(p.x + r);
          float c = s * xv / 2.f;
          if (kn == 0) c += __ldg(p.h + (size_t)r * p.E);
          atomicAdd(p.z + r, c);
          if (p.zrev) { const int b = r / p.d, i = r % p.d; atomicAdd(p.zrev + (size_t)b * p.d + (p.d - 1 - i), c); }
        }
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// Inverse by bisection (MonotonicNormalizer.inverse_transform, MonotonicNormalizer.py:69-83): the reference runs 20 full
// forward passes, halving [-20, 20] around x_middle after each.  Here the whole search of a row lives in one CTA: a tile
// holds ALL quadrature nodes of floor(64 / (S+1)) rows, so z(x_middle) is a shared-memory segment sum (no atomics, no
// global round trip) and the interval update, the next abscissae and the next forward pass follow in the same launch.
// ------------------------------------------------------------------------------------------------
struct UmnnInvParams {
  const float* z; const float* h; const float* ccw; const float* ccn;
  float* x;
  int R, E, S, iters;
  float lo, hi;
  UmnnPacked pk;
};

template <int TN>
__global__ void __launch_bounds__(kUThreads) umnn_invert_kernel(UmnnInvParams p) {
  constexpr int NP = 16 * TN;
  GNF_SMEM(float, smem);
  float* act0 = smem;                       // [NP][kLDR]
  float* act1 = act0 + NP * kLDR;           // [NP][kLDR]
  float* wp = act1 + NP * kLDR;             // [2][16][NP]
  float* red = wp + 2 * kKC * NP;           // [256]
  float* yout = red + 256;                  // [64]
  float* xlo = yout + 64;                   // [64] search interval and target of the tile's rows
  float* xhi = xlo + 64;
  float* zt = xhi + 64;
  const int t = threadIdx.x;
  const int nodes = p.S + 1;
  const int rows_per = kTileM / nodes;      // >= 1 (checked by the launcher)
  const int KP0 = p.pk.kpad[0];
  const int ntiles = (p.R + rows_per - 1) / rows_per;
  const float blast = __ldg(p.pk.blast_ptr);

  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int r0 = tile * rows_per;
    const int nr = (p.R - r0 < rows_per) ? p.R - r0 : rows_per;
    if (t < kTileM) {
      xlo[t] = p.lo; xhi[t] = p.hi;
      zt[t] = t < nr ? __ldg(p.z + r0 + t) : 0.f;
    }
    __syncthreads();
    for (int it = 0; it < p.iters; ++it) {
      // ---- input tile [KP0][64]: k=0 -> node abscissa of x_middle, k=1..E -> h[r, k-1]
      for (int idx = t; idx < KP0 * kTileM; idx += kUThreads) {
        const int row = idx & 63, k = idx >> 6;
        const int lr = row / nodes, kn = row - lr * nodes;
        float v = 0.f;
        if (lr < nr && k <= p.E) {
          if (k == 0) v = (((xhi[lr] + xlo[lr]) / 2.f) * (__ldg(p.ccn + kn) + 1.f)) / 2.f;
          else v = __ldg(p.h + (size_t)(r0 + lr) * p.E + (k - 1));
        }
        act0[(size_t)k * kLDR + row] = v;
      }
      __syncthreads();
      float* cur = act0;
      float* nxt = act1;
      float acc[4][TN];
      for (int l = 0; l < p.pk.L; ++l) {
        tile_gemm<TN>(acc, cur, p.pk.Wt[l], p.pk.kpad[l] / kKC, wp);
        store_bias_relu<TN>(acc, p.pk.bias[l], nxt);
        float* tmp = cur; cur = nxt; nxt = tmp;
        __syncthreads();
      }
      last_layer(cur, p.pk.wlast, blast, NP, red, yout);
      if (t < kTileM) {
        const float y = yout[t];
        const float f = (y > 0.f ? y : expm1f(y)) + 1.05f;
        const int lr = t / nodes, kn = t - lr * nodes;
        red[t] = lr < nr ? __ldg(p.ccw + kn) * f : 0.f;
      }
      __syncthreads();
      if (t < nr) {
        float sacc = 0.f;
        for (int i = 0; i < nodes; ++i) sacc += red[t * nodes + i];
        const float xm = (xhi[t] + xlo[t]) / 2.f;
        const float zm = sacc * xm / 2.f + __ldg(p.h + (size_t)(r0 + t) * p.E);
        if (zm > zt[t]) xhi[t] = xm; else xlo[t] = xm;          // left = (z_middle > z): x_max = x_middle, else x_min = x_middle
      }
      __syncthreads();
    }
    if (t < nr) p.x[r0 + t] = (xhi[t] + xlo[t]) / 2.f;
    __syncthreads();
  }
}

template <int TN>
static int launch_invert(const UmnnInvParams& p, cudaStream_t s) {
  const size_t smem = fwd_smem_bytes_for(16 * TN) + 3 * 64 * sizeof(float);
  if (smem > 227 * 1024) return fail(GNF_ERR_UNSUPPORTED, "umnn invert: shared memory %zu B exceeds 227 KB", smem);
#ifndef GNF_EMU
  cudaFuncSetAttribute(umnn_invert_kernel<TN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
  const int rows_per = kTileM / (p.S + 1);
  const long long ntiles = ((long long)p.R + rows_per - 1) / rows_per;
  const int per_sm = (int)((227 * 1024) / (smem + 1024));
  long long grid = (long long)kNumSMs * (per_sm < 1 ? 1 : (per_sm > 2 ? 2 : per_sm));
  if (grid > ntiles) grid = ntiles;
  GNF_LAUNCH(umnn_invert_kernel<TN>, (unsigned)grid, kUThreads, smem, s, p);
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Backward
// ------------------------------------------------------------------------------------------------
struct UmnnBwdParams {
  const float* x; const float* h; const float* ccw; const float* ccn; const float* jac;
  const float* gz; const float* gzrev; const float* gjac; const float* glogdet;
  float* dx; float* dh;
  float* dW[GNF_MAX_LAYERS]; float* db[GNF_MAX_LAYERS];
  const float* saved;   // nullable: the forward's hidden activations [R*(S+1)][L*NP]; NULL -> recompute
  int R, d, E, S;
  long long Q;  // R*(S+2)
  UmnnPacked pk;
};

// dW[n][k] += sum_row dlt[n][row] * a[k][row]   for n < Nn, k < Kk ; K range covered = 16*TK columns
template <int CH, int TK>
__device__ __forceinline__ void tile_wgrad(const float* __restrict__ dlt, const float* __restrict__ a, float* __restrict__ dW, int Nn, int Kk, int ldw, int n_groups) {
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  for (int i0 = 0; i0 < n_groups; i0 += CH) {
    float acc[CH][TK];
#pragma unroll
    for (int i = 0; i < CH; ++i)
#pragma unroll
      for (int j = 0; j < TK; ++j) acc[i][j] = 0.f;
#pragma unroll 2
    for (int r4 = 0; r4 < kTileM / 4; ++r4) {
      float4 dn[CH], ak[TK];
#pragma unroll
      for (int i = 0; i < CH; ++i) {
        const int ni = ty + 16 * (i0 + i);
        dn[i] = (i0 + i < n_groups) ? *reinterpret_cast<const float4*>(dlt + (size_t)ni * kLDR + 4 * r4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int j = 0; j < TK; ++j) ak[j] = *reinterpret_cast<const float4*>(a + (size_t)(tx + 16 * j) * kLDR + 4 * r4);
#pragma unroll
      for (int i = 0; i < CH; ++i)
#pragma unroll
        for (int j = 0; j < TK; ++j) {
          float s = acc[i][j];
          s = fmaf(dn[i].x, ak[j].x, s);
          s = fmaf(dn[i].y, ak[j].y, s);
          s = fmaf(dn[i].z, ak[j].z, s);
          s = fmaf(dn[i].w, ak[j].w, s);
          acc[i][j] = s;
        }
    }
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      const int n = ty + 16 * (i0 + i);
      if (i0 + i < n_groups && n < Nn) {
#pragma unroll
        for (int j = 0; j < TK; ++j) {
          const int k = tx + 16 * j;
          if (k < Kk) atomicAdd(dW + (size_t)n * ldw + k, acc[i][j]);
        }
      }
    }
  }
}

template <int TN> struct WgradChunk { static constexpr int CH = (TN <= 7) ? TN : (TN == 10 ? 5 : (TN == 13 ? 7 : 4)); };

template <int TN>
__global__ void __launch_bounds__(kUThreads) umnn_bwd_kernel(UmnnBwdParams p) {
  constexpr int NP = 16 * TN;
  constexpr int CH = WgradChunk<TN>::CH;
  GNF_SMEM(float, smem);
  const int L = p.pk.L;
  const int KP0 = p.pk.kb0;
  // act[0]: [KB0][kLDR] input tile; act[l], l=1..L: [NP][kLDR]
  float* actb[GNF_MAX_LAYERS + 1];
  actb[0] = smem;
  for (int l = 1; l <= L; ++l) actb[l] = smem + KP0 * kLDR + (size_t)(l - 1) * NP * kLDR;
  float* wp = smem + KP0 * kLDR + (size_t)L * NP * kLDR;  // [2][16][NP]
  float* red = wp + 2 * kKC * NP;                           // [256]
  float* yout = red + 256;                                  // [64]
  float* dy = yout + 64;                                    // [64]
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int nodes = p.S + 2;  // S+1 quadrature nodes + one plain evaluation at x (the jac output)
  const long long ntiles = (p.Q + kTileM - 1) / kTileM;
  const float blast = __ldg(p.pk.blast_ptr);

  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long q0 = tile * kTileM;
    for (int idx = t; idx < KP0 * kTileM; idx += kUThreads) {
      const int row = idx & 63, k = idx >> 6;
      const long long q = q0 + row;
      float v = 0.f;
      if (q < p.Q && k <= p.E) {
        const int r = (int)(q / nodes), kn = (int)(q % nodes);
        if (k == 0) {
          const float xv = __ldg(p.x + r);
          v = (kn <= p.S) ? (xv * (__ldg(p.ccn + kn) + 1.f)) / 2.f : xv;
        } else {
          v = __ldg(p.h + (size_t)r * p.E + (k - 1));
        }
      }
      actb[0][(size_t)k * kLDR + row] = v;
    }
    __syncthreads();
    // ---- hidden activations of every layer: reload the ones the forward kept (180 GB of HBM buys back a third of
    //      the backward's FLOPs), or recompute them like UMNN does when the caller passed no buffer
    if (p.saved) {
      const int row = t & 63, part = t >> 6;
      const long long q = q0 + row;
      const bool ok = q < p.Q;
      long long qf = 0;
      if (ok) {
        const long long r = q / nodes;
        const int kn = (int)(q % nodes);
        qf = r * (p.S + 1) + (kn <= p.S ? kn : 0);       // the extra node evaluates the integrand at x = node 0
      }
      const float4* src = reinterpret_cast<const float4*>(p.saved + (size_t)qf * (L * NP));
      for (int l = 0; l < L; ++l) {
        float* dst = actb[l + 1] + row;
#pragma unroll 2
        for (int c4 = part; c4 < NP / 4; c4 += 4) {
          const float4 v = ok ? __ldg(src + (size_t)l * (NP / 4) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
          dst[(size_t)(4 * c4 + 0) * kLDR] = v.x;
          dst[(size_t)(4 * c4 + 1) * kLDR] = v.y;
          dst[(size_t)(4 * c4 + 2) * kLDR] = v.z;
          dst[(size_t)(4 * c4 + 3) * kLDR] = v.w;
        }
      }
      __syncthreads();
    } else {
      float acc[4][TN];
      for (int l = 0; l < L; ++l) {
        tile_gemm<TN>(acc, actb[l], p.pk.Wt[l], p.pk.kpad[l] / kKC, wp);
        store_bias_relu<TN>(acc, p.pk.bias[l], actb[l + 1]);
        __syncthreads();
      }
    }
    last_layer(actb[L], p.pk.wlast, blast, NP, red, yout);
    // ---- cotangent of the pre-ELU output per node-row
    if (t < 64) {
      const long long q = q0 + t;
      float g = 0.f;
      if (q < p.Q) {
        const int r = (int)(q / nodes), kn = (int)(q % nodes);
        const int b = r / p.d, i = r % p.d;
        if (kn <= p.S) {
          float gzt = p.gz ? __ldg(p.gz + r) : 0.f;
          if (p.gzrev) gzt += __ldg(p.gzrev + (size_t)b * p.d + (p.d - 1 - i));
          g = (gzt * __ldg(p.x + r) / 2.f) * __ldg(p.ccw + kn);
        } else {
          g = p.gjac ? __ldg(p.gjac + r) : 0.f;
          if (p.glogdet) g += __ldg(p.glogdet + b) / __ldg(p.jac + r);
        }
        const float y = yout[t];
        g *= (y > 0.f) ? 1.f : expf(y);
      }
      dy[t] = g;
    }
    __syncthreads();
    // ---- last layer: dWlast[k] += sum_row dy*a_L[k][row]; dblast += sum dy; delta_L in place
    {
      const int KL = p.pk.dims[L];
      float* aL = actb[L];
      const float* wl = p.pk.wlast;
      for (int k = t; k < NP; k += kUThreads) {
        float s = 0.f;
        const float wk = __ldg(wl + k);
        float* col = aL + (size_t)k * kLDR;
        for (int row = 0; row < kTileM; ++row) {
          const float a = col[row], g = dy[row];
          s = fmaf(g, a, s);
          col[row] = (a > 0.f) ? g * wk : 0.f;
        }
        if (k < KL) atomicAdd(p.dW[L] + k, s);
      }
      if (t == 0) {
        float s = 0.f;
        for (int row = 0; row < kTileM; ++row) s += dy[row];
        atomicAdd(p.db[L], s);
      }
    }
    __syncthreads();
    // ---- hidden layers, top down: wgrad, bias grad, then dgrad (in place over the layer input)
    for (int l = L - 1; l >= 0; --l) {
      const int Nn = p.pk.dims[l + 1], Kk = p.pk.dims[l];
      const float* dlt = actb[l + 1];
      // bias
      for (int n = t; n < Nn; n += kUThreads) {
        float s = 0.f;
        const float* col = dlt + (size_t)n * kLDR;
        for (int row = 0; row < kTileM; ++row) s += col[row];
        atomicAdd(p.db[l] + n, s);
      }
      if (l > 0) {
        tile_wgrad<CH, TN>(dlt, actb[l], p.dW[l], Nn, Kk, Kk, TN);
        __syncthreads();
        float acc[4][TN];
        tile_gemm<TN>(acc, dlt, p.pk.Wn[l], round16(Nn) / kKC, wp);
        float* ain = actb[l];
#pragma unroll
        for (int j = 0; j < TN; ++j) {
          float4* ptr = reinterpret_cast<float4*>(ain + (size_t)(tx + 16 * j) * kLDR + 4 * ty);
          const float4 a = *ptr;
          float4 o;
          o.x = a.x > 0.f ? acc[0][j] : 0.f;
          o.y = a.y > 0.f ? acc[1][j] : 0.f;
          o.z = a.z > 0.f ? acc[2][j] : 0.f;
          o.w = a.w > 0.f ? acc[3][j] : 0.f;
          *ptr = o;
        }
        __syncthreads();
      } else {
        // first layer: the 1+E input columns are handled in blocks of 32 (TK = 2 groups of 16)
        for (int c0 = 0; c0 < KP0; c0 += 32) tile_wgrad<CH, 2>(dlt, actb[0] + (size_t)c0 * kLDR, p.dW[0] + c0, Nn, Kk - c0, Kk, TN);
        __syncthreads();
        for (int c0 = 0; c0 < KP0; c0 += 32) {
          float acc2[4][2];
          tile_gemm<2>(acc2, dlt, p.pk.Wn[0] + (size_t)(c0 / 32) * NP * 32, round16(Nn) / kKC, wp);
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            float4 o;
            o.x = acc2[0][j]; o.y = acc2[1][j]; o.z = acc2[2][j]; o.w = acc2[3][j];
            *reinterpret_cast<float4*>(actb[0] + (size_t)(c0 + tx + 16 * j) * kLDR + 4 * ty) = o;
          }
        }
        __syncthreads();
      }
    }
    // ---- input cotangents: dh (segment sums over the node-rows of one r), dx (Leibniz + chain on the extra node)
    {
      const float* din = actb[0];
      for (int idx = t; idx < (p.E + 1) * kTileM; idx += kUThreads) {
        const int row = idx & 63, k = idx >> 6;
        const long long q = q0 + row;
        if (q >= p.Q) continue;
        const int r = (int)(q / nodes), kn = (int)(q % nodes);
        if (k == 0) {
          if (kn == nodes - 1) atomicAdd(p.dx + r, din[row]);
          if (kn == 0) {
            const int b = r / p.d, i = r % p.d;
            float gzt = p.gz ? __ldg(p.gz + r) : 0.f;
            if (p.gzrev) gzt += __ldg(p.gzrev + (size_t)b * p.d + (p.d - 1 - i));
            atomicAdd(p.dx + r, __ldg(p.jac + r) * gzt);
            atomicAdd(p.dh + (size_t)r * p.E, gzt);  // z = integral + h[...,0]
          }
        } else if (kn == 0 || row == 0) {
          int rem = nodes - kn;
          if (rem > 64 - row) rem = 64 - row;
          if ((long long)rem > p.Q - q) rem = (int)(p.Q - q);
          float s = 0.f;
          const float* col = din + (size_t)k * kLDR + row;
          for (int i = 0; i < rem; ++i) s += col[i];
          atomicAdd(p.dh + (size_t)r * p.E + (k - 1), s);
        }
      }
    }
    __syncthreads();
  }
}

static size_t fwd_smem_bytes(int NP) { return fwd_smem_bytes_for(NP); }
static size_t bwd_smem_bytes(int NP, int KP0, int L) { return ((size_t)KP0 * kLDR + (size_t)L * NP * kLDR + 2 * kKC * NP + 256 + 128) * sizeof(float); }
// The backward keeps every hidden layer's tile in shared memory: deep or wide integrands (e.g. [256, 256, 256]) do not fit.
static int bwd_smem_check(int NP, int KB0, int L) {
  const size_t smem = bwd_smem_bytes(NP, KB0, L);
  if (smem > 227 * 1024) return fail(GNF_ERR_UNSUPPORTED, "umnn bwd: %d hidden layers of padded width %d need %zu B of shared memory (> 227 KB)", L, NP, smem);
  return 0;
}

template <int TN>
static int launch_fwd(const UmnnFwdParams& p, cudaStream_t s) {
  const size_t smem = fwd_smem_bytes(16 * TN);
  if (smem > 227 * 1024) return fail(GNF_ERR_UNSUPPORTED, "umnn fwd: shared memory %zu B exceeds 227 KB", smem);
#ifndef GNF_EMU
  cudaFuncSetAttribute(umnn_fwd_kernel<TN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
  const long long ntiles = (p.Q + kTileM - 1) / kTileM;
  const int per_sm = (int)((227 * 1024) / (smem + 1024));
  long long grid = (long long)kNumSMs * (per_sm < 1 ? 1 : (per_sm > 2 ? 2 : per_sm));
  if (grid > ntiles) grid = ntiles;
  GNF_LAUNCH(umnn_fwd_kernel<TN>, (unsigned)grid, kUThreads, smem, s, p);
  return 0;
}
template <int TN>
static int launch_bwd(const UmnnBwdParams& p, cudaStream_t s) {
  if (int e = bwd_smem_check(16 * TN, p.pk.kb0, p.pk.L)) return e;
  const size_t smem = bwd_smem_bytes(16 * TN, p.pk.kb0, p.pk.L);
#ifndef GNF_EMU
  cudaFuncSetAttribute(umnn_bwd_kernel<TN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
  const long long ntiles = (p.Q + kTileM - 1) / kTileM;
  long long grid = kNumSMs;
  if (grid > ntiles) grid = ntiles;
  GNF_LAUNCH(umnn_bwd_kernel<TN>, (unsigned)grid, kUThreads, smem, s, p);
  return 0;
}

}  // namespace gnf

using namespace gnf;

extern "C" {

size_t gnf_umnn_workspace_bytes(const gnf_mlp_t* net) {
  PackPlan pl;
  int TN;
  if (make_plan(net, &pl, &TN)) return 0;
  return pl.total * sizeof(float);
}

size_t gnf_umnn_bwd_workspace_bytes(const gnf_mlp_t* net) {
  PackPlan pl;
  int TN;
  if (make_plan(net, &pl, &TN)) return 0;
  if (bwd_smem_check(pl.NP, pl.KB0, net->n_layers - 1)) return 0;
  return pl.total * sizeof(float);
}

size_t gnf_umnn_saved_floats_per_node_row(const gnf_mlp_t* net) {
  PackPlan pl;
  int TN;
  if (make_plan(net, &pl, &TN)) return 0;
  return (size_t)(net->n_layers - 1) * pl.NP;
}

int gnf_umnn_fwd(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn, float* z,
                 float* zrev, float* jac, float* logdet, float* saved, int R, int d, void* work, size_t work_bytes,
                 gnf_stream_t stream) {
  if (!x || !h || !net || !ccw || !ccn || !z || !jac || R < 0 || d <= 0 || S < 1 || (R % d) != 0) return fail(GNF_ERR_INVALID, "gnf_umnn_fwd: bad arguments");
  PackPlan pl;
  int TN;
  if (int e = make_plan(net, &pl, &TN)) return e;
  if (!work || work_bytes < pl.total * sizeof(float)) return fail(GNF_ERR_WORKSPACE, "gnf_umnn_fwd: workspace too small (%zu < %zu)", work_bytes, pl.total * sizeof(float));
  cudaStream_t s = (cudaStream_t)stream;
  if (R == 0) return 0;
  launch_pack(net, pl, (float*)work, s);
  cudaMemsetAsync(z, 0, (size_t)R * sizeof(float), s);
  if (zrev) cudaMemsetAsync(zrev, 0, (size_t)R * sizeof(float), s);
  if (logdet) cudaMemsetAsync(logdet, 0, (size_t)(R / d) * sizeof(float), s);
  UmnnFwdParams p;
  p.x = x; p.h = h; p.ccw = ccw; p.ccn = ccn; p.z = z; p.zrev = zrev; p.jac = jac; p.logdet = logdet; p.saved = saved;
  p.R = R; p.d = d; p.E = net->dims[0] - 1; p.S = S; p.Q = (long long)R * (S + 1);
  fill_packed(net, pl, (float*)work, &p.pk);
  int e = 0;
  switch (TN) {
    case 2: e = launch_fwd<2>(p, s); break;
    case 4: e = launch_fwd<4>(p, s); break;
    case 7: e = launch_fwd<7>(p, s); break;
    case 10: e = launch_fwd<10>(p, s); break;
    case 13: e = launch_fwd<13>(p, s); break;
    default: e = launch_fwd<16>(p, s); break;
  }
  if (e) return e;
  return check_launch("gnf_umnn_fwd");
}

int gnf_umnn_invert(const float* z, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn, float* x, int iters,
                    float lo, float hi, int R, void* work, size_t work_bytes, gnf_stream_t stream) {
  if (!z || !h || !net || !ccw || !ccn || !x || R < 0 || S < 1 || iters < 0) return fail(GNF_ERR_INVALID, "gnf_umnn_invert: bad arguments");
  if (S + 1 > kTileM) return fail(GNF_ERR_UNSUPPORTED, "gnf_umnn_invert: %d quadrature nodes do not fit one %d-row tile", S + 1, kTileM);
  PackPlan pl;
  int TN;
  if (int e = make_plan(net, &pl, &TN)) return e;
  if (!work || work_bytes < pl.total * sizeof(float)) return fail(GNF_ERR_WORKSPACE, "gnf_umnn_invert: workspace too small (%zu < %zu)", work_bytes, pl.total * sizeof(float));
  cudaStream_t s = (cudaStream_t)stream;
  if (R == 0) return 0;
  launch_pack(net, pl, (float*)work, s);
  UmnnInvParams p;
  p.z = z; p.h = h; p.ccw = ccw; p.ccn = ccn; p.x = x; p.R = R; p.E = net->dims[0] - 1; p.S = S; p.iters = iters; p.lo = lo; p.hi = hi;
  fill_packed(net, pl, (float*)work, &p.pk);
  int e = 0;
  switch (TN) {
    case 2: e = launch_invert<2>(p, s); break;
    case 4: e = launch_invert<4>(p, s); break;
    case 7: e = launch_invert<7>(p, s); break;
    case 10: e = launch_invert<10>(p, s); break;
    case 13: e = launch_invert<13>(p, s); break;
    default: e = launch_invert<16>(p, s); break;
  }
  if (e) return e;
  return check_launch("gnf_umnn_invert");
}

int gnf_umnn_bwd(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn,
                 const float* jac, const float* gz, const float* gzrev, const float* gjac, const float* glogdet,
                 const float* saved, float* dx, float* dh, const gnf_mlp_grad_t* grads, int R, int d, void* work,
                 size_t work_bytes, gnf_stream_t stream) {
  if (!x || !h || !net || !ccw || !ccn || !jac || !dx || !dh || !grads || R < 0 || d <= 0 || S < 1 || (R % d) != 0) return fail(GNF_ERR_INVALID, "gnf_umnn_bwd: bad arguments");
  PackPlan pl;
  int TN;
  if (int e = make_plan(net, &pl, &TN)) return e;
  if (!work || work_bytes < pl.total * sizeof(float)) return fail(GNF_ERR_WORKSPACE, "gnf_umnn_bwd: workspace too small");
  cudaStream_t s = (cudaStream_t)stream;
  const int E = net->dims[0] - 1;
  for (int l = 0; l < net->n_layers; ++l) {
    if (!grads->dW[l] || !grads->db[l]) return fail(GNF_ERR_INVALID, "gnf_umnn_bwd: gradient pointer %d is NULL", l);
    cudaMemsetAsync(grads->dW[l], 0, (size_t)net->dims[l] * net->dims[l + 1] * sizeof(float), s);
    cudaMemsetAsync(grads->db[l], 0, (size_t)net->dims[l + 1] * sizeof(float), s);
  }
  if (R == 0) return check_launch("gnf_umnn_bwd");
  cudaMemsetAsync(dx, 0, (size_t)R * sizeof(float), s);
  cudaMemsetAsync(dh, 0, (size_t)R * E * sizeof(float), s);
  launch_pack(net, pl, (float*)work, s);
  UmnnBwdParams p;
  p.x = x; p.h = h; p.ccw = ccw; p.ccn = ccn; p.jac = jac; p.gz = gz; p.gzrev = gzrev; p.gjac = gjac; p.glogdet = glogdet;
  p.dx = dx; p.dh = dh; p.saved = saved;
  for (int l = 0; l < GNF_MAX_LAYERS; ++l) { p.dW[l] = grads->dW[l]; p.db[l] = grads->db[l]; }
  p.R = R; p.d = d; p.E = E; p.S = S; p.Q = (long long)R * (S + 2);
  fill_packed(net, pl, (float*)work, &p.pk);
  int e = 0;
  switch (TN) {
    case 2: e = launch_bwd<2>(p, s); break;
    case 4: e = launch_bwd<4>(p, s); break;
    case 7: e = launch_bwd<7>(p, s); break;
    case 10: e = launch_bwd<10>(p, s); break;
    case 13: e = launch_bwd<13>(p, s); break;
    default: e = launch_bwd<16>(p, s); break;
  }
  if (e) return e;
  return check_launch("gnf_umnn_bwd");
}

}  // extern "C"
