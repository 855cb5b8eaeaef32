// K4: AffineNormalizer + log-det + base density (HBM-bound elementwise + per-row warp reductions),
// and the small elementwise helpers of the host side.  One warp per sample row, lanes stride the
// feature axis so every global access is coalesced; row sums by shuffle reduction.
#include "common.cuh"

namespace gnf {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr int kRowsPerBlock = 8;  // 8 warps = 256 threads

__global__ void __launch_bounds__(256) affine_fwd_kernel(const float* __restrict__ x, float* __restrict__ h, int H, float* __restrict__ z,
                                                          float* __restrict__ zrev, float* __restrict__ jac, float* __restrict__ logdet,
                                                          uint8_t* __restrict__ cmask, int B, int d) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int b = blockIdx.x * kRowsPerBlock + warp; b < B; b += gridDim.x * kRowsPerBlock) {
    float acc = 0.f;
    for (int i = lane; i < d; i += 32) {
      const size_t e = (size_t)b * d + i;
      float* hp = h + e * H;
      const float h0 = hp[0], h1 = hp[1];
      const float mu = fminf(fmaxf(h0, -5.f), 5.f);
      const float ls = fminf(fmaxf(h1, -5.f), 2.f);
      hp[0] = mu;  // clamp_ is in place on h (AffineNormalizer.py:10)
      hp[1] = ls;
      const float sg = expf(ls);
      const float zv = fmaf(x[e], sg, mu);
      z[e] = zv;
      if (zrev) zrev[(size_t)b * d + (d - 1 - i)] = zv;
      if (jac) jac[e] = sg;
      if (cmask) cmask[e] = (uint8_t)((h0 >= -5.f && h0 <= 5.f ? 1 : 0) | (h1 >= -5.f && h1 <= 2.f ? 2 : 0));
      acc += ls;
    }
    acc = warp_sum(acc);
    if (lane == 0 && logdet) logdet[b] = acc;
  }
}

__global__ void __launch_bounds__(256) affine_bwd_kernel(const float* __restrict__ x, const float* __restrict__ h, int H,
                                                          const uint8_t* __restrict__ cmask, const float* __restrict__ gz,
                                                          const float* __restrict__ gzrev, const float* __restrict__ gjac,
                                                          const float* __restrict__ glogdet, float* __restrict__ gx, float* __restrict__ gh,
                                                          int B, int d) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int b = blockIdx.x * kRowsPerBlock + warp; b < B; b += gridDim.x * kRowsPerBlock) {
    const float gl = glogdet ? glogdet[b] : 0.f;
    const int n = d * H;
    for (int idx = lane; idx < n; idx += 32) {
      const int i = idx / H, k = idx % H;
      const size_t e = (size_t)b * d + i;
      float out = 0.f;
      if (k < 2) {
        float g = gz ? gz[e] : 0.f;
        if (gzrev) g += gzrev[(size_t)b * d + (d - 1 - i)];
        const uint8_t m = cmask[e];
        if (k == 0) {
          out = (m & 1) ? g : 0.f;
          const float sg = expf(h[e * H + 1]);
          gx[e] = g * sg;
        } else {
          const float sg = expf(h[e * H + 1]);
          float t = g * x[e] * sg + gl;
          if (gjac) t += gjac[e] * sg;
          out = (m & 2) ? t : 0.f;
        }
      }
      gh[e * H + k] = out;
    }
  }
}

__global__ void __launch_bounds__(256) normal_ll_fwd_kernel(const float* __restrict__ z, const float* __restrict__ logdet, float* __restrict__ out, int B, int d) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float log2pi = 1.8378770664093453f;
  for (int b = blockIdx.x * kRowsPerBlock + warp; b < B; b += gridDim.x * kRowsPerBlock) {
    float acc = 0.f;
    for (int i = lane; i < d; i += 32) {
      const float v = z[(size_t)b * d + i];
      acc += log2pi + v * v;
    }
    acc = warp_sum(acc);
    if (lane == 0) out[b] = (logdet ? logdet[b] : 0.f) + (-.5f) * acc;
  }
}

__global__ void normal_ll_bwd_kernel(const float* __restrict__ z, const float* __restrict__ gout, float* __restrict__ gz, int B, int d) {
  const size_t n = (size_t)B * d;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) gz[i] = -z[i] * gout[i / d];
}

// Training loss in one launch (NormalizingFlow.py:144-146 + NormalizingFlowFactories.py:15-16): out = constraint - mean_b(ll_b),
// ll_b = logdet_b - 0.5 sum_i (log 2pi + z_bi^2).  Every block writes the sum of its rows to work[block]; the last block to finish
// (a self-resetting counter behind the partial sums) adds them in block order: deterministic, no memset, graph-replayable.
__global__ void __launch_bounds__(256) nll_loss_fwd_kernel(const float* __restrict__ z, const float* __restrict__ logdet, const float* __restrict__ constraint,
                                                           float* __restrict__ out, float* __restrict__ work, int B, int d) {
  GNF_SMEM(float, s_part);                    // kRowsPerBlock partial sums + the "last block" flag
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float log2pi = 1.8378770664093453f;
  float rows = 0.f;
  for (int b = blockIdx.x * kRowsPerBlock + warp; b < B; b += gridDim.x * kRowsPerBlock) {
    float acc = 0.f;
    for (int i = lane; i < d; i += 32) {
      const float v = z[(size_t)b * d + i];
      acc += log2pi + v * v;
    }
    acc = warp_sum(acc);
    rows += (logdet ? logdet[b] : 0.f) + (-.5f) * acc;
  }
  if (lane == 0) s_part[warp] = rows;
  __syncthreads();
  unsigned* counter = reinterpret_cast<unsigned*>(work + gridDim.x);
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < kRowsPerBlock; ++w) t += s_part[w];
    work[blockIdx.x] = t;
    __threadfence();
    s_part[kRowsPerBlock] = atomicAdd(counter, 1u) == gridDim.x - 1 ? 1.f : 0.f;
  }
  __syncthreads();
  if (threadIdx.x == 0 && s_part[kRowsPerBlock] != 0.f) {
    __threadfence();
    float t = 0.f;
    for (unsigned k = 0; k < gridDim.x; ++k) t += reinterpret_cast<volatile float*>(work)[k];
    *out = (constraint ? *constraint : 0.f) - t / (float)B;
    *counter = 0u;
  }
}

// gz[b,i] = z[b,i] * g / B, glogdet[b] = -g / B  (g = the loss cotangent, a device scalar; NULL = 1)
__global__ void nll_loss_bwd_kernel(const float* __restrict__ z, const float* __restrict__ g, float* __restrict__ gz, float* __restrict__ glogdet, int B, int d) {
  const float s = (g ? *g : 1.f) / (float)B;
  const size_t n = (size_t)B * d;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) gz[i] = z[i] * s;
  if (glogdet)
    for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < (size_t)B; b += (size_t)gridDim.x * blockDim.x) glogdet[b] = -s;
}

__global__ void reverse_cols_kernel(const float* __restrict__ src, float* __restrict__ dst, int B, int d) {
  const size_t n = (size_t)B * d;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i / d;
    const int c = (int)(i % d);
    dst[b * d + (d - 1 - c)] = src[i];
  }
}

__global__ void broadcast_rows_kernel(const float* __restrict__ c, float* __restrict__ h, int B, int d, int indep, int H) {
  const size_t per = (size_t)indep * H, n = (size_t)B * per;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i / per, r = i % per;
    h[b * (size_t)d * H + r] = c[r];
  }
}

__global__ void counter_add_kernel(unsigned long long* c, unsigned long long inc) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *c += inc;
}

static inline int row_blocks(int B) {
  int b = ceil_div(B, kRowsPerBlock);
  if (b > 16 * kNumSMs) b = 16 * kNumSMs;
  return b < 1 ? 1 : b;
}
static inline int flat_blocks(size_t n) {
  size_t b = (n + 255) / 256;
  if (b > (size_t)16 * kNumSMs) b = (size_t)16 * kNumSMs;
  return b < 1 ? 1 : (int)b;
}

// DAGConditioner.loss (DAGConditioner.py:268-271) in one launch:
//   out = dag_const * (lambd * t + c / 2 * t^2) + l1_weight * mean(|A|)        (t = power trace, all scalars on the device)
// evaluated in fp32 in the reference's order, so that t^2 overflows to inf exactly where the reference does (SURVEY Q16).
__global__ void dag_loss_fwd_kernel(const float* __restrict__ A, int n, const float* __restrict__ t, const float* __restrict__ lambd,
                                    const float* __restrict__ c, const float* __restrict__ dag_const, const float* __restrict__ l1w,
                                    float* __restrict__ out) {
  GNF_SMEM(float, red);
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += fabsf(A[i]);
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = blockDim.x / 2; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float tv = *t;
    *out = *dag_const * (*lambd * tv + *c / 2.f * (tv * tv)) + *l1w * (red[0] / (float)n);
  }
}

// dA[i] = g * l1_weight * sign(A[i]) / n;  dt = g * dag_const * (lambd + c * t)
__global__ void dag_loss_bwd_kernel(const float* __restrict__ A, int n, const float* __restrict__ t, const float* __restrict__ lambd,
                                    const float* __restrict__ c, const float* __restrict__ dag_const, const float* __restrict__ l1w,
                                    const float* __restrict__ g, float* __restrict__ dA, float* __restrict__ dt) {
  const float gv = *g;
  const float k = gv * *l1w / (float)n;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float a = A[i];
    dA[i] = a > 0.f ? k : (a < 0.f ? -k : 0.f);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) *dt = gv * *dag_const * (*lambd + *c * *t);
}

__global__ void __launch_bounds__(256) zero_many_kernel(ZeroList z) {
  for (int k = 0; k < z.count; ++k) {
    float* __restrict__ p = z.p[k];
    const long long n = z.n[k];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = 0.f;
  }
}

void zero_many(const ZeroList& z, cudaStream_t s) {
  if (z.count == 0) return;
  long long most = 0;
  for (int k = 0; k < z.count; ++k) most = z.n[k] > most ? z.n[k] : most;
  long long blocks = (most + 255) / 256;
  if (blocks > 4 * kNumSMs) blocks = 4 * kNumSMs;
  GNF_LAUNCH(zero_many_kernel, (int)blocks, 256, 0, s, z);
}

}  // namespace gnf

using namespace gnf;

extern "C" {

int gnf_affine_fwd(const float* x, float* h, int H, float* z, float* zrev, float* jac, float* logdet, uint8_t* clampmask,
                   int B, int d, gnf_stream_t stream) {
  if (!x || !h || !z || B < 0 || d <= 0 || H < 2) return fail(GNF_ERR_INVALID, "gnf_affine_fwd: bad arguments (need H >= 2)");
  if (B == 0) return 0;
  GNF_LAUNCH(affine_fwd_kernel, row_blocks(B), 256, 0, (cudaStream_t)stream, x, h, H, z, zrev, jac, logdet, clampmask, B, d);
  return check_launch("gnf_affine_fwd");
}

int gnf_affine_bwd(const float* x, const float* h, int H, const uint8_t* clampmask, const float* gz, const float* gzrev,
                   const float* gjac, const float* glogdet, float* gx, float* gh, int B, int d, gnf_stream_t stream) {
  if (!x || !h || !clampmask || !gx || !gh || B < 0 || d <= 0 || H < 2) return fail(GNF_ERR_INVALID, "gnf_affine_bwd: bad arguments");
  if (B == 0) return 0;
  GNF_LAUNCH(affine_bwd_kernel, row_blocks(B), 256, 0, (cudaStream_t)stream, x, h, H, clampmask, gz, gzrev, gjac, glogdet, gx, gh, B, d);
  return check_launch("gnf_affine_bwd");
}

int gnf_normal_ll_fwd(const float* z, const float* logdet, float* out, int B, int d, gnf_stream_t stream) {
  if (!z || !out || B < 0 || d <= 0) return fail(GNF_ERR_INVALID, "gnf_normal_ll_fwd: bad arguments");
  if (B == 0) return 0;
  GNF_LAUNCH(normal_ll_fwd_kernel, row_blocks(B), 256, 0, (cudaStream_t)stream, z, logdet, out, B, d);
  return check_launch("gnf_normal_ll_fwd");
}

int gnf_normal_ll_bwd(const float* z, const float* gout, float* gz, int B, int d, gnf_stream_t stream) {
  if (!z || !gout || !gz || B < 0 || d <= 0) return fail(GNF_ERR_INVALID, "gnf_normal_ll_bwd: bad arguments");
  if (B == 0) return 0;
  GNF_LAUNCH(normal_ll_bwd_kernel, flat_blocks((size_t)B * d), 256, 0, (cudaStream_t)stream, z, gout, gz, B, d);
  return check_launch("gnf_normal_ll_bwd");
}

size_t gnf_nll_loss_work_floats(int B) { return (size_t)(B > 0 ? row_blocks(B) : 1) + 1; }

int gnf_nll_loss_fwd(const float* z, const float* logdet, const float* constraint, float* out, float* work, int B, int d, gnf_stream_t stream) {
  if (!z || !out || !work || B <= 0 || d <= 0) return fail(GNF_ERR_INVALID, "gnf_nll_loss_fwd: bad arguments (B >= 1; work = gnf_nll_loss_work_floats(B) floats whose last word is zero)");
  GNF_LAUNCH(nll_loss_fwd_kernel, row_blocks(B), 256, (kRowsPerBlock + 1) * sizeof(float), (cudaStream_t)stream, z, logdet, constraint, out, work, B, d);
  return check_launch("gnf_nll_loss_fwd");
}

int gnf_nll_loss_bwd(const float* z, const float* g, float* gz, float* glogdet, int B, int d, gnf_stream_t stream) {
  if (!z || !gz || B <= 0 || d <= 0) return fail(GNF_ERR_INVALID, "gnf_nll_loss_bwd: bad arguments");
  GNF_LAUNCH(nll_loss_bwd_kernel, flat_blocks((size_t)B * d), 256, 0, (cudaStream_t)stream, z, g, gz, glogdet, B, d);
  return check_launch("gnf_nll_loss_bwd");
}

int gnf_reverse_cols(const float* src, float* dst, int B, int d, gnf_stream_t stream) {
  if (!src || !dst || B < 0 || d <= 0) return fail(GNF_ERR_INVALID, "gnf_reverse_cols: bad arguments");
  if (B == 0) return 0;
  GNF_LAUNCH(reverse_cols_kernel, flat_blocks((size_t)B * d), 256, 0, (cudaStream_t)stream, src, dst, B, d);
  return check_launch("gnf_reverse_cols");
}

int gnf_broadcast_rows(const float* constants, float* h, int B, int d, int indep, int H, gnf_stream_t stream) {
  if (!constants || !h || B < 0 || d <= 0 || indep < 0 || indep > d || H <= 0) return fail(GNF_ERR_INVALID, "gnf_broadcast_rows: bad arguments");
  if (B == 0 || indep == 0) return 0;
  GNF_LAUNCH(broadcast_rows_kernel, flat_blocks((size_t)B * indep * H), 256, 0, (cudaStream_t)stream, constants, h, B, d, indep, H);
  return check_launch("gnf_broadcast_rows");
}

int gnf_counter_add(uint64_t* counter, uint64_t inc, gnf_stream_t stream) {
  if (!counter) return fail(GNF_ERR_INVALID, "gnf_counter_add: bad arguments");
  GNF_LAUNCH(counter_add_kernel, 1, 32, 0, (cudaStream_t)stream, reinterpret_cast<unsigned long long*>(counter), (unsigned long long)inc);
  return check_launch("gnf_counter_add");
}

int gnf_dag_loss_fwd(const float* A, int d, const float* t, const float* lambd, const float* c, const float* dag_const,
                     const float* l1_weight, float* out, gnf_stream_t stream) {
  if (!A || !t || !lambd || !c || !dag_const || !l1_weight || !out || d <= 0) return fail(GNF_ERR_INVALID, "gnf_dag_loss_fwd: bad arguments");
  const int threads = d * d >= 16384 ? 1024 : 256;       // one block: the reduction is over d^2 <= 6e5 elements
  GNF_LAUNCH(dag_loss_fwd_kernel, 1, threads, threads * sizeof(float), (cudaStream_t)stream, A, d * d, t, lambd, c, dag_const, l1_weight, out);
  return check_launch("gnf_dag_loss_fwd");
}

int gnf_dag_loss_bwd(const float* A, int d, const float* t, const float* lambd, const float* c, const float* dag_const,
                     const float* l1_weight, const float* gout, float* dA, float* dt, gnf_stream_t stream) {
  if (!A || !t || !lambd || !c || !dag_const || !l1_weight || !gout || !dA || !dt || d <= 0) return fail(GNF_ERR_INVALID, "gnf_dag_loss_bwd: bad arguments");
  GNF_LAUNCH(dag_loss_bwd_kernel, flat_blocks((size_t)d * d), 256, 0, (cudaStream_t)stream, A, d * d, t, lambd, c, dag_const, l1_weight, gout, dA, dt);
  return check_launch("gnf_dag_loss_bwd");
}

}  // extern "C"
