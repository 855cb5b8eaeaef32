// Weight gradient of a narrow layer over all node-rows, on tcgen05 / TMEM, for the layer-wise UMNN engine:
//     dW[n, k] = sum_q dY[q, n] * X[q, k],     n < N <= 160,  k < K <= 160,   q < Q = B*d*(S+2)  (10^5 .. 10^7)
// in 3xTF32 (fp32-equivalent) or single-pass TF32.  (IntegrandNet hidden layers, MonotonicNormalizer.py:12-38: the wgrad of
// UMNN's backward, SURVEY App. B.)
//
// The generic engine (gnf_linear_wgrad_tc) tiles the 150 output rows as 128 + 22, so half of its CTAs run a tile that is 83 %
// padding and the activation plane X is streamed twice; both operands go through the shared-memory hi/lo split.  Here:
//   * the reduction runs over q, and dY[q, :] is contiguous in n: with TMEM lane = output row n, a warp's 32 lanes read
//     dY[q, n0 .. n0+31] as one 128-byte line per q -- the A operand (dY^T) needs NO transposition at all.  Each loader
//     thread gathers 32 consecutive q of its own n, splits them into TF32 hi / lo in registers and stores them as 32 TMEM
//     columns (TS-form MMA: A from TMEM);
//   * rows 128..159 are a second accumulator fed by the first loader warp's lanes (the other lanes of that operand stay
//     zero), so X is streamed once for both;
//   * X chunks (32 q x NP, contiguous in global memory because the plane is dense) arrive by ONE bulk async copy each;
//     eight stager warps turn a landed chunk into the UMMA canonical K-major images [(q/4)][k][q%4] of hi and lo;
//   * every CTA owns a contiguous q range and writes its partial [160 x NP] tile (coalesced through a swizzled staging
//     block); a second kernel sums the partial tiles into dW -- deterministic, no atomics.
#include "tc_common.cuh"
#include "tc_rw.h"

#ifndef GNF_EMU
namespace gnf {

constexpr int kWgQC = 16;                 // reduction rows (q) per chunk: two 8-q MMA k-steps
constexpr int kWgThreads = 15 * 32;       // warps 0-3 loaders of rows 0..127 (+ epilogue), 4 loader of rows 128..159, 5-12 stagers, 13 issuer, 14 producer
constexpr int kWgRawStages = 6, kWgImgStages = 3;
constexpr int kWgDyStages = 6, kWgDyFloats = kWgQC * 160;   // dY chunks by bulk copy (dense planes): six in flight, no registers
constexpr int kWgColD0 = 0, kWgColD1 = 160, kWgColA = 320;   // A buffer b at 320 + 64 b: A0hi, A0lo, A1hi, A1lo (16 columns each)
constexpr int kWgPartRows = 160;

__device__ __forceinline__ uint32_t wg_rn_tf32(uint32_t u) { return (u + 0x1000u) & 0xffffe000u; }
__device__ __forceinline__ void wg_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ float wg_ldg(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// Measurement: role r of CTA 0 appends SM-clock stamps to row r of the trace buffer (256 stamps per role).
struct WgTrace {
  long long* buf; int n;
  __device__ __forceinline__ void stamp() { if (buf && n < 256) buf[n++] = clock64(); }
};
static long long* g_wg_trace = nullptr;

struct RwWgradParams {
  long long* trace;
  const float* dY; long long lddy;     // [Q][lddy], N columns used
  RwRankOne r1;                        // r1.g != NULL: dY is the masked rank-one product instead (dY unused)
  int bulk_dy;                         // dY rows are 16-byte aligned and at most 160 floats: its chunks arrive by bulk copies
  const float* X;                      // [Q][NP] dense (row stride NP), padding columns finite
  float* partial;                      // [gridDim.x][kWgPartRows][NP]
  int Q, N, chunks_per_cta, passes;
};

template <int NB>
__global__ void __launch_bounds__(kWgThreads, 1) rw_wgrad_kernel(RwWgradParams p) {
  using namespace tc;
  constexpr int NP = NB * 32;
  constexpr int kRawFloats = kWgQC * NP, kImgFloats = 2 * kWgQC * NP;      // one raw chunk; hi + lo images of one chunk
  GNF_SMEM(float, smem);
  float* raw = smem;                                                       // [kWgRawStages][16][NP]
  float* img = raw + kWgRawStages * kRawFloats;                            // [kWgImgStages][hi | lo][4][NP][4]
  uint64_t* bars = reinterpret_cast<uint64_t*>(img + kWgImgStages * kImgFloats);
  uint64_t* raw_full = bars;                        // bulk copy landed (transaction bytes)
  uint64_t* raw_empty = raw_full + kWgRawStages;    // stagers are done with the raw chunk (8 arrives)
  uint64_t* img_full = raw_empty + kWgRawStages;    // stagers -> issuer (8 arrives)
  uint64_t* img_empty = img_full + kWgImgStages;    // issuer -> stagers (tcgen05.commit)
  uint64_t* a_full = img_empty + kWgImgStages;      // [2] loaders -> issuer (one arrive per loader warp)
  uint64_t* a_empty = a_full + 2;                   // [2] issuer -> loaders (tcgen05.commit)
  uint64_t* d_full = a_empty + 2;                   // issuer -> epilogue (tcgen05.commit)
  uint64_t* dy_full = d_full + 1;                   // [kWgDyStages] dY chunk landed (transaction bytes)
  uint64_t* dy_empty = dy_full + kWgDyStages;       // [kWgDyStages] loaders have the chunk in registers (one arrive per loader warp)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dy_empty + kWgDyStages);
  float* dyraw = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 127) & ~(uintptr_t)127);   // [kWgDyStages][16][lddy], bulk-copy target
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  const int nchunks_all = (p.Q + kWgQC - 1) / kWgQC;
  const int c0 = blockIdx.x * p.chunks_per_cta;
  const int nloc = min(p.chunks_per_cta, nchunks_all - c0);                // >= 1 by construction of the grid
  const bool split = p.passes == 3;
  const bool two = p.N > 128;                                              // second accumulator: output rows 128..159

  if (warp == 0) tmem_alloc(tmem_slot, 512);
  if (tid == 32) {
    for (int s = 0; s < kWgRawStages; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], 8); }
    for (int s = 0; s < kWgImgStages; ++s) { mbar_init(&img_full[s], 8); mbar_init(&img_empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&a_full[b], two ? 5 : 4); mbar_init(&a_empty[b], 1); }
    mbar_init(d_full, 1);
    for (int s = 0; s < kWgDyStages; ++s) { mbar_init(&dy_full[s], 1); mbar_init(&dy_empty[s], two ? 5 : 4); }
    fence_mbar_init();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();

  if (warp == 14) {
    // ===================== bulk-copy producer =====================
    if (lane == 0) {
      for (int j = 0; j < nloc; ++j) {
        const int s = j % kWgRawStages;
        mbar_wait(&raw_empty[s], (uint32_t)(((j / kWgRawStages) & 1) ^ 1));
        const int q0 = (c0 + j) * kWgQC;
        const int rows = min(kWgQC, p.Q - q0);
        const uint32_t bytes = (uint32_t)rows * NP * 4u;
        mbar_expect_tx(&raw_full[s], bytes);
        bulk_g2s(raw + s * kRawFloats, p.X + (size_t)q0 * NP, bytes, &raw_full[s]);
        if (p.bulk_dy) {
          const int sd = j % kWgDyStages;
          mbar_wait(&dy_empty[sd], (uint32_t)(((j / kWgDyStages) & 1) ^ 1));
          const uint32_t dbytes = (uint32_t)rows * (uint32_t)p.lddy * 4u;
          mbar_expect_tx(&dy_full[sd], dbytes);
          bulk_g2s(dyraw + sd * kWgDyFloats, p.dY + (size_t)q0 * p.lddy, dbytes, &dy_full[sd]);
        }
      }
    }
  } else if (warp == 13) {
    // ===================== MMA issuer =====================
    {   // the whole warp runs the loop converged; one elected lane issues (tc_common.cuh: mma_*_w)
      const uint32_t idesc = make_idesc_tf32(128, NP);
      const uint64_t dstep = (uint64_t)((2u * NP * 16u) >> 4);             // one k-step (8 q) = two 16-byte q-quads of the image
      const uint32_t tD0 = tmem_base + kWgColD0, tD1 = tmem_base + kWgColD1;
      WgTrace tr = {(p.trace && blockIdx.x == 0 && lane == 0) ? p.trace : nullptr, 0};
      for (int j = 0; j < nloc; ++j) {
        const int i = j % kWgImgStages, b = j & 1;
        tr.stamp();                                                        // per chunk: start, A full, image full, issued
        mbar_wait(&a_full[b], (uint32_t)((j >> 1) & 1));
        tr.stamp();
        mbar_wait(&img_full[i], (uint32_t)((j / kWgImgStages) & 1));
        fence_after_sync();
        tr.stamp();
        const uint32_t ib = smem_u32(img + i * kImgFloats);
        const uint64_t bhi = make_smem_desc(ib, NP * 16u, 128u), blo = make_smem_desc(ib + kWgQC * NP * 4u, NP * 16u, 128u);
        const uint32_t tA = tmem_base + kWgColA + 64 * b;                  // A0hi +0, A0lo +16, A1hi +32, A1lo +48
#pragma unroll
        for (int ks = 0; ks < kWgQC / 8; ++ks) {
          const uint32_t acc = (j > 0 || ks > 0) ? 1u : 0u;
          if (split) {
            mma_tf32_ts_w(tD0, tA + 16 + ks * 8, bhi + dstep * ks, idesc, acc);
            mma_tf32_ts_w(tD0, tA + 0 + ks * 8, blo + dstep * ks, idesc, 1u);
            mma_tf32_ts_w(tD0, tA + 0 + ks * 8, bhi + dstep * ks, idesc, 1u);
            if (two) {
              mma_tf32_ts_w(tD1, tA + 48 + ks * 8, bhi + dstep * ks, idesc, acc);
              mma_tf32_ts_w(tD1, tA + 32 + ks * 8, blo + dstep * ks, idesc, 1u);
              mma_tf32_ts_w(tD1, tA + 32 + ks * 8, bhi + dstep * ks, idesc, 1u);
            }
          } else {
            mma_tf32_ts_w(tD0, tA + 0 + ks * 8, bhi + dstep * ks, idesc, acc);
            if (two) mma_tf32_ts_w(tD1, tA + 32 + ks * 8, bhi + dstep * ks, idesc, acc);
          }
        }
        mma_commit_w(&a_empty[b]);
        mma_commit_w(&img_empty[i]);
        tr.stamp();
      }
      mma_commit_w(d_full);
    }
  } else if (warp >= 5) {
    // ===================== stagers: raw [16 q][NP] -> canonical K-major images [(q/4)][k][q%4] of hi and lo =====================
    const int st = tid - 5 * 32;                                           // 0..255
    WgTrace tr = {(p.trace && blockIdx.x == 0 && st == 0) ? p.trace + 256 : nullptr, 0};
    for (int j = 0; j < nloc; ++j) {
      const int s = j % kWgRawStages, i = j % kWgImgStages;
      const int rows = min(kWgQC, p.Q - (c0 + j) * kWgQC);
      tr.stamp();                                                          // per chunk: start, raw landed, image free, published
      mbar_wait(&raw_full[s], (uint32_t)((j / kWgRawStages) & 1));
      tr.stamp();
      mbar_wait(&img_empty[i], (uint32_t)(((j / kWgImgStages) & 1) ^ 1));
      tr.stamp();
      const float* rw = raw + s * kRawFloats;
      float* ihi = img + i * kImgFloats;
      float* ilo = ihi + kWgQC * NP;
      constexpr int kItems = (kWgQC / 4) * NP;
#pragma unroll
      for (int it = 0; it < (kItems + 255) / 256; ++it) {
        const int item = st + it * 256;
        if (item < kItems) {
          const int qq = item / NP, k = item - qq * NP;
          float hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float v = (4 * qq + e < rows) ? rw[(4 * qq + e) * NP + k] : 0.f;   // rows past Q were not copied
            hi[e] = __uint_as_float(wg_rn_tf32(__float_as_uint(v)));
            lo[e] = __uint_as_float(wg_rn_tf32(__float_as_uint(v - hi[e])));
          }
          *reinterpret_cast<float4*>(ihi + (size_t)item * 4) = make_float4(hi[0], hi[1], hi[2], hi[3]);
          if (split) *reinterpret_cast<float4*>(ilo + (size_t)item * 4) = make_float4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // generic-proxy writes -> visible to the tensor core
      __syncwarp();
      if (lane == 0) { wg_mbar_arrive(&img_full[i]); wg_mbar_arrive(&raw_empty[s]); }
      tr.stamp();
    }
  } else {
    // ===================== loaders (TMEM lane = output row n), then epilogue =====================
    // warps 0-3: rows n = 32 warp + lane of the first accumulator; warp 4 (TMEM lanes 0-31 as well): rows 128 + lane of the second
    const int tile = warp == 4 ? 1 : 0;
    const uint32_t lane_sel = (uint32_t)((warp & 3) * 32) << 16;
    const int n = tile ? 128 + lane : warp * 32 + lane;
    if (tile == 0 || two) {
    if (two && tile == 0 && warp != 0) {                                   // rows 160.. of the second operand do not exist: zeros
      uint32_t z[16];
#pragma unroll
      for (int c = 0; c < 16; ++c) z[c] = 0u;
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        tmem_st16p(tmem_base + lane_sel + kWgColA + 64 * b + 32, z);
        tmem_st16p(tmem_base + lane_sel + kWgColA + 64 * b + 48, z);
      }
      tmem_wait_st();
    }
    // Loads are unconditional (addresses clamped into the tensor) and masked when they are used: a conditional around an
    // asm load is a branch per load, and the loads of a chunk then took thousands of clocks to issue (scripts/wg_trace.py).
    float va[kWgQC], vb[kWgQC];                                            // two chunks in flight
    const int nc = n < p.N ? n : 0;
    const bool row_ok = n < p.N;
    // Rank-one mode (p.r1.g): dY[q][n] = g_q w_n where bit n of the row's ReLU mask is set.  g_q and the mask word of this warp's
    // 32 columns are warp-uniform: lanes 0-15 fetch g of the chunk's 16 node-rows, lanes 16-31 their mask words (ONE load per lane
    // and chunk, prefetched two chunks ahead like the plane loads), and the values are handed round by shuffles when the chunk is split.
    const bool r1 = p.r1.g != nullptr;
    const float w_n = r1 ? __ldg(p.r1.w + nc) : 0.f;
    const int wword = (tile ? 128 : warp * 32) >> 5;
    // The loaders are latency-bound (scripts/wg_trace.py: a cold dY load takes ~3.9 k clocks, two chunks of register prefetch covered
    // 2 x 1.6 k): dense dY planes now arrive by bulk copies, six chunks in flight and no registers; the rank-one words are prefetched
    // four chunks ahead (one register each); only dY with unaligned rows keeps the two-chunk register path.
    const bool bulk = p.bulk_dy != 0;
    const int dist = r1 ? 4 : 2;
    uint32_t r0 = 0u, r1w = 0u, r2 = 0u, r3 = 0u;
    auto load = [&](int j, float (&v)[kWgQC], uint32_t& raw) {
      if (bulk) return;
      const long long q0 = (long long)(c0 + (j < nloc ? j : 0)) * kWgQC;
      if (r1) {
        const long long qq = q0 + (lane & 15);
        const long long q = qq < p.Q ? qq : (long long)p.Q - 1;
        raw = lane < 16 ? __float_as_uint(__ldg(p.r1.g + q)) : __ldg(p.r1.bits + q * p.r1.bits_ld + wword);
        return;
      }
#pragma unroll
      for (int c = 0; c < kWgQC; ++c) {
        const long long q = (q0 + c < p.Q) ? q0 + c : (long long)p.Q - 1;
        v[c] = wg_ldg(p.dY + q * p.lddy + nc);
      }
    };
    WgTrace tr = {(p.trace && blockIdx.x == 0 && tid == 0) ? p.trace + 512 : nullptr, 0};
    auto step = [&](int j, float (&v)[kWgQC], uint32_t& raw) {
      const int b = j & 1;
      const long long q0 = (long long)(c0 + j) * kWgQC;
      tr.stamp();                                                          // per chunk: start, split + A free, handed over, next loads issued
      uint32_t hi[kWgQC], lo[kWgQC];
      if (bulk) {                                                          // column nc of the landed [16 q][lddy] chunk: conflict-free
        const int sd = j % kWgDyStages;
        mbar_wait(&dy_full[sd], (uint32_t)((j / kWgDyStages) & 1));
        const float* src = dyraw + sd * kWgDyFloats + nc;
#pragma unroll
        for (int c = 0; c < kWgQC; ++c) v[c] = src[c * (int)p.lddy];
        __syncwarp();
        if (lane == 0) wg_mbar_arrive(&dy_empty[sd]);
      } else if (r1) {                                                     // all 32 shuffles first (independent), then the selects
        uint32_t gs[kWgQC], ms[kWgQC];
#pragma unroll
        for (int c = 0; c < kWgQC; ++c) { gs[c] = __shfl_sync(0xffffffffu, raw, c); ms[c] = __shfl_sync(0xffffffffu, raw, 16 + c); }
#pragma unroll
        for (int c = 0; c < kWgQC; ++c) v[c] = ((ms[c] >> lane) & 1u) ? __uint_as_float(gs[c]) * w_n : 0.f;
      }
#pragma unroll
      for (int c = 0; c < kWgQC; ++c) {
        const float x = (row_ok && q0 + c < p.Q) ? v[c] : 0.f;
        const uint32_t h = wg_rn_tf32(__float_as_uint(x));
        hi[c] = h;
        lo[c] = wg_rn_tf32(__float_as_uint(x - __uint_as_float(h)));
      }
      load(j + dist, v, raw);                                              // this buffer's next chunk
      if (j >= 2) {                                                        // the MMAs of chunk j-2 must be done with this A buffer
        mbar_wait(&a_empty[b], (uint32_t)(((j >> 1) - 1) & 1));
        fence_after_sync();
      }
      tr.stamp();
      const uint32_t tA = tmem_base + lane_sel + kWgColA + 64 * b + 32 * tile;
      tmem_st16p(tA, hi);
      if (split) tmem_st16p(tA + 16, lo);
      tmem_wait_st();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) wg_mbar_arrive(&a_full[b]);
      tr.stamp();
    };
    load(0, va, r0);
    load(1, vb, r1w);
    if (r1) { load(2, va, r2); load(3, vb, r3); }
    for (int j = 0; j < nloc; j += 4) {
      step(j, va, r0);
      if (j + 1 < nloc) step(j + 1, vb, r1w);
      if (j + 2 < nloc) step(j + 2, va, r1 ? r2 : r0);
      if (j + 3 < nloc) step(j + 3, vb, r1 ? r3 : r1w);
    }
    // ---- epilogue: partial tile of this CTA, row-owner -> coalesced through a swizzled 32 x 32 block (the rings are idle now)
    mbar_wait(d_full, 0);
    fence_after_sync();
    float* stage = raw + warp * 1024;
    float* out = p.partial + (size_t)blockIdx.x * kWgPartRows * NP;
    const int sub = lane >> 3, piece = lane & 7;
    const uint32_t tD = tmem_base + lane_sel + (tile ? kWgColD1 : kWgColD0);
    const int rbase = tile ? 128 : warp * 32;
#pragma unroll 1
    for (int cb = 0; cb < NB; ++cb) {
      uint32_t acc[32];
      tmem_ld32p(tD + cb * 32, acc);
      tmem_wait_ld();
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4)
        *reinterpret_cast<uint4*>(stage + lane * 32 + 4 * (j4 ^ (lane & 7))) = make_uint4(acc[4 * j4], acc[4 * j4 + 1], acc[4 * j4 + 2], acc[4 * j4 + 3]);
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int R = 4 * i + sub;
        const uint4 q = *reinterpret_cast<const uint4*>(stage + R * 32 + 4 * (piece ^ (R & 7)));
        if (rbase + R < p.N) *reinterpret_cast<uint4*>(out + (size_t)(rbase + R) * NP + cb * 32 + 4 * piece) = q;
      }
      __syncwarp();
    }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// dW[n][k] = sum_b partial[b][n][k]: eight lanes per output element (each sums every eighth partial tile, two accumulators),
// combined by shuffles in a fixed order -- deterministic.  (One thread per element left 88 blocks walking 147 strided loads each:
// 28 us for 13 MB.)
__global__ void rw_wgrad_reduce_kernel(const float* __restrict__ partial, int nblk, int NP, float* __restrict__ dW, long long lddw, int N, int K) {
  const int total = N * K;
  const int sub = threadIdx.x & 7, grp = (threadIdx.x & 31) >> 3;
  const int stride = (gridDim.x * blockDim.x) >> 3;
  // warp-uniform trip count (the shuffles are warp-wide): `base` is the element of the warp's first 8-lane group
  for (int base = ((blockIdx.x * blockDim.x + threadIdx.x) >> 3) - grp; base < total; base += stride) {
    const int i = base + grp;
    const bool valid = i < total;
    const int n = valid ? i / K : 0, k = valid ? i - n * K : 0;
    const float* src = partial + (size_t)n * NP + k;
    float s0 = 0.f, s1 = 0.f;
    if (valid) {
      int b = sub;
      for (; b + 8 < nblk; b += 16) {
        s0 += src[(size_t)b * kWgPartRows * NP];
        s1 += src[(size_t)(b + 8) * kWgPartRows * NP];
      }
      if (b < nblk) s0 += src[(size_t)b * kWgPartRows * NP];
    }
    float s = s0 + s1;
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (valid && sub == 0) dW[(long long)n * lddw + k] = s;
  }
}

static size_t wg_smem_bytes(int NP) {
  size_t fl = (size_t)kWgRawStages * kWgQC * NP + (size_t)kWgImgStages * 2 * kWgQC * NP;
  if (fl < 5 * 1024) fl = 5 * 1024;                       // the epilogue's five 4 KB staging blocks reuse the rings
  return fl * sizeof(float) + (24 + 2 * kWgDyStages) * sizeof(uint64_t) + 16 + 128 + (size_t)kWgDyStages * kWgDyFloats * sizeof(float);
}

size_t rw_wgrad_partial_floats(int K) { return (size_t)kNumSMs * kWgPartRows * ((K + 31) / 32 * 32); }

bool rw_wgrad_supported(int N, int K) {
  const int NP = (K + 31) / 32 * 32;
  return N >= 1 && N <= kWgPartRows && K >= 1 && NP <= 160 && wg_smem_bytes(NP) <= 227 * 1024;
}

int launch_rw_wgrad(const float* dY, long long lddy, const float* X, long long ldx, float* dW, long long lddw, int Q, int N, int K, int passes,
                    float* partial, cudaStream_t s, const Branches* br, int side, const RwRankOne* rank_one) {
  if (passes != 1 && passes != 3) return fail(GNF_ERR_INVALID, "resident wgrad: passes must be 1 or 3");
  // The kernel multiplies all ldx columns of X: the activation planes of a mixed-width integrand share the row stride of its widest
  // layer, so a narrower layer's plane carries columns past round_up(K, 32); the reduction keeps the first K.  `partial` holds
  // rw_wgrad_partial_floats(ldx) floats.
  const int NP = (int)ldx;
  if (K < 1 || ldx % 32 != 0 || ldx < (K + 31) / 32 * 32 || !rw_wgrad_supported(N, NP) || lddy < N || (reinterpret_cast<uintptr_t>(X) & 15) ||
      (reinterpret_cast<uintptr_t>(partial) & 15))
    return fail(GNF_ERR_UNSUPPORTED, "resident wgrad: needs N <= 160, K <= 160 and a dense 16-byte aligned activation plane (ld = %lld, K = %d)", ldx, K);
  if (Q <= 0) { cudaMemset2DAsync(dW, (size_t)lddw * sizeof(float), 0, (size_t)K * sizeof(float), (size_t)N, s); return 0; }
  const int nchunks = (Q + kWgQC - 1) / kWgQC;
  const int cpc = (nchunks + kNumSMs - 1) / kNumSMs;
  const int grid = (nchunks + cpc - 1) / cpc;
  RwWgradParams p;
  p.trace = g_wg_trace;
  p.r1 = rank_one ? *rank_one : RwRankOne{nullptr, nullptr, nullptr, 0};
  p.bulk_dy = (!rank_one && (lddy % 4) == 0 && lddy <= 160 && (reinterpret_cast<uintptr_t>(dY) & 15) == 0) ? 1 : 0;
  p.dY = dY; p.lddy = lddy; p.X = X; p.partial = partial; p.Q = Q; p.N = N; p.chunks_per_cta = cpc; p.passes = passes;
  const size_t smem = wg_smem_bytes(NP);
#define WG_CASE(nb)                                                                                                      \
  case nb:                                                                                                               \
    cudaFuncSetAttribute(rw_wgrad_kernel<nb>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                   \
    GNF_LAUNCH_PDL(rw_wgrad_kernel<nb>, grid, kWgThreads, smem, s, p);                                                       \
    break;
  switch (NP / 32) { WG_CASE(1) WG_CASE(2) WG_CASE(3) WG_CASE(4) default: WG_CASE(5) }
#undef WG_CASE
  int rb = (N * K * 8 + 255) / 256;
  if (rb > 8 * kNumSMs) rb = 8 * kNumSMs;
  if (br) s = br->begin(s, side);       // the second stage as a branch: it overlaps whatever the caller enqueues next (the caller joins: br->end)
  GNF_LAUNCH(rw_wgrad_reduce_kernel, rb, 256, 0, s, partial, grid, NP, dW, lddw, N, K);
  return 0;
}

}  // namespace gnf
using namespace gnf;
#endif

extern "C" {

size_t gnf_linear_wgrad_rw_workspace_bytes(int N, int K) {
#ifdef GNF_EMU
  (void)N; (void)K;
  gnf::set_error("tensor-core kernels have no host-simulator flavour");
  return 0;
#else
  if (!rw_wgrad_supported(N, K)) { set_error("resident wgrad: %d x %d is out of range (N, K <= 160)", N, K); return 0; }
  return rw_wgrad_partial_floats(K) * sizeof(float);
#endif
}

#ifdef GNF_DEVTOOLS
int gnf_linear_wgrad_rw_set_trace(long long* buf) {
#ifndef GNF_EMU
  gnf::g_wg_trace = buf;
#else
  (void)buf;
#endif
  return 0;
}
#endif

int gnf_linear_wgrad_rw(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, int M, int N, int K, int passes,
                        void* work, size_t work_bytes, gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!dY || !X || !dW || M < 0 || N <= 0 || K <= 0 || lddw < K) return fail(GNF_ERR_INVALID, "gnf_linear_wgrad_rw: bad arguments");
  if (!rw_wgrad_supported(N, K)) return fail(GNF_ERR_UNSUPPORTED, "gnf_linear_wgrad_rw: %d x %d is out of range (N, K <= 160)", N, K);
  if (ldx != (K + 31) / 32 * 32) return fail(GNF_ERR_UNSUPPORTED, "gnf_linear_wgrad_rw: X must be a dense plane (ldx = %d)", (K + 31) / 32 * 32);
  if (!work || work_bytes < rw_wgrad_partial_floats(K) * sizeof(float)) return fail(GNF_ERR_WORKSPACE, "gnf_linear_wgrad_rw: workspace too small");
  if (int e = launch_rw_wgrad(dY, lddy, X, ldx, dW, lddw, M, N, K, passes, (float*)work, (cudaStream_t)stream)) return e;
  return check_launch("gnf_linear_wgrad_rw");
#endif
}

}  // extern "C"
