// Conditioner MLP engine on the 5th-generation tensor cores (tcgen05 / TMEM), TF32 operands with fp32
// accumulation, in two precisions:
//   passes = 1 : single-pass TF32            (fast mode: log-likelihood tolerance 2e-3)
//   passes = 3 : 3xTF32 split  a = a_hi + a_lo,  a_hi*b_hi + a_lo*b_hi + a_hi*b_lo   (fp32-equivalent: strict mode)
//
// One persistent, warp-specialised kernel serves Linear forward, dgrad and wgrad:
//   warps 0-3  epilogue   : thread t <-> accumulator row (TMEM lane) t; TMEM -> registers -> fused epilogue -> global
//   warp  4    MMA issuer : one thread issues tcgen05.mma, commits to mbarriers
//   warps 5-12 stagers    : (a) 16-byte-aligned operands: wait for the TMA tile, produce the hi/lo split in place;
//                           (b) unaligned operands: cp.async the tile themselves (zero-filling ragged tails), then split
//   warps 13,14 TMA issuers: one thread each (A tiles / B tiles) issues cp.async.bulk.tensor loads a ring ahead
// Both operand orientations (k-contiguous or row-contiguous global memory) land as canonical 128B-swizzled UMMA tiles:
// K-major = SWIZZLE_128B, MN-major = SWIZZLE_128B_BASE32B (TMA: CU_TENSOR_MAP_SWIZZLE_128B / _128B_ATOM_32B).
// A k-chunk is 32 fp32 = one 128-byte swizzle atom per tile row.  Accumulators are double buffered in TMEM
// (2 x <=256 columns) so a tile's epilogue overlaps the next tile's MMAs; the epilogue transposes 32x16 blocks through
// shared memory so that global stores / ReLU-mask loads / atomics touch 64 contiguous bytes per row instead of 16.
#include "tc_common.cuh"
#include "tc_gemm.h"
#ifndef GNF_EMU
#include <cuda.h>
#include <cudaTypedefs.h>
#endif

#ifndef GNF_EMU
namespace gnf {

constexpr int kGemmBM = 128;
constexpr int kGemmKC = 32;              // k-chunk: 32 fp32 = 128 bytes = one swizzle atom
constexpr int kEpiThreads = 128, kProdThreads = 256, kGemmThreads = kEpiThreads + 32 + kProdThreads + 64;
constexpr int kMaxStages = 6;
constexpr int kEpiLd = 20;                               // floats per staged epilogue row (16 + 4 pad: conflict-free STS.128)
constexpr int kEpiStageBytes = 4 * 32 * kEpiLd * 4;      // one 32 x 16 block per epilogue warp
constexpr size_t kSmemBudget = 227 * 1024;

// K-major fp32 tiles use SWIZZLE_128B (16-byte chunks XOR (row & 7), 8-row atoms: SBO = 1024).  MN-major tiles of
// a 32-bit type must use SWIZZLE_128B_BASE32B (32-byte granules XOR (row & 3), 4-row atoms: SBO = 512); LBO is the
// stride between 32-element MN slabs.
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr, bool mn_major) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)(((mn_major ? 4096u : 0u) >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(((mn_major ? 512u : 1024u) >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;                            // descriptor version (sm_100)
  d |= (uint64_t)(mn_major ? 1 : 2) << 61;           // SWIZZLE_128B_BASE32B : SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Fill one operand tile (rows x 32 k) for one k-chunk.  Tile image: 128-byte rows, 16-byte chunks XOR-swizzled by
// (row & 7).  K-major: tile row = operand row.  MN-major: slabs of 32 operand rows; tile row = k index inside the chunk.
// cp.async (LDGSTS) straight into the swizzled tile: no register staging, so a producer thread can have every
// vector of several stages in flight.  src_bytes < VEC*4 zero-fills the remainder (ragged K / row tails).
template <int VEC>
__device__ __forceinline__ void cp_async_vec(char* smem_dst, const float* gmem_src, int src_bytes) {
  const uint32_t d = tc::smem_u32(smem_dst);
  if (VEC == 4) asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gmem_src), "r"(src_bytes) : "memory");
  else if (VEC == 2) asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(gmem_src), "r"(src_bytes) : "memory");
  else asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(gmem_src), "r"(src_bytes) : "memory");
}
// 3xTF32 split of a landed raw fp32 tile, in place:  hi = rn_tf32(x) (overwrites the raw value), lo = rn_tf32(x - hi).
// The tensor core truncates the fp32 bits it reads (measured: scripts/tf32_round_probe.py); feeding it operands that
// already sit on the TF32 grid makes that truncation a no-op, and round-to-nearest keeps the representation error of
// hi + lo at ~2^-22 |x| and unbiased (truncating both would leave a one-sided 2^-20 error that survives cancellation).
__device__ __forceinline__ float rn_tf32(float x) {
  // cvt.rna.tf32.f32 (round to nearest, ties away) with two full-rate integer ops instead of the quarter-rate convert:
  // add half an ulp of the 13 dropped mantissa bits to the magnitude, clear them.
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}
template <int VEC>
__device__ __forceinline__ void split_vec(char* img_hi, char* img_lo, int off) {
  float v[VEC];
  if (VEC == 4) { const float4 q = *reinterpret_cast<const float4*>(img_hi + off); v[0] = q.x; v[1 % VEC] = q.y; v[2 % VEC] = q.z; v[3 % VEC] = q.w; }
  else if (VEC == 2) { const float2 q = *reinterpret_cast<const float2*>(img_hi + off); v[0] = q.x; v[1 % VEC] = q.y; }
  else v[0] = *reinterpret_cast<const float*>(img_hi + off);
  float hi[VEC], lo[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) { hi[j] = rn_tf32(v[j]); lo[j] = rn_tf32(v[j] - hi[j]); }
  if (VEC == 4) {
    *reinterpret_cast<float4*>(img_hi + off) = make_float4(hi[0], hi[1 % VEC], hi[2 % VEC], hi[3 % VEC]);
    *reinterpret_cast<float4*>(img_lo + off) = make_float4(lo[0], lo[1 % VEC], lo[2 % VEC], lo[3 % VEC]);
  } else if (VEC == 2) {
    *reinterpret_cast<float2*>(img_hi + off) = make_float2(hi[0], hi[1 % VEC]);
    *reinterpret_cast<float2*>(img_lo + off) = make_float2(lo[0], lo[1 % VEC]);
  } else {
    *reinterpret_cast<float*>(img_hi + off) = hi[0];
    *reinterpret_cast<float*>(img_lo + off) = lo[0];
  }
}

// K-major operand (global memory contiguous along k): tile row = operand row, 128 bytes (32 k) per row, 16-byte chunks
// XOR-swizzled by (row & 7).  Thread -> (row within a pass, vector within the row); passes advance by a multiple of
// 8 rows, so the swizzle term and the in-row offset are per-thread constants.
// kSplitPass = false: issue the cp.async copies of the raw tile.  true: produce the lo tile from the landed raw tile.
template <int VEC, bool kSplitPass>
__device__ __forceinline__ void fill_k(char* img_hi, char* img_lo, const float* __restrict__ g, long long ld, int r0, int r_end,
                                       int k0, int k_end, int rows, int ptid) {
  constexpr int VPR = 32 / VEC, STEP = kProdThreads / VPR;
  const int cv = ptid % VPR, rb = ptid / VPR, e = cv * VEC;
  const int soff0 = rb * 128 + ((((e >> 2) ^ (rb & 7)) << 4) | ((e & 3) << 2));
  const int npass = rows / STEP;
  if (kSplitPass) {
#pragma unroll 4
    for (int ps = 0; ps < npass; ++ps) split_vec<VEC>(img_hi, img_lo, soff0 + ps * STEP * 128);
    return;
  }
  int nk = k_end - (k0 + e);                             // valid elements of this thread's vector along k
  nk = nk < 0 ? 0 : (nk > VEC ? VEC : nk);
  const float* p0 = g + (long long)(r0 + rb) * ld + k0 + e;
#pragma unroll 4
  for (int ps = 0; ps < npass; ++ps) {
    const bool ok = (r0 + rb + ps * STEP) < r_end && nk > 0;
    cp_async_vec<VEC>(img_hi + soff0 + ps * STEP * 128, ok ? p0 + (long long)ps * STEP * ld : g, ok ? nk * 4 : 0);
  }
}

// MN-major operand (global memory contiguous along the operand-row index): slabs of 32 operand rows; tile row = k index
// inside the chunk (32 per chunk), 32-byte granules XOR-swizzled by (k & 3) (SWIZZLE_128B_BASE32B).  Producer warp w
// owns k rows w, w+8, w+16, w+24; lanes sweep the operand rows.
template <int VEC, bool kSplitPass>
__device__ __forceinline__ void fill_mn(char* img_hi, char* img_lo, const float* __restrict__ g, long long ld, int r0, int r_end,
                                        int k0, int k_end, int rows, int ptid) {
  const int w = ptid >> 5, lane = ptid & 31;
  const int per = rows / VEC;                            // vectors per k row
  for (int rv = lane; rv < per; rv += 32) {
    const int r = rv * VEC;
    const int slab = r >> 5, e = r & 31;
    int nr = r_end - (r0 + r);
    nr = nr < 0 ? 0 : (nr > VEC ? VEC : nr);
    const float* p0 = g + (long long)(k0 + w) * ld + r0 + r;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int kk = w + 8 * u;
      const int off = slab * 4096 + kk * 128 + ((((e >> 2) ^ ((kk & 3) << 1)) << 4) | ((e & 3) << 2));
      if (kSplitPass) {
        split_vec<VEC>(img_hi, img_lo, off);
      } else {
        const bool ok = (k0 + kk) < k_end && nr > 0;
        cp_async_vec<VEC>(img_hi + off, ok ? p0 + (long long)(8 * u) * ld : g, ok ? nr * 4 : 0);
      }
    }
  }
}

template <bool kSplitPass>
__device__ __forceinline__ void fill_dispatch(int vec, char* hi, char* lo, const float* g, long long ld, int src, int r0, int r_end,
                                              int k0, int k_end, int rows, int ptid) {
  if (src == TCG_SRC_K) {
    if (vec == 4) fill_k<4, kSplitPass>(hi, lo, g, ld, r0, r_end, k0, k_end, rows, ptid);
    else if (vec == 2) fill_k<2, kSplitPass>(hi, lo, g, ld, r0, r_end, k0, k_end, rows, ptid);
    else fill_k<1, kSplitPass>(hi, lo, g, ld, r0, r_end, k0, k_end, rows, ptid);
  } else {
    if (vec == 4) fill_mn<4, kSplitPass>(hi, lo, g, ld, r0, r_end, k0, k_end, rows, ptid);
    else if (vec == 2) fill_mn<2, kSplitPass>(hi, lo, g, ld, r0, r_end, k0, k_end, rows, ptid);
    else fill_mn<1, kSplitPass>(hi, lo, g, ld, r0, r_end, k0, k_end, rows, ptid);
  }
}

// One 2-D tiled TMA load: box (32 fp32 along the contiguous global index) x (box rows), completing on an mbarrier.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c_inner, int c_outer, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   tc::smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(c_inner), "r"(c_outer), "r"(tc::smem_u32(bar))
               : "memory");
}

// Measurement: role r of CTA 0 stamps event i with the SM clock (rows of 256 stamps per role).
constexpr int kTraceRoles = 8, kTraceLen = 256;
__device__ __forceinline__ void trace_stamp(long long* trace, int role, long long i) {
  if (trace && blockIdx.x == 0 && i < kTraceLen) trace[role * kTraceLen + i] = clock64();
}

__global__ void __launch_bounds__(kGemmThreads) tc_gemm_kernel(TcGemmParams p, int vecA, int vecB, const __grid_constant__ CUtensorMap tmA,
                                                               const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmBlo) {
  using namespace tc;
  GNF_SMEM(char, smem);
  const int BN = p.BN;
  const bool split = p.passes == 3;
  const bool presplit = split && p.B_lo != nullptr;      // B arrives as separate hi / lo tiles (only with TMA)
  const uint32_t a_bytes = kGemmBM * 128u, b_bytes = (uint32_t)BN * 128u;
  const uint32_t stage_bytes = (a_bytes + b_bytes) * (split ? 2u : 1u);
  // stage layout: [A_hi][B_hi]([A_lo][B_lo]); then the epilogue transpose blocks; then the barriers
  float* epi_stage = reinterpret_cast<float*>(smem + (size_t)p.stages * stage_bytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes + kEpiStageBytes);
  uint64_t* full = bars;                       // [stages]  stagers -> MMA     (count 8: one arrive per stager warp)
  uint64_t* empty = bars + kMaxStages;         // [stages]  MMA -> loaders     (tcgen05.commit)
  uint64_t* landed = bars + 2 * kMaxStages;    // [stages]  TMA -> stagers / MMA (transaction bytes)
  uint64_t* tfull = bars + 3 * kMaxStages;     // [2]       MMA -> epilogue
  uint64_t* tempty = tfull + 2;                // [2]       epilogue -> MMA    (count 4: one arrive per epilogue warp)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) tmem_alloc(tmem_slot, 512);
  if (tid == 32) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], kProdThreads / 32); mbar_init(&empty[s], 1); mbar_init(&landed[s], 2); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], kEpiThreads / 32); }
    fence_mbar_init();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();

  const int tiles_m = (p.M + kGemmBM - 1) / kGemmBM, tiles_n = (p.N + BN - 1) / BN;
  const long long total = (long long)tiles_m * tiles_n * p.splits;

  if (warp >= 13) {
    // ===================== TMA issuers: warp 13 loads the A tiles, warp 14 the B tiles =====================
    if (p.use_tma && lane == 0) {
      const bool isA = warp == 13;
      long long it = 0;
      for (long long w = blockIdx.x; w < total; w += gridDim.x) {
        const int tm = (int)(w % tiles_m), tn = (int)((w / tiles_m) % tiles_n), sp = (int)(w / ((long long)tiles_m * tiles_n));
        const int kbeg = sp * p.k_per_split, kend = min(p.K, kbeg + p.k_per_split);
        for (int k0 = kbeg; k0 < kend; k0 += kGemmKC, ++it) {
          const int s = (int)(it % p.stages);
          mbar_wait(&empty[s], (uint32_t)(((it / p.stages) & 1) ^ 1));
          char* st = smem + (size_t)s * stage_bytes;
          if (isA) {
            mbar_expect_tx(&landed[s], a_bytes);
            if (p.a_src == TCG_SRC_K) tma_load_2d(st, &tmA, k0, tm * kGemmBM, &landed[s]);
            else for (int sl = 0; sl < kGemmBM / 32; ++sl) tma_load_2d(st + sl * 4096, &tmA, tm * kGemmBM + 32 * sl, k0, &landed[s]);
            trace_stamp(p.trace, 0, it);
          } else {
            mbar_expect_tx(&landed[s], presplit ? 2u * b_bytes : b_bytes);
            if (p.b_src == TCG_SRC_K) tma_load_2d(st + a_bytes, &tmB, k0, tn * BN, &landed[s]);
            else for (int sl = 0; sl < BN / 32; ++sl) tma_load_2d(st + a_bytes + sl * 4096, &tmB, tn * BN + 32 * sl, k0, &landed[s]);
            if (presplit) {                                // the lo tile goes straight to its slot: [A_hi][B_hi][A_lo][B_lo]
              char* lo = st + 2 * a_bytes + b_bytes;
              if (p.b_src == TCG_SRC_K) tma_load_2d(lo, &tmBlo, k0, tn * BN, &landed[s]);
              else for (int sl = 0; sl < BN / 32; ++sl) tma_load_2d(lo + sl * 4096, &tmBlo, tn * BN + 32 * sl, k0, &landed[s]);
            }
          }
        }
      }
    }
  } else if (warp >= 5) {
    // ===================== stagers =====================
    const int ptid = tid - (kEpiThreads + 32);
    long long it = 0;                                    // running k-chunk counter (stage ring position)
    auto finish = [&](long long j) {                     // chunk j's raw tiles have landed: split, publish to the MMA warp
      const int s = (int)(j % p.stages);
      char* st = smem + (size_t)s * stage_bytes;
      if (split) {
        fill_dispatch<true>(vecA, st, st + a_bytes + b_bytes, nullptr, 0, p.a_src, 0, 0, 0, 0, kGemmBM, ptid);
        if (!presplit) fill_dispatch<true>(vecB, st + a_bytes, st + 2 * a_bytes + b_bytes, nullptr, 0, p.b_src, 0, 0, 0, 0, BN, ptid);
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[s]);
    };
    if (p.use_tma) {
      if (split) {                                       // 3xTF32 only: single-pass TF32 MMAs consume the landed tiles directly
        for (long long w = blockIdx.x; w < total; w += gridDim.x) {
          const int sp = (int)(w / ((long long)tiles_m * tiles_n));
          const int kbeg = sp * p.k_per_split, kend = min(p.K, kbeg + p.k_per_split);
          for (int k0 = kbeg; k0 < kend; k0 += kGemmKC, ++it) {
            mbar_wait(&landed[(int)(it % p.stages)], (uint32_t)((it / p.stages) & 1));
            if (tid == kEpiThreads + 32) trace_stamp(p.trace, 1, it);
            finish(it);
            if (tid == kEpiThreads + 32) trace_stamp(p.trace, 2, it);
          }
        }
      }
    } else {
      // Software pipeline with a lag of kLag stages: the copies of chunk `it` are issued (cp.async, one commit group per
      // chunk) before chunk it-kLag is finished (wait for its group, produce the lo tiles, proxy fence, signal the MMA).
      const int kLag = p.stages >= 3 ? 2 : 1;            // the ring must hold the in-flight chunks plus one being consumed
      for (long long w = blockIdx.x; w < total; w += gridDim.x) {
        const int tm = (int)(w % tiles_m), tn = (int)((w / tiles_m) % tiles_n), sp = (int)(w / ((long long)tiles_m * tiles_n));
        const int kbeg = sp * p.k_per_split, kend = min(p.K, kbeg + p.k_per_split);
        for (int k0 = kbeg; k0 < kend; k0 += kGemmKC, ++it) {
          const int s = (int)(it % p.stages);
          const uint32_t par = (uint32_t)((it / p.stages) & 1);
          mbar_wait(&empty[s], par ^ 1u);
          char* st = smem + (size_t)s * stage_bytes;
          fill_dispatch<false>(vecA, st, nullptr, p.A, p.lda, p.a_src, tm * kGemmBM, p.M, k0, kend, kGemmBM, ptid);
          fill_dispatch<false>(vecB, st + a_bytes, nullptr, p.B, p.ldb, p.b_src, tn * BN, p.N, k0, kend, BN, ptid);
          cp_async_commit();
          if (it >= kLag) {
            if (kLag == 2) cp_async_wait<2>(); else cp_async_wait<1>();
            finish(it - kLag);
          }
        }
      }
      // drain
      cp_async_wait<0>();
      for (long long j = (it > kLag ? it - kLag : 0); j < it; ++j) finish(j);
    }
  } else if (warp == 4) {
    // ===================== MMA issuer =====================
    {   // the whole warp runs the loop converged; one elected lane issues (tc_common.cuh: mma_*_w)
      const uint32_t idesc = make_idesc_tf32(kGemmBM, BN) | (p.a_src == TCG_SRC_MN ? (1u << 15) : 0u) | (p.b_src == TCG_SRC_MN ? (1u << 16) : 0u);
      // per k-step (8 k) descriptor advance: K-major: 32 bytes inside the swizzle atom; MN-major: 8 tile rows = 1024 bytes
      const uint32_t a_step = (p.a_src == TCG_SRC_K) ? 2u : 64u, b_step = (p.b_src == TCG_SRC_K) ? 2u : 64u;
      const bool a_mn = p.a_src == TCG_SRC_MN, b_mn = p.b_src == TCG_SRC_MN;
      uint64_t* ready = (p.use_tma && !split) ? landed : full;
      long long it = 0;
      int gcount = 0;                                    // accumulator groups issued so far (buffer = gcount & 1)
      for (long long w = blockIdx.x; w < total; w += gridDim.x) {
        const int sp = (int)(w / ((long long)tiles_m * tiles_n));
        const int kbeg = sp * p.k_per_split, kend = min(p.K, kbeg + p.k_per_split);
        for (int kg = kbeg; kg < kend; kg += p.fold * kGemmKC, ++gcount) {
          const int kg_end = min(kend, kg + p.fold * kGemmKC);
          const int acc = gcount & 1;
          mbar_wait(&tempty[acc], (uint32_t)(((gcount >> 1) & 1) ^ 1));
          fence_after_sync();
          const uint32_t d_tmem = tmem_base + (uint32_t)acc * (uint32_t)p.acc_stride;
          bool first = true;
          for (int k0 = kg; k0 < kg_end; k0 += kGemmKC, ++it) {
            const int s = (int)(it % p.stages);
            mbar_wait(&ready[s], (uint32_t)((it / p.stages) & 1));
            fence_after_sync();
            if (lane == 0) trace_stamp(p.trace, 3, it);
            const uint32_t st = smem_u32(smem + (size_t)s * stage_bytes);
            const uint64_t da_hi = make_sw128_desc(st, a_mn), db_hi = make_sw128_desc(st + a_bytes, b_mn);
            const uint64_t da_lo = make_sw128_desc(st + a_bytes + b_bytes, a_mn), db_lo = make_sw128_desc(st + 2 * a_bytes + b_bytes, b_mn);
            // 3xTF32: the correction products of the chunk first (they accumulate at 2^-11 of the result's magnitude, where the
            // tensor core's one-sided truncation of the accumulator costs nothing), then the a_hi b_hi chain
            if (split) {
#pragma unroll
              for (int ks = 0; ks < kGemmKC / 8; ++ks) {
                const uint64_t oa = (uint64_t)(a_step * ks), ob = (uint64_t)(b_step * ks);
                mma_tf32_ss_w(d_tmem, da_lo + oa, db_hi + ob, idesc, first ? 0u : 1u);
                first = false;
                mma_tf32_ss_w(d_tmem, da_hi + oa, db_lo + ob, idesc, 1u);
              }
            }
#pragma unroll
            for (int ks = 0; ks < kGemmKC / 8; ++ks) {
              mma_tf32_ss_w(d_tmem, da_hi + (uint64_t)(a_step * ks), db_hi + (uint64_t)(b_step * ks), idesc, first ? 0u : 1u);
              first = false;
            }
            mma_commit_w(&empty[s]);
          }
          mma_commit_w(&tfull[acc]);
          if (lane == 0) trace_stamp(p.trace, 4, gcount);
        }
      }
    }
  } else {
    // ===================== epilogue =====================
    // Thread t owns accumulator row t (TMEM lane t).  Each 16-column block goes through a per-warp 32 x 16 shared-memory
    // block so that global accesses are row-contiguous: lane l <-> (row (l >> 2) + 8 i, 16-byte piece l & 3).
    const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
    float* stg = epi_stage + warp * 32 * kEpiLd;
    float* my_row = stg + lane * kEpiLd;
    const int piece = (lane & 3) * 4, rsub = lane >> 2;
    // per-element side input of the epilogue, fetched one 16-column block ahead of its use:
    //   aux_tile: ReLU-mask activations (dgrad) or a periodic bias table row (bias_period > 1), as a transposed 32 x 16 block
    // whole-tile side inputs, loaded before the accumulator is waited for (their latency hides behind the main loop):
    //   bias_row: one bias vector for every row: lane l holds bias[n0 + 32 i + l], broadcast by shuffles
    //   bit_mask: the ReLU mask as one bit per element: the row owner holds its row's words
    const bool bit_mask = p.epi == TCG_EPI_MASK && p.mask_bits != nullptr;
    const bool aux_mask = p.epi == TCG_EPI_MASK && p.act != nullptr && !bit_mask;
    const bool aux_bias = p.epi == TCG_EPI_BIAS_ACT && p.bias != nullptr && p.bias_period > 1;
    const bool aux_tile = aux_mask || aux_bias;
    const bool bias_row = p.epi == TCG_EPI_BIAS_ACT && p.bias != nullptr && p.bias_period <= 1;
    int gcount = 0, tcount = 0;
    for (long long w = blockIdx.x; w < total; w += gridDim.x, ++tcount) {
      const int tm = (int)(w % tiles_m), tn = (int)((w / tiles_m) % tiles_n), sp = (int)(w / ((long long)tiles_m * tiles_n));
      const int kbeg = sp * p.k_per_split, kend = min(p.K, kbeg + p.k_per_split);
      const int ngroups = (kend - kbeg + p.fold * kGemmKC - 1) / (p.fold * kGemmKC);
      const int m_warp = tm * kGemmBM + warp * 32, n0 = tn * BN;
      const int n_lim = min(BN, p.N - n0);               // columns of this tile that exist
      const uint32_t run = tmem_base + lane_sel + 2u * (uint32_t)p.acc_stride;   // running sum region (3xTF32 only)
      const int m_row = m_warp + lane;
      float breg[8];
      uint32_t mw[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        breg[i] = (bias_row && 32 * i < n_lim && n0 + 32 * i + lane < p.N) ? __ldg(p.bias + n0 + 32 * i + lane) : 0.f;
        mw[i] = (bit_mask && 32 * i < n_lim && m_row < p.M) ? __ldg(p.mask_bits + (long long)m_row * p.mask_ld + (n0 >> 5) + i) : 0u;
      }
      uint32_t obits = 0u;
      // The tensor core accumulates with round-toward-zero: long in-core accumulation chains bias the result.  Every `fold`
      // k-chunks the partial accumulator is therefore folded into a running sum with round-to-nearest adds (TMEM -> registers
      // -> TMEM, this warp's own lanes), while the MMA warp already fills the other partial buffer.
      for (int g = 0; g + 1 < ngroups; ++g, ++gcount) {
        const int acc = gcount & 1;
        mbar_wait(&tfull[acc], (uint32_t)((gcount >> 1) & 1));
        fence_after_sync();
        const uint32_t part = tmem_base + lane_sel + (uint32_t)acc * (uint32_t)p.acc_stride;
        for (int c = 0; c < n_lim; c += 16) {
          uint32_t a[16], b[16];
          tmem_ld16_nowait(part + c, a);
          if (g > 0) tmem_ld16_nowait(run + c, b);
          tmem_wait_ld();
          if (g > 0) {
#pragma unroll
            for (int j = 0; j < 16; ++j) a[j] = __float_as_uint(__uint_as_float(a[j]) + __uint_as_float(b[j]));
          }
          tmem_st16u(run + c, a);
        }
        tmem_wait_st();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
      }
      const int acc = gcount & 1;
      const uint32_t acc_par = (uint32_t)((gcount >> 1) & 1);
      ++gcount;
      auto load_aux = [&](int c, float4 (&a)[4], float& b1) {
        const int n = n0 + c;
        if (aux_tile) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int mr = m_warp + rsub + 8 * i;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (mr < p.M && n + piece < p.N) {
              const float* ap = aux_mask ? p.act + (long long)mr * p.ldact + n + piece
                                         : p.bias + (long long)(mr % p.bias_period) * p.bias_ld + n + piece;
              if ((aux_mask ? p.act_vec : p.bias_vec) && n + piece + 4 <= p.N) v = __ldg(reinterpret_cast<const float4*>(ap));
              else {
                v.x = __ldg(ap);
                if (n + piece + 1 < p.N) v.y = __ldg(ap + 1);
                if (n + piece + 2 < p.N) v.z = __ldg(ap + 2);
                if (n + piece + 3 < p.N) v.w = __ldg(ap + 3);
              }
            }
            a[i] = v;
          }
        }
        (void)b1;
      };
      float4 aux_cur[4], aux_nxt[4];
      float b_cur = 0.f, b_nxt = 0.f;
      load_aux(0, aux_cur, b_cur);                       // independent of the accumulator: issued before the tile is complete
      mbar_wait(&tfull[acc], acc_par);
      fence_after_sync();
      if (tid == 0) trace_stamp(p.trace, 5, tcount);
      const uint32_t src = tmem_base + lane_sel + (uint32_t)acc * (uint32_t)p.acc_stride;
      const bool folded = ngroups > 1;
      uint32_t cur[16], nxt[16];
      auto load_acc = [&](int c, uint32_t (&v)[16]) {    // last partial (+ running sum), 16 columns
        tmem_ld16_nowait(src + c, v);
        if (folded) {
          uint32_t r[16];
          tmem_ld16_nowait(run + c, r);
          tmem_wait_ld();
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(r[j]));
        }
      };
      load_acc(0, cur);
      tmem_wait_ld();
      for (int c = 0; c < n_lim; c += 16) {
        const bool more = c + 16 < n_lim;
        const bool tr = p.trace && tid == 0 && tcount == 1;
        if (tr) trace_stamp(p.trace, 7, (c >> 4) * 6 + 0);
        if (more) { load_acc(c + 16, nxt); load_aux(c + 16, aux_nxt, b_nxt); }
        if (tr) trace_stamp(p.trace, 7, (c >> 4) * 6 + 1);
        const int n = n0 + c;
        float o[16];
        if (aux_tile) {
#pragma unroll
          for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(stg + (rsub + 8 * i) * kEpiLd + piece) = aux_cur[i];
          __syncwarp();
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 a = *reinterpret_cast<const float4*>(my_row + 4 * j4);
            const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float r = __uint_as_float(cur[4 * j4 + e]);
              if (aux_mask) o[4 * j4 + e] = av[e] > 0.f ? r : 0.f;
              else o[4 * j4 + e] = p.relu ? fmaxf(r + av[e], 0.f) : r + av[e];
            }
          }
          __syncwarp();
        } else if (p.epi == TCG_EPI_BIAS_ACT) {
          float bsel = breg[0];
#pragma unroll
          for (int i = 1; i < 8; ++i) if ((c >> 5) == i) bsel = breg[i];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float r = __uint_as_float(cur[j]);
            if (bias_row) r += __shfl_sync(0xffffffffu, bsel, (c & 31) + j);
            o[j] = p.relu ? fmaxf(r, 0.f) : r;
          }
        } else if (bit_mask) {
          uint32_t wsel = mw[0];
#pragma unroll
          for (int i = 1; i < 8; ++i) if ((c >> 5) == i) wsel = mw[i];
          wsel >>= (c & 31);
#pragma unroll
          for (int j = 0; j < 16; ++j) o[j] = ((wsel >> j) & 1u) ? __uint_as_float(cur[j]) : 0.f;
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) o[j] = __uint_as_float(cur[j]);
        }
        if (p.bits_out) {                                  // ReLU mask of the output, one bit per element, row-owner layout
#pragma unroll
          for (int j = 0; j < 16; ++j) obits |= (o[j] > 0.f ? 1u : 0u) << ((c & 31) + j);
          if ((c & 31) == 16 || !more) {
            if (m_row < p.M) p.bits_out[(long long)m_row * p.bits_ld + ((n0 + c) >> 5)] = obits;
            obits = 0u;
          }
        }
        if (tr) trace_stamp(p.trace, 7, (c >> 4) * 6 + 2);
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) *reinterpret_cast<float4*>(my_row + 4 * j4) = make_float4(o[4 * j4], o[4 * j4 + 1], o[4 * j4 + 2], o[4 * j4 + 3]);
        __syncwarp();
        if (tr) trace_stamp(p.trace, 7, (c >> 4) * 6 + 3);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = rsub + 8 * i, mr = m_warp + row;
          if (mr < p.M && n + piece < p.N) {
            const float4 v = *reinterpret_cast<const float4*>(stg + row * kEpiLd + piece);
            float* y = p.C + (long long)mr * p.ldc + n + piece;
            if (p.epi == TCG_EPI_ATOMIC) {
              atomicAdd(y, v.x);
              if (n + piece + 1 < p.N) atomicAdd(y + 1, v.y);
              if (n + piece + 2 < p.N) atomicAdd(y + 2, v.z);
              if (n + piece + 3 < p.N) atomicAdd(y + 3, v.w);
            } else if (p.c_vec && n + piece + 4 <= p.N) {
              *reinterpret_cast<float4*>(y) = v;
            } else {
              y[0] = v.x;
              if (n + piece + 1 < p.N) y[1] = v.y;
              if (n + piece + 2 < p.N) y[2] = v.z;
              if (n + piece + 3 < p.N) y[3] = v.w;
            }
          }
        }
        __syncwarp();
        if (tr) trace_stamp(p.trace, 7, (c >> 4) * 6 + 4);
        if (more) {
          tmem_wait_ld();
          if (tr) trace_stamp(p.trace, 7, (c >> 4) * 6 + 5);
#pragma unroll
          for (int j = 0; j < 16; ++j) cur[j] = nxt[j];
#pragma unroll
          for (int i = 0; i < 4; ++i) aux_cur[i] = aux_nxt[i];
          b_cur = b_nxt;
        }
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
      if (tid == 0) trace_stamp(p.trace, 6, tcount);
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

static inline int vec_width(const float* p, long long ld) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  if ((a & 15) == 0 && (ld % 4) == 0) return 4;
  if ((a & 7) == 0 && (ld % 2) == 0) return 2;
  return 1;
}

static int g_tc_gemm_force_bn = 0;      // measurement overrides (gnf_tc_gemm_set_tile); 0 = planned
static int g_tc_gemm_force_splits = 0;

// Tile width and split-K factor for the persistent engine, chosen per problem shape.  The kernel hands work items
// (tile x k-split) to `kNumSMs` CTAs round-robin, so its duration is  rounds x (k-chunks per item) x (chunk cadence)  plus one
// exposed epilogue: what matters is how full the LAST round is, not only the padding of N.  (The first version took the
// widest tile that fits -- 6300 x 632: 50 x 4 = 200 items = 2 rounds of which the second is 35 % full -- and ceil(SMs / tiles)
// splits for the wgrad: 20 tiles x 8 = 160 items = 2 rounds for 12 stragglers.)
// Cost unit: one k-chunk of a 128 x 160 tile.  The chunk cadence is bound by operand movement (TMA / split), which scales
// with BM + BN; the epilogue of a tile is worth ~10 such chunks at BN = 160 (profiles/r01zb_tc_gemm_trace_tma_path.txt).
static void plan_tiles(int M, int N, int K, int max_bn, bool atomic, int* bn_out, int* splits_out) {
  const int cands[7] = {64, 96, 128, 160, 192, 224, 256};
  const int tiles_m = (M + kGemmBM - 1) / kGemmBM;
  const int kchunks = (K + kGemmKC - 1) / kGemmKC;
  const int max_splits = atomic ? (K + 8 * kGemmKC - 1) / (8 * kGemmKC) : 1;
  double best_cost = -1.;
  int best_bn = 64, best_sp = 1;
  for (int i = 0; i < 7; ++i) {
    const int bn = cands[i];
    if (bn > max_bn) break;
    if (g_tc_gemm_force_bn && bn != g_tc_gemm_force_bn) continue;
    const long long tiles = (long long)tiles_m * ((N + bn - 1) / bn);
    const double chunk = (128. + bn) / 288., epi = 10. * bn / 160.;
    for (int sp = 1; sp <= (max_splits < 1 ? 1 : max_splits); ++sp) {
      if (g_tc_gemm_force_splits && sp != (g_tc_gemm_force_splits < max_splits ? g_tc_gemm_force_splits : (max_splits < 1 ? 1 : max_splits))) continue;
      const int per = (kchunks + sp - 1) / sp;
      const int eff = (kchunks + per - 1) / per;         // splits that actually get work
      if (eff != sp) continue;
      const long long items = tiles * eff;
      const long long rounds = (items + kNumSMs - 1) / kNumSMs;
      const double cost = (double)rounds * (per * chunk + 1.) + epi;
      if (best_cost < 0. || cost < best_cost * 0.999 || (cost <= best_cost * 1.001 && bn > best_bn)) { best_cost = cost; best_bn = bn; best_sp = eff; }
    }
  }
  if (best_cost < 0. && (g_tc_gemm_force_bn || g_tc_gemm_force_splits)) {   // the forced combination does not exist for this shape
    const int fb = g_tc_gemm_force_bn, fs = g_tc_gemm_force_splits;
    g_tc_gemm_force_bn = g_tc_gemm_force_splits = 0;
    plan_tiles(M, N, K, max_bn, atomic, bn_out, splits_out);
    g_tc_gemm_force_bn = fb; g_tc_gemm_force_splits = fs;
    return;
  }
  *bn_out = best_bn;
  *splits_out = best_sp;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point query (no link-time dependency on libcuda).
static PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
    cudaGetLastError();
  }
  return fn;
}

// Tensor map of one GEMM operand.  K-major source: dims {K, rows}, box {32, tile_rows}, SWIZZLE_128B.
// MN-major source: dims {rows, K}, box {32, 32} (one 32-row slab per load), SWIZZLE_128B with 32-byte atoms.
static bool make_operand_map(CUtensorMap* map, const float* base, long long ld, int src, int rows, int K, int tile_rows) {
  PFN_cuTensorMapEncodeTiled_v12000 enc = tensor_map_encoder();
  if (!enc || (reinterpret_cast<uintptr_t>(base) & 15) != 0 || (ld % 4) != 0) return false;
  cuuint64_t dims[2], strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2], estr[2] = {1, 1};
  CUtensorMapSwizzle sw;
  if (src == TCG_SRC_K) { dims[0] = (cuuint64_t)K; dims[1] = (cuuint64_t)rows; box[0] = 32; box[1] = (cuuint32_t)tile_rows; sw = CU_TENSOR_MAP_SWIZZLE_128B; }
  else { dims[0] = (cuuint64_t)rows; dims[1] = (cuuint64_t)K; box[0] = 32; box[1] = 32; sw = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B; }
  if ((long long)dims[0] > ld) return false;
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static long long* g_tc_gemm_trace = nullptr;
static int g_tc_gemm_fold = 2;      // k-chunks accumulated inside the tensor core before a round-to-nearest fold (3xTF32)
static int g_tc_gemm_fold2 = 2;     // ... of engine v2 (forward / dgrad with pre-split weights).  With the correction products first, fold 2 leaves a
                                    // relative error of 2.7e-7 (one-sided part 1.4e-7), fold 1 1.1e-7 (4e-8) = the FFMA engine's, at +15 % time
                                    // (profiles/r02q_gemm2_fold_variants.txt).  The first layer of a wide DAG flow (periodic bias table) always folds
                                    // every chunk: its rounding error passes through every later layer and through the gate derivative, and the
                                    // gradients of A / W1 at cfg5 sit on ReLU-flip noise of that size (profiles/r02p_cfg5_grad_accuracy*.txt).
static bool g_tc_gemm_fold_forced = false;   // dev build: gnf_tc_gemm_set_fold overrides both rules
static bool g_tc_gemm_tma = true;   // measurement switch (gnf_tc_gemm_set_tma): 0 forces the cp.async staging path
static int g_tc_gemm_v2 = 1;        // measurement switch (gnf_tc_gemm_set_v2, dev build): 0 keeps forward / dgrad on the engine above

// hi = rn_tf32(W), lo = rn_tf32(W - hi), both [N][ld] with zero padding columns (ld >= K)
__global__ void split_tf32_kernel(const float* __restrict__ W, long long ldw, float* __restrict__ hi, float* __restrict__ lo, int ld, int N, int K) {
  const long long total = (long long)N * ld;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / ld), k = (int)(i - (long long)n * ld);
    const float v = k < K ? W[n * ldw + k] : 0.f;
    const float h = rn_tf32(v);
    hi[i] = h;
    lo[i] = rn_tf32(v - h);
  }
}

// =====================================================================================================================
// Engine v2 for the conditioner's hidden layers (DAGMLP, DAGConditioner.py:7-20), forward and dgrad, 3xTF32 with pre-split
// weights.  What the traces of the kernel above said (profiles/r01zb_tc_gemm_trace_tma_path.txt): its k-chunk cadence is
// 2.2-2.7 k clocks against 0.77 k of MMA time -- the 8 stager warps need ~1.7 k clocks to turn a landed 16 KB activation
// tile into hi / lo tiles in shared memory -- and the 16-column transposing epilogue takes 24 k clocks per tile.  Here:
//   * the activation operand never exists as an MMA tile in shared memory: four A-writer warps (thread = tile row = TMEM
//     lane) read their row of the TMA-landed raw tile (conflict-free through the 128B swizzle), split it in registers and
//     write A_hi / A_lo into a four-deep TMEM ring (tcgen05.st); the MMAs are TS form, B = the pre-split weight tiles;
//   * a stage is 48 KB (raw A + B_hi + B_lo) instead of 64 KB: four stages in flight;
//   * same accumulation discipline as above (the tensor core truncates its accumulator after every MMA, one-sided): two
//     partial accumulators in TMEM, folded every `fold` k-chunks into a round-to-nearest running sum that EIGHT epilogue
//     warps (two per lane quarter, 64 columns each) keep in registers, so that a fold is one TMEM read + 64 additions and the
//     output pass of a tile hides behind the next tile's first groups; correction products go first inside every chunk;
//   * the final epilogue moves 32-column blocks through a 4 KB XOR-swizzled staging block per warp (rw_gemm_kernel's):
//     every global instruction covers 4 rows x 128 bytes, the dgrad ReLU mask is applied on the coalesced side.
// TMEM columns: partials 0 / 128, A ring 256 (four buffers of hi 32 + lo 32).
// =====================================================================================================================
constexpr int kG2BN = 128, kG2Stages = 4, kG2Threads = 14 * 32;   // 8 epilogue + 4 A-writer + MMA issuer + TMA producer warps
constexpr uint32_t kG2TileBytes = 128u * 128u;                    // one 128-row x 32-k fp32 tile
constexpr uint32_t kG2StageBytes = 3u * kG2TileBytes;             // raw A, B_hi, B_lo
constexpr int kG2EpiStageFloats = 32 * 32;
constexpr int kG2Parts = 2, kG2Ring = 4;   // partial accumulators of 128 TMEM columns, then A buffers of (hi 32 + lo 32) columns

__global__ void __launch_bounds__(kG2Threads, 1) tc_gemm2_kernel(TcGemmParams p, const __grid_constant__ CUtensorMap tmA,
                                                                 const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmBlo) {
  using namespace tc;
  GNF_SMEM(char, smem);
  float* epi_stage = reinterpret_cast<float*>(smem + (size_t)kG2Stages * kG2StageBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_stage + 8 * kG2EpiStageFloats);
  uint64_t* landed = bars;                     // [stages] TMA -> A-writers / MMA (transaction bytes)
  uint64_t* empty = landed + kG2Stages;        // [stages] MMA -> producer (tcgen05.commit)
  constexpr uint32_t kG2ColA = 128u * kG2Parts;
  static_assert(kG2ColA + 64u * kG2Ring <= 512u, "TMEM budget");
  uint64_t* a_full = empty + kG2Stages;        // [kG2Ring] A-writers -> MMA (one arrive per writer warp)
  uint64_t* a_empty = a_full + kG2Ring;        // [kG2Ring] MMA -> A-writers (tcgen05.commit)
  uint64_t* tfull = a_empty + kG2Ring;         // [kG2Parts] MMA -> epilogue
  uint64_t* tempty = tfull + kG2Parts;         // [kG2Parts] epilogue -> MMA (one arrive per epilogue warp)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + kG2Parts);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) tmem_alloc(tmem_slot, 512);
  if (tid == 32) {
    for (int s = 0; s < kG2Stages; ++s) { mbar_init(&landed[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < kG2Ring; ++b) { mbar_init(&a_full[b], 4); mbar_init(&a_empty[b], 1); }
    for (int b = 0; b < kG2Parts; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 8); }
    fence_mbar_init();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();

  const int tiles_m = (p.M + kGemmBM - 1) / kGemmBM, tiles_n = (p.N + kG2BN - 1) / kG2BN;
  const int total = tiles_m * tiles_n;
  const int nchunks = (p.K + kGemmKC - 1) / kGemmKC;
  const int fold = p.fold < 1 ? 1 : p.fold;
  const bool b_mn = p.b_src == TCG_SRC_MN;

  if (warp == 13) {
    // ===================== producer: one thread issues the TMA loads of a stage (raw A, B_hi, B_lo) =====================
    if (lane == 0) {
      int it = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const int tm = w % tiles_m, tn = w / tiles_m;
        for (int c = 0; c < nchunks; ++c, ++it) {
          const int s = it % kG2Stages, k0 = c * kGemmKC;
          mbar_wait(&empty[s], (uint32_t)(((it / kG2Stages) & 1) ^ 1));
          char* st = smem + (size_t)s * kG2StageBytes;
          mbar_expect_tx(&landed[s], kG2StageBytes);
          tma_load_2d(st, &tmA, k0, tm * kGemmBM, &landed[s]);
          if (!b_mn) {
            tma_load_2d(st + kG2TileBytes, &tmB, k0, tn * kG2BN, &landed[s]);
            tma_load_2d(st + 2 * kG2TileBytes, &tmBlo, k0, tn * kG2BN, &landed[s]);
          } else {
            for (int sl = 0; sl < kG2BN / 32; ++sl) {
              tma_load_2d(st + kG2TileBytes + sl * 4096, &tmB, tn * kG2BN + 32 * sl, k0, &landed[s]);
              tma_load_2d(st + 2 * kG2TileBytes + sl * 4096, &tmBlo, tn * kG2BN + 32 * sl, k0, &landed[s]);
            }
          }
          trace_stamp(p.trace, 0, it);
        }
      }
    }
  } else if (warp == 12) {
    // ===================== MMA issuer (the whole warp runs the loop converged, one elected lane issues) =====================
    const uint32_t idesc = make_idesc_tf32(kGemmBM, kG2BN) | (b_mn ? (1u << 16) : 0u);
    const uint32_t b_step = b_mn ? 64u : 2u;
    int it = 0, gcount = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
      for (int c0 = 0; c0 < nchunks; c0 += fold, ++gcount) {
        const int acc = gcount % kG2Parts;
        mbar_wait(&tempty[acc], (uint32_t)(((gcount / kG2Parts) & 1) ^ 1));
        fence_after_sync();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * kG2BN;
        const int c1 = (c0 + fold < nchunks) ? c0 + fold : nchunks;
        uint32_t first = 0u;
        for (int c = c0; c < c1; ++c, ++it) {
          const int s = it % kG2Stages, b = it % kG2Ring;
          mbar_wait(&a_full[b], (uint32_t)((it / kG2Ring) & 1));
          mbar_wait(&landed[s], (uint32_t)((it / kG2Stages) & 1));
          fence_after_sync();
          if (lane == 0) trace_stamp(p.trace, 3, it);
          const uint32_t st = smem_u32(smem + (size_t)s * kG2StageBytes);
          const uint64_t db_hi = make_sw128_desc(st + kG2TileBytes, b_mn), db_lo = make_sw128_desc(st + 2 * kG2TileBytes, b_mn);
          const uint32_t ta_hi = tmem_base + kG2ColA + (uint32_t)b * 64u, ta_lo = ta_hi + 32u;
          // The tensor core truncates its fp32 accumulator after every MMA (one-sided: profiles/r02p_gemm2_fold_cfg5_shapes.txt).
          // Correction products first: while the partial only holds a_lo b_hi + a_hi b_lo terms (2^-11 of the result) their
          // truncations cost nothing; only the a_hi b_hi MMAs accumulate at full magnitude.
#pragma unroll
          for (int ks = 0; ks < kGemmKC / 8; ++ks) {
            const uint64_t ob = (uint64_t)(b_step * ks);
            mma_tf32_ts_w(d_tmem, ta_lo + ks * 8, db_hi + ob, idesc, first);
            first = 1u;
            mma_tf32_ts_w(d_tmem, ta_hi + ks * 8, db_lo + ob, idesc, 1u);
          }
#pragma unroll
          for (int ks = 0; ks < kGemmKC / 8; ++ks) mma_tf32_ts_w(d_tmem, ta_hi + ks * 8, db_hi + (uint64_t)(b_step * ks), idesc, 1u);
          mma_commit_w(&empty[s]);
          mma_commit_w(&a_empty[b]);
        }
        mma_commit_w(&tfull[acc]);
        if (lane == 0) trace_stamp(p.trace, 4, gcount);
      }
    }
  } else if (warp >= 8) {
    // ===================== A-writers: raw tile row -> TF32 hi / lo in registers -> TMEM ring =====================
    const int q = warp - 8, row = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    int it = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
      for (int c = 0; c < nchunks; ++c, ++it) {
        const int s = it % kG2Stages, b = it % kG2Ring;
        mbar_wait(&landed[s], (uint32_t)((it / kG2Stages) & 1));
        if (tid == 256) trace_stamp(p.trace, 1, it);
        const char* rp = smem + (size_t)s * kG2StageBytes + row * 128;
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint4 v = *reinterpret_cast<const uint4*>(rp + ((j ^ (row & 7)) << 4));
          const uint32_t e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t h = (e[k] + 0x1000u) & 0xffffe000u;
            hi[4 * j + k] = h;
            lo[4 * j + k] = __float_as_uint(__uint_as_float(e[k]) - __uint_as_float(h)) + 0x1000u;   // the tensor core drops the low bits
          }
        }
        mbar_wait(&a_empty[b], (uint32_t)(((it / kG2Ring) & 1) ^ 1));
        fence_after_sync();
        const uint32_t ta = tmem_base + lane_sel + kG2ColA + (uint32_t)b * 64u;
        tmem_st32p(ta, hi);
        tmem_st32p(ta + 32, lo);
        tmem_wait_st();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[b]);
        if (tid == 256) trace_stamp(p.trace, 2, it);
      }
    }
  } else {
    // ===================== epilogue: folds of the partial accumulators, then the tile's output =====================
    // Eight warps: warp = (TMEM lane quarter, column half); each keeps the round-to-nearest running sum of its 32 rows x 64
    // columns of the tile in REGISTERS (64 per thread): a fold is one TMEM read of the partial + 64 additions, the partial is
    // released at once, and the output pass works from registers (no running sum in TMEM: its 128 columns widen the A ring).
    const int quarter = warp & 3, half = warp >> 2, ch = 64 * half;
    const uint32_t lane_sel = (uint32_t)(quarter * 32) << 16;
    float* stage = epi_stage + warp * kG2EpiStageFloats;
    const int sub = lane >> 3, piece = lane & 7;
    const bool mask = p.epi == TCG_EPI_MASK && p.act != nullptr;          // a dgrad without a ReLU behind it (act == NULL) stores the plain product
    const bool table = !mask && p.bias != nullptr && p.bias_period > 1;   // periodic bias table (DAG layer 1: one row per variable): added on the coalesced side
    const int ngroups = (nchunks + fold - 1) / fold;
    int gcount = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
      const int tm = w % tiles_m, tn = w / tiles_m;
      const int n0 = tn * kG2BN + ch, m0 = tm * kGemmBM + quarter * 32;
      float run[64];
      // dgrad: the ReLU mask of this thread's output pieces (coalesced side: rows 4 i + sub, columns 4 piece .. + 3 of both 32-column
      // blocks), fetched before the tile's first MMA group is awaited (the running sum is not live yet) and kept as 2 x 32 bits.  Loading it inside the output pass put one
      // exposed global-load latency in front of every store (dgrad 508 us against 318 us for the plain product at 64512 x 632 x 632,
      // profiles/r02ab_dgrad_probe.txt).  Clamped addresses: the loads are unconditional, out-of-range pieces are never stored.
      uint32_t mbits[2] = {0u, 0u};
      {
        if (mask) {
#pragma unroll
          for (int cb = 0; cb < 2; ++cb) {
            const int n = n0 + 32 * cb + 4 * piece, nc = n < p.N ? n : 0;
            float4 av[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int m = m0 + 4 * i + sub, mc = m < p.M ? m : p.M - 1;
              av[i] = __ldg(reinterpret_cast<const float4*>(p.act + (long long)mc * p.ldact + nc));
            }
            uint32_t bits = 0u;
#pragma unroll
            for (int i = 0; i < 8; ++i)
              bits |= ((av[i].x > 0.f ? 1u : 0u) | (av[i].y > 0.f ? 2u : 0u) | (av[i].z > 0.f ? 4u : 0u) | (av[i].w > 0.f ? 8u : 0u)) << (4 * i);
            mbits[cb] = bits;
          }
        }
      }
      for (int g = 0; g < ngroups; ++g, ++gcount) {
        const int acc = gcount % kG2Parts;
        mbar_wait(&tfull[acc], (uint32_t)((gcount / kG2Parts) & 1));
        fence_after_sync();
        if (tid == 0) trace_stamp(p.trace, 5, gcount);
        const uint32_t part = tmem_base + lane_sel + (uint32_t)acc * kG2BN + (uint32_t)ch;
#pragma unroll
        for (int c = 0; c < 64; c += 32) {
          uint32_t a[32];
          tmem_ld32p(part + c, a);
          tmem_wait_ld();
          if (g == 0) {
#pragma unroll
            for (int j = 0; j < 32; ++j) run[c + j] = __uint_as_float(a[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) run[c + j] += __uint_as_float(a[j]);
          }
        }
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
        if (tid == 0) trace_stamp(p.trace, 6, gcount);
      }
      // ---- output pass (trace row 7, per tile and 32-column block: start, staged, stored)
      int otr = (int)((w - blockIdx.x) / gridDim.x) * 6;
#pragma unroll
      for (int c = 0; c < 64; c += 32) {
        if (n0 + c < p.N) {
          if (tid == 0) trace_stamp(p.trace, 7, otr++);
          if (!mask && !table) {
            // the block's 32 bias values: unconditional loads from clamped addresses, all in flight together (the warp's lanes read the
            // same words: broadcast).  Guarded float4 loads were one exposed L2 round trip per guard -- 8 k clocks per tile in the output
            // pass (scripts/gemm_trace.py 6300 630 64 fwd 3: fold end 3.7 k -> next fold start 11.8 k), hidden only when a tile is long
            float bv[32];
            if (p.bias) {
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                const int nb = n0 + c + e;
                const float b = __ldg(p.bias + (nb < p.N ? nb : p.N - 1));
                bv[e] = nb < p.N ? b : 0.f;           // columns >= N of a piece straddling N are stored: they must stay 0
              }
            } else {
#pragma unroll
              for (int e = 0; e < 32; ++e) bv[e] = 0.f;
            }
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
              float v0 = run[c + 4 * j4] + bv[4 * j4], v1 = run[c + 4 * j4 + 1] + bv[4 * j4 + 1], v2 = run[c + 4 * j4 + 2] + bv[4 * j4 + 2],
                    v3 = run[c + 4 * j4 + 3] + bv[4 * j4 + 3];
              if (p.relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f); }
              *reinterpret_cast<float4*>(stage + lane * 32 + 4 * (j4 ^ (lane & 7))) = make_float4(v0, v1, v2, v3);
            }
          } else {
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4)
              *reinterpret_cast<float4*>(stage + lane * 32 + 4 * (j4 ^ (lane & 7))) =
                  make_float4(run[c + 4 * j4], run[c + 4 * j4 + 1], run[c + 4 * j4 + 2], run[c + 4 * j4 + 3]);
          }
          __syncwarp();
          if (tid == 0) trace_stamp(p.trace, 7, otr++);
          const int n = n0 + c + 4 * piece;
          float4 tb[8];                                  // periodic bias table: the eight pieces of this thread, unconditional loads in flight together
          if (table) {
            const int ncl = n < p.N ? n : 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int m = m0 + 4 * i + sub, mc = m < p.M ? m : p.M - 1;
              tb[i] = __ldg(reinterpret_cast<const float4*>(p.bias + (long long)(mc % p.bias_period) * p.bias_ld + ncl));
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int R = 4 * i + sub, m = m0 + R;
            uint4 o = *reinterpret_cast<const uint4*>(stage + R * 32 + 4 * (piece ^ (R & 7)));
            // pieces straddling N end in the row's padding (ldc >= round_up(N, 4)): their columns >= N get zeros (the accumulator is
            // zero there -- B's rows >= N are TMA zero fill -- and so are the bias values selected for them)
            if (m < p.M && n < p.N) {
              if (mask) {
                const uint32_t mb = mbits[c >> 5] >> (4 * i);
                o.x = (mb & 1u) ? o.x : 0u; o.y = (mb & 2u) ? o.y : 0u; o.z = (mb & 4u) ? o.z : 0u; o.w = (mb & 8u) ? o.w : 0u;
              } else if (table) {                        // bias_ld >= round_up(N, 4) (g2_eligible): the piece is inside the padded table row,
                const float4 b4 = tb[i];                 // whose padding columns hold anything
                float v0 = __uint_as_float(o.x) + b4.x, v1 = __uint_as_float(o.y) + (n + 1 < p.N ? b4.y : 0.f),
                      v2 = __uint_as_float(o.z) + (n + 2 < p.N ? b4.z : 0.f), v3 = __uint_as_float(o.w) + (n + 3 < p.N ? b4.w : 0.f);
                if (p.relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f); }
                o = make_uint4(__float_as_uint(v0), __float_as_uint(v1), __float_as_uint(v2), __float_as_uint(v3));
              }
              *reinterpret_cast<uint4*>(p.C + (long long)m * p.ldc + n) = o;
            }
          }
          __syncwarp();
          if (tid == 0) trace_stamp(p.trace, 7, otr++);
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

static bool g2_eligible(const TcGemmParams& p) {
  if (p.passes != 3 || !p.B_lo || p.a_src != TCG_SRC_K || p.epi == TCG_EPI_ATOMIC || p.bits_out || p.mask_bits) return false;
  if (p.epi == TCG_EPI_BIAS_ACT && p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15) != 0) return false;
  if (p.epi == TCG_EPI_BIAS_ACT && p.bias && p.bias_period > 1 && ((p.bias_ld % 4) != 0 || p.bias_ld < (p.N + 3) / 4 * 4)) return false;   // 16-byte pieces inside the (padded) table row
  if (p.epi == TCG_EPI_MASK && p.act && ((reinterpret_cast<uintptr_t>(p.act) & 15) != 0 || (p.ldact % 4) != 0)) return false;
  const int N4 = (p.N + 3) / 4 * 4;                        // 16-byte pieces: a row's last piece may reach into its padding columns
  if (p.ldc < N4 || (p.ldc % 4) != 0 || (reinterpret_cast<uintptr_t>(p.C) & 15) != 0) return false;
  if (p.epi == TCG_EPI_MASK && p.act && p.ldact < N4) return false;
  if (p.M < 1024) return false;                            // small problems: the planned tiling of the engine above
  if (p.N >= 256 && p.K >= 128) return true;
  // layer 1 of a narrow DAG flow against the gate planes: a short reduction with a wide output (forward: two k-chunks per tile -- the
  // engine above spends 24 k clocks per tile in its transposing epilogue) and a long reduction with ONE narrow output tile (input cotangent)
  return (p.K >= 32 && p.K <= 64 && p.N >= 256) || (p.N >= 32 && p.N <= 64 && p.K >= 256);
}

// =====================================================================================================================
// Engine v2, weight gradient: dW[n, k] = sum_m dY[m, n] X[m, k] (3xTF32, split-K over m with atomic accumulation).  Both
// operands are activations, contiguous along the OUTPUT index (MN-major sources), so neither can be pre-split per call.
// The engine above turns both landed tiles into hi / lo tiles in shared memory with eight stager warps (4.4 k clocks per
// 32-m chunk at 6300 x 632 x 632 against 0.96 k of MMA time).  Here, per chunk:
//   * dY^T is the A operand and goes through registers into TMEM: thread = output row n = TMEM lane reads its column of the
//     landed [32 m][128 n] tile (conflict-free: a warp's 32 lanes read one 128-byte row per m), splits it and writes A_hi /
//     A_lo columns (tcgen05.st) into a four-deep ring; the MMAs are TS form;
//   * only X is split in shared memory, elementwise and in place (hi) + a lo tile, by two stager warps;
//   * a stage is raw dY (16 KB) + X hi (16 KB, TMA-loaded raw) + X lo (16 KB): 32 KB of L2 traffic per chunk instead of 36-40;
//   * partial accumulators are folded into a register running sum by eight epilogue warps (as in the forward engine), the
//     finished partial tile of a (tile, split) work item is added to dW with coalesced atomics through the staging blocks.
// TMEM columns: partials 0 / 128, A ring 256 (four buffers of hi 32 + lo 32).
// =====================================================================================================================
constexpr int kW2Threads = 16 * 32;              // 8 epilogue + 4 A-writer + 2 X-stager + MMA issuer + TMA producer warps
constexpr int kW2Ring = 4;
constexpr uint32_t kW2ColA = 256;

__global__ void __launch_bounds__(kW2Threads, 1) tc_wgrad2_kernel(TcGemmParams p, const __grid_constant__ CUtensorMap tmA,
                                                                  const __grid_constant__ CUtensorMap tmB) {
  using namespace tc;
  GNF_SMEM(char, smem);
  float* epi_stage = reinterpret_cast<float*>(smem + (size_t)kG2Stages * kG2StageBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_stage + 8 * kG2EpiStageFloats);
  uint64_t* landed = bars;                     // [stages] TMA -> A-writers / stagers (transaction bytes)
  uint64_t* empty = landed + kG2Stages;        // [stages] MMA -> producer (tcgen05.commit)
  uint64_t* b_full = empty + kG2Stages;        // [stages] X-stagers -> MMA (one arrive per stager warp)
  uint64_t* a_full = b_full + kG2Stages;       // [ring] A-writers -> MMA (one arrive per writer warp)
  uint64_t* a_empty = a_full + kW2Ring;        // [ring] MMA -> A-writers (tcgen05.commit)
  uint64_t* tfull = a_empty + kW2Ring;         // [2] MMA -> epilogue
  uint64_t* tempty = tfull + 2;                // [2] epilogue -> MMA (one arrive per epilogue warp)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) tmem_alloc(tmem_slot, 512);
  if (tid == 32) {
    for (int s = 0; s < kG2Stages; ++s) { mbar_init(&landed[s], 1); mbar_init(&empty[s], 1); mbar_init(&b_full[s], 2); }
    for (int b = 0; b < kW2Ring; ++b) { mbar_init(&a_full[b], 4); mbar_init(&a_empty[b], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 8); }
    fence_mbar_init();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();

  // GEMM view: rows = dW rows n (p.M of them), columns = dW columns k (p.N), reduction = the batch rows m (p.K)
  const int tiles_m = (p.M + kGemmBM - 1) / kGemmBM, tiles_n = (p.N + kG2BN - 1) / kG2BN;
  const int tiles = tiles_m * tiles_n;
  const int total = tiles * p.splits;
  const int fold = p.fold < 1 ? 1 : p.fold;
  auto item_chunks = [&](int w) {                                      // k-chunks of work item w = (tile, split)
    const int sp = w / tiles;
    const int kbeg = sp * p.k_per_split, kend = min(p.K, kbeg + p.k_per_split);
    return (kend - kbeg + kGemmKC - 1) / kGemmKC;
  };

  if (warp == 15) {
    // ===================== producer: raw dY tile (four 32-row slabs) + raw X tile =====================
    if (lane == 0) {
      int it = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const int t = w % tiles, sp = w / tiles, tm = t % tiles_m, tn = t / tiles_m;
        const int kbeg = sp * p.k_per_split, nch = item_chunks(w);
        for (int c = 0; c < nch; ++c, ++it) {
          const int s = it % kG2Stages, k0 = kbeg + c * kGemmKC;
          mbar_wait(&empty[s], (uint32_t)(((it / kG2Stages) & 1) ^ 1));
          char* st = smem + (size_t)s * kG2StageBytes;
          mbar_expect_tx(&landed[s], 2u * kG2TileBytes);
#pragma unroll
          for (int sl = 0; sl < 4; ++sl) {
            tma_load_2d(st + sl * 4096, &tmA, tm * kGemmBM + 32 * sl, k0, &landed[s]);
            tma_load_2d(st + kG2TileBytes + sl * 4096, &tmB, tn * kG2BN + 32 * sl, k0, &landed[s]);
          }
          trace_stamp(p.trace, 0, it);
        }
      }
    }
  } else if (warp == 14) {
    // ===================== MMA issuer (warp-converged) =====================
    const uint32_t idesc = make_idesc_tf32(kGemmBM, kG2BN) | (1u << 16);     // B MN-major
    int it = 0, gcount = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
      const int nch = item_chunks(w);
      for (int c0 = 0; c0 < nch; c0 += fold, ++gcount) {
        const int acc = gcount & 1;
        mbar_wait(&tempty[acc], (uint32_t)(((gcount >> 1) & 1) ^ 1));
        fence_after_sync();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * kG2BN;
        const int c1 = (c0 + fold < nch) ? c0 + fold : nch;
        uint32_t first = 0u;
        for (int c = c0; c < c1; ++c, ++it) {
          const int s = it % kG2Stages, b = it % kW2Ring;
          mbar_wait(&a_full[b], (uint32_t)((it / kW2Ring) & 1));
          mbar_wait(&b_full[s], (uint32_t)((it / kG2Stages) & 1));
          fence_after_sync();
          if (lane == 0) trace_stamp(p.trace, 3, it);
          const uint32_t st = smem_u32(smem + (size_t)s * kG2StageBytes);
          const uint64_t db_hi = make_sw128_desc(st + kG2TileBytes, true), db_lo = make_sw128_desc(st + 2 * kG2TileBytes, true);
          const uint32_t ta_hi = tmem_base + kW2ColA + (uint32_t)b * 64u, ta_lo = ta_hi + 32u;
#pragma unroll
          for (int ks = 0; ks < kGemmKC / 8; ++ks) {                          // correction products first (see tc_gemm2_kernel)
            mma_tf32_ts_w(d_tmem, ta_lo + ks * 8, db_hi + (uint64_t)(64u * ks), idesc, first);
            first = 1u;
            mma_tf32_ts_w(d_tmem, ta_hi + ks * 8, db_lo + (uint64_t)(64u * ks), idesc, 1u);
          }
#pragma unroll
          for (int ks = 0; ks < kGemmKC / 8; ++ks) mma_tf32_ts_w(d_tmem, ta_hi + ks * 8, db_hi + (uint64_t)(64u * ks), idesc, 1u);
          mma_commit_w(&empty[s]);
          mma_commit_w(&a_empty[b]);
        }
        mma_commit_w(&tfull[acc]);
        if (lane == 0) trace_stamp(p.trace, 4, gcount);
      }
    }
  } else if (warp >= 12) {
    // ===================== X-stagers: landed raw tile -> hi in place + lo tile (elementwise: the swizzled layout is kept) =====================
    const int ptid = tid - 12 * 32;
    int it = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
      const int nch = item_chunks(w);
      for (int c = 0; c < nch; ++c, ++it) {
        const int s = it % kG2Stages;
        mbar_wait(&landed[s], (uint32_t)((it / kG2Stages) & 1));
        char* hi = smem + (size_t)s * kG2StageBytes + kG2TileBytes;
#pragma unroll 4
        for (int i = 0; i < (int)(kG2TileBytes / 16) / 64; ++i) split_vec<4>(hi, hi + kG2TileBytes, (ptid + 64 * i) * 16);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&b_full[s]);
      }
    }
  } else if (warp >= 8) {
    // ===================== A-writers: column n of the landed dY tile -> TF32 hi / lo in registers -> TMEM ring =====================
    const int q = warp - 8;                                              // slab = TMEM lane quarter
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const uint32_t col_off = (uint32_t)(q * 4096) + (uint32_t)((lane & 3) << 2);
    const uint32_t g16 = (uint32_t)(lane >> 2);                          // 16-byte group of this lane inside a 128-byte row
    int it = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
      const int nch = item_chunks(w);
      // bias gradient for free: this thread sees every dY[m, n] of its output row n; the work items of the first tile column add
      // their share of db[n] = sum_m dY[m, n] (rows beyond the batch are TMA zero fill)
      const int t = w % tiles;
      const bool want_sum = p.rowsum != nullptr && t / tiles_m == 0;
      float bs0 = 0.f, bs1 = 0.f, bs2 = 0.f, bs3 = 0.f;
      for (int c = 0; c < nch; ++c, ++it) {
        const int s = it % kG2Stages, b = it % kW2Ring;
        mbar_wait(&landed[s], (uint32_t)((it / kG2Stages) & 1));
        if (tid == 256) trace_stamp(p.trace, 1, it);
        const char* base = smem + (size_t)s * kG2StageBytes + col_off;
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int kk = 0; kk < 32; ++kk) {                                // row kk of the slab: 32-byte atoms swizzled by (kk & 3)
          const uint32_t e = *reinterpret_cast<const uint32_t*>(base + kk * 128 + ((g16 ^ (uint32_t)((kk & 3) << 1)) << 4));
          const uint32_t h = (e + 0x1000u) & 0xffffe000u;
          hi[kk] = h;
          lo[kk] = __float_as_uint(__uint_as_float(e) - __uint_as_float(h)) + 0x1000u;   // the tensor core drops the low bits
          if ((kk & 3) == 0) bs0 += __uint_as_float(e);
          else if ((kk & 3) == 1) bs1 += __uint_as_float(e);
          else if ((kk & 3) == 2) bs2 += __uint_as_float(e);
          else bs3 += __uint_as_float(e);
        }
        mbar_wait(&a_empty[b], (uint32_t)(((it / kW2Ring) & 1) ^ 1));
        fence_after_sync();
        const uint32_t ta = tmem_base + lane_sel + kW2ColA + (uint32_t)b * 64u;
        tmem_st32p(ta, hi);
        tmem_st32p(ta + 32, lo);
        tmem_wait_st();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[b]);
        if (tid == 256) trace_stamp(p.trace, 2, it);
      }
      if (want_sum) {
        const int n = (t % tiles_m) * kGemmBM + q * 32 + lane;
        if (n < p.M) atomicAdd(p.rowsum + n, (bs0 + bs1) + (bs2 + bs3));
      }
    }
  } else {
    // ===================== epilogue: register running sum per work item, then coalesced atomics =====================
    const int quarter = warp & 3, half = warp >> 2, ch = 64 * half;
    const uint32_t lane_sel = (uint32_t)(quarter * 32) << 16;
    float* stage = epi_stage + warp * kG2EpiStageFloats;
    const int sub = lane >> 3, piece = lane & 7;
    int gcount = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
      const int t = w % tiles, tm = t % tiles_m, tn = t / tiles_m;
      const int n0 = tn * kG2BN + ch, m0 = tm * kGemmBM + quarter * 32;
      const int ngroups = (item_chunks(w) + fold - 1) / fold;
      float run[64];
      for (int g = 0; g < ngroups; ++g, ++gcount) {
        const int acc = gcount & 1;
        mbar_wait(&tfull[acc], (uint32_t)((gcount >> 1) & 1));
        fence_after_sync();
        if (tid == 0) trace_stamp(p.trace, 5, gcount);
        const uint32_t part = tmem_base + lane_sel + (uint32_t)acc * kG2BN + (uint32_t)ch;
#pragma unroll
        for (int c = 0; c < 64; c += 32) {
          uint32_t a[32];
          tmem_ld32p(part + c, a);
          tmem_wait_ld();
          if (g == 0) {
#pragma unroll
            for (int j = 0; j < 32; ++j) run[c + j] = __uint_as_float(a[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) run[c + j] += __uint_as_float(a[j]);
          }
        }
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[acc]);
        if (tid == 0) trace_stamp(p.trace, 6, gcount);
      }
      if (ngroups == 0) continue;
#pragma unroll
      for (int c = 0; c < 64; c += 32) {
        if (n0 + c < p.N) {
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4)
            *reinterpret_cast<float4*>(stage + lane * 32 + 4 * (j4 ^ (lane & 7))) =
                make_float4(run[c + 4 * j4], run[c + 4 * j4 + 1], run[c + 4 * j4 + 2], run[c + 4 * j4 + 3]);
          __syncwarp();
          const int n = n0 + c + 4 * piece;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int R = 4 * i + sub, m = m0 + R;
            const float4 o = *reinterpret_cast<const float4*>(stage + R * 32 + 4 * (piece ^ (R & 7)));
            if (m < p.M) {
              float* dst = p.C + (long long)m * p.ldc + n;
              if (n < p.N) atomicAdd(dst, o.x);
              if (n + 1 < p.N) atomicAdd(dst + 1, o.y);
              if (n + 2 < p.N) atomicAdd(dst + 2, o.z);
              if (n + 3 < p.N) atomicAdd(dst + 3, o.w);
            }
          }
          __syncwarp();
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

static bool w2_eligible(const TcGemmParams& p) {
  if (p.passes != 3 || p.epi != TCG_EPI_ATOMIC || p.a_src != TCG_SRC_MN || p.b_src != TCG_SRC_MN || p.B_lo) return false;
  if (p.M < 256 || p.K < 2048) return false;               // small problems: the planned tiling of the first engine
  return p.N >= 256 || (p.N >= 32 && p.N <= 64);           // ... or ONE narrow tile column (layer 1 of a narrow DAG flow against the gate plane)
}

// splits of the reduction for the weight-gradient engine: work items = tiles x splits over the persistent grid, cost of a round =
// its k-chunks + ~6 chunks' worth of fold / atomic epilogue
static int w2_plan_splits(int tiles, int kchunks) {
  int best = 1;
  double best_cost = -1.;
  const int max_sp = kchunks / 8 < 1 ? 1 : kchunks / 8;
  for (int sp = 1; sp <= max_sp && sp <= 64; ++sp) {
    const int per = (kchunks + sp - 1) / sp;
    if ((kchunks + per - 1) / per != sp) continue;
    const long long rounds = ((long long)tiles * sp + kNumSMs - 1) / kNumSMs;
    const double cost = (double)rounds * (per + 6.);
    if (best_cost < 0. || cost < best_cost * 0.999) { best_cost = cost; best = sp; }
  }
  return best;
}

int launch_tc_gemm(TcGemmParams p, cudaStream_t s) {
  if (p.M <= 0 || p.N <= 0) return 0;
  if (p.passes != 1 && p.passes != 3) return fail(GNF_ERR_INVALID, "tensor-core GEMM: passes must be 1 or 3");
  // 3xTF32: two partial accumulators + the round-to-nearest running sum must fit the 512 TMEM columns (3 x 160);
  // single-pass TF32: two accumulators of up to 256 columns, no folding
  int plan_splits = 1;
  plan_tiles(p.M, p.N, p.K, p.passes == 3 ? 160 : 256, p.epi == TCG_EPI_ATOMIC, &p.BN, &plan_splits);
  p.acc_stride = p.passes == 3 ? 160 : 256;
  p.fold = p.passes == 3 ? g_tc_gemm_fold : (1 << 20);
  // every candidate is a multiple of 32: K-major fills advance 8/16/32 rows per pass, MN-major tiles are 32-row slabs
  const uint32_t stage_bytes = (uint32_t)(kGemmBM + p.BN) * 128u * (p.passes == 3 ? 2u : 1u);
  const size_t fixed = kEpiStageBytes + (3 * kMaxStages + 4) * sizeof(uint64_t) + 16;
  int stages = (int)((kSmemBudget - fixed) / stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  if (stages < 2) return fail(GNF_ERR_UNSUPPORTED, "tensor-core GEMM: tile does not fit shared memory");
  p.stages = stages;
  const int tiles = ((p.M + kGemmBM - 1) / kGemmBM) * ((p.N + p.BN - 1) / p.BN);
  const int splits = plan_splits;
  const int kchunks = (p.K + kGemmKC - 1) / kGemmKC;
  p.k_per_split = ((kchunks + splits - 1) / splits) * kGemmKC;
  p.splits = (p.K + p.k_per_split - 1) / p.k_per_split;
  if (p.splits < 1) p.splits = 1;
  p.c_vec = ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0 && (p.ldc % 4) == 0) ? 1 : 0;
  p.act_vec = (p.act && (reinterpret_cast<uintptr_t>(p.act) & 15) == 0 && (p.ldact % 4) == 0) ? 1 : 0;
  p.bias_vec = (p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0 && (p.bias_ld % 4) == 0) ? 1 : 0;
  CUtensorMap tmA, tmB, tmBlo;
  memset(&tmA, 0, sizeof(tmA));
  memset(&tmB, 0, sizeof(tmB));
  memset(&tmBlo, 0, sizeof(tmBlo));
  p.use_tma = (g_tc_gemm_tma && make_operand_map(&tmA, p.A, p.lda, p.a_src, p.M, p.K, kGemmBM) &&
               make_operand_map(&tmB, p.B, p.ldb, p.b_src, p.N, p.K, p.BN)) ? 1 : 0;
  if (p.passes != 3) p.B_lo = nullptr;
  if (p.B_lo && !(p.use_tma && make_operand_map(&tmBlo, p.B_lo, p.ldb, p.b_src, p.N, p.K, p.BN)))
    return fail(GNF_ERR_UNSUPPORTED, "tensor-core GEMM: pre-split weights need TMA-loadable operands (16-byte aligned rows)");
  if (g_tc_gemm_v2 && p.use_tma && w2_eligible(p)) {
    // engine v2, weight gradient: BN = 128, its own split plan (MN-major maps have 32 x 32 boxes whatever the tile width)
    p.BN = kG2BN;
    const int tiles2 = ((p.M + kGemmBM - 1) / kGemmBM) * ((p.N + kG2BN - 1) / kG2BN);
    const int sp2 = g_tc_gemm_force_splits ? g_tc_gemm_force_splits : w2_plan_splits(tiles2, kchunks);
    p.k_per_split = ((kchunks + sp2 - 1) / sp2) * kGemmKC;
    p.splits = (p.K + p.k_per_split - 1) / p.k_per_split;
    p.fold = g_tc_gemm_fold;
    p.trace = g_tc_gemm_trace;
    const size_t smem2 = (size_t)kG2Stages * kG2StageBytes + 8 * kG2EpiStageFloats * sizeof(float) + (3 * kG2Stages + 2 * kW2Ring + 4) * sizeof(uint64_t) + 16;
    const long long total2 = (long long)tiles2 * p.splits;
    cudaFuncSetAttribute(tc_wgrad2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
    GNF_LAUNCH_PDL(tc_wgrad2_kernel, (int)(total2 < kNumSMs ? total2 : kNumSMs), kW2Threads, smem2, s, p, tmA, tmB);
    return 0;
  }
  if (p.rowsum) {      // only the kernel above sums the rows of A on its way: shapes of the first engine take the column-sum kernel (overwrites)
    if (int e = gnf_colsum(p.A, (int)p.lda, p.rowsum, p.K, p.M, 1, (gnf_stream_t)s)) return e;
    p.rowsum = nullptr;
  }
  if (g_tc_gemm_v2 && p.use_tma && g2_eligible(p)) {
    // engine v2: BN = 128, A through registers into TMEM (the maps of A and of the pre-split B built above already have the
    // right boxes when the plan chose BN = 128; rebuild B's for that width otherwise)
    if (p.BN != kG2BN && !(make_operand_map(&tmB, p.B, p.ldb, p.b_src, p.N, p.K, kG2BN) && make_operand_map(&tmBlo, p.B_lo, p.ldb, p.b_src, p.N, p.K, kG2BN)))
      return fail(GNF_ERR_UNSUPPORTED, "tensor-core GEMM v2: operand maps");
    p.BN = kG2BN;
    p.fold = (!g_tc_gemm_fold_forced && p.epi == TCG_EPI_BIAS_ACT && p.bias && p.bias_period > 1) ? 1 : g_tc_gemm_fold2;
    p.trace = g_tc_gemm_trace;
    const size_t smem2 = (size_t)kG2Stages * kG2StageBytes + 8 * kG2EpiStageFloats * sizeof(float) +
                         (2 * kG2Stages + 2 * kG2Ring + 2 * kG2Parts) * sizeof(uint64_t) + 16;
    const int total2 = ((p.M + kGemmBM - 1) / kGemmBM) * ((p.N + kG2BN - 1) / kG2BN);
    const int grid2 = total2 < kNumSMs ? total2 : kNumSMs;
    cudaFuncSetAttribute(tc_gemm2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);
    GNF_LAUNCH_PDL(tc_gemm2_kernel, grid2, kG2Threads, smem2, s, p, tmA, tmB, tmBlo);
    return 0;
  }
  p.trace = g_tc_gemm_trace;
  const long long total = (long long)tiles * p.splits;
  const size_t smem = (size_t)stages * stage_bytes + fixed;
  // per launch: the attribute is per DEVICE, a process-wide "done" flag breaks the second GPU of a process (and is racy)
  cudaFuncSetAttribute(tc_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget);
  const int grid = (int)(total < kNumSMs ? total : kNumSMs);
  GNF_LAUNCH_PDL(tc_gemm_kernel, grid, kGemmThreads, smem, s, p, vec_width(p.A, p.lda), vec_width(p.B, p.ldb), tmA, tmB, tmBlo);
  return 0;
}

}  // namespace gnf
using namespace gnf;
#endif

extern "C" {

int gnf_linear_fwd_tc(const float* X, int ldx, const float* W, int ldw, const float* bias, int bias_period, float* Y, int ldy,
                      int M, int N, int K, int relu, int passes, gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!X || !W || !Y || M < 0 || N <= 0 || K <= 0 || ldx < K || ldw < K || ldy < N) return fail(GNF_ERR_INVALID, "gnf_linear_fwd_tc: bad arguments");
  TcGemmParams p = {};
  p.A = X; p.lda = ldx; p.a_src = TCG_SRC_K;
  p.B = W; p.ldb = ldw; p.b_src = TCG_SRC_K;
  p.M = M; p.N = N; p.K = K; p.passes = passes;
  p.epi = TCG_EPI_BIAS_ACT; p.C = Y; p.ldc = ldy; p.bias = bias; p.bias_ld = N; p.bias_period = bias_period < 1 ? 1 : bias_period; p.relu = relu;
  if (int e = launch_tc_gemm(p, (cudaStream_t)stream)) return e;
  return check_launch("gnf_linear_fwd_tc");
#endif
}

int gnf_linear_dgrad_tc(const float* dY, int lddy, const float* W, int ldw, const float* act, int ldact, float* dX, int lddx,
                        int M, int N, int K, int passes, gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!dY || !W || !dX || M < 0 || N <= 0 || K <= 0 || lddy < N || ldw < K || lddx < K) return fail(GNF_ERR_INVALID, "gnf_linear_dgrad_tc: bad arguments");
  TcGemmParams p = {};
  p.A = dY; p.lda = lddy; p.a_src = TCG_SRC_K;         // A(m, n): reduction over n, contiguous
  p.B = W; p.ldb = ldw; p.b_src = TCG_SRC_MN;          // B(k_out, n) = W[n*ldw + k_out]: contiguous along the output index
  p.M = M; p.N = K; p.K = N; p.passes = passes;
  p.epi = TCG_EPI_MASK; p.C = dX; p.ldc = lddx; p.act = act; p.ldact = ldact;
  if (int e = launch_tc_gemm(p, (cudaStream_t)stream)) return e;
  return check_launch("gnf_linear_dgrad_tc");
#endif
}

int gnf_split_tf32(const float* W, int ldw, float* hi, float* lo, int ld, int N, int K, gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!W || !hi || !lo || N <= 0 || K <= 0 || ldw < K || ld < K) return fail(GNF_ERR_INVALID, "gnf_split_tf32: bad arguments");
  long long blocks = ((long long)N * ld + 255) / 256;
  if (blocks > 4 * kNumSMs) blocks = 4 * kNumSMs;
  GNF_LAUNCH(split_tf32_kernel, (int)blocks, 256, 0, (cudaStream_t)stream, W, (long long)ldw, hi, lo, ld, N, K);
  return check_launch("gnf_split_tf32");
#endif
}

int gnf_linear_fwd_tc_ps(const float* X, int ldx, const float* W_hi, const float* W_lo, int ldw, const float* bias, int bias_period, float* Y,
                         int ldy, int M, int N, int K, int relu, gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!X || !W_hi || !W_lo || !Y || M < 0 || N <= 0 || K <= 0 || ldx < K || ldw < K || ldy < N) return fail(GNF_ERR_INVALID, "gnf_linear_fwd_tc_ps: bad arguments");
  TcGemmParams p = {};
  p.A = X; p.lda = ldx; p.a_src = TCG_SRC_K;
  p.B = W_hi; p.B_lo = W_lo; p.ldb = ldw; p.b_src = TCG_SRC_K;
  p.M = M; p.N = N; p.K = K; p.passes = 3;
  p.epi = TCG_EPI_BIAS_ACT; p.C = Y; p.ldc = ldy; p.bias = bias; p.bias_ld = N; p.bias_period = bias_period < 1 ? 1 : bias_period; p.relu = relu;
  if (int e = launch_tc_gemm(p, (cudaStream_t)stream)) return e;
  return check_launch("gnf_linear_fwd_tc_ps");
#endif
}

int gnf_linear_fwd_tc_ps_tb(const float* X, int ldx, const float* W_hi, const float* W_lo, int ldw, const float* table, int ldt, int period, float* Y,
                            int ldy, int M, int N, int K, int relu, gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!X || !W_hi || !W_lo || !Y || !table || M < 0 || N <= 0 || K <= 0 || ldx < K || ldw < K || ldy < N || ldt < N || period < 1) return fail(GNF_ERR_INVALID, "gnf_linear_fwd_tc_ps_tb: bad arguments");
  TcGemmParams p = {};
  p.A = X; p.lda = ldx; p.a_src = TCG_SRC_K;
  p.B = W_hi; p.B_lo = W_lo; p.ldb = ldw; p.b_src = TCG_SRC_K;
  p.M = M; p.N = N; p.K = K; p.passes = 3;
  p.epi = TCG_EPI_BIAS_ACT; p.C = Y; p.ldc = ldy; p.bias = table; p.bias_ld = ldt; p.bias_period = period; p.relu = relu;
  if (int e = launch_tc_gemm(p, (cudaStream_t)stream)) return e;
  return check_launch("gnf_linear_fwd_tc_ps_tb");
#endif
}

int gnf_linear_dgrad_tc_ps(const float* dY, int lddy, const float* W_hi, const float* W_lo, int ldw, const float* act, int ldact, float* dX,
                           int lddx, int M, int N, int K, gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!dY || !W_hi || !W_lo || !dX || M < 0 || N <= 0 || K <= 0 || lddy < N || ldw < K || lddx < K) return fail(GNF_ERR_INVALID, "gnf_linear_dgrad_tc_ps: bad arguments");
  TcGemmParams p = {};
  p.A = dY; p.lda = lddy; p.a_src = TCG_SRC_K;
  p.B = W_hi; p.B_lo = W_lo; p.ldb = ldw; p.b_src = TCG_SRC_MN;
  p.M = M; p.N = K; p.K = N; p.passes = 3;
  p.epi = TCG_EPI_MASK; p.C = dX; p.ldc = lddx; p.act = act; p.ldact = ldact;
  if (int e = launch_tc_gemm(p, (cudaStream_t)stream)) return e;
  return check_launch("gnf_linear_dgrad_tc_ps");
#endif
}

#ifdef GNF_DEVTOOLS
int gnf_tc_gemm_set_trace(long long* buf) {
#ifdef GNF_EMU
  (void)buf;
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  g_tc_gemm_trace = buf;
  return 0;
#endif
}
#endif

#ifdef GNF_DEVTOOLS
int gnf_tc_gemm_set_fold(int chunks) {
#ifdef GNF_EMU
  (void)chunks;
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (chunks < 1) return fail(GNF_ERR_INVALID, "gnf_tc_gemm_set_fold: need >= 1 k-chunk per fold");
  g_tc_gemm_fold = chunks > (1 << 20) ? (1 << 20) : chunks;
  g_tc_gemm_fold2 = g_tc_gemm_fold;
  g_tc_gemm_fold_forced = true;
  return 0;
#endif
}
#endif

#ifdef GNF_DEVTOOLS
int gnf_tc_gemm_set_tile(int bn, int splits) {
#ifdef GNF_EMU
  (void)bn; (void)splits;
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (bn != 0 && (bn < 64 || bn > 256 || bn % 32 != 0)) return fail(GNF_ERR_INVALID, "gnf_tc_gemm_set_tile: tile width must be 0 (planned) or 64, 96, ... 256");
  if (splits < 0) return fail(GNF_ERR_INVALID, "gnf_tc_gemm_set_tile: splits must be >= 0 (0 = planned)");
  g_tc_gemm_force_bn = bn;
  g_tc_gemm_force_splits = splits;
  return 0;
#endif
}
#endif

int gnf_tc_gemm_plan(int M, int N, int K, int passes, int wgrad, int* bn, int* splits) {
#ifdef GNF_EMU
  (void)M; (void)N; (void)K; (void)passes; (void)wgrad; (void)bn; (void)splits;
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (M <= 0 || N <= 0 || K <= 0 || !bn || !splits || (passes != 1 && passes != 3)) return fail(GNF_ERR_INVALID, "gnf_tc_gemm_plan: bad arguments");
  plan_tiles(M, N, K, passes == 3 ? 160 : 256, wgrad != 0, bn, splits);
  return 0;
#endif
}

#ifdef GNF_DEVTOOLS
int gnf_tc_gemm_set_v2(int enable) {
  if (enable != 0 && enable != 1) return gnf::fail(GNF_ERR_INVALID, "gnf_tc_gemm_set_v2: 0 (first engine) or 1 (engine v2)");
#ifndef GNF_EMU
  gnf::g_tc_gemm_v2 = enable;
#else
  (void)enable;
#endif
  return 0;
}
#endif
#ifdef GNF_DEVTOOLS
int gnf_tc_gemm_set_tma(int enable) {
#ifdef GNF_EMU
  (void)enable;
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  g_tc_gemm_tma = enable != 0;
  return 0;
#endif
}
#endif

int gnf_linear_wgrad_tc(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, int M, int N, int K, int passes,
                        gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!dY || !X || !dW || M < 0 || N <= 0 || K <= 0 || lddy < N || ldx < K || lddw < K) return fail(GNF_ERR_INVALID, "gnf_linear_wgrad_tc: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  if (lddw == K) cudaMemsetAsync(dW, 0, (size_t)N * K * sizeof(float), s);
  else cudaMemset2DAsync(dW, (size_t)lddw * sizeof(float), 0, (size_t)K * sizeof(float), (size_t)N, s);
  if (M == 0) return check_launch("gnf_linear_wgrad_tc");
  TcGemmParams p = {};
  p.A = dY; p.lda = lddy; p.a_src = TCG_SRC_MN;        // A(n, m) = dY[m*lddy + n]: contiguous along the output row index
  p.B = X; p.ldb = ldx; p.b_src = TCG_SRC_MN;          // B(k, m) = X[m*ldx + k]
  p.M = N; p.N = K; p.K = M; p.passes = passes;
  p.epi = TCG_EPI_ATOMIC; p.C = dW; p.ldc = lddw;
  if (int e = launch_tc_gemm(p, s)) return e;
  return check_launch("gnf_linear_wgrad_tc");
#endif
}

int gnf_linear_wgrad_bias_tc(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, float* db, int M, int N, int K,
                             gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!dY || !X || !dW || !db || M < 0 || N <= 0 || K <= 0 || lddy < N || ldx < K || lddw < K) return fail(GNF_ERR_INVALID, "gnf_linear_wgrad_bias_tc: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  TcGemmParams p = {};
  p.A = dY; p.lda = lddy; p.a_src = TCG_SRC_MN;
  p.B = X; p.ldb = ldx; p.b_src = TCG_SRC_MN;
  p.M = N; p.N = K; p.K = M; p.passes = 3;
  p.epi = TCG_EPI_ATOMIC; p.C = dW; p.ldc = lddw;
  if (M == 0) {
    if (int e = gnf_colsum(dY, lddy, db, M, N, 1, stream)) return e;
    return gnf_linear_wgrad_tc(dY, lddy, X, ldx, dW, lddw, M, N, K, 3, stream);
  }
  if (lddw == K) {
    ZeroList zl;
    zl.add(dW, (size_t)N * K);
    zl.add(db, (size_t)N);
    zero_many(zl, s);
  } else {
    cudaMemset2DAsync(dW, (size_t)lddw * sizeof(float), 0, (size_t)K * sizeof(float), (size_t)N, s);
    cudaMemsetAsync(db, 0, (size_t)N * sizeof(float), s);
  }
  p.rowsum = db;
  if (int e = launch_tc_gemm(p, s)) return e;
  return check_launch("gnf_linear_wgrad_bias_tc");
#endif
}

}  // extern "C"
