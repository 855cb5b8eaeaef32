// K3, strict (3xTF32 = fp32-equivalent) and fused on the 5th-generation tensor cores: the whole Clenshaw-Curtis UMNN
// integral of MonotonicNormalizer.forward (models/Normalizers/MonotonicNormalizer.py:51-66; UMNN==1.0
// ParallelNeuralIntegral forward, SURVEY.md App. B) in ONE kernel -- the training-mode forward of the integrand
// network over all (row, quadrature node) pairs, with no activation round trip through HBM between the layers.
//
// Why not the resident-weight scheme of tc_umnn.cu (single-pass TF32): 3xTF32 needs the hi AND lo image of every hidden
// layer (2 x 96 KB per 150x150 layer), two layers do not fit 227 KB of shared memory.  So the weights STREAM: the
// hi/lo images are packed once per call in K-chunks of 32 (40 KB per chunk at NP = 160), every CTA pulls them through
// a 4-stage shared-memory ring with bulk async copies (all 148 CTAs read the same 0.4 MB, which lives in L2), and the
// activation chain stays on chip:
//   * thread pair (t, t+128) owns tile row t = TMEM lane t (even / odd 32-column blocks): layer-1 activations
//     a1 = relu(t_q W0[:,0] + P[r]) (P = h W0[:,1:]^T + b0, once per row r) are generated in registers, split into
//     TF32 hi / lo (round to nearest) and written to TMEM columns [0,NP) / [NP,2NP) -- the A operand (TS form);
//   * one issuer thread runs, per streamed chunk, a_lo*b_hi, a_hi*b_lo, a_hi*b_hi into the accumulator in TMEM columns
//     [2NP,3NP) and releases the ring stage with tcgen05.commit; (order = 1: all correction products of a layer first,
//     then the a_hi*b_hi chain, streaming the hi images twice);
//   * the epilogue drains the accumulator (tcgen05.ld), adds the bias, applies ReLU and rewrites the A region for the
//     next layer; after the last hidden layer it takes the output Linear as a dot product, ELU + 1.05, the CC
//     weighting and the per-row segment reduction, emitting z, jac, logdet (+ zrev).
// Training keeps what the backward (gnf_umnn_bwd_tc3) consumes, in the layer-wise engine's layout: the activation planes,
// the pre-ELU outputs and the ReLU bit masks, written with full 128-byte lines through a per-warp XOR-swizzled staging
// block (row-owner global stores are poison: DESIGN §4, "What the measurements said").
#include "tc_common.cuh"

#ifndef GNF_EMU
namespace gnf {

constexpr int kU3Rows = 128;
constexpr int kU3Stages = 4;
constexpr int kU3StageBlock = 32 * 16;              // floats of one warp's transposition block (a 32 x 32 block goes in two passes)
constexpr int kU3PRows = 12;                        // rows of P staged per tile (a 128-node-row tile spans <= 127/nodes + 2 rows)
constexpr int kU3MaxNodes = 256;                    // quadrature nodes + weights staged in shared memory

__device__ __forceinline__ uint32_t u3_rn_tf32(uint32_t u) { return (u + 0x1000u) & 0xffffe000u; }
__device__ __forceinline__ void u3_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}

struct U3Plan {
  int L, NP, E, N1;
  int kp[GNF_MAX_LAYERS], nch[GNF_MAX_LAYERS];     // hidden GEMM layers l = 1..L-1: K padded to 8, number of 32-k chunks
  size_t off_img[GNF_MAX_LAYERS];                  // float offset of layer l's chunk sequence inside the image
  size_t chunk_floats, off_tail, image_floats, off_P, total_floats;
};

static int u3_plan(const gnf_mlp_t* net, int R, U3Plan* pl) {
  if (!net || net->n_layers < 3 || net->n_layers > GNF_MAX_LAYERS) return fail(GNF_ERR_UNSUPPORTED, "umnn tc3: integrand needs 3..%d linear layers", GNF_MAX_LAYERS);
  if (net->dims[net->n_layers] != 1) return fail(GNF_ERR_UNSUPPORTED, "umnn tc3: integrand output size must be 1");
  if (net->dims[0] < 2) return fail(GNF_ERR_UNSUPPORTED, "umnn tc3: needs at least one conditioning feature");
  const int L = net->n_layers - 1;
  int maxh = 0;
  for (int l = 1; l <= L; ++l) maxh = net->dims[l] > maxh ? net->dims[l] : maxh;
  const int NP = (maxh + 31) / 32 * 32;
  if (NP > 160) return fail(GNF_ERR_UNSUPPORTED, "umnn tc3: hidden width %d > 160 (A_hi + A_lo + D must fit 512 TMEM columns)", maxh);
  pl->L = L; pl->NP = NP; pl->E = net->dims[0] - 1; pl->N1 = net->dims[1];
  pl->chunk_floats = (size_t)2 * 8 * NP * 4;
  size_t off = 0;
  for (int l = 0; l < GNF_MAX_LAYERS; ++l) { pl->kp[l] = 0; pl->nch[l] = 0; pl->off_img[l] = 0; }
  for (int l = 1; l < L; ++l) {
    pl->kp[l] = (net->dims[l] + 7) / 8 * 8;
    pl->nch[l] = (pl->kp[l] + 31) / 32;
    pl->off_img[l] = off;
    off += (size_t)pl->nch[l] * pl->chunk_floats;
  }
  pl->off_tail = off;
  off += (size_t)(L + 1) * NP;                     // bias of layers 1..L-1, w_L, W0[:,0]
  pl->image_floats = off;
  pl->off_P = (off + 3) / 4 * 4;
  pl->total_floats = pl->off_P + (size_t)(R > 0 ? R : 0) * NP;
  return 0;
}

struct U3PackArgs {
  const float* W[GNF_MAX_LAYERS];
  const float* b[GNF_MAX_LAYERS];
  int dims[GNF_MAX_LAYERS + 1], nch[GNF_MAX_LAYERS];
  unsigned off_img[GNF_MAX_LAYERS], chunk_floats, off_tail, total;
  int L, NP;
};

// chunk c of layer l: [hi: (k/4 within the chunk)][n][k%4], then the same for lo  (UMMA canonical K-major, no swizzle)
__global__ void u3_pack_kernel(U3PackArgs a, float* __restrict__ img) {
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < a.total; i += gridDim.x * blockDim.x) {
    float out = 0.f;
    if (i >= a.off_tail) {
      const int e = (int)(i - a.off_tail), j = e / a.NP, n = e % a.NP;
      if (j < a.L - 1) { if (n < a.dims[j + 2]) out = a.b[j + 1][n]; }                       // bias of hidden GEMM layer j+1
      else if (j == a.L - 1) { if (n < a.dims[a.L]) out = a.W[a.L][n]; }                     // output Linear [1, dims[L]]
      else { if (n < a.dims[1]) out = a.W[0][(size_t)n * a.dims[0]]; }                       // W0[:, 0]
    } else {
      int l = 1;
      while (l + 1 < a.L && i >= a.off_img[l + 1]) ++l;
      const unsigned e = i - a.off_img[l];
      const unsigned c = e / a.chunk_floats, e2 = e % a.chunk_floats;
      const unsigned half = 8u * a.NP * 4u;
      const unsigned part = e2 / half, e3 = e2 % half;
      const int k4 = (int)(e3 / (a.NP * 4u)), n = (int)((e3 / 4u) % a.NP), kk = (int)(e3 % 4u);
      const int k = (int)c * 32 + k4 * 4 + kk;
      float v = 0.f;
      if (n < a.dims[l + 1] && k < a.dims[l]) v = a.W[l][(size_t)n * a.dims[l] + k];
      const float hi = __uint_as_float(u3_rn_tf32(__float_as_uint(v)));
      out = part ? __uint_as_float(u3_rn_tf32(__float_as_uint(v - hi))) : hi;
    }
    img[i] = out;
  }
}

struct U3Params {
  const float *x, *h, *ccw, *ccn, *P, *image, *blast;
  float *z, *zrev, *jac, *logdet, *saved;
  int R, d, E, S, nodes, L, N1, train, order, p_smem, debug;
  long long Q;
  int kp[GNF_MAX_LAYERS], nch[GNF_MAX_LAYERS];
  unsigned off_img[GNF_MAX_LAYERS], off_tail, chunk_floats;
  long long* trace;
};

#ifdef GNF_DEVTOOLS
#define U3_STAMP(row) do { if (tr_on && tr_n < 256) p.trace[(row) * 256 + tr_n++] = clock64(); } while (0)
#else
#define U3_STAMP(row) do { } while (0)
#endif

template <int NB>
__global__ void __launch_bounds__((4 * NB + 2) * 32, 1) umnn_fwd_tc3_kernel(U3Params p) {
  using namespace tc;
  constexpr int NP = NB * 32;
  constexpr int EW = 4 * NB;                                    // epilogue warps: one per (TMEM lane quarter, 32-column block)
  constexpr int NT = (EW + 2) * 32;
  constexpr uint32_t kChunkBytes = 2u * 8u * NP * 16u;          // hi + lo image of one 32-k chunk
  constexpr uint32_t kHalfBytes = 8u * NP * 16u;
  GNF_SMEM(float, smem);
  float* ring = smem;                                           // [kU3Stages][chunk]
  float* tail = ring + (size_t)kU3Stages * (kChunkBytes / 4);   // bias[L-1][NP], w_L[NP], w0col[NP]
  float* stage_all = tail + (GNF_MAX_LAYERS + 1) * NP;          // [EW][32 x 16] transposition blocks
  float* pbuf = stage_all + EW * kU3StageBlock;                 // [2][kU3PRows][NP]: the tile's rows of P
  float* ypart = pbuf + 2 * kU3PRows * NP;                      // [NB][128]
  float* red = ypart + NB * kU3Rows;                            // [128]
  float* ccs = red + kU3Rows;                                   // ccn[S+1], ccw[S+1] (padded to kU3MaxNodes each)
  uint64_t* bars = reinterpret_cast<uint64_t*>(ccs + 2 * kU3MaxNodes);
  uint64_t* w_full = bars;                   // [stages] chunk landed (expect_tx)
  uint64_t* w_empty = w_full + kU3Stages;    // [stages] chunk's MMAs done (tcgen05.commit)
  uint64_t* a_full = w_empty + kU3Stages;    // [NB] epilogue -> issuer: A columns of k-chunk c staged (4 quarter warps)
  uint64_t* a_free = a_full + NB;            // [NB] issuer -> generator: last layer's MMAs are done with k-chunk c (commit)
  uint64_t* d_full = a_free + NB;            // issuer -> epilogue: layer's MMAs done
  uint64_t* d_empty = d_full + 1;            // epilogue -> issuer: accumulator drained into registers
  uint64_t* p_full = d_empty + 1;            // [2] P rows of a tile landed
  uint64_t* p_empty = p_full + 2;            // [2] generator warps are done with them
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p_empty + 2);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) tmem_alloc(tmem_slot, 512);
  if (tid == 32) {
    for (int s = 0; s < kU3Stages; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
    for (int c = 0; c < NB; ++c) { mbar_init(&a_full[c], 4); mbar_init(&a_free[c], 1); }
    mbar_init(d_full, 1);
    mbar_init(d_empty, EW);
    for (int b = 0; b < 2; ++b) { mbar_init(&p_full[b], 1); mbar_init(&p_empty[b], EW); }
    fence_mbar_init();
  }
  pdl_prologue_done();                // the weight image read next comes from the previous kernel of the stream (u3_pack_kernel)
  for (int i = tid; i < (p.L + 1) * NP; i += NT) tail[i] = __ldg(p.image + p.off_tail + i);
  for (int i = tid; i <= p.S; i += NT) { ccs[i] = __ldg(p.ccn + i); ccs[kU3MaxNodes + i] = __ldg(p.ccw + i); }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int Q = (int)p.Q, nodes = p.nodes;
  const int ntiles = (Q + kU3Rows - 1) / kU3Rows;
  const int n_local = (ntiles > (int)blockIdx.x) ? (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int L = p.L;
#ifdef GNF_DEVTOOLS
  int tr_n = 0;
  const bool tr_on = p.trace != nullptr && blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 4 * (NB - 1) || warp >= EW);
#endif

  if (warp == EW + 1) {
    // ===================== producer (one thread): weight chunks + the tiles' rows of P =====================
    if (lane == 0) {
      auto issue_P = [&](int tl) {                               // rows r_first..r_last of P -> pbuf[tl & 1]: one contiguous copy
        const int q0 = ((int)blockIdx.x + tl * (int)gridDim.x) * kU3Rows;
        const int q1 = (q0 + kU3Rows - 1 < Q - 1) ? q0 + kU3Rows - 1 : Q - 1;
        const int r0 = q0 / nodes, r1 = q1 / nodes;
        const uint32_t bytes = (uint32_t)(r1 - r0 + 1) * NP * 4u;
        const int b = tl & 1;
        if (tl >= 2) mbar_wait(&p_empty[b], (uint32_t)(((tl >> 1) - 1) & 1));
        mbar_expect_tx(&p_full[b], bytes);
        bulk_g2s(pbuf + (size_t)b * kU3PRows * NP, p.P + (size_t)r0 * NP, bytes, &p_full[b]);
      };
      if (p.p_smem && n_local > 0) issue_P(0);
      int g = 0;
      for (int tl = 0; tl < n_local; ++tl) {
        if (p.p_smem && tl + 1 < n_local) issue_P(tl + 1);
        for (int l = 1; l < L; ++l) {
          const int nch = p.nch[l], nseq = p.order ? 2 * nch : nch, nk = p.kp[l] / 8;
          const char* src0 = reinterpret_cast<const char*>(p.image + p.off_img[l]);
          for (int i = 0; i < nseq; ++i, ++g) {
            const int c = i < nch ? i : i - nch;
            const bool want_lo = !(p.order && i >= nch);
            const int ks = (nk - c * 4 < 4) ? nk - c * 4 : 4;                  // k-steps of this chunk
            const uint32_t bytes = (uint32_t)ks * 2u * NP * 16u;
            const int s = g % kU3Stages;
            if (g >= kU3Stages) mbar_wait(&w_empty[s], (uint32_t)(((g / kU3Stages) - 1) & 1));
            char* dst = reinterpret_cast<char*>(ring) + (size_t)s * kChunkBytes;
            const char* src = src0 + (size_t)c * kChunkBytes;
            mbar_expect_tx(&w_full[s], want_lo ? 2u * bytes : bytes);
            bulk_g2s(dst, src, bytes, &w_full[s]);
            if (want_lo) bulk_g2s(dst + kHalfBytes, src + kHalfBytes, bytes, &w_full[s]);
            U3_STAMP(2);
          }
        }
      }
    }
  } else if (warp == EW) {
    // ===================== MMA issuer: the whole warp runs the loop converged, one elected lane issues =====================
    constexpr uint32_t idesc = make_idesc_tf32(kU3Rows, NP);
    constexpr uint32_t dstep = (2u * NP * 16u) >> 4;                           // one k-step = two 16-byte K groups of the image
    const uint32_t tAhi = tmem_base, tAlo = tmem_base + NP, tD = tmem_base + 2 * NP;
    const uint32_t ring_addr = smem_u32(ring);
    int g = 0, it = 0;
    for (int tl = 0; tl < n_local; ++tl)
      for (int l = 1; l < L; ++l, ++it) {
        const int nch = p.nch[l], nseq = p.order ? 2 * nch : nch, nk = p.kp[l] / 8;
        const bool release_a = (l == L - 1) && (tl + 1 < n_local);            // the next tile's layer 1 is generated under this layer's MMAs
        if (it > 0) mbar_wait(d_empty, (uint32_t)((it - 1) & 1));
        U3_STAMP(0);
        uint32_t acc = 0u;
        for (int i = 0; i < nseq; ++i, ++g) {
          const int c = i < nch ? i : i - nch;
          const int kind = p.order ? (i < nch ? 0 : 1) : 2;                    // 0 corrections, 1 main, 2 both
          const int ks = (nk - c * 4 < 4) ? nk - c * 4 : 4;
          const int s = g % kU3Stages;
          if (i < nch) mbar_wait(&a_full[c], (uint32_t)(it & 1));
          mbar_wait(&w_full[s], (uint32_t)((g / kU3Stages) & 1));
          fence_after_sync();
          U3_STAMP(0);
          const uint32_t base = ring_addr + (uint32_t)s * kChunkBytes;
          const uint64_t dhi = make_smem_desc(base, NP * 16u, 128u), dlo = make_smem_desc(base + kHalfBytes, NP * 16u, 128u);
          const uint32_t a0 = (uint32_t)c * 32u;
          if (kind != 1) {
#pragma unroll 4
            for (int kk = 0; kk < ks; ++kk) { mma_tf32_ts_w(tD, tAlo + a0 + kk * 8, dhi + (uint64_t)(dstep * kk), idesc, acc); acc = 1u; }
#pragma unroll 4
            for (int kk = 0; kk < ks; ++kk) mma_tf32_ts_w(tD, tAhi + a0 + kk * 8, dlo + (uint64_t)(dstep * kk), idesc, 1u);
          }
          if (kind != 0) {
#pragma unroll 4
            for (int kk = 0; kk < ks; ++kk) { mma_tf32_ts_w(tD, tAhi + a0 + kk * 8, dhi + (uint64_t)(dstep * kk), idesc, acc); acc = 1u; }
          }
          mma_commit_w(&w_empty[s]);
          if (release_a && kind != 0) mma_commit_w(&a_free[c]);
        }
        if (release_a)                                                         // k-chunks beyond this layer's K are free at once
          for (int c = nch; c < NB; ++c) mma_commit_w(&a_free[c]);
        mma_commit_w(d_full);
        U3_STAMP(0);
      }
  } else {
    // ===================== epilogue / generator warps: warp = (column block ci, lane quarter) =====================
    const int quarter = warp & 3, ci = warp >> 2, c = ci * 32;
    const int t = quarter * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(quarter * 32) << 16;
    const uint32_t tAhi = tmem_base + lane_sel + c, tAlo = tAhi + NP, tD = tAhi + 2 * NP;
    float* stage = stage_all + warp * kU3StageBlock;
    const float* bias = tail + c;                          // [(l-1)*NP + n] for hidden GEMM layer l
    const float* wlast = tail + (L - 1) * NP + c;
    const float* w0col = tail + L * NP + c;
    const float blast = __ldg(p.blast);
    const size_t plane = (size_t)Q * NP;
    float* ysave = p.saved ? p.saved + (size_t)L * plane : nullptr;
    uint32_t* bits = (p.saved && p.train && L > 1) ? reinterpret_cast<uint32_t*>(p.saved + (size_t)L * plane + Q) : nullptr;
#ifdef GNF_DEVTOOLS
    if (p.debug & 4) { bits = nullptr; ysave = nullptr; }
#endif
    const bool full_block = c + 32 <= p.N1;                // no padding column in this warp's block of layer 1

    // row context of a tile (q may exceed Q - 1 in the last tile: such rows compute on clamped inputs, store nothing)
    struct Row { int q, r, kn, r_first; float xv; };
    auto row_of = [&](int tl) {
      Row w;
      const int q0 = ((int)blockIdx.x + tl * (int)gridDim.x) * kU3Rows;
      w.q = q0 + t;
      const int qc = w.q < Q ? w.q : Q - 1;
      w.r = qc / nodes; w.kn = qc - w.r * nodes;
      w.r_first = q0 / nodes;
      w.xv = ldg_pinned(p.x + w.r);
      return w;
    };
    // coalesced store of this warp's 32 x 32 block (row-owner registers v) into plane columns [c, c+32): two 32 x 16 passes
    // through the 2 KB staging block (16-byte slots XOR-swizzled by (row >> 1) & 3), 8 rows x 64 bytes per store instruction
    auto store_block = [&](float* dstplane, const uint32_t* v, int q_row) {
#ifdef GNF_DEVTOOLS
      if (p.debug & 2) return;
#endif
      const int sub = lane >> 2, piece = lane & 3;
      const int row0 = q_row - lane + sub;
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4)
          *reinterpret_cast<uint4*>(stage + lane * 16 + 4 * (j4 ^ ((lane >> 1) & 3))) =
              make_uint4(v[16 * hb + 4 * j4], v[16 * hb + 4 * j4 + 1], v[16 * hb + 4 * j4 + 2], v[16 * hb + 4 * j4 + 3]);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int Rr = 8 * i + sub;
          const uint4 o = *reinterpret_cast<const uint4*>(stage + Rr * 16 + 4 * (piece ^ ((Rr >> 1) & 3)));
#ifdef GNF_DEVTOOLS
          if (p.debug & 1) continue;
#endif
          if (row0 + 8 * i < Q) *reinterpret_cast<uint4*>(dstplane + (size_t)(row0 + 8 * i) * NP + c + 16 * hb + 4 * piece) = o;
        }
        __syncwarp();
      }
    };
    // fp32 block -> TF32 hi (round to nearest) / lo -> TMEM A columns [c, c+32).  lo keeps its low mantissa bits after the
    // rounding increment: the tensor core ignores them, which completes the round-to-nearest of lo.
    auto split_store = [&](const uint32_t* v) {
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          hi[j] = u3_rn_tf32(v[16 * hb + j]);
          lo[j] = __float_as_uint(__uint_as_float(v[16 * hb + j]) - __uint_as_float(hi[j])) + 0x1000u;
        }
        tmem_st16p(tAhi + 16 * hb, hi);
        tmem_st16p(tAlo + 16 * hb, lo);
      }
    };
    auto mask_word = [&](const uint32_t* v) {            // v >= +0 after the ReLU: positive <=> non-zero bits
      uint32_t w = 0u;
#pragma unroll
      for (int j = 0; j < 32; ++j) w |= (v[j] != 0u ? 1u : 0u) << j;
      return w;
    };
    // layer 1 of tile tl, this warp's block: a1[q][n] = relu(t_q W0[n][0] + P[r][n]) -> A (+ plane, mask)
    auto gen_a1 = [&](int tl, const Row& w) {
      const float tq = (w.kn <= p.S) ? (w.xv * (ccs[w.kn] + 1.f)) / 2.f : w.xv;
      const float* Prow;
      if (p.p_smem) {
        mbar_wait(&p_full[tl & 1], (uint32_t)((tl >> 1) & 1));
        Prow = pbuf + (size_t)(tl & 1) * kU3PRows * NP + (size_t)(w.r - w.r_first) * NP + c;
      } else {
        Prow = p.P + (size_t)w.r * NP + c;
      }
      uint32_t v[32];
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        const float4 pv = p.p_smem ? *reinterpret_cast<const float4*>(Prow + 4 * j4) : __ldg(reinterpret_cast<const float4*>(Prow + 4 * j4));
        const float4 w4 = *reinterpret_cast<const float4*>(w0col + 4 * j4);
        v[4 * j4 + 0] = __float_as_uint(fmaxf(fmaf(tq, w4.x, pv.x), 0.f));
        v[4 * j4 + 1] = __float_as_uint(fmaxf(fmaf(tq, w4.y, pv.y), 0.f));
        v[4 * j4 + 2] = __float_as_uint(fmaxf(fmaf(tq, w4.z, pv.z), 0.f));
        v[4 * j4 + 3] = __float_as_uint(fmaxf(fmaf(tq, w4.w, pv.w), 0.f));
      }
      if (!full_block) {                                   // P's padding columns are never written: select, do not multiply
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = (c + j < p.N1) ? v[j] : 0u;
      }
      split_store(v);
      tmem_wait_st();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) {
        u3_arrive(&a_full[ci]);
        if (p.p_smem) u3_arrive(&p_empty[tl & 1]);
      }
      if (bits && w.q < Q) bits[(size_t)w.q * NB + ci] = mask_word(v);
      if (p.saved) store_block(p.saved, v, w.q);
    };

    Row cur = {0, 0, 0, 0, 0.f};
    if (n_local > 0) { cur = row_of(0); gen_a1(0, cur); }
    int it = 0;
    for (int tl = 0; tl < n_local; ++tl) {
      for (int l = 1; l < L; ++l, ++it) {
        const float* bl = bias + (l - 1) * NP;
        Row nxt = cur;
        const bool gen_next = (l == L - 1) && (tl + 1 < n_local);
        // The next tile's layer 1 is generated under this layer's MMAs: k-chunk ci of A is free as soon as its MMAs have
        // completed.  The warps of the LAST k-chunk get it back together with the accumulator: they drain first (the next
        // tile's first MMA waits for the drain; its chunk ci is needed four chunks later).
        const bool gen_late = gen_next && ci >= p.nch[l] - 1;
        if (gen_next) nxt = row_of(tl + 1);
        if (gen_next && !gen_late) {
          mbar_wait(&a_free[ci], (uint32_t)(tl & 1));
          fence_after_sync();
          gen_a1(tl + 1, nxt);
        }
        mbar_wait(d_full, (uint32_t)(it & 1));
        fence_after_sync();
        U3_STAMP(warp == 0 ? 1 : 3);
        uint32_t v[32];
        tmem_ld32p(tD, v);
        tmem_wait_ld();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) u3_arrive(d_empty);
        if (gen_late) {
          mbar_wait(&a_free[ci], (uint32_t)(tl & 1));
          fence_after_sync();
          gen_a1(tl + 1, nxt);
        }
        if (l < L - 1) {
          // hidden epilogue: a_{l+1} = relu(D + b_l) -> A for the next layer (+ plane, mask)
#pragma unroll
          for (int j4 = 0; j4 < 32; j4 += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(bl + j4);
            v[j4 + 0] = __float_as_uint(fmaxf(__uint_as_float(v[j4 + 0]) + b4.x, 0.f));
            v[j4 + 1] = __float_as_uint(fmaxf(__uint_as_float(v[j4 + 1]) + b4.y, 0.f));
            v[j4 + 2] = __float_as_uint(fmaxf(__uint_as_float(v[j4 + 2]) + b4.z, 0.f));
            v[j4 + 3] = __float_as_uint(fmaxf(__uint_as_float(v[j4 + 3]) + b4.w, 0.f));
          }
          split_store(v);
          tmem_wait_st();
          fence_before_sync();
          __syncwarp();
          if (lane == 0) u3_arrive(&a_full[ci]);
          U3_STAMP(warp == 0 ? 1 : 3);
          if (bits && cur.q < Q) bits[(size_t)l * Q * NB + (size_t)cur.q * NB + ci] = mask_word(v);
          if (p.saved) store_block(p.saved + (size_t)l * plane, v, cur.q);
        } else {
          // last hidden layer: a_L = relu(D + b), y = a_L . w_L + b_L
          float y0 = 0.f, y1 = 0.f, y2 = 0.f, y3 = 0.f;
#pragma unroll
          for (int j4 = 0; j4 < 32; j4 += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(bl + j4);
            const float4 w4 = *reinterpret_cast<const float4*>(wlast + j4);
            const float a0 = fmaxf(__uint_as_float(v[j4 + 0]) + b4.x, 0.f), a1 = fmaxf(__uint_as_float(v[j4 + 1]) + b4.y, 0.f);
            const float a2 = fmaxf(__uint_as_float(v[j4 + 2]) + b4.z, 0.f), a3 = fmaxf(__uint_as_float(v[j4 + 3]) + b4.w, 0.f);
            y0 = fmaf(a0, w4.x, y0); y1 = fmaf(a1, w4.y, y1); y2 = fmaf(a2, w4.z, y2); y3 = fmaf(a3, w4.w, y3);
            v[j4 + 0] = __float_as_uint(a0); v[j4 + 1] = __float_as_uint(a1); v[j4 + 2] = __float_as_uint(a2); v[j4 + 3] = __float_as_uint(a3);
          }
          ypart[ci * kU3Rows + t] = (y0 + y1) + (y2 + y3);
          if (bits && cur.q < Q) bits[(size_t)l * Q * NB + (size_t)cur.q * NB + ci] = mask_word(v);   // mask of a_L: the fused backward starts from it
          if (p.saved) store_block(p.saved + (size_t)l * plane, v, cur.q);
          named_bar_sync(1, EW * 32);
          const bool cur_valid = cur.q < Q;
          if (ci == 0) {
            float y = blast;
#pragma unroll
            for (int k = 0; k < NB; ++k) y += ypart[k * kU3Rows + t];
            const float f = (y > 0.f ? y : expm1f(y)) + 1.05f;
            float wv = 0.f;
            if (cur_valid) {
              if (ysave) ysave[cur.q] = y;
              if (cur.kn <= p.S) wv = ccs[kU3MaxNodes + cur.kn] * f;
              if (cur.kn == 0) {
                p.jac[cur.r] = f;
                if (p.logdet) atomicAdd(p.logdet + cur.r / p.d, logf(f));
              }
            }
            red[t] = wv;
          }
          named_bar_sync(1, EW * 32);
          if (ci == 0 && cur_valid && (cur.kn == 0 || t == 0)) {
            float sacc = 0.f;
            int rem = nodes - cur.kn;
            if (rem > kU3Rows - t) rem = kU3Rows - t;
            for (int k = 0; k < rem; ++k) sacc += red[t + k];
            float cz = sacc * cur.xv / 2.f;
            if (cur.kn == 0) cz += __ldg(p.h + (size_t)cur.r * p.E);
            atomicAdd(p.z + cur.r, cz);
            if (p.zrev) { const int b = cur.r / p.d, ii = cur.r % p.d; atomicAdd(p.zrev + (size_t)b * p.d + (p.d - 1 - ii), cz); }
          }
          U3_STAMP(warp == 0 ? 1 : 3);
        }
        cur = nxt;
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// =====================================================================================================================
// Backward chain (UMNN NeuralIntegral.backward's dgrad pass over all quadrature node-rows, SURVEY App. B): from the cotangent of
// the integrand's pre-ELU output down to the first layer, in ONE kernel with the same structure as the forward:
//   delta_L = (g_q w_L) o relu'(a_L)            generated in registers from the saved ReLU bit mask of a_L and the saved y
//   delta_l = (delta_{l+1} W_l) o relu'(a_l)    l = L-1 .. 1: 3xTF32 tcgen05 GEMMs, A = delta in TMEM, W_l^T streamed as hi/lo chunks
// What leaves the chip: the delta_l planes the weight-gradient GEMMs (tc_rw_wgrad.cu) consume (l >= 2), the column sums
// db_{l-1} = sum_q delta_l, and the first-layer reductions D[r] = sum_k delta_1[(r,k)], dW0[:,0] = sum_q delta_1[q] t_q,
// dx[r] = delta_1[(r,S+1)] . W0[:,0] + jac[r] gz[r] -- taken with warp shuffles (16 columns x 32 rows per pass) and atomics.
// Replaces the dgrad GEMMs, the colsum passes and the layer-1 reduction pass of gnf_umnn_bwd_lw.
// =====================================================================================================================
struct U3BParams {
  const float *x, *ccw, *ccn, *jac, *gz, *gzrev, *gjac, *glogdet, *image, *saved;
  float* dplanes;                       // [L-2][Q][NP]: delta_{L-1} .. delta_2 (delta_l at plane L-1-l)
  float *D, *dx, *dW0;                  // D [R][NP], dx [R], dW0 = W0 gradient (column 0 written, row stride ldw0): atomic accumulation
  float* db[GNF_MAX_LAYERS];            // db[l-1] for l = 2..L-1 (atomic)
  int R, d, E, S, nodes, L, ldw0;
  long long Q;
  int dims[GNF_MAX_LAYERS + 1];
  int kp[GNF_MAX_LAYERS], nch[GNF_MAX_LAYERS];      // per GEMM layer l: reduction = dims[l+1] padded to 8, its 32-chunks
  unsigned off_img[GNF_MAX_LAYERS], off_tail, chunk_floats;
};

// sum over the 32 lanes of each of 16 columns held as w[16]; lane i (and i + 16) ends with column (i & 15)
__device__ __forceinline__ float u3_colsum16(float (&w)[16], int lane) {
#pragma unroll
  for (int i = 0; i < 16; ++i) w[i] += __shfl_xor_sync(0xffffffffu, w[i], 16);
#pragma unroll
  for (int o = 8; o >= 1; o >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const float send = up ? w[i] : w[i + o];
      const float keep = up ? w[i + o] : w[i];
      w[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return w[0];
}

template <int NB>
__global__ void __launch_bounds__((4 * NB + 2) * 32, 1) umnn_bwd_tc3_kernel(U3BParams p) {
  using namespace tc;
  constexpr int NP = NB * 32;
  constexpr int EW = 4 * NB;
  constexpr int NT = (EW + 2) * 32;
  constexpr uint32_t kChunkBytes = 2u * 8u * NP * 16u;
  constexpr uint32_t kHalfBytes = 8u * NP * 16u;
  GNF_SMEM(float, smem);
  float* ring = smem;
  float* tail = ring + (size_t)kU3Stages * (kChunkBytes / 4);   // w_L[NP], W0[:,0][NP]
  float* stage_all = tail + 2 * NP;
  float* ccs = stage_all + EW * kU3StageBlock;                  // ccn, ccw
  uint64_t* bars = reinterpret_cast<uint64_t*>(ccs + 2 * kU3MaxNodes);
  uint64_t* w_full = bars;
  uint64_t* w_empty = w_full + kU3Stages;
  uint64_t* a_full = w_empty + kU3Stages;
  uint64_t* a_free = a_full + NB;
  uint64_t* d_full = a_free + NB;
  uint64_t* d_empty = d_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d_empty + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (warp == 0) tmem_alloc(tmem_slot, 512);
  if (tid == 32) {
    for (int s = 0; s < kU3Stages; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 1); }
    for (int c = 0; c < NB; ++c) { mbar_init(&a_full[c], 4); mbar_init(&a_free[c], 1); }
    mbar_init(d_full, 1);
    mbar_init(d_empty, EW);
    fence_mbar_init();
  }
  pdl_prologue_done();
  for (int i = tid; i < 2 * NP; i += NT) tail[i] = __ldg(p.image + p.off_tail + i);
  for (int i = tid; i <= p.S; i += NT) { ccs[i] = __ldg(p.ccn + i); ccs[kU3MaxNodes + i] = __ldg(p.ccw + i); }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  const int Q = (int)p.Q, nodes = p.nodes;
  const int ntiles = (Q + kU3Rows - 1) / kU3Rows;
  const int n_local = (ntiles > (int)blockIdx.x) ? (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int L = p.L;

  if (warp == EW + 1) {
    // ===================== producer: W_l^T chunks, l = L-1 .. 1 per tile =====================
    if (lane == 0) {
      int g = 0;
      for (int tl = 0; tl < n_local; ++tl)
        for (int l = L - 1; l >= 1; --l) {
          const int nch = p.nch[l], nk = p.kp[l] / 8;
          const char* src0 = reinterpret_cast<const char*>(p.image + p.off_img[l]);
          for (int i = 0; i < 2 * nch; ++i, ++g) {                             // corrections first, then the a_hi * b_hi chain
            const int c = i < nch ? i : i - nch;
            const bool want_lo = i < nch;
            const int ks = (nk - c * 4 < 4) ? nk - c * 4 : 4;
            const uint32_t bytes = (uint32_t)ks * 2u * NP * 16u;
            const int s = g % kU3Stages;
            if (g >= kU3Stages) mbar_wait(&w_empty[s], (uint32_t)(((g / kU3Stages) - 1) & 1));
            char* dst = reinterpret_cast<char*>(ring) + (size_t)s * kChunkBytes;
            const char* src = src0 + (size_t)c * kChunkBytes;
            mbar_expect_tx(&w_full[s], want_lo ? 2u * bytes : bytes);
            bulk_g2s(dst, src, bytes, &w_full[s]);
            if (want_lo) bulk_g2s(dst + kHalfBytes, src + kHalfBytes, bytes, &w_full[s]);
          }
        }
    }
  } else if (warp == EW) {
    // ===================== MMA issuer (warp-converged) =====================
    constexpr uint32_t idesc = make_idesc_tf32(kU3Rows, NP);
    constexpr uint32_t dstep = (2u * NP * 16u) >> 4;
    const uint32_t tAhi = tmem_base, tAlo = tmem_base + NP, tD = tmem_base + 2 * NP;
    const uint32_t ring_addr = smem_u32(ring);
    int g = 0, it = 0;
    for (int tl = 0; tl < n_local; ++tl)
      for (int l = L - 1; l >= 1; --l, ++it) {
        const int nch = p.nch[l], nk = p.kp[l] / 8;
        const bool release_a = (l == 1) && (tl + 1 < n_local);
        if (it > 0) mbar_wait(d_empty, (uint32_t)((it - 1) & 1));
        uint32_t acc = 0u;
        for (int i = 0; i < 2 * nch; ++i, ++g) {
          const int c = i < nch ? i : i - nch;
          const bool corr = i < nch;
          const int ks = (nk - c * 4 < 4) ? nk - c * 4 : 4;
          const int s = g % kU3Stages;
          if (corr) mbar_wait(&a_full[c], (uint32_t)(it & 1));
          mbar_wait(&w_full[s], (uint32_t)((g / kU3Stages) & 1));
          fence_after_sync();
          const uint32_t base = ring_addr + (uint32_t)s * kChunkBytes;
          const uint64_t dhi = make_smem_desc(base, NP * 16u, 128u), dlo = make_smem_desc(base + kHalfBytes, NP * 16u, 128u);
          const uint32_t a0 = (uint32_t)c * 32u;
          if (corr) {
#pragma unroll 4
            for (int kk = 0; kk < ks; ++kk) { mma_tf32_ts_w(tD, tAlo + a0 + kk * 8, dhi + (uint64_t)(dstep * kk), idesc, acc); acc = 1u; }
#pragma unroll 4
            for (int kk = 0; kk < ks; ++kk) mma_tf32_ts_w(tD, tAhi + a0 + kk * 8, dlo + (uint64_t)(dstep * kk), idesc, 1u);
          } else {
#pragma unroll 4
            for (int kk = 0; kk < ks; ++kk) mma_tf32_ts_w(tD, tAhi + a0 + kk * 8, dhi + (uint64_t)(dstep * kk), idesc, 1u);
          }
          mma_commit_w(&w_empty[s]);
          if (release_a && !corr) mma_commit_w(&a_free[c]);
        }
        if (release_a)
          for (int c = nch; c < NB; ++c) mma_commit_w(&a_free[c]);
        mma_commit_w(d_full);
      }
  } else {
    // ===================== epilogue / generator warps: warp = (column block ci, lane quarter) =====================
    const int quarter = warp & 3, ci = warp >> 2, c = ci * 32;
    const int t = quarter * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(quarter * 32) << 16;
    const uint32_t tAhi = tmem_base + lane_sel + c, tAlo = tAhi + NP, tD = tAhi + 2 * NP;
    float* stage = stage_all + warp * kU3StageBlock;
    const float* wL = tail + c;
    const float* w0col = tail + NP + c;
    const size_t plane = (size_t)Q * NP;
    const float* ysave = p.saved + (size_t)L * plane;
    const uint32_t* bits = reinterpret_cast<const uint32_t*>(p.saved + (size_t)L * plane + Q);   // [L][Q][NB]: masks of a_1 .. a_L
    const size_t bplane = (size_t)Q * NB;

    struct Row { int q, r, kn; float gq, tq, jg; uint32_t mtop; };
    // row context of tile tl: cotangent of the pre-ELU output (lw_out_bwd_kernel's formula), node abscissa, top-layer mask word
    auto row_of = [&](int tl) {
      Row w;
      const int q0 = ((int)blockIdx.x + tl * (int)gridDim.x) * kU3Rows;
      w.q = q0 + t;
      const bool valid = w.q < Q;
      const int qc = valid ? w.q : Q - 1;
      w.r = qc / nodes; w.kn = qc - w.r * nodes;
      const int r = w.r;
      const float xv = ldg_pinned(p.x + r);
      float gzt = p.gz ? ldg_pinned(p.gz + r) : 0.f;
      if (p.gzrev) { const int b = r / p.d, i = r - b * p.d; gzt += ldg_pinned(p.gzrev + (size_t)b * p.d + (p.d - 1 - i)); }
      const float y = ldg_pinned(ysave + qc);
      float gq;
      if (w.kn <= p.S) {
        gq = (gzt * xv / 2.f) * ccs[kU3MaxNodes + w.kn];
        w.tq = (xv * (ccs[w.kn] + 1.f)) / 2.f;
      } else {
        gq = p.gjac ? ldg_pinned(p.gjac + r) : 0.f;
        if (p.glogdet) gq += ldg_pinned(p.glogdet + r / p.d) / ldg_pinned(p.jac + r);
        w.tq = xv;
      }
      gq *= (y > 0.f) ? 1.f : expf(y);
      w.gq = valid ? gq : 0.f;
      w.jg = ldg_pinned(p.jac + r) * gzt;
      w.mtop = valid ? __ldg(bits + (size_t)(L - 1) * bplane + (size_t)qc * NB + ci) : 0u;
      return w;
    };
    auto store_block = [&](float* dstplane, const uint32_t* v, int q_row) {
      const int sub = lane >> 2, piece = lane & 3;
      const int row0 = q_row - lane + sub;
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4)
          *reinterpret_cast<uint4*>(stage + lane * 16 + 4 * (j4 ^ ((lane >> 1) & 3))) =
              make_uint4(v[16 * hb + 4 * j4], v[16 * hb + 4 * j4 + 1], v[16 * hb + 4 * j4 + 2], v[16 * hb + 4 * j4 + 3]);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int Rr = 8 * i + sub;
          const uint4 o = *reinterpret_cast<const uint4*>(stage + Rr * 16 + 4 * (piece ^ ((Rr >> 1) & 3)));
          if (row0 + 8 * i < Q) *reinterpret_cast<uint4*>(dstplane + (size_t)(row0 + 8 * i) * NP + c + 16 * hb + 4 * piece) = o;
        }
        __syncwarp();
      }
    };
    auto split_store = [&](const uint32_t* v) {
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          hi[j] = u3_rn_tf32(v[16 * hb + j]);
          lo[j] = __float_as_uint(__uint_as_float(v[16 * hb + j]) - __uint_as_float(hi[j])) + 0x1000u;
        }
        tmem_st16p(tAhi + 16 * hb, hi);
        tmem_st16p(tAlo + 16 * hb, lo);
      }
    };
    // top of the chain: delta_L[q][n] = g_q w_L[n] where a_L[q][n] > 0
    auto gen_top = [&](const Row& w) {
      uint32_t v[32];
#pragma unroll
      for (int j4 = 0; j4 < 8; ++j4) {
        const float4 w4 = *reinterpret_cast<const float4*>(wL + 4 * j4);
        v[4 * j4 + 0] = ((w.mtop >> (4 * j4 + 0)) & 1u) ? __float_as_uint(w.gq * w4.x) : 0u;
        v[4 * j4 + 1] = ((w.mtop >> (4 * j4 + 1)) & 1u) ? __float_as_uint(w.gq * w4.y) : 0u;
        v[4 * j4 + 2] = ((w.mtop >> (4 * j4 + 2)) & 1u) ? __float_as_uint(w.gq * w4.z) : 0u;
        v[4 * j4 + 3] = ((w.mtop >> (4 * j4 + 3)) & 1u) ? __float_as_uint(w.gq * w4.w) : 0u;
      }
      split_store(v);
      tmem_wait_st();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) u3_arrive(&a_full[ci]);
    };

    Row cur;
    cur.q = 0; cur.r = 0; cur.kn = 0; cur.gq = 0.f; cur.tq = 0.f; cur.jg = 0.f; cur.mtop = 0u;
    if (n_local > 0) { cur = row_of(0); gen_top(cur); }
    int it = 0;
    for (int tl = 0; tl < n_local; ++tl) {
      for (int l = L - 1; l >= 1; --l, ++it) {
        Row nxt = cur;
        const bool gen_next = (l == 1) && (tl + 1 < n_local);
        const bool gen_late = gen_next && ci >= p.nch[l] - 1;
        // ReLU mask of a_l for this row / column block (dependent global load: issued before the waits)
        const bool valid = cur.q < Q;
        const uint32_t m = valid ? __ldg(bits + (size_t)(l - 1) * bplane + (size_t)cur.q * NB + ci) : 0u;
        if (gen_next) nxt = row_of(tl + 1);
        if (gen_next && !gen_late) {
          mbar_wait(&a_free[ci], (uint32_t)(tl & 1));
          fence_after_sync();
          gen_top(nxt);
        }
        mbar_wait(d_full, (uint32_t)(it & 1));
        fence_after_sync();
        uint32_t v[32];
        tmem_ld32p(tD, v);
        tmem_wait_ld();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) u3_arrive(d_empty);
        if (gen_late) {
          mbar_wait(&a_free[ci], (uint32_t)(tl & 1));
          fence_after_sync();
          gen_top(nxt);
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = ((m >> j) & 1u) ? v[j] : 0u;        // delta_l = (delta_{l+1} W_l) o relu'(a_l); rows >= Q: 0
        if (l > 1) {
          split_store(v);
          tmem_wait_st();
          fence_before_sync();
          __syncwarp();
          if (lane == 0) u3_arrive(&a_full[ci]);
          // db_{l-1} = column sums of delta_l; the plane goes to the weight-gradient GEMM of W_{l-1}
#pragma unroll
          for (int hb = 0; hb < 2; ++hb) {
            float w16[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) w16[j] = __uint_as_float(v[16 * hb + j]);
            const float sum = u3_colsum16(w16, lane);
            const int n = c + 16 * hb + (lane & 15);
            if (lane < 16 && n < p.dims[l]) atomicAdd(p.db[l - 1] + n, sum);
          }
          store_block(p.dplanes + (size_t)(L - 1 - l) * plane, v, cur.q);
        } else {
          // first layer: dx (the row of node S+1 carries the jac output's chain rule), dW0[:,0], D[r] = sum over the row's nodes
          float dot = 0.f;
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 w4 = *reinterpret_cast<const float4*>(w0col + 4 * j4);
            dot = fmaf(__uint_as_float(v[4 * j4 + 0]), w4.x, dot); dot = fmaf(__uint_as_float(v[4 * j4 + 1]), w4.y, dot);
            dot = fmaf(__uint_as_float(v[4 * j4 + 2]), w4.z, dot); dot = fmaf(__uint_as_float(v[4 * j4 + 3]), w4.w, dot);
          }
          if (valid && cur.kn == p.S + 1) atomicAdd(p.dx + cur.r, dot + (ci == 0 ? cur.jg : 0.f));
          const int r_lo = __shfl_sync(0xffffffffu, cur.r, 0), r_hi = __shfl_sync(0xffffffffu, cur.r, 31);
#pragma unroll
          for (int hb = 0; hb < 2; ++hb) {
            const int n = c + 16 * hb + (lane & 15);
            const bool col_ok = lane < 16 && n < p.dims[1];
            float w16[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) w16[j] = __uint_as_float(v[16 * hb + j]) * cur.tq;
            const float st = u3_colsum16(w16, lane);
            if (col_ok) atomicAdd(p.dW0 + (size_t)n * p.ldw0, st);
            for (int rr = r_lo; rr <= r_hi; ++rr) {                    // warp-uniform trip count: the rows this warp's 32 node-rows span
#pragma unroll
              for (int j = 0; j < 16; ++j) w16[j] = (cur.r == rr) ? __uint_as_float(v[16 * hb + j]) : 0.f;
              const float sd = u3_colsum16(w16, lane);
              if (col_ok) atomicAdd(p.D + (size_t)rr * NP + n, sd);
            }
          }
        }
        cur = nxt;
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

static size_t u3b_smem_bytes(int NP) {
  const int NB = NP / 32, EW = 4 * NB;
  return ((size_t)kU3Stages * 2 * 8 * NP * 4 + (size_t)2 * NP + (size_t)EW * kU3StageBlock + 2 * kU3MaxNodes) * sizeof(float) +
         (2 * kU3Stages + 2 * NB + 2) * sizeof(uint64_t) + 16;
}

// Packed operands of the chain: for GEMM layer l the image of W_l^T (B[n'][k'] = W_l[k'][n'], n' = in-feature, reduction k' =
// out-feature) in the forward's chunk format, then w_L and W0[:,0].
struct U3BPlan {
  int L, NP;
  int kp[GNF_MAX_LAYERS], nch[GNF_MAX_LAYERS];
  size_t off_img[GNF_MAX_LAYERS], chunk_floats, off_tail, image_floats;
};
static int u3b_plan(const gnf_mlp_t* net, U3BPlan* pl) {
  U3Plan f;
  if (int e = u3_plan(net, 0, &f)) return e;
  pl->L = f.L; pl->NP = f.NP; pl->chunk_floats = f.chunk_floats;
  size_t off = 0;
  for (int l = 0; l < GNF_MAX_LAYERS; ++l) { pl->kp[l] = 0; pl->nch[l] = 0; pl->off_img[l] = 0; }
  for (int l = 1; l < f.L; ++l) {
    pl->kp[l] = (net->dims[l + 1] + 7) / 8 * 8;
    pl->nch[l] = (pl->kp[l] + 31) / 32;
    pl->off_img[l] = off;
    off += (size_t)pl->nch[l] * pl->chunk_floats;
  }
  pl->off_tail = off;
  pl->image_floats = off + (size_t)2 * f.NP;
  return 0;
}

__global__ void u3_pack_bwd_kernel(U3PackArgs a, float* __restrict__ img) {
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < a.total; i += gridDim.x * blockDim.x) {
    float out = 0.f;
    if (i >= a.off_tail) {
      const int e = (int)(i - a.off_tail), j = e / a.NP, n = e % a.NP;
      if (j == 0) { if (n < a.dims[a.L]) out = a.W[a.L][n]; }                                 // output Linear [1, dims[L]]
      else { if (n < a.dims[1]) out = a.W[0][(size_t)n * a.dims[0]]; }                        // W0[:, 0]
    } else {
      int l = 1;
      while (l + 1 < a.L && i >= a.off_img[l + 1]) ++l;
      const unsigned e = i - a.off_img[l];
      const unsigned c = e / a.chunk_floats, e2 = e % a.chunk_floats;
      const unsigned half = 8u * a.NP * 4u;
      const unsigned part = e2 / half, e3 = e2 % half;
      const int k4 = (int)(e3 / (a.NP * 4u)), n = (int)((e3 / 4u) % a.NP), kk = (int)(e3 % 4u);
      const int k = (int)c * 32 + k4 * 4 + kk;                                                // k = out-feature (reduction), n = in-feature
      float v = 0.f;
      if (n < a.dims[l] && k < a.dims[l + 1]) v = a.W[l][(size_t)k * a.dims[l] + n];
      const float hi = __uint_as_float(u3_rn_tf32(__float_as_uint(v)));
      out = part ? __uint_as_float(u3_rn_tf32(__float_as_uint(v - hi))) : hi;
    }
    img[i] = out;
  }
}

size_t u3_bwd_image_floats(const gnf_mlp_t* net) {
  U3BPlan pl;
  if (u3b_plan(net, &pl)) return 0;
  return (pl.image_floats + 3) / 4 * 4;
}

// image: u3_bwd_image_floats(net) floats of scratch; dplanes: (L-2) planes; D, dx and the db / dW0 targets must be zeroed by the caller.
int launch_u3_bwd_chain(const float* x, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn, const float* jac, const float* gz,
                        const float* gzrev, const float* gjac, const float* glogdet, const float* saved, float* image, float* dplanes, float* D,
                        float* dx, const gnf_mlp_grad_t* grads, int R, int d, cudaStream_t s, const Branches* br, int side, cudaStream_t pack_stream) {
  U3BPlan pl;
  if (int e = u3b_plan(net, &pl)) return e;
  const int NP = pl.NP, L = pl.L;
  const int nodes = S + 2;
  const long long Q = (long long)R * nodes;
  if (Q > 0x7fffffffLL - 2 * kU3Rows || S + 1 > kU3MaxNodes) return fail(GNF_ERR_UNSUPPORTED, "umnn tc3 backward: problem size out of range");
  U3PackArgs a;
  for (int l = 0; l < GNF_MAX_LAYERS; ++l) { a.W[l] = nullptr; a.b[l] = nullptr; a.nch[l] = pl.nch[l]; a.off_img[l] = (unsigned)pl.off_img[l]; }
  for (int l = 0; l <= L; ++l) { a.W[l] = net->W[l]; a.b[l] = net->b[l]; }
  for (int l = 0; l <= net->n_layers; ++l) a.dims[l] = net->dims[l];
  a.chunk_floats = (unsigned)pl.chunk_floats; a.off_tail = (unsigned)pl.off_tail; a.total = (unsigned)pl.image_floats; a.L = L; a.NP = NP;
  int blocks = (int)((pl.image_floats + 255) / 256);
  if (blocks > 2 * kNumSMs) blocks = 2 * kNumSMs;
  // the weight images depend on nothing of this call: the caller forked `pack_stream` before its output pass, joined here
  GNF_LAUNCH(u3_pack_bwd_kernel, blocks, 256, 0, (br && pack_stream) ? pack_stream : s, a, image);
  if (br && pack_stream) br->end(s, side);
  U3BParams p;
  p.x = x; p.ccw = ccw; p.ccn = ccn; p.jac = jac; p.gz = gz; p.gzrev = gzrev; p.gjac = gjac; p.glogdet = glogdet; p.image = image; p.saved = saved;
  p.dplanes = dplanes; p.D = D; p.dx = dx; p.dW0 = grads->dW[0]; p.ldw0 = net->dims[0];
  for (int l = 0; l < GNF_MAX_LAYERS; ++l) p.db[l] = grads->db[l];
  p.R = R; p.d = d; p.E = net->dims[0] - 1; p.S = S; p.nodes = nodes; p.L = L; p.Q = Q;
  for (int l = 0; l <= GNF_MAX_LAYERS; ++l) p.dims[l] = l <= net->n_layers ? net->dims[l] : 0;
  for (int l = 0; l < GNF_MAX_LAYERS; ++l) { p.kp[l] = pl.kp[l]; p.nch[l] = pl.nch[l]; p.off_img[l] = (unsigned)pl.off_img[l]; }
  p.off_tail = (unsigned)pl.off_tail; p.chunk_floats = (unsigned)pl.chunk_floats;
  const size_t smem = u3b_smem_bytes(NP);
  const long long ntiles = (Q + kU3Rows - 1) / kU3Rows;
  const int grid = (int)(ntiles < kNumSMs ? ntiles : kNumSMs);
#define U3B_CASE(nb)                                                                                             \
  case nb:                                                                                                       \
    cudaFuncSetAttribute(umnn_bwd_tc3_kernel<nb>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);       \
    GNF_LAUNCH_PDL(umnn_bwd_tc3_kernel<nb>, grid, (4 * nb + 2) * 32, smem, s, p);                                    \
    break;
  switch (NP / 32) { U3B_CASE(1) U3B_CASE(2) U3B_CASE(3) U3B_CASE(4) U3B_CASE(5) default: return fail(GNF_ERR_UNSUPPORTED, "umnn tc3 backward: width"); }
#undef U3B_CASE
  return 0;
}

static size_t u3_smem_bytes(int NP) {
  const int NB = NP / 32, EW = 4 * NB;
  return ((size_t)kU3Stages * 2 * 8 * NP * 4 + (size_t)(GNF_MAX_LAYERS + 1) * NP + (size_t)EW * kU3StageBlock + (size_t)2 * kU3PRows * NP +
          (size_t)(NB + 1) * kU3Rows + 2 * kU3MaxNodes) * sizeof(float) + (2 * kU3Stages + 2 * NB + 6) * sizeof(uint64_t) + 16;
}

#ifdef GNF_DEVTOOLS
static long long* g_u3_trace = nullptr;
static int g_u3_debug = 0;      // ablation: bit0 skip the global stores of the planes, bit1 skip their staging too, bit2 skip masks / y
#endif

}  // namespace gnf
using namespace gnf;
#endif  // !GNF_EMU

extern "C" {

size_t gnf_umnn_tc3_workspace_bytes(const gnf_mlp_t* net, int R) {
#ifdef GNF_EMU
  (void)net; (void)R;
  gnf::set_error("tensor-core kernels have no host-simulator flavour");
  return 0;
#else
  U3Plan pl;
  if (u3_plan(net, R, &pl)) return 0;
  return pl.total_floats * sizeof(float);
#endif
}

int gnf_umnn_fwd_tc3(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn, float* z,
                     float* zrev, float* jac, float* logdet, float* saved, int train, int order, int R, int d, void* work,
                     size_t work_bytes, gnf_stream_t stream) {
#ifdef GNF_EMU
  return gnf::fail(GNF_ERR_UNSUPPORTED, "tensor-core kernels have no host-simulator flavour");
#else
  if (!x || !h || !net || !ccw || !ccn || !z || !jac || R < 0 || d <= 0 || S < 1 || (R % d) != 0) return fail(GNF_ERR_INVALID, "gnf_umnn_fwd_tc3: bad arguments");
  if (train && !saved) return fail(GNF_ERR_INVALID, "gnf_umnn_fwd_tc3: training needs the saved-activation buffer");
  U3Plan pl;
  if (int e = u3_plan(net, R, &pl)) return e;
  if (!work || work_bytes < pl.total_floats * sizeof(float)) return fail(GNF_ERR_WORKSPACE, "gnf_umnn_fwd_tc3: workspace too small (%zu < %zu)", work_bytes, pl.total_floats * sizeof(float));
  if ((reinterpret_cast<uintptr_t>(work) & 15) != 0 || (saved && (reinterpret_cast<uintptr_t>(saved) & 15) != 0)) return fail(GNF_ERR_INVALID, "gnf_umnn_fwd_tc3: workspace / saved must be 16-byte aligned");
  const int nodes = S + 1 + (train ? 1 : 0);
  const long long Q = (long long)R * nodes;
  if (Q > 0x7fffffffLL - 2 * kU3Rows) return fail(GNF_ERR_UNSUPPORTED, "gnf_umnn_fwd_tc3: %lld node-rows exceed the index range", Q);
  if (S + 1 > kU3MaxNodes) return fail(GNF_ERR_UNSUPPORTED, "gnf_umnn_fwd_tc3: more than %d quadrature nodes", kU3MaxNodes);
  cudaStream_t s = (cudaStream_t)stream;
  if (R == 0) return 0;
  float* ws = (float*)work;
  const int NP = pl.NP, L = pl.L, E = pl.E;
  // packed hi/lo chunk images + biases + w_L + W0[:,0]
  U3PackArgs a;
  for (int l = 0; l < GNF_MAX_LAYERS; ++l) { a.W[l] = nullptr; a.b[l] = nullptr; a.nch[l] = pl.nch[l]; a.off_img[l] = (unsigned)pl.off_img[l]; }
  for (int l = 0; l <= L; ++l) { a.W[l] = net->W[l]; a.b[l] = net->b[l]; }
  for (int l = 0; l <= net->n_layers; ++l) a.dims[l] = net->dims[l];
  a.chunk_floats = (unsigned)pl.chunk_floats; a.off_tail = (unsigned)pl.off_tail; a.total = (unsigned)pl.image_floats; a.L = L; a.NP = NP;
  int blocks = (int)((pl.image_floats + 255) / 256);
  if (blocks > 2 * kNumSMs) blocks = 2 * kNumSMs;
  // branch 0: the weight images and the zero-fills (they depend on nothing of this call) next to the P GEMM
  const Branches& br = branches();
  cudaStream_t s0 = br.begin(s, 0);
  GNF_LAUNCH(u3_pack_kernel, blocks, 256, 0, s0, a, ws);
  ZeroList zl;
  zl.add(z, (size_t)R);
  zl.add(zrev, (size_t)R);
  zl.add(logdet, (size_t)(R / d));
  zero_many(zl, s0);
  // P = h W0[:,1:]^T + b0, once per row (strict fp32 on the FFMA engine: R x N1 x E is tiny)
  float* P = ws + pl.off_P;
  if (int e = gnf_linear_fwd(h, E, net->W[0] + 1, 1 + E, net->b[0], 1, P, NP, R, net->dims[1], E, 0, stream)) return e;
  br.end(s, 0);
  U3Params p;
  p.x = x; p.h = h; p.ccw = ccw; p.ccn = ccn; p.P = P; p.image = ws; p.blast = net->b[L];
  p.z = z; p.zrev = zrev; p.jac = jac; p.logdet = logdet; p.saved = saved;
  p.R = R; p.d = d; p.E = E; p.S = S; p.nodes = nodes; p.L = L; p.N1 = pl.N1; p.train = train; p.order = order ? 1 : 0;
  p.Q = Q;
  p.p_smem = ((kU3Rows - 1) / nodes + 2 <= kU3PRows) ? 1 : 0;       // else the generator reads P from global memory
  for (int l = 0; l < GNF_MAX_LAYERS; ++l) { p.kp[l] = pl.kp[l]; p.nch[l] = pl.nch[l]; p.off_img[l] = (unsigned)pl.off_img[l]; }
  p.off_tail = (unsigned)pl.off_tail; p.chunk_floats = (unsigned)pl.chunk_floats;
#ifdef GNF_DEVTOOLS
  p.trace = g_u3_trace; p.debug = g_u3_debug;
#else
  p.trace = nullptr; p.debug = 0;
#endif
  const size_t smem = u3_smem_bytes(NP);
  const long long ntiles = (Q + kU3Rows - 1) / kU3Rows;
  const int grid = (int)(ntiles < kNumSMs ? ntiles : kNumSMs);
#define U3_CASE(nb)                                                                                              \
  case nb:                                                                                                       \
    cudaFuncSetAttribute(umnn_fwd_tc3_kernel<nb>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);       \
    GNF_LAUNCH_PDL(umnn_fwd_tc3_kernel<nb>, grid, (4 * nb + 2) * 32, smem, s, p);                                           \
    break;
  switch (NP / 32) { U3_CASE(1) U3_CASE(2) U3_CASE(3) U3_CASE(4) U3_CASE(5) default: return fail(GNF_ERR_UNSUPPORTED, "gnf_umnn_fwd_tc3: width"); }
#undef U3_CASE
  return check_launch("gnf_umnn_fwd_tc3");
#endif
}

#ifdef GNF_DEVTOOLS
/* Measurement (dev build only): CTA 0 records SM-clock stamps into buf[4][256]; NULL disables.
 * row 0 issuer: per layer instance [input ready, each chunk landed..., committed];  row 2 producer: each chunk issued;
 * rows 1 / 3 epilogue warps 0 / 4: hidden layer [accumulator full, input of next layer staged]; last layer
 * [accumulator full, drained (+ plane stored), next tile's layer-1 staged, reduction done]. */
int gnf_umnn_tc3_set_trace(long long* buf) {
#ifndef GNF_EMU
  gnf::g_u3_trace = buf;
#else
  (void)buf;
#endif
  return 0;
}
int gnf_umnn_tc3_set_debug(int bits) {
#ifndef GNF_EMU
  gnf::g_u3_debug = bits;
#else
  (void)bits;
#endif
  return 0;
}
#endif

}  // extern "C"
