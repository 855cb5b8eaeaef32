/* libgnf_sm100 — C-ABI of the B200-native Graphical-Normalizing-Flows hot path.
 *
 * One shared library (nvcc -gencode arch=compute_100a,code=sm_100a), loaded with ctypes by the
 * Python package.  The entry points replace, one for one, the device work that the
 * reference's plugin hierarchy launches through ATen / UMNN on its hot path; the reference
 * file:line each one stands in for is cited on the declaration (paths relative to the
 * reference checkout, see SURVEY.md §8a/§8b).
 *
 * Conventions (SURVEY.md §8b)
 *  - every pointer is a DEVICE pointer to fp32 unless stated, row-major, caller-owned;
 *    the library never allocates or frees device memory and keeps no pointer after return;
 *  - scratch space is passed in by the caller (gnf_*_workspace_bytes tells how much);
 *  - all entry points are asynchronous on `stream` (a cudaStream_t) and re-entrant;
 *  - return 0 on success, non-zero on error (a cudaError_t value, or GNF_ERR_*);
 *    gnf_last_error() gives a thread-local message; an unsupported shape / mode is an
 *    error, never a silent fallback;
 *  - the product library has NO process-global switches: measurement knobs (traces, ablation bits, tiling / engine overrides)
 *    exist only in the development build (-DGNF_DEVTOOLS, libgnf_sm100_dev.so, declared in include/gnf_devtools.h).
 */
#ifndef GNF_H_
#define GNF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* gnf_stream_t; /* cudaStream_t */

#define GNF_ERR_INVALID 1001     /* bad argument */
#define GNF_ERR_UNSUPPORTED 1002 /* shape or mode outside what the kernels cover */
#define GNF_ERR_WORKSPACE 1003   /* workspace too small */
#define GNF_ERR_PEER 1004        /* peer memory (CUDA IPC between the ranks of one node) unavailable */

#define GNF_MAX_LAYERS 8

int gnf_version(void);
const char* gnf_last_error(void);
/* 1 when this build contains device code (always, for the product library). */
int gnf_has_device_code(void);

/* --------------------------------------------------------------------------------------------
 * K4 — AffineNormalizer + log-det + base density
 * ------------------------------------------------------------------------------------------ */

/* AffineNormalizer.forward (models/Normalizers/AffineNormalizer.py:9-12) fused with
 * NormalizingFlowStep.forward's log(jac).sum(1) (models/NormalizingFlow.py:70).
 *   mu = clamp(h[b,i,0],-5,5); ls = clamp(h[b,i,1],-5,2)  (written back into h: in-place
 *   semantics of clamp_);  z = x*exp(ls)+mu;  jac = exp(ls);  logdet[b] = sum_i ls.
 * h: [B,d,H] (H >= 2).  clampmask: [B,d] uint8, bit0 = h0 was inside [-5,5], bit1 = h1 inside
 * [-5,2] (saved for backward).  zrev (nullable): z with reversed columns
 * (FCNormalizingFlow.forward's z[:, inv_idx], NormalizingFlow.py:120,123).  jac nullable. */
int gnf_affine_fwd(const float* x, float* h, int H, float* z, float* zrev, float* jac, float* logdet,
                   uint8_t* clampmask, int B, int d, gnf_stream_t stream);

/* Backward of the above.  gz, gzrev, gjac, glogdet are cotangents (each nullable);
 * gx: [B,d]; gh: [B,d,H] fully written (zeros beyond channel 1). */
int gnf_affine_bwd(const float* x, const float* h, int H, const uint8_t* clampmask, const float* gz,
                   const float* gzrev, const float* gjac, const float* glogdet, float* gx, float* gh, int B,
                   int d, gnf_stream_t stream);

/* NormalLogDensity.forward (models/NormalizingFlowFactories.py:15-16), optionally fused with the
 * `+ jac` of the log-likelihood (UCIExperiments.py:160): out[b] = (logdet? logdet[b]:0) - 0.5*sum_i(log(2pi)+z^2). */
int gnf_normal_ll_fwd(const float* z, const float* logdet, float* out, int B, int d, gnf_stream_t stream);
/* gz[b,i] = -z[b,i]*gout[b]. */
int gnf_normal_ll_bwd(const float* z, const float* gout, float* gz, int B, int d, gnf_stream_t stream);

/* The training loss in one launch (FCNormalizingFlow.loss, NormalizingFlow.py:144-146: constraintsLoss() - log_p_x.mean() with
 * log_p_x = jac + z_log_density(z)): *out = (constraint ? *constraint : 0) - mean_b ll_b.  work: gnf_nll_loss_work_floats(B) floats,
 * caller-owned and reusable across calls; its LAST word is a block counter that must be zero before the first call (the kernel
 * leaves it zero).  Deterministic (block-ordered sum). */
size_t gnf_nll_loss_work_floats(int B);
int gnf_nll_loss_fwd(const float* z, const float* logdet, const float* constraint, float* out, float* work, int B, int d,
                     gnf_stream_t stream);
/* gz[b,i] = z[b,i] g / B, glogdet[b] = -g / B (nullable); g: device scalar cotangent of the loss (NULL = 1). */
int gnf_nll_loss_bwd(const float* z, const float* g, float* gz, float* glogdet, int B, int d, gnf_stream_t stream);

/* --------------------------------------------------------------------------------------------
 * K2 — acyclicity term  tr((I + alpha A∘A)^p) - d
 * (DAGConditioner.get_power_trace, models/Conditionners/DAGConditioner.py:176-194)
 * ------------------------------------------------------------------------------------------ */
size_t gnf_power_trace_workspace_bytes(int d);
/* t_out: device scalar.  Multiplication order follows torch.matrix_power. */
int gnf_power_trace_fwd(const float* A, int d, float alpha, int p, float* t_out, void* work, size_t work_bytes,
                        gnf_stream_t stream);
/* dA = gt * 2*alpha*p * A ∘ ((I+alpha A∘A)^(p-1))^T ;  gt: device scalar. */
int gnf_power_trace_bwd(const float* A, int d, float alpha, int p, const float* gt, float* dA, void* work,
                        size_t work_bytes, gnf_stream_t stream);

/* Training flavour for d <= 64: the forward also leaves G = (I+alpha A∘A)^(p-1) [d,d] in G_out (t = tr(G B) - d as a dot product:
 * the last product's rounding order differs from torch.matrix_power's by ~1e-6 relative), and the backward is one elementwise
 * pass over it instead of a second single-CTA chain of matrix products. */
int gnf_power_trace_fwd_save(const float* A, int d, float alpha, int p, float* t_out, float* G_out, gnf_stream_t stream);
int gnf_power_trace_bwd_saved(const float* A, const float* G, int d, float alpha, int p, const float* gt, float* dA,
                              gnf_stream_t stream);

/* --------------------------------------------------------------------------------------------
 * Conditioner MLP engine (K1 layers 2..L, K5, K6): nn.Linear / ReLU stacks
 * (DAGConditioner.py:7-20, AutoregressiveConditioner.py:24-25, CouplingConditioner.py:6-18)
 * ------------------------------------------------------------------------------------------ */

/* Y[m,n] = act( sum_k X[m,k] W[n,k] + bias[(m % bias_period), n] ),  act = relu or identity.
 * bias: [bias_period, N] (bias_period = 1 -> ordinary bias). */
int gnf_linear_fwd(const float* X, int ldx, const float* W, int ldw, const float* bias, int bias_period, float* Y,
                   int ldy, int M, int N, int K, int relu, gnf_stream_t stream);
/* dX[m,k] = (sum_n dY[m,n] W[n,k]) * (act? act[m,k] > 0 : 1)   (act = the ReLU output feeding this layer). */
int gnf_linear_dgrad(const float* dY, int lddy, const float* W, int ldw, const float* act, int ldact, float* dX,
                     int lddx, int M, int N, int K, gnf_stream_t stream);
/* dW[n,k] = sum_m dY[m,n] X[m,k]  (overwrites dW). */
int gnf_linear_wgrad(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, int M, int N, int K,
                     gnf_stream_t stream);
/* gnf_linear_fwd for a skinny layer with a long reduction (N <= 32, M >= 1024, K >= 128: the conditioner's output layer,
 * DAGConditioner.py:7-20 with out_size = 30): split-K into partial tiles in `work` + a fixed-order sum with bias / ReLU
 * (deterministic).  gnf_linear_fwd_splitk_workspace_bytes returns 0 for shapes it does not take. */
size_t gnf_linear_fwd_splitk_workspace_bytes(int M, int N, int K);
int gnf_linear_fwd_splitk(const float* X, int ldx, const float* W, int ldw, const float* bias, float* Y, int ldy, int M, int N, int K,
                          int relu, void* work, size_t work_bytes, gnf_stream_t stream);
/* out[p,n] = sum_{m % period == p} Y[m,n]  (bias gradients; one-hot column gradients). */
int gnf_colsum(const float* Y, int ldy, float* out, int M, int N, int period, gnf_stream_t stream);

/* The same three GEMMs on the tensor cores (tcgen05.mma kind::tf32, fp32 accumulation in TMEM; warp-specialised
 * persistent kernel, operands staged into 128B-swizzled UMMA tiles by producer warps).
 *   passes = 1: single-pass TF32 (fast mode, log-likelihood tolerance 2e-3);
 *   passes = 3: 3xTF32 hi/lo split, fp32-equivalent (strict mode: ll 1e-4, gradients 1e-3).
 * Forward and dgrad (here and in the _ps / _ps_tb flavours below) store rows in 16-byte pieces: when ldy / lddx leave room for
 * them, they may write zeros into the output columns [N, round_up(N, 4)) (dgrad: [K, round_up(K, 4))), and never write past
 * them.  The weight gradients write the first K columns of dW only. */
int gnf_linear_fwd_tc(const float* X, int ldx, const float* W, int ldw, const float* bias, int bias_period, float* Y,
                      int ldy, int M, int N, int K, int relu, int passes, gnf_stream_t stream);
int gnf_linear_dgrad_tc(const float* dY, int lddy, const float* W, int ldw, const float* act, int ldact, float* dX,
                        int lddx, int M, int N, int K, int passes, gnf_stream_t stream);
int gnf_linear_wgrad_tc(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, int M, int N, int K,
                        int passes, gnf_stream_t stream);
/* Weight AND bias gradient of one nn.Linear in 3xTF32 (autograd of DAGConditioner.py:7-20): dW as gnf_linear_wgrad_tc, and
 * db[n] = sum_m dY[m, n] taken by the weight-gradient engine from the dY tiles it streams anyway (no separate column-sum pass;
 * shapes the engine does not take fall back to gnf_colsum + gnf_linear_wgrad_tc inside).  db: [N], overwritten. */
int gnf_linear_wgrad_bias_tc(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, float* db, int M, int N, int K,
                             gnf_stream_t stream);
/* DAGMLP / MADE / CouplingMLP hidden layers (DAGConditioner.py:7-20, AutoregressiveConditioner.py:24-25, CouplingConditioner.py:6-18)
 * in 3xTF32 with the weights split ONCE per call instead of per tile in shared memory: gnf_split_tf32 writes W_hi = rn_tf32(W) and
 * W_lo = rn_tf32(W - W_hi) as [N][ld] (ld a multiple of 4 floats, 16-byte aligned: both are TMA-loaded); the _ps flavours of
 * forward / dgrad take the pair.  The in-kernel split is bound by shared-memory bandwidth (DESIGN.md §4): dropping the weight
 * half of it shortens the k-chunk cadence. */
int gnf_split_tf32(const float* W, int ldw, float* W_hi, float* W_lo, int ld, int N, int K, gnf_stream_t stream);
int gnf_linear_fwd_tc_ps(const float* X, int ldx, const float* W_hi, const float* W_lo, int ldw, const float* bias, int bias_period,
                         float* Y, int ldy, int M, int N, int K, int relu, gnf_stream_t stream);
/* ... with a periodic bias TABLE of explicit row stride (row m of Y takes row m % period of table [period, ldt]; ldt a multiple of 4
 * floats lets the engine read it in 16-byte pieces whatever N is: DAG layer 1 with the one-hot half as a per-variable bias). */
int gnf_linear_fwd_tc_ps_tb(const float* X, int ldx, const float* W_hi, const float* W_lo, int ldw, const float* table, int ldt,
                            int period, float* Y, int ldy, int M, int N, int K, int relu, gnf_stream_t stream);
int gnf_linear_dgrad_tc_ps(const float* dY, int lddy, const float* W_hi, const float* W_lo, int ldw, const float* act, int ldact,
                           float* dX, int lddx, int M, int N, int K, gnf_stream_t stream);
/* Host-only query of that plan for a GEMM of M x N outputs reduced over K (wgrad != 0: the split-K orientation, where M x N is
 * the weight shape and K the number of rows): writes the tile width and the split-K factor the engine would use. */
int gnf_tc_gemm_plan(int M, int N, int K, int passes, int wgrad, int* bn, int* splits);

/* MaskedLinear's `mask * weight` (AutoregressiveConditioner.py:24-25) fused with the output-row
 * permutation that turns MADE's view(B,out,d).permute(0,2,1) (:108-109) into a plain row-major
 * h[b,i,k]:  out[r,k] = W[perm[r],k] * mask[perm[r],k]   (mask, perm nullable; perm int32 [R]). */
int gnf_pack_rows(const float* W, const float* mask, const int32_t* perm, float* out, int R, int K,
                  gnf_stream_t stream);
/* Scatter for the gradient: dW[perm[r],k] = dWp[r,k]*mask[perm[r],k]; dW [N,K] is zero-filled first. */
int gnf_unpack_rows(const float* dWp, const float* mask, const int32_t* perm, float* dW, int R, int N, int K,
                    gnf_stream_t stream);
/* dst[perm[r]] = src[r] (bias gradient un-permutation; dst [N] zero-filled first; perm nullable = copy). */
int gnf_unpack_vec(const float* src, const int32_t* perm, float* dst, int R, int N, gnf_stream_t stream);

/* --------------------------------------------------------------------------------------------
 * K1 — DAGConditioner masked embedding fused into the first Linear
 * (DAGConditioner.forward, models/Conditionners/DAGConditioner.py:94-169)
 * The [B,d,d] masked tensor e[b,i,j] = x[b,j]*G[b,i,j] is generated inside the GEMM's operand
 * loader and never written to memory.
 * ------------------------------------------------------------------------------------------ */
enum {
  GNF_GATE_TABLE = 0,  /* G[b,i,j] = P[i,j]  (deterministic soft/hard threshold, or raw A after post_process) */
  GNF_GATE_GUMBEL = 1, /* G = z1/(z1+z2), Gumbel relaxed Bernoulli (DAGConditioner.py:94-103) */
  GNF_GATE_NOISER = 2  /* e = P*(x + n*|1-P|)  (noiser_gate, DAGConditioner.py:114-116) */
};
enum { GNF_IMP_RAW = 0, GNF_IMP_SOFT = 1, GNF_IMP_HARD_SOFT = 2, GNF_IMP_HARD_SQ = 3 };

typedef struct {
  int32_t mode;        /* GNF_GATE_* */
  float temperature;   /* gumble_T */
  uint64_t seed;       /* Philox key when noise pointers are NULL */
  uint64_t offset;     /* Philox counter offset (advanced by the caller per forward) */
  const float* noise1; /* optional replay of the reference's draws: u1 (Gumbel) or n (noiser), [B,d,d] */
  const float* noise2; /* u2 (Gumbel), [B,d,d] */
  const uint64_t* offset_dev; /* optional device counter added to `offset` (lets a captured CUDA graph draw fresh
                                 noise on every replay: the counter is bumped by gnf_counter_add inside the graph) */
} gnf_gate_t;

/* Importance table P[d,d] and dP/dA[d,d] from A (DAGConditioner.py:118-124).
 * imp: RAW P=A; SOFT P=2(sigmoid(2A^2)-.5); HARD_SOFT P=soft*[soft>h]; HARD_SQ P=A^2*[A^2>h]. */
int gnf_dag_importance(const float* A, int d, int imp, float h_thresh, float* P, float* dPdA, gnf_stream_t stream);
/* T[i,n] = W1[n, d+i] + b1[n]  (one-hot half of layer 1 as a per-variable bias, hot_encoding=True),
 * or T[0,n] = b1[n] when hot == 0.  W1: [N, ldw]. */
int gnf_dag_bias_table(const float* W1, int ldw, const float* b1, float* T, int d, int N, int hot,
                       gnf_stream_t stream);
/* Gradient of the bias table: dW1[n, d+i] = dT[i,n] (hot), db1[n] = sum_i dT[i,n]. */
/* The same table with an explicit row stride ldt >= N (padding columns zero). */
int gnf_dag_bias_table_ld(const float* W1, int ldw, const float* b1, float* T, int ldt, int d, int N, int hot, gnf_stream_t stream);
int gnf_dag_bias_table_bwd(const float* dT, float* dW1, int ldw, float* db1, int d, int N, int hot,
                           gnf_stream_t stream);
/* Y[b*d+i, n] = act( sum_j x[b,j] G[b,i,j] W1[n,j] + T[i or 0, n] ). */
int gnf_dag_l1_fwd(const float* x, const float* P, const gnf_gate_t* gate, const float* W1, int ldw, const float* T,
                   int bias_period, float* Y, int ldy, int B, int d, int N, int relu, gnf_stream_t stream);
/* dW1[n,j] = sum_{b,i} dY[b*d+i,n] e[b,i,j]  (first d columns of dW1; overwrites them). */
int gnf_dag_l1_wgrad(const float* dY, int lddy, const float* x, const float* P, const gnf_gate_t* gate, float* dW1,
                     int ldw, int B, int d, int N, gnf_stream_t stream);
/* Fused input-cotangent GEMM + reductions; the [B,d,d] cotangent never leaves the SM:
 *   ebar[b,i,j] = sum_n dY[b*d+i,n] W1[n,j];  dx[b,j] = sum_i ebar*de/dx;  dP[i,j] = sum_b ebar*de/dP.
 * dx [B,d] and dP [d,d] are zero-filled by the call. */
int gnf_dag_l1_dgrad(const float* dY, int lddy, const float* W1, int ldw, const float* x, const float* P,
                     const gnf_gate_t* gate, float* dx, float* dP, int B, int d, int N, gnf_stream_t stream);
/* Narrow flows (d <= 64), training with a stochastic gate: gnf_dag_l1_fwd that also leaves e[b,i,j], de/dx and de/dP as planes
 * E / DX / DP ([B*d, 64] floats each, 16-byte aligned, columns >= d zero), and the two backward entry points that read them instead
 * of drawing and evaluating every gate again (autograd of DAGConditioner.py:94-169; same results as the regenerating flavours:
 * the planes hold exactly the values those would recompute). */
int gnf_dag_l1_fwd_save(const float* x, const float* P, const gnf_gate_t* gate, const float* W1, int ldw, const float* T,
                        int bias_period, float* Y, int ldy, float* E, float* DX, float* DP, int B, int d, int N, int relu,
                        gnf_stream_t stream);
/* ... the three planes alone (layer 1's forward then is gnf_linear_fwd_tc_ps against E with the bias table as a periodic bias). */
int gnf_dag_gate_planes(const float* x, const float* P, const gnf_gate_t* gate, float* E, float* DX, float* DP, int B, int d,
                        gnf_stream_t stream);
int gnf_dag_l1_wgrad_saved(const float* dY, int lddy, const float* E, float* dW1, int ldw, int B, int d, int N, gnf_stream_t stream);
int gnf_dag_l1_dgrad_saved(const float* dY, int lddy, const float* W1, int ldw, const float* DX, const float* DP, float* dx,
                           float* dP, int B, int d, int N, gnf_stream_t stream);
/* ... or, with the input-cotangent GEMM dE = dY W1[:, :d] run elsewhere (gnf_linear_dgrad_tc into a [B*d, 64] plane whose columns
 * >= d are zero or finite), only the reductions: dx[b,j] = sum_i dE DX (overwritten), dP[i,j] = sum_b dE DP (zero-filled, atomics). */
int gnf_dag_l1_reduce_saved(const float* dE, const float* DX, const float* DP, float* dx, float* dP, int B, int d, gnf_stream_t stream);
/* Wide flows on the tensor-core GEMM engine (d > 64, cfg5): the masked embedding of DAGConditioner.forward
 * (DAGConditioner.py:126-153: x.unsqueeze(1).expand(-1,d,-1) * gate) written once as a plane
 *   E[b*d+i, j] = x[b,j] G[b,i,j]   ([B*d, lde], lde % 4 == 0, padding columns zero)
 * so that layer 1's forward / weight-gradient / input-cotangent GEMMs run on gnf_linear_*_tc against it.  DX / DP (nullable,
 * both or neither; same shape as E): training also keeps the gate's partial derivatives de/dx and de/dP ... */
int gnf_dag_embed_fwd(const float* x, const float* P, const gnf_gate_t* gate, float* E, float* DX, float* DP, int lde, int B,
                      int d, gnf_stream_t stream);
/* ... for the reduction of the cotangent plane dE = dY W1[:, :d] those GEMMs leave (autograd through the same lines):
 *   dx[b,j] = sum_i dE[b*d+i,j] de/dx(b,i,j);  dP[i,j] = sum_b dE[b*d+i,j] de/dP(b,i,j).  dx is zero-filled by the call.
 * With DX / DP the pass streams the three planes; without them (NULL) the gate is regenerated from x, P and the same Philox
 * counters. */
int gnf_dag_embed_bwd(const float* dE, int lde, const float* x, const float* P, const gnf_gate_t* gate, const float* DX,
                      const float* DP, float* dx, float* dP, int B, int d, gnf_stream_t stream);
/* dA[i,j] (+)= dP[i,j]*dPdA[i,j]. */
int gnf_dag_finish_dA(const float* dP, const float* dPdA, float* dA, int d, int accumulate, gnf_stream_t stream);
/* Debug / parity hook: materialise the in-kernel Philox draws for (seed, offset) as [B,d,d] tensors. */
int gnf_dag_dump_noise(const gnf_gate_t* gate, float* n1, float* n2, int B, int d, gnf_stream_t stream);

/* --------------------------------------------------------------------------------------------
 * K3 — MonotonicNormalizer: fused Clenshaw-Curtis UMNN integral
 * (MonotonicNormalizer.forward, models/Normalizers/MonotonicNormalizer.py:12-66; UMNN==1.0
 * NeuralIntegral / ParallelNeuralIntegral forward + recompute backward, SURVEY.md App. B)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t n_layers;                 /* number of nn.Linear layers (hidden layers + 1) */
  int32_t dims[GNF_MAX_LAYERS + 1]; /* dims[0] = 1 + E, dims[n_layers] = 1 */
  const float* W[GNF_MAX_LAYERS];   /* W[l]: [dims[l+1], dims[l]] row-major (nn.Linear.weight) */
  const float* b[GNF_MAX_LAYERS];   /* b[l]: [dims[l+1]] */
} gnf_mlp_t;

typedef struct {
  float* dW[GNF_MAX_LAYERS]; /* same shapes as gnf_mlp_t; zero-filled by the call, then accumulated */
  float* db[GNF_MAX_LAYERS];
} gnf_mlp_grad_t;

size_t gnf_umnn_workspace_bytes(const gnf_mlp_t* net);
/* x: [R] (R = B*d rows, row r = b*d+i), h: [R,E] -> z[r] = int_0^x f(t;h_r)dt + h[r,0], jac[r] = f(x;h_r).
 * ccw / ccn: [S+1] Clenshaw-Curtis weights and nodes cos(k pi/S) (fp32, computed in float64 by the
 * caller exactly like UMNN's compute_cc_weights).  zrev (nullable): z with the d columns reversed.
 * logdet (nullable): [R/d], logdet[b] = sum_i log jac[b,i].
 * saved (nullable): [R*(S+1), gnf_umnn_saved_floats_per_node_row(net)] buffer in which the forward keeps every hidden
 * activation; handing it to gnf_umnn_bwd replaces the backward's forward recompute (UMNN's memory-saving choice) by a
 * reload — HBM capacity traded for a third of the backward's FLOPs. */
size_t gnf_umnn_saved_floats_per_node_row(const gnf_mlp_t* net);
int gnf_umnn_fwd(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn,
                 float* z, float* zrev, float* jac, float* logdet, float* saved, int R, int d, void* work,
                 size_t work_bytes, gnf_stream_t stream);
/* Inverse of the monotonic transform by bisection (MonotonicNormalizer.inverse_transform, MonotonicNormalizer.py:69-83:
 * 20 halvings of [-20, 20], one full forward pass each; the sampling path FCNormalizingFlow.invert, NormalizingFlow.py:98-107):
 * x[r] such that int_0^x f(t;h_r)dt + h[r,0] = z[r].  All `iters` forward passes of a row run inside one launch (a tile holds
 * every quadrature node of its rows: needs S + 1 <= 64); lo / hi = the initial interval, x = midpoint of the final one. */
int gnf_umnn_invert(const float* z, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn, float* x,
                    int iters, float lo, float hi, int R, void* work, size_t work_bytes, gnf_stream_t stream);
/* Cotangents: gz [R], gzrev [R], gjac [R], glogdet [R/d], each nullable (NULL = zero cotangent).
 * Gradient convention = UMNN's: dtheta, dh by quadrature of the integrand's gradients with weights
 * w_k*gz*x/2; dx by the Leibniz rule f(x)*gz; the jac output is differentiated by the plain chain rule. */
int gnf_umnn_bwd(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn,
                 const float* jac, const float* gz, const float* gzrev, const float* gjac, const float* glogdet,
                 const float* saved, float* dx, float* dh, const gnf_mlp_grad_t* grads, int R, int d, void* work,
                 size_t work_bytes, gnf_stream_t stream);

/* Tensor-core ("fast", single-pass TF32 operands / fp32 TMEM accumulation) forward of the same integral:
 * tcgen05.mma with the activation chain resident in TMEM and all weights resident in shared memory.
 * Same arguments and outputs as gnf_umnn_fwd; per-sample log-likelihood tolerance 2e-3 (north_star's
 * TF32 bar).  Returns GNF_ERR_UNSUPPORTED when the integrand's weights do not fit in shared memory. */
size_t gnf_umnn_tc_workspace_bytes(const gnf_mlp_t* net);
int gnf_umnn_fwd_tc(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn,
                    float* z, float* zrev, float* jac, float* logdet, int R, int d, void* work, size_t work_bytes,
                    gnf_stream_t stream);
/* Layer-wise flavour of the same integral and of its backward: every integrand layer is one pass over all node-rows,
 * the hidden x hidden layers run on the tensor-core GEMM engine (passes = 3: 3xTF32, fp32-equivalent; 1: TF32;
 * 0: the strict FFMA tile GEMM), the conditioning half of the first layer is evaluated once per row instead of once
 * per quadrature node, and hidden activations live in HBM between the passes.
 * saved: [gnf_umnn_lw_saved_floats(net, R, S, train)] floats, written by the forward (L planes [Q, NP] + y [Q]);
 * train != 0 adds the node-row that carries the chain rule of the jac output and is required by gnf_umnn_bwd_lw.
 * Outputs, cotangents and gradient conventions are those of gnf_umnn_fwd / gnf_umnn_bwd. */
size_t gnf_umnn_lw_saved_floats(const gnf_mlp_t* net, int R, int S, int train);
size_t gnf_umnn_lw_workspace_bytes(const gnf_mlp_t* net, int R, int S, int backward);
int gnf_umnn_fwd_lw(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn,
                    float* z, float* zrev, float* jac, float* logdet, float* saved, int train, int passes, int R, int d,
                    void* work, size_t work_bytes, gnf_stream_t stream);
int gnf_umnn_bwd_lw(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn,
                    const float* jac, const float* gz, const float* gzrev, const float* gjac, const float* glogdet,
                    const float* saved, float* dx, float* dh, const gnf_mlp_grad_t* grads, int passes, int R, int d,
                    void* work, size_t work_bytes, gnf_stream_t stream);

/* Fused strict forward of the same integral on the tensor cores (tc_umnn3.cu): 3xTF32 (fp32-equivalent, round-to-nearest
 * hi/lo split), the activation chain of a 128-node-row tile resident in TMEM from the first to the last hidden layer, the
 * hidden weights streamed through shared memory as pre-split hi/lo K-chunks.  Replaces the per-layer passes of
 * gnf_umnn_fwd_lw (MonotonicNormalizer.py:51-66 / UMNN ParallelNeuralIntegral forward): same outputs, and -- when
 * `saved` is given -- the same saved-activation buffer, so that gnf_umnn_bwd_lw consumes it unchanged; in training
 * (train != 0) the buffer holds gnf_umnn_tc3_saved_floats(net, R, S) floats: the layer-wise layout followed by the ReLU bit
 * mask of the last hidden activation, which gnf_umnn_bwd_tc3 starts from.  saved == NULL (evaluation): no activation touches HBM.
 * order: 0 = per K-chunk a_lo*b_hi, a_hi*b_lo, a_hi*b_hi; 1 = all correction products of a layer first (the hi images
 * are streamed twice).  Hidden widths <= 160, >= 3 linear layers; otherwise GNF_ERR_UNSUPPORTED.
 * work: gnf_umnn_tc3_workspace_bytes(net, R) bytes, 16-byte aligned. */
size_t gnf_umnn_tc3_workspace_bytes(const gnf_mlp_t* net, int R);
size_t gnf_umnn_tc3_saved_floats(const gnf_mlp_t* net, int R, int S);
int gnf_umnn_fwd_tc3(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn,
                     float* z, float* zrev, float* jac, float* logdet, float* saved, int train, int order, int R, int d,
                     void* work, size_t work_bytes, gnf_stream_t stream);

/* One Adam step over a list of parameter tensors in one launch (per 48 tensors): the optimizer of the reference's training
 * loops (torch.optim.Adam(model.parameters(), lr, weight_decay), UCIExperiments.py:100, ToyExperiments.py:59; L2 weight decay,
 * no amsgrad):  g += wd*p;  m += (1-b1)(g-m);  v = b2 v + (1-b2) g^2;  p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
 * with t = *step_dev + 1.  `tensors` is a HOST array (device pointers inside); step_dev a device int64 counter of the steps done
 * so far -- the caller increments it after the call (gnf_counter_add), which keeps the pair capturable in a CUDA graph. */
typedef struct {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int64_t numel;
} gnf_adam_tensor_t;
int gnf_adam_step(const gnf_adam_tensor_t* tensors, int n_tensors, const int64_t* step_dev, float lr, float beta1, float beta2,
                  float eps, float weight_decay, gnf_stream_t stream);

/* --------------------------------------------------------------------------------------------
 * Data-parallel gradient exchange over NVLink peer memory (one process per GPU; replaces the gradient gather of the
 * reference's nn.DataParallel, ImageExperiments.py:168, and the NCCL all-reduce of the flat bucket): every rank allocates its
 * bucket and a flag block with gnf_peer_alloc (the one place where the library allocates device memory: cudaIpc needs a
 * cudaMalloc base), exports 64-byte handles, imports its peers' and passes the pointer tables to gnf_peer_allreduce_avg:
 * ONE kernel = barrier, reduce-scatter by peer loads, all-gather by peer stores, barrier; in place, bit-identical on every
 * rank, replayable inside a CUDA graph (the barrier epoch lives in the flag block).
 * -------------------------------------------------------------------------------------------- */
int gnf_peer_alloc(size_t bytes, void** out);                    /* zero-filled */
int gnf_peer_free(void* p);
int gnf_peer_export(const void* p, unsigned char* handle64);     /* cudaIpcGetMemHandle */
int gnf_peer_import(const unsigned char* handle64, void** out);  /* cudaIpcOpenMemHandle with lazy peer access */
int gnf_peer_close(void* p);
size_t gnf_peer_flag_bytes(void);
/* bufs / flags: [world] device pointers (entry `rank` = this rank's own allocations), numel % 4 == 0, world <= 16.
 * Every rank of the group must make the call once per step; bufs[rank][0..numel) becomes the mean over ranks. */
int gnf_peer_allreduce_avg(float* const* bufs, unsigned* const* flags, int rank, int world, long long numel,
                           gnf_stream_t stream);

/* Backward of the integral with the dgrad chain fused on the tensor cores (UMNN NeuralIntegral.backward, SURVEY App. B; same
 * cotangents, outputs and gradient conventions as gnf_umnn_bwd / gnf_umnn_bwd_lw; 3xTF32): the cotangent of the pre-ELU output is
 * pushed from the last hidden layer down to the first in ONE kernel (delta planes for the weight-gradient GEMMs, bias gradients and
 * the first layer's per-row reductions leave the chip; no dgrad activation plane is re-read), followed by the resident
 * weight-gradient GEMMs.  `saved` must have been written by gnf_umnn_fwd_tc3 with train != 0.
 * work: gnf_umnn_bwd_tc3_workspace_bytes(net, R, S) bytes (0 = integrand not covered, see gnf_last_error), 16-byte aligned. */
size_t gnf_umnn_bwd_tc3_workspace_bytes(const gnf_mlp_t* net, int R, int S);
int gnf_umnn_bwd_tc3(const float* x, const float* h, const gnf_mlp_t* net, int S, const float* ccw, const float* ccn,
                     const float* jac, const float* gz, const float* gzrev, const float* gjac, const float* glogdet,
                     const float* saved, float* dx, float* dh, const gnf_mlp_grad_t* grads, int R, int d, void* work,
                     size_t work_bytes, gnf_stream_t stream);

/* DAGConditioner.loss (DAGConditioner.py:268-271) fused:  out = dag_const*(lambd*t + c/2*t^2) + l1_weight*mean|A|, with the
 * dual variables read from their device buffers (lambd, c, dag_const, l1_weight: one float each, as registered by the
 * reference's constructor :86-91) and t = the power trace (gnf_power_trace_fwd).  fp32, reference evaluation order (t^2
 * overflows to inf where the reference's does).  Backward: dA = g*l1_weight*sign(A)/d^2 (the l1 term only; the trace's own
 * dependence on A flows through gnf_power_trace_bwd), dt = g*dag_const*(lambd + c*t). */
int gnf_dag_loss_fwd(const float* A, int d, const float* t, const float* lambd, const float* c, const float* dag_const,
                     const float* l1_weight, float* out, gnf_stream_t stream);
int gnf_dag_loss_bwd(const float* A, int d, const float* t, const float* lambd, const float* c, const float* dag_const,
                     const float* l1_weight, const float* gout, float* dA, float* dt, gnf_stream_t stream);


/* Resident-weight tensor-core layer GEMM (tc_rw.cu) -- the hidden x hidden layers of IntegrandNet
 * (MonotonicNormalizer.py:12-38) over all quadrature node-rows, forward and dgrad.  The layer's weights (N, K <= 160) are
 * split into TF32 hi / lo images once per call and stay resident in shared memory; the activations stream global ->
 * registers -> TMEM (no shared-memory staging), TS-form tcgen05.mma, row-owner epilogue.  passes as gnf_linear_*_tc.
 * Operand contract (what the layer-wise engine's padded planes satisfy): X / dY / Y / dX rows 32-byte aligned (leading dimensions multiples of 8), X / dY with
 * round_up(K or N, 32) readable columns whose padding is zero; Y / dX receive round_up(N or K, 32) columns per row.
 * bits_out (nullable): ReLU bit mask of Y, [M][round_up(N,32)/32] words; mask_bits (nullable, same layout) or act select
 * the ReLU mask of dgrad.  work: gnf_linear_rw_workspace_bytes(N, K) bytes (0 = shape unsupported, see gnf_last_error). */
size_t gnf_linear_rw_workspace_bytes(int N, int K);
int gnf_linear_fwd_rw(const float* X, int ldx, const float* W, int ldw, const float* bias, float* Y, int ldy, uint32_t* bits_out,
                      int M, int N, int K, int relu, int passes, void* work, size_t work_bytes, gnf_stream_t stream);
int gnf_linear_dgrad_rw(const float* dY, int lddy, const float* W, int ldw, const float* act, int ldact,
                        const uint32_t* mask_bits, float* dX, int lddx, int M, int N, int K, int passes, void* work,
                        size_t work_bytes, gnf_stream_t stream);

/* Weight gradient of an IntegrandNet hidden layer (MonotonicNormalizer.py:12-38) over all quadrature node-rows -- the parameter
 * gradient UMNN's NeuralIntegral.backward accumulates node by node (SURVEY App. B) -- (tc_rw_wgrad.cu): dW[N,K] = dY^T X,
 * N, K <= 160, M rows.  TMEM lane =
 * output row, so dY^T is gathered straight from the row-major dY (a warp reads dY[q, n0..n0+31]); X must be a dense
 * [M][round_up(K,32)] plane (ldx = round_up(K,32), 16-byte aligned) and is streamed once by bulk async copies; per-CTA partial
 * tiles in `work` (gnf_linear_wgrad_rw_workspace_bytes(N, K)) are summed by a second kernel (deterministic). */
size_t gnf_linear_wgrad_rw_workspace_bytes(int N, int K);
int gnf_linear_wgrad_rw(const float* dY, int lddy, const float* X, int ldx, float* dW, int lddw, int M, int N, int K,
                        int passes, void* work, size_t work_bytes, gnf_stream_t stream);

/* Self-test of the tcgen05 conventions: C[128,N] = A[128,K] W[N,K]^T on one CTA (mode 0: A staged in TMEM,
 * mode 1: A staged in shared memory).  N, K <= 256. */
int gnf_tc_selftest(const float* A, const float* W, float* C, int N, int K, int mode, gnf_stream_t stream);

/* --------------------------------------------------------------------------------------------
 * Small elementwise helpers used by the host side
 * ------------------------------------------------------------------------------------------ */
/* dst[b, d-1-i] = src[b,i]. */
int gnf_reverse_cols(const float* src, float* dst, int B, int d, gnf_stream_t stream);
/* CouplingConditioner: h[b,i,:] = constants[i,:] for i < indep (CouplingConditioner.py:33). h: [B,d,H]. */
int gnf_broadcast_rows(const float* constants, float* h, int B, int d, int indep, int H, gnf_stream_t stream);
/* *counter += inc  (device-side Philox offset for graph-captured training steps). */
int gnf_counter_add(uint64_t* counter, uint64_t inc, gnf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GNF_H_ */
