/* libgnf_sm100_dev.so ONLY (built with -DGNF_DEVTOOLS by `python graphical-normalizing-flows_b200/build.py --dev`):
 * measurement knobs used by scripts/ -- SM-clock traces of the warp roles, ablation bits, tiling and engine overrides, hardware
 * probes.  They are process-global switches, which is exactly why the product library (include/gnf.h) does not contain them:
 * it is stateless and re-entrant (SURVEY.md 8b).  scripts/devlib.py loads the development build in place of the product one. */
#ifndef GNF_DEVTOOLS_H_
#define GNF_DEVTOOLS_H_

#include "gnf.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Measurement switch: 0 makes the tensor-core GEMM stage every operand with cp.async (the path taken anyway by operands
 * whose base / leading dimension are not 16-byte aligned) instead of TMA tensor maps.  Default 1. */
int gnf_tc_gemm_set_tma(int enable);

/* Measurement switch: force the tensor-core GEMM's tile width (64, 96, ... 256 columns; 3xTF32 is capped at 160) and / or the
 * split-K factor of the wgrad orientation; 0 = planned per shape (fill of the last round of work items over the SMs). */
int gnf_tc_gemm_set_tile(int bn, int splits);

/* 3xTF32 accuracy knob: k-chunks (of 32) accumulated inside the tensor core (round-toward-zero accumulation) before the
 * partial sum is folded into a round-to-nearest running sum.  Default 2; a huge value disables folding. */
int gnf_tc_gemm_set_fold(int chunks);

/* Measurement: later tensor-core GEMM launches write SM-clock stamps of CTA 0's warp roles into buf (8 x 256 int64, device;
 * rows: TMA issue, stager landed, stager published, MMA chunk ready, MMA tile committed, epilogue start, epilogue end). */
int gnf_tc_gemm_set_trace(long long* buf);

/* Measurement switch: 1 (default) = narrow flows (d <= 64) run layer 1 on the kernels that keep the gate tile of a row block
 * resident in shared memory (every gate evaluated once per direction); 0 = functor-loader tile GEMM for every d. */
int gnf_dag_l1_set_resident(int enable);

/* Measurement switch: 0 routes the layer-wise engine's hidden GEMMs to the generic tensor-core engine (gnf_linear_*_tc)
 * instead of the resident-weight kernels below; 3 keeps forward/dgrad resident but runs wgrad on the generic engine.  Default 1. */
int gnf_umnn_lw_set_rw(int enable);

/* Measurement: later resident-weight GEMM launches write SM-clock stamps of CTA 0 into buf (4 x 256 int64, device; rows:
 * MMA issuer, loader of even chunks, loader of odd chunks, epilogue).  NULL disables. */
int gnf_linear_rw_set_trace(long long* buf);

/* Measurement: bit0 skips the kernel's global stores, bit1 its global loads, bit2 its MMAs (results are then garbage). */
int gnf_linear_rw_set_debug(int bits);

/* Measurement: later gnf_linear_wgrad_rw launches write SM-clock stamps of CTA 0 into buf (3 x 256 int64, device; rows: MMA
 * issuer, first stager thread, first loader thread).  NULL disables. */
int gnf_linear_wgrad_rw_set_trace(long long* buf);

/* Measurement tool (not on the product path): TMEM-read bandwidth / MMA issue rate / overlap probe on one CTA.
 * mode bit0: stream tcgen05.ld; bit1: issue TF32 MMAs; out[0], out[1]: elapsed SM clocks of the two roles. */
int gnf_tc_probe(int mode, int iters, long long* out, gnf_stream_t stream);

/* Debug / measurement: later gnf_umnn_fwd_tc calls write per-phase SM-clock stamps of CTA 0 into buf (48*8 int64). */
int gnf_tc_set_trace(long long* buf);

/* Measurement switch: 0 keeps the pre-split forward / dgrad GEMMs on the first engine (stagers split the activation tile in shared
 * memory); 1 (default) = engine v2.  Any other value is GNF_ERR_INVALID. */
int gnf_tc_gemm_set_v2(int enable);
/* Fused strict UMNN forward (tc_umnn3.cu): CTA 0 records SM-clock stamps into buf[4][256] (rows: issuer, epilogue warp 0,
 * producer, epilogue warp of the last column block); NULL disables. */
int gnf_umnn_tc3_set_trace(long long* buf);
/* 0: skinny layers (one weight dimension <= 32) run on the register-tiled GEMM instead of the kernels of csrc/thin.cuh. */
int gnf_linear_set_thin(int enable);
/* Ablation: bit0 skip the global stores of the saved planes, bit1 skip their staging too, bit2 skip masks / pre-ELU outputs. */
int gnf_umnn_tc3_set_debug(int bits);

#ifdef __cplusplus
}
#endif
#endif
