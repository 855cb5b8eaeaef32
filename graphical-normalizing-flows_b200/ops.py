"""torch.autograd.Function wrappers over the C-ABI (include/gnf.h).

Operator layer of the drop-in boundary (SURVEY.md §8b): the same role the reference gives to
``UMNN.NeuralIntegral.apply`` — custom forward/backward pairs whose arithmetic lives in the
hand-written sm_100a kernels.  Tensors, workspaces and saved-for-backward buffers are torch
allocations handed to the library as raw device pointers on torch's current stream.
"""
import ctypes as C
import math
import weakref

import numpy as np
import torch

from . import _lib as L
from ._lib import check, lib, ptr, require, stream_ptr

_LAUNCHES = 0  # number of C-ABI compute calls issued (bench.py reports it as gpu_launches evidence)


def _count(n=1):
    global _LAUNCHES
    _LAUNCHES += n


_TIMING = False
_TIMES = {}


def enable_kernel_timing(flag):
    """bench.py: bracket every C-ABI call with CUDA events on the launching stream."""
    global _TIMING
    _TIMING = bool(flag)
    if flag:
        _TIMES.clear()
        _FLOPS.clear()
        _SHAPES.clear()


def collect_kernel_timing():
    """{entry point: [ms per call]} — synchronises."""
    torch.cuda.synchronize()
    return {k: [a.elapsed_time(b) for a, b in v] for k, v in _TIMES.items()}


_FLOPS = {}


def collect_call_flops():
    """{entry point: [algorithmic FLOPs per call]} for the GEMM entry points timed since enable_kernel_timing(True)."""
    return {k: list(v) for k, v in _FLOPS.items()}


_SHAPES = {}


def collect_call_shapes():
    """{entry point: [(M, N, K) per call]} for the GEMM entry points timed since enable_kernel_timing(True)."""
    return {k: list(v) for k, v in _SHAPES.items()}


def _note_flops(name, flops, shape=None):
    if _TIMING:
        _FLOPS.setdefault(name, []).append(float(flops))
        _SHAPES.setdefault(name, []).append(shape)


def tc_kernel_name(op, M, N, K, passes=3):
    """Which kernel of the tcgen05 GEMM engine a layer call of this shape launches (mirrors g2_eligible / w2_eligible in
    csrc/tc_gemm.cu for TMA-loadable operands, and for bias tables / context terms with rows of 16-byte pieces, as DagMlpFn
    makes them): op 'fwd' / 'dgrad' (M rows, N out-features, K in-features) or 'wgrad'."""
    if passes == 3:
        if op == "wgrad":
            return "tc_wgrad2_kernel" if (N >= 256 and (K >= 256 or 32 <= K <= 64) and M >= 2048) else "tc_gemm_kernel"
        n, k = (N, K) if op == "fwd" else (K, N)
        return "tc_gemm2_kernel" if (M >= 1024 and ((n >= 256 and k >= 128) or (32 <= k <= 64 and n >= 256) or (32 <= n <= 64 and k >= 256))) else "tc_gemm_kernel"
    return "tc_gemm_kernel"


_TIMES_ALIAS = {}    # entry point -> the name its timings are filed under (flavours of one kernel)


def _call(name, *args):
    fn = getattr(lib(), name)
    if _TIMING and not L._SIMULATOR:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        _TIMES.setdefault(_TIMES_ALIAS.get(name, name), []).append((e0, e1))
    else:
        rc = fn(*args)
    check(rc)


def launch_count():
    return _LAUNCHES


# Independent pieces of one backward (a layer's weight gradient, bias-table gradient and input cotangent; the wgrad and dgrad of a
# skinny layer) are enqueued on side streams between a fork and a join: inside a captured step they become parallel branches of the
# graph, and kernels that fill a fraction of the SMs run next to each other.  Discipline (caching allocator): a fork always waits for
# the forking stream, every tensor a branch reads or writes stays referenced until the join.
PARALLEL_BRANCHES = True
_SIDE_STREAMS = {}


class _Fork:
    def __init__(self, k, like):
        self.on = PARALLEL_BRANCHES and like.is_cuda and not L._SIMULATOR
        if self.on:
            key = (like.device.index, k)
            if key not in _SIDE_STREAMS:
                _SIDE_STREAMS[key] = torch.cuda.Stream(device=like.device)
            self.side = _SIDE_STREAMS[key]

    def __enter__(self):
        if self.on:
            self.cur = torch.cuda.current_stream()
            self.side.wait_stream(self.cur)
            self.ctx = torch.cuda.stream(self.side)
            self.ctx.__enter__()
        return self

    def __exit__(self, *a):
        if self.on:
            self.ctx.__exit__(*a)

    def join(self):
        if self.on:
            self.cur.wait_stream(self.side)


def _contig(t):
    return t if t.is_contiguous() else t.contiguous()


# ----------------------------------------------------------------------------------------------
# K4: affine normalizer, base density
# ----------------------------------------------------------------------------------------------
class AffineFn(torch.autograd.Function):
    """AffineNormalizer.forward + log(jac).sum(1) (AffineNormalizer.py:9-12, NormalizingFlow.py:70).

    Returns (z, jac, logdet, zrev).  Like the reference's clamp_, the clamped mu / log-sigma are written
    back into h's storage; h's autograd version counter is bumped so that an upstream op that saved h for
    its own backward fails loudly instead of silently using modified values."""

    @staticmethod
    def forward(ctx, x, h, want_rev):
        require(x, "x"), require(h, "h")
        B, d = x.shape
        H = h.shape[2]
        if h.shape[0] != B or h.shape[1] != d or H < 2:
            raise ValueError(f"AffineNormalizer: h must be [B, d, >=2], got {tuple(h.shape)} for x {tuple(x.shape)}")
        z = torch.empty_like(x)
        jac = torch.empty_like(x)
        zrev = torch.empty_like(x) if want_rev else None
        logdet = torch.empty(B, device=x.device, dtype=x.dtype)
        mask = torch.empty(B, d, device=x.device, dtype=torch.uint8)
        _call("gnf_affine_fwd", ptr(x), ptr(h), H, ptr(z), ptr(zrev), ptr(jac), ptr(logdet), ptr(mask), B, d, stream_ptr())
        _count()
        torch.autograd.graph.increment_version(h)
        ctx.save_for_backward(x, h, mask)
        ctx.want_rev = want_rev
        ctx.set_materialize_grads(False)
        if zrev is None:
            zrev = x.new_empty(0)
            ctx.mark_non_differentiable(zrev)
        return z, jac, logdet, zrev

    @staticmethod
    def backward(ctx, gz, gjac, glogdet, gzrev):
        x, h, mask = ctx.saved_tensors
        B, d = x.shape
        H = h.shape[2]
        gz = _contig(gz) if gz is not None else None
        gjac = _contig(gjac) if gjac is not None else None
        glogdet = _contig(glogdet) if glogdet is not None else None
        gzrev = _contig(gzrev) if (gzrev is not None and ctx.want_rev) else None
        gx = torch.empty_like(x)
        gh = torch.empty_like(h)
        _call("gnf_affine_bwd", ptr(x), ptr(h), H, ptr(mask), ptr(gz), ptr(gzrev), ptr(gjac), ptr(glogdet), ptr(gx), ptr(gh),
                                   B, d, stream_ptr())
        _count()
        return gx, gh, None


class NormalLLFn(torch.autograd.Function):
    """out[b] = (logdet[b]) - 0.5 * sum_i (log 2pi + z^2)  (NormalizingFlowFactories.py:15-16)."""

    @staticmethod
    def forward(ctx, z, logdet):
        require(z, "z")
        B, d = z.shape
        if logdet is not None:
            require(logdet, "logdet")
        out = torch.empty(B, device=z.device, dtype=z.dtype)
        _call("gnf_normal_ll_fwd", ptr(z), ptr(logdet), ptr(out), B, d, stream_ptr())
        _count()
        ctx.save_for_backward(z)
        ctx.has_logdet = logdet is not None
        return out

    @staticmethod
    def backward(ctx, gout):
        (z,) = ctx.saved_tensors
        gout = _contig(gout)
        gz = torch.empty_like(z)
        _call("gnf_normal_ll_bwd", ptr(z), ptr(gout), ptr(gz), z.shape[0], z.shape[1], stream_ptr())
        _count()
        return gz, (gout if ctx.has_logdet else None)


_NLL_WORK = {}


class NllLossFn(torch.autograd.Function):
    """FCNormalizingFlow.loss (NormalizingFlow.py:144-146) with the standard-normal base density: constraint - mean_b(logdet_b +
    log N(z_b)) as ONE kernel per direction instead of the density kernel + mean / neg / add (and their autograd nodes).
    forward(z [B,d], logdet [B], constraint: 0-dim tensor or None) -> 0-dim loss."""

    @staticmethod
    def forward(ctx, z, logdet, constraint):
        require(z, "z"), require(logdet, "logdet")
        B, d = z.shape
        if constraint is not None:
            require(constraint, "constraint")
        # one persistent buffer per (device, stream): calls on one stream are ordered, calls on different streams must not share the
        # partial sums (made by the eager warm-up steps before any graph capture)
        key = (z.device, torch.cuda.current_stream().cuda_stream if z.is_cuda else 0)
        n = lib().gnf_nll_loss_work_floats(B)
        work = _NLL_WORK.get(key)
        if work is None or work.numel() < n or L._SIMULATOR:
            work = torch.zeros(max(n, 256), device=z.device, dtype=torch.float32)      # the trailing block counter starts at zero and is left at zero
            _NLL_WORK[key] = work
        out = torch.empty((), device=z.device, dtype=z.dtype)
        _call("gnf_nll_loss_fwd", ptr(z), ptr(logdet), ptr(constraint), ptr(out), ptr(work[work.numel() - n:]), B, d, stream_ptr())
        _count()
        ctx.save_for_backward(z)
        ctx.has_constraint = constraint is not None
        return out

    @staticmethod
    def backward(ctx, g):
        (z,) = ctx.saved_tensors
        g = _contig(g)
        gz = torch.empty_like(z)
        glogdet = torch.empty(z.shape[0], device=z.device, dtype=z.dtype)
        _call("gnf_nll_loss_bwd", ptr(z), ptr(g), ptr(gz), ptr(glogdet), z.shape[0], z.shape[1], stream_ptr())
        _count()
        return gz, glogdet, (g if ctx.has_constraint else None)


def reverse_cols(z):
    require(z, "z")
    out = torch.empty_like(z)
    _call("gnf_reverse_cols", ptr(z), ptr(out), z.shape[0], z.shape[1], stream_ptr())
    _count()
    return out


class ReverseColsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z):
        return reverse_cols(z)

    @staticmethod
    def backward(ctx, g):
        return reverse_cols(_contig(g))


# ----------------------------------------------------------------------------------------------
# K2: acyclicity term
# ----------------------------------------------------------------------------------------------
def _pt_workspace(d, device):
    n = lib().gnf_power_trace_workspace_bytes(d)
    return torch.empty((n + 3) // 4, device=device, dtype=torch.float32), n


POWER_TRACE_SAVE_MAX_D = 64   # d <= 64 and A needs a gradient: the forward leaves (I + alpha A∘A)^(p-1) for the backward


class PowerTraceFn(torch.autograd.Function):
    """tr((I + alpha A∘A)^p) - d  (DAGConditioner.get_power_trace, DAGConditioner.py:176-194)."""

    @staticmethod
    def forward(ctx, A, alpha, p):
        require(A, "A")
        d = A.shape[0]
        t = torch.empty((), device=A.device, dtype=A.dtype)
        ctx.alpha, ctx.p = float(alpha), int(p)
        if d <= POWER_TRACE_SAVE_MAX_D and ctx.needs_input_grad[0]:
            G = torch.empty(d, d, device=A.device, dtype=A.dtype)
            _TIMES_ALIAS["gnf_power_trace_fwd_save"] = "gnf_power_trace_fwd"
            _call("gnf_power_trace_fwd_save", ptr(A), d, float(alpha), int(p), ptr(t), ptr(G), stream_ptr())
            _count()
            ctx.save_for_backward(A, G)
            return t
        ws, n = _pt_workspace(d, A.device)
        _call("gnf_power_trace_fwd", ptr(A), d, float(alpha), int(p), ptr(t), ptr(ws), n, stream_ptr())
        _count()
        ctx.save_for_backward(A)
        return t

    @staticmethod
    def backward(ctx, gt):
        A = ctx.saved_tensors[0]
        d = A.shape[0]
        gt = _contig(gt)
        dA = torch.empty_like(A)
        if len(ctx.saved_tensors) == 2:
            _TIMES_ALIAS["gnf_power_trace_bwd_saved"] = "gnf_power_trace_bwd"
            _call("gnf_power_trace_bwd_saved", ptr(A), ptr(ctx.saved_tensors[1]), d, ctx.alpha, ctx.p, ptr(gt), ptr(dA), stream_ptr())
            _count()
            return dA, None, None
        ws, n = _pt_workspace(d, A.device)
        _call("gnf_power_trace_bwd", ptr(A), d, ctx.alpha, ctx.p, ptr(gt), ptr(dA), ptr(ws), n, stream_ptr())
        _count()
        return dA, None, None


class DagLossFn(torch.autograd.Function):
    """DAGConditioner.loss (DAGConditioner.py:268-271): dag_const*(lambd*t + c/2*t^2) + l1_weight*mean|A| in one launch
    per direction (a dozen scalar torch kernels otherwise).  lambd / c / dag_const / l1_weight are the module's device
    buffers; they receive no gradient (the reference's are buffers too)."""

    @staticmethod
    def forward(ctx, A, t, lambd, c, dag_const, l1_weight):
        require(A, "A"), require(t, "t")
        duals = [require(_contig(v.detach()), "dual variable") for v in (lambd, c, dag_const, l1_weight)]
        out = torch.empty((), device=A.device, dtype=A.dtype)
        _call("gnf_dag_loss_fwd", ptr(A), A.shape[0], ptr(t), *[ptr(v) for v in duals], ptr(out), stream_ptr())
        _count()
        ctx.save_for_backward(A, t, *duals)
        return out

    @staticmethod
    def backward(ctx, g):
        A, t, lambd, c, dag_const, l1_weight = ctx.saved_tensors
        g = _contig(g)
        dA = torch.empty_like(A)
        dt = torch.empty_like(t)
        _call("gnf_dag_loss_bwd", ptr(A), A.shape[0], ptr(t), ptr(lambd), ptr(c), ptr(dag_const), ptr(l1_weight), ptr(g), ptr(dA),
              ptr(dt), stream_ptr())
        _count()
        return dA, dt, None, None, None, None


# ----------------------------------------------------------------------------------------------
# Conditioner MLP engine
# ----------------------------------------------------------------------------------------------
_GEMM_MODE = "ffma"
_GEMM_MODES = ("ffma", "tf32", "tf32x3", "auto", "auto-fast")


def set_gemm_mode(mode):
    """Select the conditioner-MLP GEMM engine.
      'ffma'      fp32 CUDA-core tile GEMM (strict);
      'tf32x3'    tensor cores (tcgen05), 3xTF32 split, fp32-equivalent (strict);
      'tf32'      tensor cores, single-pass TF32 (ll tolerance 2e-3; not for gradient parity);
      'auto'      strict: tf32x3 where it beats the FFMA engine (large M*N*K, N and K >= 256), else ffma;
      'auto-fast' tf32 where N and K >= 128, else ffma."""
    global _GEMM_MODE
    if mode not in _GEMM_MODES:
        raise ValueError(f"gemm mode must be one of {_GEMM_MODES}")
    _GEMM_MODE = mode


def get_gemm_mode():
    return _GEMM_MODE


def _gemm_passes(M, N, K, op="fwd"):
    """0 = FFMA engine, 1 / 3 = tensor-core engine passes; thresholds from scripts/gemm_bench.py on B200 with
    TMA-loadable operands (16-byte aligned rows: activations are allocated with padded row strides and weights get a
    padded copy, see _rows / _tma_weight): 3xTF32 beats the FFMA engine from ~0.4 GFLOP-sized layers on, e.g.
    6300 x 632 x 632: 78 vs 144 us, 10000 x 212 x 212: 37 vs 55 us (profiles/r01y_gemm_bench_generic.txt)."""
    if _GEMM_MODE == "ffma":
        return 0
    if _GEMM_MODE == "tf32":
        return 1
    if _GEMM_MODE == "tf32x3":
        return 3
    if _GEMM_MODE == "auto":
        if op == "wgrad":
            return 3 if (min(N, K) >= 128 and M >= 4096) else 0
        return 3 if (min(N, K) >= 128 and float(M) * N * K >= 4e8) else 0
    return 1 if min(N, K) >= 128 else 0


def _pad4(n):
    return (n + 3) // 4 * 4


def _rows(M, N, like):
    """[M, N] activation buffer whose rows start 16-byte aligned (row stride padded to 4 floats): what the tensor-core
    engine's TMA tensor maps need; every kernel takes the row stride explicitly."""
    t = torch.empty(M, _pad4(N), device=like.device, dtype=like.dtype)
    return t if t.shape[1] == N else t[:, :N]


def _tma_weight(W):
    """W itself if its rows are 16-byte aligned, else a copy with the row stride padded to 4 floats (630 -> 632): the
    unaligned staging path of the tensor-core engine is 2x slower than TMA (148 vs 78 us at 6300 x 630 x 630)."""
    if W.stride(0) % 4 == 0 and W.data_ptr() % 16 == 0:
        return W
    Wp = _rows(W.shape[0], W.shape[1], W)
    Wp.copy_(W)
    return Wp


SPLITK_SKINNY = True         # skinny layers with a long reduction (630 -> 30) on the FFMA engine: deterministic split-K (gnf_linear_fwd_splitk)


_SPLIT_CACHE = {}


def _split_weight(W):
    """(W_hi, W_lo) with rows padded to 4 floats, for the *_tc_ps entry points: in 3xTF32 the weights are split once per call
    (gnf_split_tf32) instead of per tile in shared memory.  The forward's split is reused by the same
    step's dgrad: keyed by storage and version (optimizers update in place, which bumps the version), and by the stream
    capture state so that a captured step never refers to tensors made outside its graph."""
    key = (W.data_ptr(), W._version, tuple(W.shape), torch.cuda.is_current_stream_capturing() if W.is_cuda else False)
    hit = _SPLIT_CACHE.get(key)
    if hit is not None and hit[2]() is W:
        return hit[0], hit[1]
    N, K = W.shape
    hi = torch.empty(N, _pad4(K), device=W.device, dtype=W.dtype)
    lo = torch.empty_like(hi)
    _call("gnf_split_tf32", ptr(W), W.stride(0), ptr(hi), ptr(lo), hi.stride(0), N, K, stream_ptr())
    _count()
    if len(_SPLIT_CACHE) >= 16:
        _SPLIT_CACHE.clear()
    _SPLIT_CACHE[key] = (hi, lo, weakref.ref(W))
    return hi, lo


def _tma_ok(t, ld):
    return t.data_ptr() % 16 == 0 and ld % 4 == 0


def linear_fwd(X, W, bias, relu, bias_period=1, out=None, ldy=None, K=None, ldx=None):
    """Y = act(X[:, :K] @ W^T + bias).  X may be a row-strided view described by (ldx, K)."""
    M = X.shape[0]
    N = W.shape[0]
    K = W.shape[1] if K is None else K
    ldx = X.stride(0) if ldx is None else ldx
    if out is None:
        out = _rows(M, N, X)
        ldy = out.stride(0)
    passes = _gemm_passes(M, N, K)
    if passes == 3 and _tma_ok(X, ldx) and K == W.shape[1]:
        hi, lo = _split_weight(W)
        _note_flops("gnf_linear_fwd_tc", 2. * M * N * K, (M, N, K))
        _TIMES_ALIAS["gnf_linear_fwd_tc_ps"] = "gnf_linear_fwd_tc"
        _call("gnf_linear_fwd_tc_ps", ptr(X), ldx, ptr(hi), ptr(lo), hi.stride(0), ptr(bias), bias_period, ptr(out), ldy, M, N, K,
              int(relu), stream_ptr())
    elif passes:
        W = _tma_weight(W)
        _note_flops("gnf_linear_fwd_tc", 2. * M * N * K, (M, N, K))
        _call("gnf_linear_fwd_tc", ptr(X), ldx, ptr(W), W.stride(0), ptr(bias), bias_period, ptr(out), ldy, M, N, K, int(relu),
              passes, stream_ptr())
    else:
        nbytes = lib().gnf_linear_fwd_splitk_workspace_bytes(M, N, K) if (SPLITK_SKINNY and bias_period <= 1 and (X.is_cuda or L._SIMULATOR)) else 0
        if nbytes:
            work = torch.empty(nbytes // 4, device=X.device, dtype=torch.float32)
            _TIMES_ALIAS["gnf_linear_fwd_splitk"] = "gnf_linear_fwd"
            _call("gnf_linear_fwd_splitk", ptr(X), ldx, ptr(W), W.stride(0), ptr(bias), ptr(out), ldy, M, N, K, int(relu), ptr(work), nbytes,
                  stream_ptr())
            _count()
        else:
            _call("gnf_linear_fwd", ptr(X), ldx, ptr(W), W.stride(0), ptr(bias), bias_period, ptr(out), ldy, M, N, K, int(relu),
                  stream_ptr())
    _count()
    return out


def linear_dgrad(dY, lddy, W, act, M, out=None, lddx=None):
    N, K = W.shape
    if out is None:
        out = _rows(M, K, dY)
        lddx = out.stride(0)
    passes = _gemm_passes(M, N, K)
    if passes == 3 and _tma_ok(dY, lddy):
        hi, lo = _split_weight(W)
        _note_flops("gnf_linear_dgrad_tc", 2. * M * N * K, (M, N, K))
        _TIMES_ALIAS["gnf_linear_dgrad_tc_ps"] = "gnf_linear_dgrad_tc"
        _call("gnf_linear_dgrad_tc_ps", ptr(dY), lddy, ptr(hi), ptr(lo), hi.stride(0), ptr(act), (act.stride(0) if act is not None else 0),
              ptr(out), lddx, M, N, K, stream_ptr())
    elif passes:
        W = _tma_weight(W)
        _note_flops("gnf_linear_dgrad_tc", 2. * M * N * K, (M, N, K))
        _call("gnf_linear_dgrad_tc", ptr(dY), lddy, ptr(W), W.stride(0), ptr(act), (act.stride(0) if act is not None else 0),
              ptr(out), lddx, M, N, K, passes, stream_ptr())
    else:
        _call("gnf_linear_dgrad", ptr(dY), lddy, ptr(W), W.stride(0), ptr(act), (act.stride(0) if act is not None else 0),
              ptr(out), lddx, M, N, K, stream_ptr())
    _count()
    return out


def linear_wgrad(dY, lddy, X, ldx, M, N, K, out=None, lddw=None):
    """dW[n, k] = sum_m dY[m, n] X[m, k]; `out` / `lddw`: write into the first K columns of a wider [N, lddw] matrix."""
    dW = torch.empty(N, K, device=dY.device, dtype=dY.dtype) if out is None else out
    lddw = K if out is None else lddw
    passes = _gemm_passes(M, N, K, "wgrad")
    if passes:
        _note_flops("gnf_linear_wgrad_tc", 2. * M * N * K, (M, N, K))
        _call("gnf_linear_wgrad_tc", ptr(dY), lddy, ptr(X), ldx, ptr(dW), lddw, M, N, K, passes, stream_ptr())
    else:
        _call("gnf_linear_wgrad", ptr(dY), lddy, ptr(X), ldx, ptr(dW), lddw, M, N, K, stream_ptr())
    _count()
    return dW


def linear_wgrad_bias(dY, lddy, X, ldx, M, N, K):
    """(dW, db) of one Linear layer; in 3xTF32 the weight-gradient engine takes db from the dY tiles it streams (one launch)."""
    if _gemm_passes(M, N, K, "wgrad") == 3 and M > 0:
        dW = torch.empty(N, K, device=dY.device, dtype=dY.dtype)
        db = torch.empty(N, device=dY.device, dtype=dY.dtype)
        _note_flops("gnf_linear_wgrad_tc", 2. * M * N * K, (M, N, K))
        _TIMES_ALIAS["gnf_linear_wgrad_bias_tc"] = "gnf_linear_wgrad_tc"
        _call("gnf_linear_wgrad_bias_tc", ptr(dY), lddy, ptr(X), ldx, ptr(dW), K, ptr(db), M, N, K, stream_ptr())
        _count()
        return dW, db
    db = colsum(dY, lddy, M, N).view(N)
    return linear_wgrad(dY, lddy, X, ldx, M, N, K), db


def colsum(Y, ldy, M, N, period=1):
    out = torch.empty(period, N, device=Y.device, dtype=Y.dtype)
    _call("gnf_colsum", ptr(Y), ldy, ptr(out), M, N, period, stream_ptr())
    _count()
    return out


def _mlp_backward(gout, ldg, acts, x_in, ldx, K0, weights, need_dx, first_layer_done=False):
    """Shared backward of a Linear/ReLU stack.

    gout: cotangent of the last layer's (un-activated) output [M, N_last] with row stride ldg.
    acts: ReLU outputs of layers 0..n-2.  Returns (dW list, db list, d_input or None, delta_first)
    where delta_first is the cotangent of layer 0's pre-activation (already ReLU-masked)."""
    n = len(weights)
    M = gout.shape[0]
    dWs, dbs = [None] * n, [None] * n
    delta, ldd = gout, ldg
    for l in range(n - 1, 0, -1):
        W = weights[l]
        N, K = W.shape
        a_prev = acts[l - 1]
        if _gemm_passes(M, N, K, "wgrad") == 0 and M > 0:
            # a skinny layer on the FFMA engine (cfg4's 630 -> 30 output layer: ~20 us each, a fraction of the SMs): the weight / bias
            # gradient and the input cotangent run side by side
            with _Fork(0, delta) as f:
                dWs[l], dbs[l] = linear_wgrad_bias(delta, ldd, a_prev, a_prev.stride(0), M, N, K)
            delta_in, delta = delta, linear_dgrad(delta, ldd, W, a_prev, M)
            f.join()
            del delta_in
        else:
            dWs[l], dbs[l] = linear_wgrad_bias(delta, ldd, a_prev, a_prev.stride(0), M, N, K)
            delta = linear_dgrad(delta, ldd, W, a_prev, M)
        ldd = delta.stride(0)
    if first_layer_done:
        return dWs, dbs, None, delta
    W = weights[0]
    N = W.shape[0]
    dbs[0] = colsum(delta, ldd, M, N).view(N)
    dWs[0] = linear_wgrad(delta, ldd, x_in, ldx, M, N, K0)
    dx = linear_dgrad(delta, ldd, W, None, M) if need_dx else None
    return dWs, dbs, dx, delta


class MlpFn(torch.autograd.Function):
    """Plain nn.Linear/ReLU stack on the MLP engine (CouplingMLP, CouplingConditioner.py:6-18; MADE with
    pre-masked weights).  forward(x2d, out_or_None, ldy, *params) with params = W0, b0, W1, b1, ..."""

    @staticmethod
    def forward(ctx, x, K0, *params):
        require(x, "x")
        weights = [require(_contig(p), "weight") for p in params[0::2]]
        biases = [require(_contig(p), "bias") for p in params[1::2]]
        n = len(weights)
        _SPLIT_CACHE.clear()     # weight splits live from a forward to its own backward only
        if weights[0].shape[1] != K0 or x.shape[1] < K0:
            raise ValueError(f"MLP: first layer expects {weights[0].shape[1]} inputs, got {K0} (x has {x.shape[1]} columns)")
        acts = []
        cur, ldx, K = x, x.stride(0), K0
        for l in range(n):
            out = None
            if l == n - 1:   # the result leaves the Function: plain contiguous rows
                out = torch.empty(x.shape[0], weights[l].shape[0], device=x.device, dtype=x.dtype)
            cur = linear_fwd(cur, weights[l], biases[l], relu=(l < n - 1), K=K, ldx=ldx, out=out, ldy=weights[l].shape[0])
            ldx, K = cur.stride(0), cur.shape[1]
            if l < n - 1:
                acts.append(cur)
        ctx.save_for_backward(x, *weights, *acts)
        ctx.n, ctx.K0 = n, K0
        ctx.need_dx = x.requires_grad
        return cur

    @staticmethod
    def backward(ctx, gout):
        saved = ctx.saved_tensors
        n = ctx.n
        x, weights, acts = saved[0], list(saved[1:1 + n]), list(saved[1 + n:])
        gout = _contig(gout)
        dWs, dbs, dx, _ = _mlp_backward(gout, gout.stride(0), acts, x, x.stride(0), ctx.K0, weights, ctx.need_dx)
        gx = None
        if dx is not None:
            if x.shape[1] == ctx.K0:
                gx = dx
            else:
                gx = torch.zeros_like(x)
                gx[:, :ctx.K0] = dx
        out = [gx, None]
        for l in range(n):
            out += [dWs[l], dbs[l]]
        return tuple(out)


def pack_rows(W, mask=None, perm=None, R=None):
    R = W.shape[0] if R is None else R
    K = W.shape[1]
    out = torch.empty(R, K, device=W.device, dtype=W.dtype)
    _call("gnf_pack_rows", ptr(W), ptr(mask), ptr(perm), ptr(out), R, K, stream_ptr())
    _count()
    return out


class PackRowsFn(torch.autograd.Function):
    """out[r,:] = (mask*W)[perm[r],:] — MaskedLinear's mask*weight (AutoregressiveConditioner.py:24-25) fused
    with the row permutation that makes MADE's output land directly in [B, d, H] order (:108-109)."""

    @staticmethod
    def forward(ctx, W, mask, perm):
        W = require(_contig(W), "W")
        ctx.mask, ctx.perm, ctx.shape = mask, perm, W.shape
        return pack_rows(W, mask, perm, R=(perm.numel() if perm is not None else None))

    @staticmethod
    def backward(ctx, g):
        g = _contig(g)
        N, K = ctx.shape
        dW = torch.empty(N, K, device=g.device, dtype=g.dtype)
        _call("gnf_unpack_rows", ptr(g), ptr(ctx.mask), ptr(ctx.perm), ptr(dW), g.shape[0], N, K, stream_ptr())
        _count()
        return dW, None, None


class PackVecFn(torch.autograd.Function):
    """out[r] = b[perm[r]]."""

    @staticmethod
    def forward(ctx, b, perm):
        b = require(_contig(b), "bias")
        ctx.perm, ctx.n = perm, b.numel()
        return pack_rows(b.view(-1, 1), None, perm, R=perm.numel()).view(-1)

    @staticmethod
    def backward(ctx, g):
        g = _contig(g)
        db = torch.empty(ctx.n, device=g.device, dtype=g.dtype)
        _call("gnf_unpack_vec", ptr(g), ptr(ctx.perm), ptr(db), g.numel(), ctx.n, stream_ptr())
        _count()
        return db, None


def broadcast_rows(constants, h, indep):
    B, d, H = h.shape
    _call("gnf_broadcast_rows", ptr(constants), ptr(h), B, d, indep, H, stream_ptr())
    _count()


# ----------------------------------------------------------------------------------------------
# K1: DAG conditioner
# ----------------------------------------------------------------------------------------------
class GateSpec:
    """Host description of DAGConditioner's gating branch (DAGConditioner.py:126-153)."""

    def __init__(self, mode, imp, h_thresh=0., T=1., seed=0, offset=0, noise=None, offset_dev=None):
        self.mode, self.imp, self.h_thresh, self.T = mode, imp, float(h_thresh), float(T)
        self.seed, self.offset, self.noise = int(seed), int(offset), noise
        self.offset_dev = offset_dev        # optional device int64 counter added to `offset` (CUDA-graph replays)

    def c_struct(self):
        g = L.GateT()
        g.mode, g.temperature, g.seed, g.offset = self.mode, self.T, self.seed, self.offset
        n = self.noise or ()
        g.noise1 = n[0].data_ptr() if len(n) > 0 else None
        g.noise2 = n[1].data_ptr() if len(n) > 1 else None
        g.offset_dev = self.offset_dev.data_ptr() if self.offset_dev is not None else None
        return g


def dag_dump_noise(gate, B, d, device):
    """Materialise the in-kernel Philox draws of a GateSpec (parity / debugging hook)."""
    n1 = torch.empty(B, d, d, device=device, dtype=torch.float32)
    n2 = torch.empty(B, d, d, device=device, dtype=torch.float32) if gate.mode == L.GATE_GUMBEL else None
    g = GateSpec(gate.mode, gate.imp, gate.h_thresh, gate.T, gate.seed, gate.offset, None, gate.offset_dev).c_struct()
    _call("gnf_dag_dump_noise", C.byref(g), ptr(n1), ptr(n2), B, d, stream_ptr())
    _count()
    return (n1, n2) if n2 is not None else (n1,)


# Wide DAG flows (d > DAG_L1_PLANE_MIN_D, e.g. MNIST d = 784) with a tensor-core GEMM mode: layer 1 runs as three GEMMs of the
# tcgen05 engine against the masked embedding written once as a [B*d, d] plane (gnf_dag_embed_fwd / _bwd) instead of the FFMA
# kernels that generate the gate inside their operand loaders: cfg5 layer 1 30 ms -> ~4 ms per step (profiles/r02p_*).
DAG_L1_PLANE = True
DAG_L1_PLANE_MIN_D = 65
DAG_L1_PLANE_KEEP_DERIVATIVES = True      # training keeps the de/dx and de/dP planes (2 x 246 MB at cfg5) instead of regenerating the gates


# Narrow DAG flows (d <= 64) with a stochastic gate, training: the forward kernel also leaves e, de/dx and de/dP as [B d, 64] planes
# and the two backward kernels read them instead of drawing and evaluating every gate again (the gate math was most of each kernel)
DAG_L1_KEEP_GATES = True


def _narrow_l1_tc(M, N1, delta):
    """Backward GEMMs of a narrow flow's layer 1 against the saved planes on the tensor-core engine (3xTF32)?  cfg4 (6300 x 630 x 64):
    weight gradient 42 -> 23 us, input cotangent 49 -> 26 + 5 us (profiles/r02ag_*)."""
    return (DAG_L1_NARROW_TC and _GEMM_MODE in ("auto", "tf32x3") and not L._SIMULATOR and M >= 2048 and N1 >= 128
            and _tma_ok(delta, delta.stride(0)))


DAG_L1_NARROW_TC = True
# ... and the forward GEMM too (gnf_dag_gate_planes + gnf_linear_fwd_tc_ps_tb with the periodic bias table).  On the planned-tile engine
# (K = 64: two k-chunks per tile against its 24 k-clock transposing epilogue) this measured 5 + 40 us against 46 us for the resident-gate
# kernel (profiles/r02ah_*); engine v2 takes the shape since (g2_eligible: short reduction, wide output)
DAG_L1_NARROW_TC_FWD = True


def _dag_l1_plane(M, N1, d):
    # narrow flows (d <= 64) stay on the resident-gate kernels: through the plane + the register-tiled GEMM layer 1 of cfg4 measured
    # 43 / 45 / 73 us (forward / wgrad / dgrad) against 45 / 51 / 55 us, plus the plane kernels (profiles/r02aa_*)
    return DAG_L1_PLANE and d >= DAG_L1_PLANE_MIN_D and M > 0 and _gemm_passes(M, N1, d) != 0 and not L._SIMULATOR


def _dag_context_term(context, W1, in_net, N1):
    """U = context W1[:, in_net:]^T ([B, N1], rows padded to 16-byte pieces): the per-sample term of a conditional flow's layer 1."""
    B, c = context.shape
    U = _rows(B, N1, context)
    if B > 0:
        _call("gnf_linear_fwd", ptr(context), c, ptr(W1[:, in_net:]), W1.stride(0), None, 1, ptr(U), U.stride(0), B, N1, c, 0, stream_ptr())
        _count()
    return U


class DagMlpFn(torch.autograd.Function):
    """DAGConditioner.forward (DAGConditioner.py:126-169): gate/threshold of A, masked expansion of x,
    optional one-hot encoding, embedding MLP — with the [B,d,d] masked tensor generated inside the first
    GEMM's operand loader.  forward(x, A, gate, hot, *params) -> h [B, d, H], params = W0, b0, W1, b1, ...

    Conditional flows: params may end with a context [B, c] after the last bias (an odd count).  Layer 1 then has in_net + c
    inputs, in_net = 2 d (hot) or d, and its input row for sample b, variable i is [e[b,i,:] | onehot(i) | context[b,:]]:
    y1[b*d+i] = act(e[b,i,:] W1[:, :d]^T + T[i] + U[b]) with the bias table T (one-hot columns + b1) and
    U = context W1[:, in_net:]^T, added in the epilogue of whichever layer-1 kernel runs."""

    @staticmethod
    def forward(ctx, x, A, gate, hot, *params):
        require(x, "x")
        A = require(_contig(A), "A")
        context = None
        if len(params) % 2:
            params, context = params[:-1], require(params[-1], "context")
        weights = [require(_contig(p), "weight") for p in params[0::2]]
        biases = [require(_contig(p), "bias") for p in params[1::2]]
        B, d = x.shape
        n = len(weights)
        _SPLIT_CACHE.clear()     # weight splits live from a forward to its own backward only
        in_net = 2 * d if hot else d
        c = weights[0].shape[1] - in_net
        if c < 0 or (c > 0) != (context is not None):
            raise ValueError(f"DAGConditioner: first layer expects {weights[0].shape[1]} inputs, d={d}, hot_encoding={hot}, "
                             f"context={'none' if context is None else tuple(context.shape)}")
        if context is not None and tuple(context.shape) != (B, c):
            raise ValueError(f"DAGConditioner: context must be [B, cond_in] = [{B}, {c}], got {tuple(context.shape)}")
        for t in (gate.noise or ()):
            require(t, "noise")
            if tuple(t.shape) != (B, d, d):
                raise ValueError("replayed gate noise must be [B, d, d]")
        st = stream_ptr()
        P = torch.empty_like(A)
        dPdA = torch.empty_like(A)
        _call("gnf_dag_importance", ptr(A), d, gate.imp, gate.h_thresh, ptr(P), ptr(dPdA), st)
        N1 = weights[0].shape[0]
        # narrow flow, stochastic gate, training, tensor-core GEMM mode: gate planes by one kernel (one gate per thread, every SM) + layer 1 as
        # a GEMM of engine v2 against the plane with the bias table in its epilogue (the table rows padded to 16-byte pieces)
        tc_fwd = (DAG_L1_NARROW_TC_FWD and DAG_L1_KEEP_GATES and d <= 64 and gate.mode != L.GATE_TABLE and B > 0 and n > 1 and hot
                  and DAG_L1_NARROW_TC and _GEMM_MODE in ("auto", "tf32x3", "auto-fast", "tf32") and not L._SIMULATOR
                  and B * d >= 2048 and N1 >= 256 and d >= 32)        # evaluation (no gradient) takes it as well
        U = None
        if context is not None:
            # conditional: the table keeps rows of 16-byte pieces on every route (engine v2 reads it so, period 1 included)
            T = torch.empty(d if hot else 1, _pad4(N1), device=x.device, dtype=x.dtype)
            _call("gnf_dag_bias_table_ld", ptr(weights[0]), weights[0].stride(0), ptr(biases[0]), ptr(T), T.stride(0), d, N1, int(hot), st)
            U = _dag_context_term(context, weights[0], in_net, N1)
        elif tc_fwd:
            T = torch.empty(d, _pad4(N1), device=x.device, dtype=x.dtype)
            _call("gnf_dag_bias_table_ld", ptr(weights[0]), weights[0].stride(0), ptr(biases[0]), ptr(T), T.stride(0), d, N1, 1, st)
        else:
            T = torch.empty(d if hot else 1, N1, device=x.device, dtype=x.dtype)
            _call("gnf_dag_bias_table", ptr(weights[0]), weights[0].stride(0), ptr(biases[0]), ptr(T), d, N1, int(hot), st)
        g = gate.c_struct()
        # the weight splits of the hidden layers depend on nothing of this step: a side branch next to layer 1
        f_split = None
        if B > 0:
            todo = [weights[l] for l in range(1, n) if _gemm_passes(B * d, weights[l].shape[0], weights[l].shape[1]) == 3]
            if todo:
                with _Fork(0, x) as f_split:
                    for W in todo:
                        _split_weight(W)
        y = _rows(B * d, N1, x) if n > 1 else torch.empty(B * d, N1, device=x.device, dtype=x.dtype)
        E = W1e = narrow = None
        gate_planes = (None, None)
        if _dag_l1_plane(B * d, N1, d):
            E = _rows(B * d, d, x)
            if DAG_L1_PLANE_KEEP_DERIVATIVES and (ctx.needs_input_grad[0] or ctx.needs_input_grad[1]):
                gate_planes = (_rows(B * d, d, x), _rows(B * d, d, x))        # de/dx, de/dP (same row stride as E): the backward reduction streams them
            _call("gnf_dag_embed_fwd", ptr(x), ptr(P), C.byref(g), ptr(E), ptr(gate_planes[0]), ptr(gate_planes[1]), E.stride(0), B, d, st)
            W1e = weights[0][:, :d]                 # the masked-input half of layer 1; the one-hot half is the bias table T
            if U is not None:
                passes = _gemm_passes(B * d, N1, d)
                if passes == 3 and _tma_ok(E, E.stride(0)):
                    hi, lo = _split_weight(W1e)
                else:
                    hi, lo = _tma_weight(W1e), None
                _note_flops("gnf_linear_fwd_tc", 2. * B * d * N1 * d, (B * d, N1, d))
                _TIMES_ALIAS["gnf_linear_fwd_tc_cond"] = "gnf_linear_fwd_tc"
                _call("gnf_linear_fwd_tc_cond", ptr(E), E.stride(0), ptr(hi), ptr(lo), hi.stride(0), ptr(T), T.stride(0), (d if hot else 1),
                      ptr(U), U.stride(0), d, ptr(y), y.stride(0), B * d, N1, d, int(n > 1), passes, st)
                _count()
            else:
                linear_fwd(E, W1e, T, relu=(n > 1), bias_period=(d if hot else 1), out=y, ldy=y.stride(0), K=d, ldx=E.stride(0))
            _count(2)
        elif (DAG_L1_KEEP_GATES and d <= 64 and gate.mode != L.GATE_TABLE and B > 0 and (any(ctx.needs_input_grad) or tc_fwd)):
            # narrow flow, stochastic gate, training: the forward leaves e, de/dx, de/dP ([B d, 64] each) for the two backward kernels
            narrow = tuple(torch.empty(B * d, 64, device=x.device, dtype=x.dtype) for _ in range(3))
            if tc_fwd:
                _TIMES_ALIAS["gnf_dag_gate_planes"] = "gnf_dag_l1_fwd"
                _call("gnf_dag_gate_planes", ptr(x), ptr(P), C.byref(g), ptr(narrow[0]), ptr(narrow[1]), ptr(narrow[2]), B, d, st)
                hi, lo = _split_weight(weights[0][:, :d])
                if U is not None:
                    _TIMES_ALIAS["gnf_linear_fwd_tc_cond"] = "gnf_dag_l1_fwd"
                    _call("gnf_linear_fwd_tc_cond", ptr(narrow[0]), 64, ptr(hi), ptr(lo), hi.stride(0), ptr(T), T.stride(0), d, ptr(U), U.stride(0), d,
                          ptr(y), y.stride(0), B * d, N1, d, 1, 3, st)
                else:
                    _TIMES_ALIAS["gnf_linear_fwd_tc_ps_tb"] = "gnf_dag_l1_fwd"
                    _call("gnf_linear_fwd_tc_ps_tb", ptr(narrow[0]), 64, ptr(hi), ptr(lo), hi.stride(0), ptr(T), T.stride(0), d, ptr(y), y.stride(0),
                          B * d, N1, d, 1, st)
                _count(4)
            elif U is not None:
                _TIMES_ALIAS["gnf_dag_l1_fwd_cond"] = "gnf_dag_l1_fwd"
                _call("gnf_dag_l1_fwd_cond", ptr(x), ptr(P), C.byref(g), ptr(weights[0]), weights[0].stride(0), ptr(T), T.stride(0), (d if hot else 1),
                      ptr(U), U.stride(0), ptr(y), y.stride(0), ptr(narrow[0]), ptr(narrow[1]), ptr(narrow[2]), B, d, N1, int(n > 1), st)
                _count(3)
            else:
                _TIMES_ALIAS["gnf_dag_l1_fwd_save"] = "gnf_dag_l1_fwd"
                _call("gnf_dag_l1_fwd_save", ptr(x), ptr(P), C.byref(g), ptr(weights[0]), weights[0].stride(0), ptr(T), (d if hot else 1),
                      ptr(y), y.stride(0), ptr(narrow[0]), ptr(narrow[1]), ptr(narrow[2]), B, d, N1, int(n > 1), st)
                _count(3)
        elif U is not None:
            _TIMES_ALIAS["gnf_dag_l1_fwd_cond"] = "gnf_dag_l1_fwd"
            _call("gnf_dag_l1_fwd_cond", ptr(x), ptr(P), C.byref(g), ptr(weights[0]), weights[0].stride(0), ptr(T), T.stride(0), (d if hot else 1),
                  ptr(U), U.stride(0), ptr(y), y.stride(0), None, None, None, B, d, N1, int(n > 1), st)
            _count(3)
        else:
            _call("gnf_dag_l1_fwd", ptr(x), ptr(P), C.byref(g), ptr(weights[0]), weights[0].stride(0), ptr(T), (d if hot else 1),
                                       ptr(y), y.stride(0), B, d, N1, int(n > 1), st)
            _count(3)
        if f_split is not None:
            f_split.join()
        acts = []
        cur = y
        for l in range(1, n):
            acts.append(cur)
            out = None
            if l == n - 1:   # final layer writes straight into the [B, d, H] result (no view of an internal tensor)
                out = torch.empty(B, d, weights[l].shape[0], device=x.device, dtype=x.dtype)
            cur = linear_fwd(cur, weights[l], biases[l], relu=(l < n - 1), out=out, ldy=weights[l].shape[0])
        ctx.E, ctx.W1e = (E, W1e) if any(ctx.needs_input_grad) else (None, None)
        ctx.gate_planes = gate_planes
        ctx.narrow = narrow if any(ctx.needs_input_grad) else None
        ctx.save_for_backward(x, A, P, dPdA, *weights, *acts)
        ctx.gate, ctx.hot, ctx.n = gate, hot, n
        ctx.context, ctx.in_net = context, in_net
        if n == 1:
            cur = cur.view(B, d, -1).clone()
        return cur

    @staticmethod
    def backward(ctx, gh):
        saved = ctx.saved_tensors
        n, hot, gate = ctx.n, ctx.hot, ctx.gate
        needs = ctx.needs_input_grad
        x, A, P, dPdA = saved[:4]
        weights, acts = list(saved[4:4 + n]), list(saved[4 + n:])
        B, d = x.shape
        M = B * d
        gh = _contig(gh).view(M, -1)
        dWs, dbs, _, delta = _mlp_backward(gh, gh.stride(0), acts, None, 0, 0, weights, False, first_layer_done=True)
        W1 = weights[0]
        N1 = W1.shape[0]
        g = gate.c_struct()
        dW1 = torch.empty_like(W1)
        E, W1e = ctx.E, ctx.W1e           # set iff the forward ran layer 1 against the embedding plane: the backward follows it
        DXp, DPp = ctx.gate_planes
        ctx.E = ctx.W1e = None
        ctx.gate_planes = (None, None)
        narrow, ctx.narrow = ctx.narrow, None
        narrow_tc = narrow is not None and _narrow_l1_tc(M, N1, delta)
        # three independent pieces: [weight gradient of the masked half] | [bias table -> one-hot half of dW1, db1] | [input cotangent]
        with _Fork(0, x) as f_w:
            st = stream_ptr()
            if E is not None:
                linear_wgrad(delta, delta.stride(0), E, E.stride(0), M, N1, d, out=dW1, lddw=dW1.stride(0))
            elif narrow_tc:
                # dW1[:, :d] = delta^T E on the tensor-core engine (3xTF32) against the saved plane
                _TIMES_ALIAS["gnf_linear_wgrad_tc"] = "gnf_dag_l1_wgrad"
                _call("gnf_linear_wgrad_tc", ptr(delta), delta.stride(0), ptr(narrow[0]), 64, ptr(dW1), W1.stride(0), M, N1, d, 3, st)
                _TIMES_ALIAS.pop("gnf_linear_wgrad_tc")
            elif narrow is not None:
                _TIMES_ALIAS["gnf_dag_l1_wgrad_saved"] = "gnf_dag_l1_wgrad"
                _call("gnf_dag_l1_wgrad_saved", ptr(delta), delta.stride(0), ptr(narrow[0]), ptr(dW1), W1.stride(0), B, d, N1, st)
            else:
                _call("gnf_dag_l1_wgrad", ptr(delta), delta.stride(0), ptr(x), ptr(P), C.byref(g), ptr(dW1), W1.stride(0), B, d, N1, st)
        context, in_net = ctx.context, ctx.in_net
        ctx.context = None
        dctx = None
        with _Fork(1, x) as f_b:
            if context is None:
                dT = colsum(delta, delta.stride(0), M, N1, period=(d if hot else 1))
            else:
                # conditional: the table's gradient and the per-sample sums S[b] = sum_i delta[b*d+i] from one read of delta, then
                # dW1[:, in_net:] = S^T context and dcontext = S W1[:, in_net:] (FFMA engine: B x N1 x c, strict fp32 in every mode)
                c = context.shape[1]
                dT = torch.empty(d if hot else 1, N1, device=x.device, dtype=x.dtype)
                S = _rows(B, N1, x)
                stb = stream_ptr()
                _call("gnf_dag_l1_bias_sums", ptr(delta), delta.stride(0), ptr(dT), ptr(S), S.stride(0), B, d, N1, (d if hot else 1), stb)
                _call("gnf_linear_wgrad", ptr(S), S.stride(0), ptr(context), c, ptr(dW1[:, in_net:]), dW1.stride(0), B, N1, c, stb)
                _count(2)
                if needs[4 + 2 * n]:
                    dctx = torch.empty_like(context)
                    if B > 0:
                        _call("gnf_linear_dgrad", ptr(S), S.stride(0), ptr(W1[:, in_net:]), W1.stride(0), None, 0, ptr(dctx), c, B, N1, c, stb)
                        _count()
            db1 = torch.empty(N1, device=x.device, dtype=x.dtype)
            _call("gnf_dag_bias_table_bwd", ptr(dT), ptr(dW1), W1.stride(0), ptr(db1), d, N1, int(hot), stream_ptr())
        _count(2)
        dWs[0], dbs[0] = dW1, db1
        st = stream_ptr()
        dx = dA = dE = dP = hi = lo = None
        if needs[0] or needs[1]:
            dx = torch.empty_like(x)
            dP = torch.empty_like(A)
            if E is not None:
                dE = linear_dgrad(delta, delta.stride(0), W1e, None, M)
                _call("gnf_dag_embed_bwd", ptr(dE), dE.stride(0), ptr(x), ptr(P), C.byref(g), ptr(DXp), ptr(DPp), ptr(dx), ptr(dP), B, d, st)
            elif narrow_tc:
                # ebar = delta W1[:, :d] on the tensor-core engine, then the two reductions against the saved derivative planes
                hi, lo = _split_weight(W1[:, :d])
                dE = torch.empty(M, 64, device=x.device, dtype=x.dtype)
                _TIMES_ALIAS["gnf_linear_dgrad_tc_ps"] = "gnf_dag_l1_dgrad"
                _call("gnf_linear_dgrad_tc_ps", ptr(delta), delta.stride(0), ptr(hi), ptr(lo), hi.stride(0), None, 0, ptr(dE), 64, M, N1, d, st)
                _TIMES_ALIAS["gnf_linear_dgrad_tc_ps"] = "gnf_linear_dgrad_tc"
                _TIMES_ALIAS["gnf_dag_l1_reduce_saved"] = "gnf_dag_l1_dgrad"
                _call("gnf_dag_l1_reduce_saved", ptr(dE), ptr(narrow[1]), ptr(narrow[2]), ptr(dx), ptr(dP), B, d, st)
                _count(2)
            elif narrow is not None:
                _TIMES_ALIAS["gnf_dag_l1_dgrad_saved"] = "gnf_dag_l1_dgrad"
                _call("gnf_dag_l1_dgrad_saved", ptr(delta), delta.stride(0), ptr(W1), W1.stride(0), ptr(narrow[1]), ptr(narrow[2]), ptr(dx),
                      ptr(dP), B, d, N1, st)
            else:
                _call("gnf_dag_l1_dgrad", ptr(delta), delta.stride(0), ptr(W1), W1.stride(0), ptr(x), ptr(P), C.byref(g), ptr(dx),
                                             ptr(dP), B, d, N1, st)
            dA = torch.empty_like(A)
            _call("gnf_dag_finish_dA", ptr(dP), ptr(dPdA), ptr(dA), d, 0, st)
            _count(2)
        f_w.join()
        f_b.join()
        del dE, DXp, DPp, narrow, E, dT, hi, lo          # (everything the branches touched stayed referenced until the joins)
        out = [dx if needs[0] else None, dA if needs[1] else None, None, None]
        for l in range(n):
            out += [dWs[l], dbs[l]]
        if context is not None:
            out.append(dctx)
        return tuple(out)


# ----------------------------------------------------------------------------------------------
# K3: UMNN integral
# ----------------------------------------------------------------------------------------------
_CC_CACHE = {}

# The strict UMNN forward keeps its hidden activations for the backward when they fit in this many bytes (else the
# backward recomputes them, as UMNN does).  0 disables.
SAVE_ACTIVATIONS_MAX_BYTES = 48 << 30
# ... and never more than this fraction of the device memory that is free at the time of the call (an N-step flow keeps N sets of
# activations alive until its backward; a smaller GPU falls back to the recomputing backward instead of running out of memory)
SAVE_ACTIVATIONS_FREE_FRACTION = 0.5


def _activation_budget(device):
    if SAVE_ACTIVATIONS_MAX_BYTES <= 0:
        return 0
    if L._SIMULATOR or torch.cuda.is_current_stream_capturing():
        return SAVE_ACTIVATIONS_MAX_BYTES
    free, _ = torch.cuda.mem_get_info(device)
    return min(SAVE_ACTIVATIONS_MAX_BYTES, int(free * SAVE_ACTIVATIONS_FREE_FRACTION))


# Engine of the strict UMNN integral: 'fused' = one FFMA kernel per direction (umnn.cu), 'layerwise' = per-layer passes
# with the hidden GEMMs on the GEMM engine selected by set_gemm_mode (umnn_lw.cu), 'auto' = layerwise whenever the GEMM
# mode allows tensor cores, the integrand has a hidden x hidden layer worth a GEMM and the activations fit the budget.
UMNN_ENGINE = "auto"
UMNN_LAYERWISE_MIN_NODE_ROWS = 16384
# The strict forward of the layer-wise engine runs as ONE fused tensor-core kernel (gnf_umnn_fwd_tc3) when the integrand fits it
# (>= 3 linear layers, hidden widths <= 160); False = per-layer passes (gnf_umnn_fwd_lw).  Its backward runs the dgrad chain as one
# fused tensor-core kernel too (gnf_umnn_bwd_tc3) whenever that kernel takes the shape, else gnf_umnn_bwd_lw.
UMNN_FWD_FUSED_TC3 = True
# gnf_umnn_fwd_tc3 / gnf_umnn_bwd_tc3 stage the S + 1 quadrature nodes and weights in shared memory (kU3MaxNodes, tc_umnn3.cu)
UMNN_TC3_MAX_NODES = 256


def _umnn_tc3_takes(net, R, S):
    """Does the fused strict forward (gnf_umnn_fwd_tc3) take this integrand at R rows and S quadrature steps?"""
    return UMNN_FWD_FUSED_TC3 and S + 1 <= UMNN_TC3_MAX_NODES and lib().gnf_umnn_tc3_workspace_bytes(C.byref(net), R) != 0


_UMNN_LW_PASSES = {"ffma": 0, "tf32": 1, "tf32x3": 3, "auto": 3, "auto-fast": 3}


def _umnn_fused_ffma_fallback(net, R, S, train, fast, device):
    """Route of a call that the choice above left on the fused FFMA kernels: None when they take the integrand (the forward and,
    in training, the backward, whose shared-memory tiles of every hidden layer cap depth x width); otherwise the layer-wise
    passes of the GEMM mode.  Raises, before any work is done, when no engine takes the call."""
    ffma_fwd = fast or lib().gnf_umnn_workspace_bytes(C.byref(net)) != 0
    if ffma_fwd and (not train or lib().gnf_umnn_bwd_workspace_bytes(C.byref(net)) != 0):
        return None
    why = lib().gnf_last_error().decode()
    if not fast and UMNN_ENGINE == "auto" and net.dims[0] >= 2:
        need = 4 * (lib().gnf_umnn_lw_saved_floats(C.byref(net), R, S, int(train)) +
                    (lib().gnf_umnn_lw_workspace_bytes(C.byref(net), R, S, int(train)) // 4))
        if 0 < need <= _activation_budget(device):
            return _UMNN_LW_PASSES[_GEMM_MODE]
        why += "; layer-wise engine: " + (lib().gnf_last_error().decode() if need == 0 else
                                          f"{need} B of activations exceed the budget (ops.SAVE_ACTIVATIONS_MAX_BYTES)")
    raise RuntimeError("libgnf: " + why)


def _umnn_layerwise_passes(net, R, S, train, device=None):
    """GEMM passes (0 FFMA / 1 TF32 / 3 3xTF32) for the layer-wise UMNN engine, or None for the fused FFMA kernels."""
    if UMNN_ENGINE == "fused" or net.dims[0] < 2:
        return None
    passes = _UMNN_LW_PASSES[_GEMM_MODE]
    if UMNN_ENGINE == "auto":
        hidden = [net.dims[l] for l in range(1, net.n_layers)]
        if passes == 0 or net.n_layers < 3 or min(hidden) < 64 or R * (S + 2) < UMNN_LAYERWISE_MIN_NODE_ROWS:
            return None
    need = 4 * (lib().gnf_umnn_lw_saved_floats(C.byref(net), R, S, int(train)) +
                (lib().gnf_umnn_lw_workspace_bytes(C.byref(net), R, S, int(train)) // 4))
    if need == 0 or need > _activation_budget(device):
        if UMNN_ENGINE == "layerwise" and need == 0:
            raise RuntimeError("libgnf: " + lib().gnf_last_error().decode())
        return None
    return passes


def cc_weights(nb_steps, device):
    """Clenshaw-Curtis weights / nodes, float64 numpy -> fp32, exactly as UMNN's compute_cc_weights
    (SURVEY.md App. B); cached per (S, device)."""
    key = (int(nb_steps), str(device))
    if key not in _CC_CACHE:
        S = int(nb_steps)
        k = np.arange(S + 1, dtype=np.float64)
        lam = np.cos(np.outer(k, k) * math.pi / S)
        lam[:, 0] = .5
        lam[:, -1] = .5 * lam[:, -1]
        lam = lam * 2 / S
        W = np.zeros(S + 1, dtype=np.float64)
        even = np.arange(0, S + 1, 2)
        W[even] = 2. / (1. - even.astype(np.float64) ** 2)
        W[0] = 1.
        w = torch.tensor(lam.T @ W).float().to(device)
        t = torch.tensor(np.cos(k * math.pi / S)).float().to(device)
        _CC_CACHE[key] = (w, t)
    return _CC_CACHE[key]


def _mlp_struct(weights, biases):
    n = len(weights)
    if n > L.GNF_MAX_LAYERS:
        raise ValueError(f"integrand network deeper than {L.GNF_MAX_LAYERS} linear layers is not supported")
    m = L.MlpT()
    m.n_layers = n
    m.dims[0] = weights[0].shape[1]
    for l in range(n):
        m.dims[l + 1] = weights[l].shape[0]
        m.W[l] = weights[l].data_ptr()
        m.b[l] = biases[l].data_ptr()
    return m


class UmnnFn(torch.autograd.Function):
    """MonotonicNormalizer.forward (MonotonicNormalizer.py:51-66) = UMNN (Parallel)NeuralIntegral + h[...,0]
    and the Jacobian evaluation, fused.  forward(x [B,d], h [B,d,E], S, want_rev, fast, *params)
    -> (z, jac, logdet, zrev).  fast=True runs the forward on the tensor cores (single-pass TF32, ll tolerance
    2e-3); the backward always uses the strict fp32 kernel."""

    @staticmethod
    def forward(ctx, x, h, S, want_rev, fast, *params):
        require(x, "x"), require(h, "h")
        weights = [require(_contig(p), "weight") for p in params[0::2]]
        biases = [require(_contig(p), "bias") for p in params[1::2]]
        B, d = x.shape
        E = h.shape[2]
        if weights[0].shape[1] != 1 + E:
            raise ValueError(f"integrand expects {weights[0].shape[1] - 1} conditioning features, h has {E}")
        R = B * d
        net = _mlp_struct(weights, biases)
        if fast:
            nbytes = lib().gnf_umnn_tc_workspace_bytes(C.byref(net))
            if nbytes == 0:
                raise RuntimeError("libgnf: " + lib().gnf_last_error().decode())
        train = any(ctx.needs_input_grad)
        lw_passes = None if fast else _umnn_layerwise_passes(net, R, int(S), train, x.device)
        if lw_passes is None:
            lw_passes = _umnn_fused_ffma_fallback(net, R, int(S), train, fast, x.device)
        if lw_passes is None:
            if not fast:
                nbytes = lib().gnf_umnn_workspace_bytes(C.byref(net))
            ws = torch.empty((nbytes + 3) // 4, device=x.device, dtype=torch.float32)
        ccw, ccn = cc_weights(S, x.device)
        z = torch.empty_like(x)
        jac = torch.empty_like(x)
        zrev = torch.empty_like(x) if want_rev else None
        logdet = torch.empty(B, device=x.device, dtype=x.dtype)
        saved = None
        tc3 = False
        if fast:
            _call("gnf_umnn_fwd_tc", ptr(x), ptr(h), C.byref(net), int(S), ptr(ccw), ptr(ccn), ptr(z), ptr(zrev), ptr(jac),
                  ptr(logdet), R, d, ptr(ws), nbytes, stream_ptr())
        elif lw_passes == 3 and _umnn_tc3_takes(net, R, int(S)):
            # fused strict forward (tc_umnn3.cu): 3xTF32, the activation chain of a tile stays in TMEM from the first to the
            # last hidden layer; training keeps the planes / masks gnf_umnn_bwd_tc3 consumes, evaluation keeps nothing.
            # MMA order: training = all correction products of a layer first (order 1: 20 instead of 60 truncating additions at
            # full accumulator magnitude; with order 0 the saved activations carry a one-sided 5e-7 error that the backward's
            # cancelling sums amplify to 1e-3 .. 2e-3 on the integrand's bias gradients); evaluation = per-chunk order 0
            tc3 = True
            if train:
                saved = torch.empty(lib().gnf_umnn_tc3_saved_floats(C.byref(net), R, int(S)), device=x.device, dtype=torch.float32)
            nbytes = lib().gnf_umnn_tc3_workspace_bytes(C.byref(net), R)
            ws = torch.empty((nbytes + 3) // 4, device=x.device, dtype=torch.float32)
            _call("gnf_umnn_fwd_tc3", ptr(x), ptr(h), C.byref(net), int(S), ptr(ccw), ptr(ccn), ptr(z), ptr(zrev), ptr(jac),
                  ptr(logdet), ptr(saved), int(train), int(train), R, d, ptr(ws), nbytes, stream_ptr())
            _count(6)
        elif lw_passes is not None:
            # layer-wise engine: hidden x hidden layers on the tensor-core GEMM engine, activations in HBM
            saved = torch.empty(lib().gnf_umnn_lw_saved_floats(C.byref(net), R, int(S), int(train)), device=x.device,
                                dtype=torch.float32)
            nbytes = lib().gnf_umnn_lw_workspace_bytes(C.byref(net), R, int(S), 0)
            ws = torch.empty((nbytes + 3) // 4, device=x.device, dtype=torch.float32)
            _call("gnf_umnn_fwd_lw", ptr(x), ptr(h), C.byref(net), int(S), ptr(ccw), ptr(ccn), ptr(z), ptr(zrev), ptr(jac),
                  ptr(logdet), ptr(saved), int(train), lw_passes, R, d, ptr(ws), nbytes, stream_ptr())
            _count(3 + len(weights))
            if not train:
                saved = None
        else:
            # training: keep the hidden activations for the backward when they fit the budget (B200: 180 GB of HBM)
            if train and SAVE_ACTIVATIONS_MAX_BYTES > 0:
                per_row = lib().gnf_umnn_saved_floats_per_node_row(C.byref(net))
                need = R * (int(S) + 1) * per_row * 4
                if 0 < need <= _activation_budget(x.device):
                    saved = torch.empty(R * (int(S) + 1) * per_row, device=x.device, dtype=torch.float32)
            _call("gnf_umnn_fwd", ptr(x), ptr(h), C.byref(net), int(S), ptr(ccw), ptr(ccn), ptr(z), ptr(zrev), ptr(jac),
                  ptr(logdet), ptr(saved), R, d, ptr(ws), nbytes, stream_ptr())
        ctx.lw_passes = lw_passes if (lw_passes is not None and train) else None
        ctx.tc3 = tc3
        _count(2)
        ctx.saved_acts = saved
        ctx.save_for_backward(x, h, jac, *weights, *biases)
        ctx.S, ctx.want_rev, ctx.n = int(S), want_rev, len(weights)
        ctx.set_materialize_grads(False)
        if zrev is None:
            zrev = x.new_empty(0)
            ctx.mark_non_differentiable(zrev)
        return z, jac, logdet, zrev

    @staticmethod
    def backward(ctx, gz, gjac, glogdet, gzrev):
        saved = ctx.saved_tensors
        n = ctx.n
        x, h, jac = saved[:3]
        weights, biases = list(saved[3:3 + n]), list(saved[3 + n:])
        B, d = x.shape
        R = B * d
        net = _mlp_struct(weights, biases)
        ccw, ccn = cc_weights(ctx.S, x.device)
        gz = _contig(gz) if gz is not None else None
        gjac = _contig(gjac) if gjac is not None else None
        glogdet = _contig(glogdet) if glogdet is not None else None
        gzrev = _contig(gzrev) if (gzrev is not None and ctx.want_rev) else None
        dx = torch.empty_like(x)
        dh = torch.empty_like(h)
        grads = L.MlpGradT()
        dWs = [torch.empty_like(w) for w in weights]
        dbs = [torch.empty_like(b) for b in biases]
        for l in range(n):
            grads.dW[l] = dWs[l].data_ptr()
            grads.db[l] = dbs[l].data_ptr()
        if ctx.tc3:
            # dgrad chain fused on the tensor cores (tc_umnn3.cu), then the resident weight-gradient GEMMs
            nbytes = lib().gnf_umnn_bwd_tc3_workspace_bytes(C.byref(net), R, ctx.S)
            if nbytes == 0:
                raise RuntimeError("libgnf: " + lib().gnf_last_error().decode())
            ws = torch.empty((nbytes + 3) // 4, device=x.device, dtype=torch.float32)
            _call("gnf_umnn_bwd_tc3", ptr(x), ptr(h), C.byref(net), ctx.S, ptr(ccw), ptr(ccn), ptr(jac), ptr(gz), ptr(gzrev),
                  ptr(gjac), ptr(glogdet), ptr(ctx.saved_acts), ptr(dx), ptr(dh), C.byref(grads), R, d, ptr(ws), nbytes, stream_ptr())
            _count(6 + 2 * n)
        elif ctx.lw_passes is not None:
            nbytes = lib().gnf_umnn_lw_workspace_bytes(C.byref(net), R, ctx.S, 1)
            ws = torch.empty((nbytes + 3) // 4, device=x.device, dtype=torch.float32)
            _call("gnf_umnn_bwd_lw", ptr(x), ptr(h), C.byref(net), ctx.S, ptr(ccw), ptr(ccn), ptr(jac), ptr(gz), ptr(gzrev),
                  ptr(gjac), ptr(glogdet), ptr(ctx.saved_acts), ptr(dx), ptr(dh), C.byref(grads), ctx.lw_passes, R, d, ptr(ws),
                  nbytes, stream_ptr())
            _count(4 + 3 * n)
        else:
            nbytes = lib().gnf_umnn_bwd_workspace_bytes(C.byref(net))
            ws = torch.empty((nbytes + 3) // 4, device=x.device, dtype=torch.float32)
            _call("gnf_umnn_bwd", ptr(x), ptr(h), C.byref(net), ctx.S, ptr(ccw), ptr(ccn), ptr(jac), ptr(gz), ptr(gzrev), ptr(gjac),
                  ptr(glogdet), ptr(ctx.saved_acts), ptr(dx), ptr(dh), C.byref(grads), R, d, ptr(ws), nbytes, stream_ptr())
        ctx.saved_acts = None
        _count(2)
        out = [dx, dh, None, None, None]
        for l in range(n):
            out += [dWs[l], dbs[l]]
        return tuple(out)


def umnn_forward_on_tensor_cores(params, R, S, device):
    """Would UmnnFn's evaluation forward of R rows run on the fused tcgen05 kernel (gnf_umnn_fwd_tc3) in the current GEMM mode?"""
    if L._SIMULATOR:
        return False
    weights, biases = [p.detach() for p in params[0::2]], [p.detach() for p in params[1::2]]
    net = _mlp_struct(weights, biases)
    return _umnn_layerwise_passes(net, R, int(S), False, device) == 3 and _umnn_tc3_takes(net, R, int(S))


def umnn_invert(z, h, S, weights, biases, iters=20, lo=-20., hi=20.):
    """MonotonicNormalizer.inverse_transform (MonotonicNormalizer.py:69-83): x with integral(x; h) + h[..., 0] = z by `iters`
    bisection steps on [lo, hi], every forward pass of the search inside ONE kernel launch (gnf_umnn_invert).  No autograd
    (the reference searches under torch.no_grad()).  z [B, d], h [B, d, E] -> x [B, d]."""
    require(z, "z"), require(h, "h")
    weights = [require(_contig(w.detach()), "weight") for w in weights]
    biases = [require(_contig(b.detach()), "bias") for b in biases]
    B, d = z.shape
    if weights[0].shape[1] != 1 + h.shape[2]:
        raise ValueError(f"integrand expects {weights[0].shape[1] - 1} conditioning features, h has {h.shape[2]}")
    net = _mlp_struct(weights, biases)
    nbytes = lib().gnf_umnn_workspace_bytes(C.byref(net))
    if nbytes == 0:
        raise RuntimeError("libgnf: " + lib().gnf_last_error().decode())
    ws = torch.empty((nbytes + 3) // 4, device=z.device, dtype=torch.float32)
    ccw, ccn = cc_weights(S, z.device)
    x = torch.empty_like(z)
    _call("gnf_umnn_invert", ptr(z), ptr(h), C.byref(net), int(S), ptr(ccw), ptr(ccn), ptr(x), int(iters), float(lo), float(hi), B * d,
          ptr(ws), nbytes, stream_ptr())
    _count(2)
    return x


def _pad32(v):
    return (v + 31) // 32 * 32


def linear_wgrad_rw(dY, X, N, K, passes=3):
    """dW [N, K] = dY[:, :N]^T @ X[:, :K] on the resident wgrad kernel (tc_rw_wgrad.cu).  X: dense [M, pad32(K)]."""
    require(dY, "dY"), require(X, "X")
    M = dY.shape[0]
    if X.shape[1] != _pad32(K) or X.shape[0] != M:
        raise ValueError(f"X must be [M, pad32(K) = {_pad32(K)}]")
    nbytes = lib().gnf_linear_wgrad_rw_workspace_bytes(N, K)
    if nbytes == 0:
        raise RuntimeError("libgnf: " + lib().gnf_last_error().decode())
    ws = torch.empty(nbytes // 4, device=dY.device, dtype=torch.float32)
    dW = torch.empty(N, K, device=dY.device, dtype=torch.float32)
    _call("gnf_linear_wgrad_rw", ptr(dY), dY.stride(0), ptr(X), X.stride(0), ptr(dW), K, M, N, K, int(passes), ptr(ws), nbytes,
          stream_ptr())
    _count(2)
    return dW


def counter_add(counter, inc=1):
    """*counter += inc on the device (int64 tensor with one element)."""
    _call("gnf_counter_add", ptr(counter), int(inc), stream_ptr())
    _count()


def tc_selftest(A, W, mode):
    """C = A @ W^T for A [128,K], W [N,K] through one tcgen05 CTA (mode 0: A in TMEM, 1: A in shared memory)."""
    require(A, "A"), require(W, "W")
    Cm = torch.empty(128, W.shape[0], device=A.device, dtype=A.dtype)
    _call("gnf_tc_selftest", ptr(A), ptr(W), ptr(Cm), W.shape[0], W.shape[1], int(mode), stream_ptr())
    _count()
    return Cm
