"""CPU tests: the kernels' logic, executed by the host SIMT simulator build of the same .cu sources
(tests/emu, csrc/cpu_emu.h), against the reference-generated golden vectors.  This is a debugging aid for
the GPU-less build container; the GPU parity tests (test_gpu_parity.py, -m gpu) are the real gate."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

import gnf_b200 as G
import sim_hook
from helpers import golden_names
import parity


@pytest.fixture(scope="module")
def emu():
    import build_emu
    path = build_emu.build()
    sim_hook.install(path)
    yield
    sim_hook.uninstall()


@pytest.mark.parametrize("name", golden_names())
def test_golden_case_in_simulator(emu, name):
    torch.set_num_threads(1)
    parity.run_case(name, "cpu")


@pytest.mark.parametrize("name", [n for n in golden_names() if "mono" in n])
def test_golden_monotonic_case_layerwise_engine_in_simulator(emu, name):
    """The layer-wise UMNN engine (umnn_lw.cu) with the FFMA GEMMs: per-layer passes, once-per-row conditioning half of
    the first layer, first-layer reductions, against the reference's golden vectors."""
    torch.set_num_threads(1)
    G.ops.UMNN_ENGINE = "layerwise"
    try:
        parity.run_case(name, "cpu")
    finally:
        G.ops.UMNN_ENGINE = "auto"


def _record_calls(monkeypatch):
    """Names of the C-ABI entry points UmnnFn calls (kernel timing has no simulator flavour)."""
    calls = []
    real = G.ops._call

    def rec(name, *args):
        calls.append(name)
        return real(name, *args)
    monkeypatch.setattr(G.ops, "_call", rec)
    return calls


def test_training_on_a_net_the_ffma_backward_refuses_runs_layerwise_in_simulator(emu, monkeypatch):
    """[256, 256, 256] under the default engine and GEMM mode 'ffma': the FFMA backward cannot hold its tiles in shared memory, so
    the training step runs gnf_umnn_fwd_lw + gnf_umnn_bwd_lw with FFMA GEMMs, against float64."""
    from umnn_ref import OUTS, explicit_quadrature, grad_names, make_cots, make_params, rel
    torch.set_num_threads(1)
    assert G.ops.UMNN_ENGINE == "auto" and G.ops.get_gemm_mode() == "ffma"
    B, d, E, S = 1, 2, 3, 3
    params = [p.requires_grad_(True) for p in make_params([256, 256, 256], E, 0, "cpu")]
    g = torch.Generator().manual_seed(1)
    x, h = torch.randn(B, d, generator=g).requires_grad_(True), torch.randn(B, d, E, generator=g).requires_grad_(True)
    cots = make_cots(OUTS, B, d, "cpu", 2)
    calls = _record_calls(monkeypatch)
    outs = G.ops.UmnnFn.apply(x, h, S, True, False, *params)
    grads = torch.autograd.grad(outs, [x, h] + params, [cots[k] for k in OUTS])
    assert {c for c in calls if c.startswith("gnf_umnn")} == {"gnf_umnn_fwd_lw", "gnf_umnn_bwd_lw"}, calls
    ref = explicit_quadrature(params, x, h, S, cots)
    got = dict(zip(OUTS + tuple(grad_names(4)), [o.detach() for o in outs] + list(grads)))
    errs = {k: rel(got[k], ref[k], k, d) for k in ref}
    bad = {k: e for k, e in errs.items() if not e < (1e-6 if k in OUTS else 2e-4)}
    assert not bad, bad


def test_no_umnn_engine_for_the_call_raises_before_any_work_in_simulator(emu, monkeypatch):
    """Training [256, 256, 256] with the engine forced to 'fused', or with no activation budget for the layer-wise engine: UmnnFn
    raises in its forward, before any entry point runs."""
    from umnn_ref import make_params
    params = [p.requires_grad_(True) for p in make_params([256, 256, 256], 3, 0, "cpu")]
    x, h = torch.randn(1, 2, requires_grad=True), torch.randn(1, 2, 3, requires_grad=True)
    calls = _record_calls(monkeypatch)
    for name, value in [("UMNN_ENGINE", "fused"), ("SAVE_ACTIVATIONS_MAX_BYTES", 0)]:
        old = getattr(G.ops, name)
        setattr(G.ops, name, value)
        try:
            with pytest.raises(RuntimeError, match="shared memory"):
                G.ops.UmnnFn.apply(x, h, 3, True, False, *params)
        finally:
            setattr(G.ops, name, old)
    assert not calls, calls


def test_power_trace_golden_in_simulator(emu):
    """K2 against the reference's golden power traces, both flavours: the no-grad forward (torch.matrix_power's order) and
    the training forward that leaves (I + alpha A∘A)^(p-1) for an elementwise backward (d <= 64)."""
    import numpy as np
    from helpers import GOLDEN, rel_l2
    torch.set_num_threads(1)
    f = np.load(os.path.join(GOLDEN, "power_trace.npz"))
    for key in sorted({k.rsplit(".", 1)[0] for k in f.files}):
        d, p, alpha = f[key + ".meta"]
        if int(d) > 64:
            continue                      # the host-driven GEMM chain is too slow for the simulator; covered on the GPU
        want = float(f[key + ".t"])
        tol = 2e-5 * abs(want) + 1e-5 * float(d)
        A = torch.from_numpy(f[key + ".A"])
        with torch.no_grad():
            t0 = G.ops.PowerTraceFn.apply(A, float(alpha), int(p))
        assert abs(float(t0) - want) <= tol, key
        A = A.clone().requires_grad_(True)
        t = G.ops.PowerTraceFn.apply(A, float(alpha), int(p))
        t.backward()
        assert abs(float(t.detach()) - want) <= tol, key
        assert rel_l2(A.grad, torch.from_numpy(f[key + ".dA"])) < 1e-4, key


def test_fused_bisection_inverse_in_simulator(emu):
    """gnf_umnn_invert (MonotonicNormalizer.inverse_transform's 20 bisection steps in one launch) against the reference's loop of
    20 forward passes through the same simulated forward kernel, and against the x that produced z."""
    torch.set_num_threads(1)
    torch.manual_seed(0)
    norm = G.MonotonicNormalizer([16, 16], 3, nb_steps=7, solver="CC")
    x, h = torch.randn(5, 4) * 2, torch.randn(5, 4, 3)
    with torch.no_grad():
        z, _ = norm(x, h)
        norm.fused_inverse = True
        x_fused = norm.inverse_transform(z, h)
        norm.fused_inverse = False
        x_loop = norm.inverse_transform(z, h)
    res = 40. / 2 ** 20
    assert float((x_fused - x_loop).abs().max()) <= res * 1.01
    assert float((x_fused - x).abs().max()) < 2 * res


@pytest.mark.parametrize("M_,N,K", [(520, 5, 70), (515, 70, 5), (600, 32, 33)])
def test_skinny_layer_kernels_in_simulator(emu, M_, N, K):
    """csrc/thin.cuh (one weight dimension <= 32): forward with bias + ReLU and the masked input cotangent, both weight layouts,
    against torch."""
    torch.set_num_threads(1)
    g = torch.Generator().manual_seed(M_ + N + K)
    X, W, b = torch.randn(M_, K, generator=g), torch.randn(N, K, generator=g) / K ** .5, torch.randn(N, generator=g)
    dY = torch.randn(M_, N, generator=g)
    Y = G.ops.linear_fwd(X, W, b, relu=True)
    assert torch.allclose(Y, torch.relu(X @ W.t() + b), rtol=1e-4, atol=1e-5)
    dX = G.ops.linear_dgrad(dY, N, W, X, M_)
    assert torch.allclose(dX, (dY @ W) * (X > 0), rtol=1e-4, atol=1e-5)


def _nll_loss_case(device, B, d, with_constraint):
    g = torch.Generator().manual_seed(B * 131 + d)
    z = torch.randn(B, d, generator=g).to(device).requires_grad_(True)
    logdet = torch.randn(B, generator=g).to(device).requires_grad_(True)
    c = (torch.randn((), generator=g).abs()).to(device).requires_grad_(True) if with_constraint else None
    out = G.ops.NllLossFn.apply(z, logdet, c)
    out.backward()
    z64, l64 = z.detach().double().cpu().requires_grad_(True), logdet.detach().double().cpu().requires_grad_(True)
    ll = l64 - .5 * (torch.log(torch.tensor(2 * torch.pi, dtype=torch.float64)) + z64 ** 2).sum(1)
    want = (c.detach().double().cpu() if with_constraint else 0.) - ll.mean()
    want.backward()
    assert abs(float(out.detach()) - float(want)) <= 1e-5 * max(1., abs(float(want)))
    assert torch.allclose(z.grad.cpu().double(), z64.grad, rtol=1e-6, atol=1e-9)
    assert torch.allclose(logdet.grad.cpu().double(), l64.grad, rtol=1e-6, atol=1e-9)
    if with_constraint:
        assert float(c.grad) == 1.


@pytest.mark.parametrize("B,d,with_constraint", [(1, 1, False), (100, 63, True), (37, 6, True), (300, 5, False)])
def test_fused_training_loss_in_simulator(emu, B, d, with_constraint):
    """gnf_nll_loss_{fwd,bwd} (FCNormalizingFlow.loss with the standard-normal base density, NormalizingFlow.py:144-146) against
    float64 torch; called twice through the same work buffer (the block counter must be left at zero)."""
    torch.set_num_threads(1)
    _nll_loss_case("cpu", B, d, with_constraint)
    _nll_loss_case("cpu", B, d, with_constraint)


def _narrow_reduce_case(device, B, d):
    import ctypes as C
    from gnf_b200.ops import _call, ptr, stream_ptr
    g = torch.Generator().manual_seed(B * 7 + d)
    dE, DX, DP = (torch.randn(B * d, 64, generator=g).to(device) for _ in range(3))
    DX[:, d:] = 0
    DP[:, d:] = 0
    dx = torch.full((B, d), float("nan"), device=device)
    dP = torch.full((d, d), float("nan"), device=device)
    _call("gnf_dag_l1_reduce_saved", ptr(dE), ptr(DX), ptr(DP), ptr(dx), ptr(dP), B, d, stream_ptr())
    e, vx, vp = (t.double().cpu().view(B, d, 64)[:, :, :d] for t in (dE, DX, DP))
    assert torch.allclose(dx.double().cpu(), (e * vx).sum(1), rtol=1e-5, atol=1e-5)
    assert torch.allclose(dP.double().cpu(), (e * vp).sum(0), rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("B,d", [(1, 1), (5, 6), (7, 63), (4, 64)])
def test_narrow_layer1_plane_reduction_in_simulator(emu, B, d):
    """gnf_dag_l1_reduce_saved: dx[b,j] = sum_i dE de/dx, dP[i,j] = sum_b dE de/dP over the planes the training forward kept."""
    torch.set_num_threads(1)
    _narrow_reduce_case("cpu", B, d)


def _splitk_case(device, M_, N, K, relu):
    g = torch.Generator().manual_seed(M_ + N + K)
    X = torch.randn(M_, K, generator=g).to(device)
    W = (torch.randn(N, K, generator=g) / K ** .5).to(device)
    b = torch.randn(N, generator=g).to(device)
    assert G._lib.lib().gnf_linear_fwd_splitk_workspace_bytes(M_, N, K) > 0
    Y = G.ops.linear_fwd(X, W, b, relu=relu)
    Y2 = G.ops.linear_fwd(X, W, b, relu=relu)
    assert torch.equal(Y, Y2)                                      # fixed-order sum of the partial tiles: deterministic
    ref = X.double() @ W.double().t() + b.double()
    ref = torch.relu(ref) if relu else ref
    assert torch.allclose(Y.double(), ref, rtol=1e-5, atol=1e-5)


def test_skinny_split_k_forward_in_simulator(emu):
    """gnf_linear_fwd_splitk (the conditioner's 630 -> 30 output layer): partial tiles + fixed-order sum, against float64."""
    torch.set_num_threads(1)
    _splitk_case("cpu", 1024, 5, 130, False)


def test_gate_planes_and_padded_bias_table_in_simulator(emu):
    """gnf_dag_gate_planes (one gate per thread) against the planes the resident-gate forward leaves (gnf_dag_l1_fwd_save), same
    replayed noise; gnf_dag_bias_table_ld (padded rows) against gnf_dag_bias_table."""
    import ctypes as C
    from gnf_b200.ops import _call, ptr, stream_ptr, GateSpec
    import gnf_b200._lib as L
    torch.set_num_threads(1)
    g = torch.Generator().manual_seed(9)
    B, d, N1 = 5, 7, 12
    x, A = torch.randn(B, d, generator=g), torch.randn(d, d, generator=g)
    W1, b1 = torch.randn(N1, 2 * d, generator=g), torch.randn(N1, generator=g)
    noise = (torch.rand(B, d, d, generator=g).clamp(1e-3, 1 - 1e-3), torch.rand(B, d, d, generator=g).clamp(1e-3, 1 - 1e-3))
    gate = GateSpec(L.GATE_GUMBEL, L.IMP_SOFT, 0., .5, noise=noise)
    P, dPdA = torch.empty_like(A), torch.empty_like(A)
    _call("gnf_dag_importance", ptr(A), d, gate.imp, gate.h_thresh, ptr(P), ptr(dPdA), stream_ptr())
    gs = gate.c_struct()
    planes = [torch.full((B * d, 64), float("nan")) for _ in range(3)]
    _call("gnf_dag_gate_planes", ptr(x), ptr(P), C.byref(gs), ptr(planes[0]), ptr(planes[1]), ptr(planes[2]), B, d, stream_ptr())
    T = torch.empty(d, N1)
    _call("gnf_dag_bias_table", ptr(W1), W1.stride(0), ptr(b1), ptr(T), d, N1, 1, stream_ptr())
    Tp = torch.full((d, 16), float("nan"))
    _call("gnf_dag_bias_table_ld", ptr(W1), W1.stride(0), ptr(b1), ptr(Tp), 16, d, N1, 1, stream_ptr())
    assert torch.equal(Tp[:, :N1], T) and bool((Tp[:, N1:] == 0).all())
    ref = [torch.full((B * d, 64), float("nan")) for _ in range(3)]
    y = torch.empty(B * d, N1)
    _call("gnf_dag_l1_fwd_save", ptr(x), ptr(P), C.byref(gs), ptr(W1), W1.stride(0), ptr(T), d, ptr(y), N1, ptr(ref[0]), ptr(ref[1]), ptr(ref[2]),
          B, d, N1, 1, stream_ptr())
    for a, b in zip(planes, ref):
        assert torch.equal(a, b)
    # and layer 1 itself from the plane: relu(E W1[:, :d]^T + T[i])
    want = torch.relu(planes[0][:, :d] @ W1[:, :d].t() + T.repeat(B, 1))
    assert torch.allclose(y, want, rtol=1e-5, atol=1e-5)
