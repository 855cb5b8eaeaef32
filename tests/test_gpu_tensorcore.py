"""GPU tests of the tcgen05 (tensor-core) path: the UMMA descriptor / TMEM-layout conventions via the one-CTA
self-test GEMM, then the fused TF32 UMNN forward against the strict fp32 kernel and the CPU oracle.
Tolerance: north_star's TF32 bar — per-sample log-likelihood within 2e-3 relative."""
import pytest
import torch

import gnf_b200 as G
import parity

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("N,K", [(16, 8), (160, 32), (160, 152), (112, 104), (208, 96), (256, 64), (30, 31)])
def test_tcgen05_selftest_gemm_exact_on_tf32_representable_inputs(mode, N, K):
    g = torch.Generator(device="cuda").manual_seed(N * 1000 + K + mode)
    A = torch.randint(-8, 9, (128, K), device="cuda", generator=g).float()
    W = torch.randint(-8, 9, (N, K), device="cuda", generator=g).float()
    Cm = G.ops.tc_selftest(A, W, mode)
    ref = A @ W.t()
    assert torch.equal(Cm, ref), f"max err {float((Cm - ref).abs().max())}"


@pytest.mark.parametrize("mode", [0, 1])
def test_tcgen05_selftest_gemm_tf32_accuracy(mode):
    A = torch.randn(128, 152, device="cuda")
    W = torch.randn(160, 152, device="cuda") / 152 ** .5
    Cm = G.ops.tc_selftest(A, W, mode)
    ref = (A.double() @ W.double().t()).float()
    assert float((Cm - ref).abs().max()) < 5e-3          # 10-bit mantissa operands, fp32 accumulation


@pytest.mark.parametrize("cfg,B,S", [("cfg4", 100, 20), ("cfg4", 7, 40), ("cfg2", 500, 40), ("cfg2", 3, 7)])
def test_umnn_tensorcore_forward_matches_strict(cfg, B, S):
    import model_vs_oracle as M
    model = M.build(M.CONFIGS[cfg], "cuda")
    parity.set_modes(model, dict(stoch_gate=False))
    for n in model.getNormalizers():
        n.nb_steps = S
    x = torch.randn(B, M.CONFIGS[cfg]["d"], device="cuda", generator=torch.Generator(device="cuda").manual_seed(11))
    with torch.no_grad():
        ll_s, z_s = model.compute_ll(x)
        for n in model.getNormalizers():
            n.precision = "tf32"
        ll_f, z_f = model.compute_ll(x)
    rel = float(((ll_f - ll_s).abs() / ll_s.abs().clamp_min(1e-6)).max())
    assert rel < 2e-3, f"per-sample ll relative error {rel}"
    assert float((z_f - z_s).abs().max()) < 5e-3


def test_umnn_tensorcore_forward_with_strict_backward_trains():
    """fast forward + strict backward still trains: ll within the TF32 bar of the CPU oracle, gradients finite and
    close to the strict ones (they are the strict kernel's gradients of the same weights)."""
    import model_vs_oracle as M
    spec = M.CONFIGS["cfg2"]
    model = M.build(spec, "cuda")
    parity.set_modes(model, dict(stoch_gate=False))
    x = torch.randn(64, 6, device="cuda")
    model.zero_grad()
    z, jac = model(x)
    model.loss(z, jac).backward()
    g_strict = {k: p.grad.clone() for k, p in model.named_parameters()}
    for n in model.getNormalizers():
        n.precision = "tf32"
    model.zero_grad()
    z2, jac2 = model(x)
    model.loss(z2, jac2).backward()
    assert float((z - z2).abs().max()) < 5e-3
    for k, p in model.named_parameters():
        assert torch.isfinite(p.grad).all()
        if "integrand_net" in k:
            assert float((p.grad - g_strict[k]).norm() / g_strict[k].norm().clamp_min(1e-12)) < 5e-2, k


def test_tensorcore_unsupported_width_is_loud():
    n = G.MonotonicNormalizer([200, 200, 200], 30).cuda()      # 2 x 208 x 200 fp32 weights do not fit in 227 KB
    n.precision = "tf32"
    with pytest.raises(RuntimeError):
        n(torch.randn(4, 3, device="cuda"), torch.randn(4, 3, 30, device="cuda"))


# ---------------- tensor-core conditioner GEMM engine (tcgen05, 128B-swizzled producer-staged tiles) ----------------
@pytest.fixture
def gemm_mode():
    yield G.ops.set_gemm_mode
    G.ops.set_gemm_mode("ffma")


SHAPES = [(1, 1, 1), (127, 33, 65), (300, 630, 126), (1000, 30, 630), (64, 2, 1024), (513, 210, 21), (6300, 630, 630),
          (256, 1024, 784), (300, 160, 160), (1000, 152, 64), (513, 212, 20), (129, 4, 36), (2200, 150, 150),
          (138600, 152, 148), (6300, 632, 632), (4100, 300, 260), (12544, 1024, 784)]


@pytest.mark.parametrize("M_,N,K", SHAPES)
def test_tc_gemm_exact_on_small_integers(gemm_mode, M_, N, K):
    """Integer-valued operands are exactly representable in TF32 and all partial sums in fp32: the single-pass
    engine must reproduce fwd / dgrad / wgrad bit-exactly (checks tile staging, swizzle, both operand majors)."""
    gemm_mode("tf32")
    g = torch.Generator(device="cuda").manual_seed(M_ * 7 + N * 3 + K)
    X = torch.randint(-3, 4, (M_, K), device="cuda", generator=g).float()
    W = torch.randint(-3, 4, (N, K), device="cuda", generator=g).float()
    b = torch.randint(-3, 4, (N,), device="cuda", generator=g).float()
    dY = torch.randint(-3, 4, (M_, N), device="cuda", generator=g).float()
    Y = G.ops.linear_fwd(X, W, b, relu=True)
    assert torch.equal(Y, torch.relu(X @ W.t() + b)), float((Y - torch.relu(X @ W.t() + b)).abs().max())
    dX = G.ops.linear_dgrad(dY, N, W, X, M_)
    assert torch.equal(dX, (dY @ W) * (X > 0)), float((dX - (dY @ W) * (X > 0)).abs().max())
    dW = G.ops.linear_wgrad(dY, N, X, K, M_, N, K)
    ref = (dY.double().t() @ X.double()).float()
    assert torch.equal(dW, ref), float((dW - ref).abs().max())


@pytest.mark.parametrize("M_,N,K", SHAPES)
def test_tc_gemm_3xtf32_is_fp32_equivalent(gemm_mode, M_, N, K):
    gemm_mode("tf32x3")
    g = torch.Generator(device="cuda").manual_seed(M_ + N + K)
    X = torch.randn(M_, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** .5
    b = torch.randn(N, device="cuda", generator=g)
    dY = torch.randn(M_, N, device="cuda", generator=g)
    Y = G.ops.linear_fwd(X, W, b, relu=True)
    ref = torch.relu(X.double() @ W.double().t() + b.double()).float()
    assert float((Y - ref).norm() / ref.norm().clamp_min(1e-12)) < 2e-5
    dX = G.ops.linear_dgrad(dY, N, W, X, M_)
    refdX = ((dY.double() @ W.double()) * (X > 0)).float()
    assert float((dX - refdX).norm() / refdX.norm().clamp_min(1e-12)) < 2e-5
    dW = G.ops.linear_wgrad(dY, N, X, K, M_, N, K)
    refdW = (dY.double().t() @ X.double()).float()
    assert float((dW - refdW).norm() / refdW.norm().clamp_min(1e-12)) < 2e-5


def test_tc_gemm_single_pass_tf32_accuracy(gemm_mode):
    gemm_mode("tf32")
    X = torch.randn(2000, 630, device="cuda")
    W = torch.randn(630, 630, device="cuda") / 630 ** .5
    Y = G.ops.linear_fwd(X, W, None, relu=False)
    ref = (X.double() @ W.double().t()).float()
    assert float((Y - ref).norm() / ref.norm()) < 2e-3


@pytest.mark.parametrize("cfg,B", [("cfg2", 256), ("cfg3", 48), ("cfg4", 12), ("cfg1", 100)])
def test_train_step_vs_oracle_with_3xtf32_conditioner(gemm_mode, cfg, B):
    """Strict bars (ll 1e-4, per-tensor gradients 1e-3) with the conditioner GEMMs on the tensor cores."""
    import model_vs_oracle as M
    gemm_mode("tf32x3")
    rep = M.compare(M.CONFIGS[cfg], B, "cuda", train=True)
    bad = {k: v for k, v in rep.items() if (k.startswith("grad.") and not v < 1e-3) or (k in ("ll", "loss") and not v < 1e-4)}
    assert not bad, f"out of tolerance: {bad}\n{rep}"


@pytest.mark.parametrize("cfg,B", [("cfg4", 24), ("cfg2", 512)])
def test_mixed_mode_training_gradients_vs_oracle(cfg, B):
    """Fast training mode — TF32 tensor-core UMNN forward + strict fp32 backward ("tf32" normalizer precision): per-sample
    ll within the TF32 bar (2e-3).  Gradients are the strict kernel's, evaluated at cotangents that carry the TF32
    forward error: measured 2e-5..3e-3 per tensor (cfg2 / cfg4), i.e. NOT within the strict 1e-3 bar on cfg4, which is
    why bench.py's training number uses the strict forward.  The bound asserted here documents that measurement."""
    import model_vs_oracle as M
    spec = M.CONFIGS[cfg]
    model = M.build(spec, "cuda")
    parity.set_modes(model, dict(stoch_gate=False))
    for n in model.getNormalizers():
        n.precision = "tf32"
    x = torch.randn(B, spec["d"], generator=torch.Generator().manual_seed(5)).cuda()
    model.zero_grad()
    z, jac = model(x)
    loss = model.loss(z, jac)
    loss.backward()
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    loss_o, z_o, jac_o, grads_o = M.O.train_step_grads(x.cpu(), sd, spec, [dict(stoch_gate=False)] * spec["nb_flow"], None)
    ll = (model.z_log_density(z) + jac).detach().cpu()
    ll_o = M.O.normal_log_density(z_o) + jac_o
    assert float(((ll - ll_o).abs() / ll_o.abs().clamp_min(1e-6)).max()) < 2e-3
    params = dict(model.named_parameters())
    from helpers import rel_l2
    rep = {k: rel_l2(params[k].grad.cpu(), g) for k, g in grads_o.items() if g is not None}
    bad = {k: v for k, v in rep.items() if not v < 1e-2}
    print("mixed-mode gradient errors:", {k.split("steps.0.")[-1]: float("%.2g" % v) for k, v in rep.items()})
    assert not bad, f"gradients out of tolerance: {bad}"


# ---------------- layer-wise UMNN engine (umnn_lw.cu): hidden layers on the GEMM engine, activations in HBM ----------------
@pytest.fixture
def umnn_engine():
    def set_engine(engine, gemm="auto"):
        G.ops.UMNN_ENGINE = engine
        G.ops.set_gemm_mode(gemm)
    yield set_engine
    G.ops.UMNN_ENGINE = "auto"
    G.ops.set_gemm_mode("ffma")


def _strict_check(rep):
    bad = {k: v for k, v in rep.items() if (k.startswith("grad.") and not v < 1e-3) or (k in ("ll", "loss") and not v < 1e-4)}
    assert not bad, f"out of tolerance: {bad}\n{rep}"


@pytest.mark.parametrize("gemm", ["ffma", "tf32x3"])
@pytest.mark.parametrize("name", [n for n in __import__("helpers").golden_names() if n.endswith("mono") or "mono_" in n])
def test_umnn_layerwise_golden_vectors(umnn_engine, name, gemm):
    """Reference-generated golden vectors through the layer-wise engine (strict bars), FFMA and 3xTF32 GEMMs."""
    umnn_engine("layerwise", gemm)
    parity.run_case(name, "cuda", 1e-4, 1e-3)


@pytest.mark.parametrize("cfg,B", [("cfg2", 256), ("cfg3", 48), ("cfg4", 12), ("cfg4", 100)])
def test_umnn_layerwise_train_step_vs_oracle(umnn_engine, cfg, B):
    """Strict bars (ll 1e-4, per-tensor gradients 1e-3) against the CPU oracle with the 3xTF32 layer-wise engine."""
    import model_vs_oracle as M
    umnn_engine("layerwise", "auto")
    _strict_check(M.compare(M.CONFIGS[cfg], B, "cuda", train=True))


@pytest.mark.parametrize("cfg,B,S", [("cfg4", 20, 40), ("cfg2", 33, 29), ("cfg3", 64, 40)])
def test_umnn_layerwise_eval_vs_oracle(umnn_engine, cfg, B, S):
    import model_vs_oracle as M
    umnn_engine("layerwise", "auto")
    _strict_check(M.compare(M.CONFIGS[cfg], B, "cuda", train=False, nb_steps=S))


def test_umnn_layerwise_vs_float64_quadrature(umnn_engine):
    """cfg4's integrand (30 -> 150 x 3 -> 1, S = 20) on 6300 rows, random inputs and cotangents: forward values and every
    gradient of the layer-wise 3xTF32 engine against the oracle's quadrature evaluated in float64 (on the GPU), next to the
    fused FFMA kernels.  Measured on B200: fused <= 1e-6, layer-wise <= 3e-5 (its long fp32 reductions over 138 600
    node-rows), both far inside the 1e-3 gradient bar."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import gnf_oracle as O
    torch.manual_seed(0)
    B, d, S = 100, 63, 20
    norm = G.MonotonicNormalizer([150, 150, 150], 30, nb_steps=S, solver="CC").to("cuda")
    x, h = torch.randn(B, d, device="cuda"), torch.randn(B, d, 30, device="cuda")
    cz, cj = torch.randn(B, d, device="cuda"), torch.randn(B, d, device="cuda")
    sd64 = {"n." + k: v.detach().double().requires_grad_(True) for k, v in norm.state_dict().items()}
    x64, h64 = x.double().requires_grad_(True), h.double().requires_grad_(True)
    z, jac = O.monotonic_normalizer(x64, h64, sd64, "n.integrand_net.net", 4, S)
    ((z * cz.double()).sum() + (torch.log(jac) * cj.double()).sum()).backward()
    ref = {"x": x64.grad, "h": h64.grad, "z": z.detach(), "jac": jac.detach()}
    ref.update({k[2:]: v.grad for k, v in sd64.items()})
    for engine, gemm, tol in (("fused", "ffma", 1e-5), ("layerwise", "tf32x3", 2e-4)):
        umnn_engine(engine, gemm)
        xg, hg = x.clone().requires_grad_(True), h.clone().requires_grad_(True)
        norm.zero_grad()
        z32, j32 = norm(xg, hg)
        ((z32 * cz).sum() + (torch.log(j32) * cj).sum()).backward()
        got = {"x": xg.grad, "h": hg.grad, "z": z32.detach(), "jac": j32.detach()}
        got.update({k: p.grad for k, p in norm.named_parameters()})
        for k, r in ref.items():
            err = float((got[k].double() - r).norm() / r.norm().clamp_min(1e-30))
            assert err < (1e-6 if k in ("z", "jac") else tol), (engine, k, err)


def test_umnn_layerwise_auto_engine_selection(umnn_engine):
    """'auto' keeps the fused kernels in strict-FFMA mode and for tiny problems, and switches to the layer-wise engine
    when tensor cores are allowed and the problem is large enough."""
    import model_vs_oracle as M
    _umnn_layerwise_passes, _mlp_struct = G.ops._umnn_layerwise_passes, G.ops._mlp_struct
    model = M.build(M.CONFIGS["cfg4"], "cuda")
    net_params = list(model.getNormalizers()[0].integrand_net.parameters())
    net = _mlp_struct(net_params[0::2], net_params[1::2])
    umnn_engine("auto", "ffma")
    assert _umnn_layerwise_passes(net, 6300, 20, True) is None
    umnn_engine("auto", "auto")
    assert _umnn_layerwise_passes(net, 6300, 20, True) == 3
    assert _umnn_layerwise_passes(net, 63, 20, True) is None


# ---------------------------------------------------------------------------------------------------------------
# resident weight-gradient kernel (tc_rw_wgrad.cu): the hidden-layer weight gradients of the fused UMNN backward
# ---------------------------------------------------------------------------------------------------------------
def _padded(t, cols):
    out = torch.zeros(t.shape[0], cols, device=t.device, dtype=t.dtype)
    out[:, :t.shape[1]] = t
    return out


@pytest.mark.parametrize("M_,N,K", [(1000, 150, 150), (32, 160, 160), (4133, 100, 100), (77, 30, 150), (300, 150, 31), (40000, 150, 150),
                                    (5, 128, 96), (6000, 129, 64)])
def test_rw_wgrad_exact_and_fp32_equivalent(M_, N, K):
    g = torch.Generator(device="cuda").manual_seed(M_ + 3 * N + K)
    NPn, KP = (N + 31) // 32 * 32, (K + 31) // 32 * 32
    dY = torch.randint(-4, 5, (M_, N), device="cuda", generator=g).float()
    X = torch.randint(-4, 5, (M_, K), device="cuda", generator=g).float()
    ref = dY.double().t() @ X.double()
    for passes in (1, 3):
        dW = G.ops.linear_wgrad_rw(_padded(dY, NPn), _padded(X, KP), N, K, passes=passes)
        assert torch.equal(dW.double(), ref), f"passes={passes}: max err {float((dW.double() - ref).abs().max())}"
    dY = torch.randn(M_, N, device="cuda", generator=g)
    X = torch.randn(M_, K, device="cuda", generator=g)
    ref = dY.double().t() @ X.double()
    dW = G.ops.linear_wgrad_rw(_padded(dY, NPn), _padded(X, KP), N, K, passes=3)
    err = float((dW.double() - ref).abs().max() / ref.abs().max())
    err32 = float(((dY.t() @ X).double() - ref).abs().max() / ref.abs().max())
    assert err < max(3e-6, 4 * err32), (err, err32)
    # garbage (non-finite) in the padding columns of X must not leak: the kernel only promises finite padding, so fill with large values
    Xp = _padded(X, KP)
    if KP > K:
        Xp[:, K:] = 1e30
        dW2 = G.ops.linear_wgrad_rw(_padded(dY, NPn), Xp, N, K, passes=3)
        assert torch.equal(dW2, dW)

