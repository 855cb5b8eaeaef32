"""Conditional flows (cond_in > 0) on the GPU: every layer-1 route of the DAG conditioner with the context term, forced by the module
flags at its shape limits, against the float64 oracle; the zero-context-weight identity with the unconditional flow; captured steps;
inversion; the coupling and MADE conditioners; argument errors."""
import pytest
import torch

import gnf_b200 as G
import cond_oracle as CO
import parity
from helpers import rel_l2

pytestmark = pytest.mark.gpu

TABLE = dict(stoch_gate=False, noise_gate=False, s_thresh=True)


@pytest.fixture
def flags():
    """Restores the layer-1 route flags and the GEMM mode after a test."""
    ops = G.ops
    saved = (ops.DAG_L1_KEEP_GATES, ops.DAG_L1_NARROW_TC_FWD, ops.DAG_L1_PLANE, ops.get_gemm_mode())
    yield ops
    ops.DAG_L1_KEEP_GATES, ops.DAG_L1_NARROW_TC_FWD, ops.DAG_L1_PLANE = saved[:3]
    ops.set_gemm_mode(saved[3])


def launched(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [e.name for e in prof.events()]


# route -> (gemm mode, flag overrides, train, kernel that must run for layer 1's forward)
ROUTES = {
    "narrow_ffma": ("ffma", dict(DAG_L1_KEEP_GATES=False), True, "dag_l1_fwd_kernel<false, true>"),
    "narrow_ffma_save": ("ffma", {}, True, "dag_l1_fwd_kernel<true, true>"),
    "narrow_tc": ("tf32x3", {}, True, "tc_gemm2_kernel<true>"),
    "narrow_tc_small": ("tf32x3", {}, True, "dag_l1_fwd_kernel<true, true>"),
    "narrow_tc_eval": ("tf32x3", {}, False, "tc_gemm2_kernel<true>"),
    "wide_ffma": ("ffma", {}, True, "EpiBiasCtxAct"),
    "wide_ffma_flag": ("tf32x3", dict(DAG_L1_PLANE=False), True, "EpiBiasCtxAct"),
    "wide_plane_v1": ("tf32x3", {}, True, "tc_gemm_kernel<true>"),
    "wide_plane_v2": ("tf32x3", {}, True, "tc_gemm2_kernel<true>"),
    "wide_plane_tf32_eval": ("tf32", {}, False, "tc_gemm_kernel<true>"),
}

# (route, B, d, N1, c, hot, norm)
CASES = [
    ("narrow_ffma", 31, 64, 256, 7, True, "affine"),
    ("narrow_ffma", 9, 63, 40, 1, False, "affine"),
    ("narrow_ffma_save", 31, 64, 256, 64, True, "monotonic"),
    ("narrow_ffma_save", 5, 32, 33, 1, True, "affine"),
    ("narrow_tc_small", 31, 64, 256, 1, True, "affine"),         # B d = 1984: below the tensor-core forward's 2048 rows
    ("narrow_tc", 32, 64, 256, 1, True, "affine"),               # B d = 2048
    ("narrow_tc", 64, 32, 256, 7, True, "monotonic"),            # d = 32, N1 = 256: the tensor-core forward's lower bounds
    ("narrow_tc", 33, 63, 300, 64, True, "affine"),
    ("narrow_tc_eval", 40, 64, 256, 7, True, "affine"),
    ("wide_ffma", 7, 65, 48, 7, True, "affine"),
    ("wide_ffma", 33, 65, 130, 1, False, "monotonic"),
    ("wide_ffma_flag", 32, 65, 256, 64, True, "affine"),
    ("wide_plane_v1", 32, 65, 256, 7, True, "affine"),           # the first plane shape: K = 65 is no engine v2 band
    ("wide_plane_v1", 31, 65, 300, 1, False, "monotonic"),
    ("wide_plane_v2", 16, 128, 256, 64, True, "affine"),
    ("wide_plane_v2", 17, 128, 257, 1, False, "affine"),
    ("wide_plane_tf32_eval", 32, 65, 256, 7, True, "affine"),
]


def _spec(B, d, N1, c, hot, norm):
    return CO.spec_of("DAG", d=d, c=c, hidden=(N1, 64), out=2, hot=hot, norm=norm)


@pytest.mark.parametrize("route,B,d,N1,c,hot,norm", CASES)
def test_conditional_layer1_route_matches_float64(flags, route, B, d, N1, c, hot, norm):
    gemm, over, train, kern = ROUTES[route]
    flags.set_gemm_mode(gemm)
    for k, v in over.items():
        setattr(flags, k, v)
    spec = _spec(B, d, N1, c, hot, norm)         # stochastic (Gumbel) gate: the narrow tensor-core forward takes no other
    rep, names = launched(lambda: CO.compare(spec, B, "cuda", seed=B + d + c, train=train))
    assert any(kern in n for n in names), f"{kern} did not run: {sorted(set(names))}"
    if train:
        assert any("dag_l1_bias_sums_kernel" in n for n in names)
    single = gemm == "tf32"
    CO.assert_report(rep, 2e-3 if single else 1e-4, 1e-3)
    if not single:
        assert rep["z_abs"] < 1e-3, rep


@pytest.mark.parametrize("route,B,d,N1,c,hot", [("narrow_ffma_save", 9, 63, 40, 7, True), ("narrow_tc", 32, 64, 256, 1, True),
                                                ("wide_ffma", 7, 65, 48, 7, False), ("wide_plane_v1", 32, 65, 256, 64, True),
                                                ("wide_plane_v2", 16, 128, 256, 7, False)])
def test_zero_context_weights_equal_unconditional(flags, route, B, d, N1, c, hot):
    """W1[:, in_net:] = 0: the conditional forward equals the unconditional one bit for bit (up to the sign of zero); its gradients
    agree to 1e-6 (the bias-table gradient comes from another reduction kernel)."""
    gemm, over, _, _ = ROUTES[route]
    flags.set_gemm_mode(gemm)
    for k, v in over.items():
        setattr(flags, k, v)
    spec = _spec(B, d, N1, c, hot, "affine")
    cmodel = G.build_from_spec(spec, "cuda", seed=1)
    CO.zero_context_columns(cmodel, spec)
    umodel = G.build_from_spec(dict(spec, cond_in=0), "cuda", seed=1)
    sd = cmodel.state_dict()
    key = "steps.0.conditioner.embedding_net.net.0.weight"
    with torch.no_grad():
        umodel.load_state_dict({k: (v[:, :v.shape[1] - c].contiguous() if k == key else v) for k, v in sd.items()})
    for m in (cmodel, umodel):
        m.getConditioners()[0]._noise_seed = 1234
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(B, d, device="cuda", generator=g)
    ctx = torch.randn(B, c, device="cuda", generator=g)
    xc, xu = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    zc, jc = cmodel(xc, ctx)
    zu, ju = umodel(xu)
    assert torch.equal(zc + 0., zu + 0.) and torch.equal(jc + 0., ju + 0.)
    (zc.square().sum() + jc.sum()).backward()
    (zu.square().sum() + ju.sum()).backward()
    up = dict(umodel.named_parameters())
    for k, p in cmodel.named_parameters():
        gc = p.grad if k != key else p.grad[:, :p.shape[1] - c]
        assert rel_l2(gc, up[k].grad) < 1e-6, k
    assert rel_l2(xc.grad, xu.grad) < 1e-6


def _train_setup(seed):
    spec = CO.spec_of("DAG", d=63, c=8, hidden=(256, 64), out=2, norm="monotonic")
    model = G.build_from_spec(spec, "cuda", seed=seed)
    parity.set_modes(model, dict(stoch_gate=False))
    bucket = G.dist.GradBucket(model.parameters())
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, fused=True, capturable=True)
    return spec, model, bucket, opt


@pytest.mark.parametrize("gemm", ["ffma", "tf32x3"])
def test_captured_steps_with_context_match_eager(flags, gemm):
    flags.set_gemm_mode(gemm)
    g = torch.Generator(device="cuda").manual_seed(4)
    B = 40
    xs = [torch.randn(B, 63, device="cuda", generator=g) for _ in range(4)]
    cs = [torch.randn(B, 8, device="cuda", generator=g) for _ in range(4)]
    spec, model_e, bucket_e, opt_e = _train_setup(2)
    for x, c in [(xs[0], cs[0])] * 3 + list(zip(xs[1:], cs[1:])):
        bucket_e.zero()
        z, jac = model_e(x, c)
        model_e.loss(z, jac).backward()
        opt_e.step()
    _, model_g, bucket_g, opt_g = _train_setup(2)
    step = G.GraphedTrainStep(model_g, opt_g, bucket_g, xs[0], allreduce=False, warmup=3, example_context=cs[0])
    losses = [float(step(x, c)) for x, c in zip(xs[1:], cs[1:])]
    assert all(l == l for l in losses)
    for (k, pe), (_, pg) in zip(model_e.named_parameters(), model_g.named_parameters()):
        err = float((pe - pg).norm() / pe.norm().clamp_min(1e-12))
        assert err < 2e-3, (k, err)
    with pytest.raises(ValueError):
        step(xs[1])
    ev = G.GraphedEvalStep(model_g, xs[0], example_context=cs[0])
    for x, c in zip(xs, cs):
        ll_g, z_g = (t.clone() for t in ev(x, c))
        with torch.no_grad():
            ll_e, z_e = model_g.compute_ll(x, c)
        assert float(((ll_g - ll_e).abs() / ll_e.abs().clamp_min(1e-6)).max()) < 1e-5
        assert float((z_g - z_e).abs().max()) < 1e-4


@pytest.mark.parametrize("norm", ["affine", "monotonic"])
def test_invert_recovers_x_with_context(norm):
    spec = CO.spec_of("DAG", d=6, c=4, hidden=(40, 40), out=2 if norm == "affine" else 6, norm=norm, nb_flow=2)
    model = G.build_from_spec(spec, "cuda", seed=5)
    for cond in model.getConditioners():
        cond.post_process()
    g = torch.Generator(device="cuda").manual_seed(6)
    x = torch.randn(64, 6, device="cuda", generator=g)
    ctx = torch.randn(64, 4, device="cuda", generator=g)
    with torch.no_grad():
        z, _ = model(x, ctx)
        xr = model.invert(z, ctx)
        xw = model.invert(z, torch.randn(64, 4, device="cuda", generator=g))
    err = float((xr - x).abs().max())
    assert err < (1e-5 if norm == "affine" else 1e-3), err
    assert float((xw - x).abs().max()) > 100 * max(err, 1e-6), "a different context must give a different inverse"


# ConditionnalMADE's h has out * d / (d + c) columns (MADE(nin + cond_in, ..., out * nin) in the reference): the affine normalizer only
@pytest.mark.parametrize("cond,nb_flow,norm", [("Coupling", 1, "affine"), ("Coupling", 3, "monotonic"), ("Autoregressive", 1, "affine"),
                                               ("Autoregressive", 3, "affine")])
def test_conditional_coupling_and_made_match_float64(flags, cond, nb_flow, norm):
    flags.set_gemm_mode("tf32x3")
    if cond == "Autoregressive":
        spec = CO.spec_of(cond, d=6, c=6, hidden=(60, 60), out=4, nb_flow=nb_flow, norm=norm)   # h: 4 * 6 / 12 = 2 columns
    else:
        spec = CO.spec_of(cond, d=8, c=5, hidden=(60, 60), out=2, nb_flow=nb_flow, norm=norm)
    rep = CO.compare(spec, 300, "cuda", seed=nb_flow)
    CO.assert_report(rep, 1e-4, 1e-3)


def test_conditional_argument_errors():
    for cond in ("DAG", "Coupling"):
        model = G.build_from_spec(CO.spec_of(cond, d=4, c=3), "cuda", seed=0)
        x = torch.randn(2, 4, device="cuda")
        for bad in (None, torch.randn(2, 2, device="cuda"), torch.randn(3, 3, device="cuda")):
            with pytest.raises(ValueError):
                model(x, bad)
        for bad in (torch.randn(2, 3), torch.randn(2, 3, device="cuda", dtype=torch.float64), torch.randn(3, 2, device="cuda").t()):
            with pytest.raises(TypeError):
                model(x, bad)
    # cond_in = 0: a context is ignored, as in the reference
    model = G.build_from_spec(CO.spec_of("DAG", d=4, c=0), "cuda", seed=0)
    parity.set_modes(model, TABLE)
    x = torch.randn(2, 4, device="cuda")
    with torch.no_grad():
        assert torch.equal(model(x)[0], model(x, torch.randn(2, 7, device="cuda"))[0])
