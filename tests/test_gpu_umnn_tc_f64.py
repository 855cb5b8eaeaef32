"""The tensor-core UMNN kernels against the quadrature evaluated in float64, at the shape limits of their instances:

  * gnf_umnn_fwd_tc3 + gnf_umnn_bwd_tc3 (3xTF32, strict): every template width NB = 1..5, uniform and mixed hidden widths,
    3..8 linear layers, S from 1 to 255 (both sides of the kernel's P-in-shared-memory switch at 12 nodes), node-row counts
    below one 128-row tile, one past a multiple of it and over one tile per SM, training and evaluation (they use different
    MMA orders), each of the four cotangents alone (the others reach the kernels as NULL) and all four together;
  * gnf_umnn_fwd_tc (single-pass TF32): padded widths NP = 16 .. 256 (the 256 instance is the switch's default case; past
    NP = 128 the kernel allocates 512 TMEM columns) and its two rejections;
  * the cfg4-shaped forward + backward captured in a CUDA graph and replayed on new inputs;
  * the route at S = 255 / 256: the fused kernels stage S + 1 <= 256 quadrature nodes, longer quadratures run layer-wise.

Every GPU case starts from a caching allocator whose free blocks are NaN-filled (`poison`), so a kernel that reads a workspace,
padding column or accumulator it never wrote produces NaN instead of a plausible number.

Bars (relative L2 unless noted):
  * forward outputs 1e-6 in training (MMA order 1: a layer's correction products first, ~K/8 truncating additions into the
    fp32 TMEM accumulator at full magnitude).  Evaluation runs order 0 (all three 3xTF32 products per k-step, ~3K/8 = 60
    truncating additions at K = 160), each off by up to one ulp (1.2e-7) in the same direction; through up to 7 layers this
    was measured at 1.6e-6 on jac and, since logdet adds d such one-sided errors, 4.7e-6 on logdet (B200): evaluation
    bar 1e-5;
  * single-pass TF32 forward: 2e-3 on z, jac, zrev and on the per-sample log-likelihood (the project's TF32 bar);
  * gradients: per tensor, 10x the error of the fused FFMA kernels (gnf_umnn_fwd / gnf_umnn_bwd) on the same case, floored at
    5e-5 and capped at 2e-4.  The floor: the truncating 3xTF32 accumulation leaves ~1e-6 one-sided per term, and dh / dW0 are
    sums over S + 1 nodes and the first hidden layer whose terms cancel ~20-fold (cfg4: measured 2.2e-5 on a B200, where the
    round-to-nearest FFMA kernels reach 1e-6).
"""
import pytest
import torch

import gnf_b200 as G
from umnn_ref import (EVAL_FWD_BAR, FWD_BAR, GNF_ERR_UNSUPPORTED, GRAD_CAP, OUTS, TF32_BAR, UMNN_ENTRY_POINTS, check,
                      explicit_quadrature, ffma_grad_bars, grad_names, make_cots, make_params, reference, rel, report, run_umnn)
from umnn_ref import poison  # noqa: F401  (pytest fixture)


@pytest.mark.parametrize("keys", [("z",), ("jac",), ("logdet",), ("zrev",), OUTS])
def test_float64_reference_matches_explicit_quadrature(keys):
    """CPU: the reference's custom backward (oracle) against autograd through the explicit node sum plus the Leibniz term."""
    B, d, E, S = 3, 4, 3, 7
    params = make_params([6, 5], E, 1, "cpu")
    g = torch.Generator().manual_seed(2)
    x, h = torch.randn(B, d, generator=g), torch.randn(B, d, E, generator=g)
    cots = make_cots(keys, B, d, "cpu", 3)
    a, b = reference(params, x, h, S, cots), explicit_quadrature(params, x, h, S, cots)
    assert set(a) == set(b) == set(OUTS) | set(grad_names(3))
    for k in a:
        assert rel(a[k], b[k]) < 1e-12, (k, rel(a[k], b[k]))
    assert float(b["dx"].abs().max()) > 0 and float(b["dW1"].abs().max()) > 0


def tc3_case(poison, widths, E, B, d, S, train, keys=OUTS, seed=0, engine="layerwise", gemm="tf32x3", expect="tc3"):
    """Errors of UmnnFn (strict, route `expect`: 'tc3' = gnf_umnn_fwd_tc3 [+ gnf_umnn_bwd_tc3], 'lw' = gnf_umnn_fwd_lw
    [+ gnf_umnn_bwd_lw]) against float64, with their bars."""
    params = make_params(widths, E, seed, "cuda")
    g = torch.Generator().manual_seed(seed + 1)
    x, h = torch.randn(B, d, generator=g).cuda(), torch.randn(B, d, E, generator=g).cuda()
    cots = make_cots(keys, B, d, "cuda", seed + 2) if train else {}
    ref = reference(params, x, h, S, cots)
    bars = {k: FWD_BAR if train else EVAL_FWD_BAR for k in OUTS}
    if train:
        gb, _ = ffma_grad_bars(params, x, h, S, cots, ref, poison)
        if expect != "tc3":
            gb = {k: GRAD_CAP for k in gb}       # the layer-wise engine's long fp32 reductions: its existing 2e-4 bar
        bars.update(gb)
    G.ops.UMNN_ENGINE = engine
    G.ops.set_gemm_mode(gemm)
    got, used = run_umnn(params, x, h, S, train, cots, poison=poison)
    fwd, bwd = {"tc3": ("gnf_umnn_fwd_tc3", "gnf_umnn_bwd_tc3"), "lw": ("gnf_umnn_fwd_lw", "gnf_umnn_bwd_lw")}[expect]
    assert fwd in used and (bwd in used) == train, used
    assert not (used & UMNN_ENTRY_POINTS) - {fwd, bwd}, used
    errs = {k: rel(got[k], ref[k], k, d) for k in bars}
    return errs, bars


# ---------------------------------------------------------------------------------------------------------------------
# gnf_umnn_fwd_tc3 + gnf_umnn_bwd_tc3
# ---------------------------------------------------------------------------------------------------------------------
# (widths, E, B, d, S): NB = ceil(max width / 32); nodes = S + 2 (training) / S + 1 (evaluation); Q = B d nodes node-rows.
# The deep integrands stay within what the FFMA backward that sets the gradient bars holds in shared memory (hidden layers x
# FFMA-padded width <= ~700).
TC3_SHAPES = {
    "nb1": ([32, 32], 4, 40, 5, 20),
    "nb2": ([64, 64, 64], 8, 33, 7, 11),                  # nodes 13 / 12: P staged in shared memory
    "nb2_mixed": ([64, 40], 12, 64, 21, 20),
    "nb3_mixed_many_tiles": ([64, 96], 12, 64, 21, 20),   # Q = 29568 in training: 231 tiles over 148 SMs
    "nb3": ([96, 96, 96], 6, 25, 4, 10),                  # training: 12 nodes (P in shared memory); evaluation: 11 (P from global)
    "nb4_s1": ([128, 128, 128], 16, 50, 10, 1),
    "nb4_mixed_q385": ([100, 128, 33], 9, 7, 5, 9),       # training: 11 nodes (P from global), Q = 385 = 3 * 128 + 1
    "nb5_cfg4": ([150, 150, 150], 30, 100, 63, 20),       # Q = 138600 in training: 1083 tiles
    "nb5_mixed_s255": ([160, 33, 150], 5, 5, 3, 255),
    "b1_d1": ([150, 150, 150], 30, 1, 1, 20),             # Q = 22: one partial tile
    "depth6": ([48, 64, 32, 64, 48], 3, 30, 6, 10),
    "depth7": ([96, 96, 96, 96, 96, 96], 10, 20, 4, 11),
    "depth8": ([64, 48, 64, 40, 64, 56, 64], 7, 16, 9, 20),
    "depth5_s255": ([150, 150, 150, 150], 6, 8, 8, 255),  # Q = 16448 in training: 129 tiles
}


@pytest.mark.gpu
@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("shape", list(TC3_SHAPES))
def test_tc3_vs_float64(poison, shape, train):
    widths, E, B, d, S = TC3_SHAPES[shape]
    errs, bars = tc3_case(poison, widths, E, B, d, S, train, seed=len(shape))
    report(f"tc3 {shape} {'train' if train else 'eval'}", errs, bars)
    check(errs, bars)


@pytest.mark.gpu
@pytest.mark.parametrize("key", OUTS)
@pytest.mark.parametrize("shape", ["nb2", "nb5_mixed", "depth8"])
def test_tc3_single_cotangent_vs_float64(poison, shape, key):
    """One output's cotangent, the other three None: the kernels read NULL for them."""
    widths, E, B, d, S = {"nb2": TC3_SHAPES["nb2"], "nb5_mixed": ([160, 33, 150], 5, 20, 7, 20),
                          "depth8": ([64, 48, 64, 40, 64, 56, 64], 7, 16, 9, 9)}[shape]
    errs, bars = tc3_case(poison, widths, E, B, d, S, True, keys=(key,), seed=7)
    report(f"tc3 {shape} only {key}", errs, bars)
    check(errs, bars)


# ---------------------------------------------------------------------------------------------------------------------
# S = 255 / 256: the fused kernels stage at most 256 quadrature nodes
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("engine,gemm", [("auto", "auto"), ("layerwise", "tf32x3")])
@pytest.mark.parametrize("S", [255, 256])
def test_quadrature_length_routes_past_the_fused_kernels(poison, engine, gemm, S):
    """S = 255 runs on gnf_umnn_fwd_tc3 / gnf_umnn_bwd_tc3, S = 256 on the layer-wise engine; both against float64.  R = 64
    rows: R (S + 2) > 16384 node-rows, so 'auto' picks the layer-wise family."""
    errs, bars = tc3_case(poison, [96, 96, 96], 5, 16, 4, S, True, seed=S, engine=engine, gemm=gemm,
                          expect="tc3" if S < 256 else "lw")
    report(f"route S={S} {engine}", errs, bars)
    check(errs, bars)


@pytest.mark.gpu
def test_quadrature_length_route_of_inverse_transform(poison):
    """inverse_transform's 'auto' choice asks the same predicate: at S = 256 it bisects on the layer-wise forward."""
    G.ops.UMNN_ENGINE = "auto"
    G.ops.set_gemm_mode("auto")
    norm = G.MonotonicNormalizer([96, 96, 96], 5, nb_steps=256).cuda()
    ps = norm.integrand_net.linear_params()
    assert G.ops.umnn_forward_on_tensor_cores(ps, 64, 255, "cuda")
    assert not G.ops.umnn_forward_on_tensor_cores(ps, 64, 256, "cuda")
    g = torch.Generator().manual_seed(0)
    x, h = (torch.randn(16, 4, generator=g) * 2).cuda(), torch.randn(16, 4, 5, generator=g).cuda()
    with torch.no_grad():
        z, _ = norm(x, h)
        x_rec = norm.inverse_transform(z, h)
    assert float((x_rec - x).abs().max()) < 2 * 40. / 2 ** 20 + 1e-5


@pytest.mark.gpu
def test_fused_backward_takes_160_wide_hidden_layers(poison):
    """Hidden 160 x 160 weights (the widest the fused kernels take) fit the resident weight-gradient kernel: gnf_umnn_bwd_tc3
    sizes a workspace for them, and UmnnFn runs gnf_umnn_fwd_tc3 + gnf_umnn_bwd_tc3, against float64 at the tc3 bars."""
    import ctypes as C
    params = make_params([160, 160, 160], 6, 0, "cuda")
    net = G.ops._mlp_struct(params[0::2], params[1::2])
    assert G._lib.lib().gnf_umnn_bwd_tc3_workspace_bytes(C.byref(net), 240, 20) > 0
    errs, bars = tc3_case(poison, [160, 160, 160], 6, 40, 6, 20, True, seed=9)
    report("fused backward 160 wide", errs, bars)
    check(errs, bars)


@pytest.mark.gpu
def test_tc3_rejects_more_than_256_nodes():
    """gnf_umnn_fwd_tc3 itself: GNF_ERR_UNSUPPORTED at S + 1 > 256, before any launch."""
    import ctypes as C
    params = make_params([96, 96, 96], 5, 0, "cuda")
    net = G.ops._mlp_struct(params[0::2], params[1::2])
    R, d = 64, 4
    nbytes = G._lib.lib().gnf_umnn_tc3_workspace_bytes(C.byref(net), R)
    assert nbytes > 0
    ws = torch.empty(nbytes // 4 + 4, device="cuda")
    x, out = torch.zeros(R, device="cuda"), [torch.empty(R, device="cuda") for _ in range(4)]
    h = torch.zeros(R, 5, device="cuda")
    ccw, ccn = G.ops.cc_weights(256, "cuda")
    P = G.ops.ptr
    rc = G._lib.lib().gnf_umnn_fwd_tc3(P(x), P(h), C.byref(net), 256, P(ccw), P(ccn), P(out[0]), P(out[1]), P(out[2]), P(out[3]),
                                        None, 0, 0, R, d, P(ws), nbytes, G._lib.stream_ptr())
    assert rc == GNF_ERR_UNSUPPORTED and b"quadrature nodes" in G._lib.lib().gnf_last_error()


# ---------------------------------------------------------------------------------------------------------------------
# gnf_umnn_fwd_tc (single-pass TF32 forward)
# ---------------------------------------------------------------------------------------------------------------------
# (widths, E, B, d, S): NP = max width rounded up to 16; 1 + E <= 32 runs the two-tile kernel where 3 NP <= 512 columns fit TMEM
TC_SHAPES = {
    16: ([16, 12], 7, 37, 11, 20),
    48: ([48, 40], 30, 20, 9, 9),
    80: ([80, 80, 72], 40, 13, 7, 40),
    128: ([128, 128], 30, 100, 63, 20),
    144: ([144, 136], 60, 9, 5, 7),
    176: ([176, 170], 20, 31, 3, 20),
    208: ([200], 30, 40, 6, 11),
    240: ([240], 100, 17, 4, 20),
    256: ([256], 30, 50, 10, 40),
}


@pytest.mark.gpu
@pytest.mark.parametrize("NP", list(TC_SHAPES))
def test_tf32_forward_vs_float64(poison, NP):
    widths, E, B, d, S = TC_SHAPES[NP]
    params = make_params(widths, E, NP, "cuda")
    g = torch.Generator().manual_seed(NP)
    x, h = torch.randn(B, d, generator=g).cuda(), torch.randn(B, d, E, generator=g).cuda()
    ref = reference(params, x, h, S, {})
    got, used = run_umnn(params, x, h, S, False, {}, fast=True, poison=poison)
    assert used == {"gnf_umnn_fwd_tc"}, used
    errs = {k: rel(got[k], ref[k], k) for k in ("z", "jac", "zrev")}
    ll = lambda z, logdet: -.5 * (z.double() ** 2).sum(1) - .5 * d * 1.8378770664093453 + logdet.double()
    ll_ref = ll(ref["z"], ref["logdet"])
    errs["ll"] = float(((ll(got["z"], got["logdet"]) - ll_ref).abs() / ll_ref.abs().clamp_min(1e-6)).max())
    bars = {k: TF32_BAR for k in errs}
    report(f"tf32 NP={NP}", errs, bars)
    check(errs, bars)


@pytest.mark.gpu
@pytest.mark.parametrize("widths,E,msg", [([16], 20, "widths out of range"), ([240, 240], 8, "shared memory")])
def test_tf32_forward_rejections_are_loud(widths, E, msg):
    """1 + E wider than the padded hidden width; resident weight images over 227 KB of shared memory."""
    params = make_params(widths, E, 0, "cuda")
    x, h = torch.randn(4, 3, device="cuda"), torch.randn(4, 3, E, device="cuda")
    with pytest.raises(RuntimeError, match=msg):
        G.ops.UmnnFn.apply(x, h, 20, False, True, *params)


# ---------------------------------------------------------------------------------------------------------------------
# captured forward + backward
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_tc3_captured_forward_backward_vs_float64(poison):
    """cfg4's normalizer shape (B = 100, d = 63, 30 -> 150^3 -> 1, S = 20) forward + backward of all four outputs captured in
    one CUDA graph (the library forks side streams inside both directions), replayed on two new inputs / cotangent sets."""
    widths, E, B, d, S = [150, 150, 150], 30, 100, 63, 20
    G.ops.UMNN_ENGINE = "layerwise"
    G.ops.set_gemm_mode("tf32x3")
    params = [p.requires_grad_(True) for p in make_params(widths, E, 5, "cuda")]
    names = grad_names(4)
    sx, sh = torch.zeros(B, d, device="cuda", requires_grad=True), torch.zeros(B, d, E, device="cuda", requires_grad=True)
    scots = make_cots(OUTS, B, d, "cuda", 0)

    def step():
        outs = G.ops.UmnnFn.apply(sx, sh, S, True, False, *params)
        grads = torch.autograd.grad(outs, [sx, sh] + params, [scots[k] for k in OUTS])
        return dict(zip(OUTS + tuple(names), [o.detach() for o in outs] + list(grads)))

    def load(seed):
        g = torch.Generator().manual_seed(seed)
        with torch.no_grad():
            sx.copy_(torch.randn(B, d, generator=g))
            sh.copy_(torch.randn(B, d, E, generator=g))
            for k, v in make_cots(OUTS, B, d, "cpu", seed + 1).items():
                scots[k].copy_(v)

    load(1)
    G.ops.enable_kernel_timing(True)
    step()
    used = set(G.ops.collect_kernel_timing())
    G.ops.enable_kernel_timing(False)
    assert {"gnf_umnn_fwd_tc3", "gnf_umnn_bwd_tc3"} <= used, used
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    poison()
    with torch.cuda.graph(graph):
        out = step()
    for seed in (11, 12):
        load(seed)
        graph.replay()
        torch.cuda.synchronize()
        cots = {k: v.clone() for k, v in scots.items()}
        ref = reference(params, sx, sh, S, cots)
        bars, _ = ffma_grad_bars(params, sx.detach(), sh.detach(), S, cots, ref, poison)
        bars.update({k: FWD_BAR for k in OUTS})
        errs = {k: rel(out[k], ref[k], k, d) for k in bars}
        report(f"captured replay {seed}", errs, bars)
        check(errs, bars)
        G.ops.UMNN_ENGINE = "layerwise"
        G.ops.set_gemm_mode("tf32x3")
