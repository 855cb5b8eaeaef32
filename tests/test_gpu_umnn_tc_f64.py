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
import os
import sys

import pytest
import torch

import gnf_b200 as G

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import gnf_oracle as O  # noqa: E402

OUTS = ("z", "jac", "logdet", "zrev")
FWD_BAR, EVAL_FWD_BAR, TF32_BAR, GRAD_FLOOR, GRAD_CAP = 1e-6, 1e-5, 2e-3, 5e-5, 2e-4
GNF_ERR_UNSUPPORTED = 1002                  # include/gnf.h


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference
# ---------------------------------------------------------------------------------------------------------------------
def make_params(widths, E, seed, device):
    """Integrand [1 + E] -> widths -> 1: He-uniform weights (activations keep their scale through deep ReLU stacks), small biases."""
    g = torch.Generator().manual_seed(seed)
    dims = [1 + E] + list(widths) + [1]
    params = []
    for i, o in zip(dims[:-1], dims[1:]):
        params += [(torch.rand(o, i, generator=g) * 2 - 1) * (6. / i) ** .5, torch.randn(o, generator=g) * .1]
    return [p.to(device) for p in params]


def grad_names(n):
    return ["dx", "dh"] + [f"{k}{l}" for l in range(n) for k in ("dW", "db")]


def _sd(p64):
    return {f"n.{2 * (i // 2)}.{('weight', 'bias')[i % 2]}": p for i, p in enumerate(p64)}


def reference(params, x, h, S, cots):
    """z, jac, logdet = log(jac).sum(1), zrev = z.flip(1) in float64 (oracle/gnf_oracle.monotonic_normalizer, UMNN's gradient
    convention) and, for the cotangents given in `cots` (output name -> tensor), the gradients of x, h and every parameter."""
    n = len(params) // 2
    p64 = [p.detach().double().requires_grad_(True) for p in params]
    x64 = x.detach().double().requires_grad_(True)
    h64 = h.detach().double().requires_grad_(True)
    z, jac = O.monotonic_normalizer(x64, h64, _sd(p64), "n", n, S)
    outs = {"z": z, "jac": jac, "logdet": torch.log(jac).sum(1), "zrev": z.flip(1)}
    ref = {k: v.detach() for k, v in outs.items()}
    keys = [k for k in OUTS if cots.get(k) is not None]
    if keys:
        grads = torch.autograd.grad([outs[k] for k in keys], [x64, h64] + p64, [cots[k].double() for k in keys])
        ref.update(zip(grad_names(n), grads))
    return ref


def explicit_quadrature(params, x, h, S, cots):
    """The same quantities from plain autograd through an explicit float64 sum over the quadrature nodes.  The nodes are
    detached from x: UMNN differentiates the integral's upper limit by the Leibniz rule, dx += f(x) * (gz + gzrev flipped)."""
    n = len(params) // 2
    p64 = [p.detach().double().requires_grad_(True) for p in params]
    x64 = x.detach().double().requires_grad_(True)
    h64 = h.detach().double().requires_grad_(True)
    sd = _sd(p64)
    B, d = x.shape
    hr, xr = h64.reshape(B * d, -1), x64.reshape(B * d)
    xc = xr.detach()
    w, t = O.cc_weights_nodes(S)
    acc = sum(w[k] * O.integrand(xc * (t[k] + 1) / 2, hr, sd, "n", n) for k in range(S + 1))
    z = (acc * xc / 2).view(B, d) + h64[:, :, 0]
    jac = O.integrand(xr, hr, sd, "n", n).view(B, d)
    outs = {"z": z, "jac": jac, "logdet": torch.log(jac).sum(1), "zrev": z.flip(1)}
    ref = {k: v.detach() for k, v in outs.items()}
    keys = [k for k in OUTS if cots.get(k) is not None]
    grads = torch.autograd.grad([outs[k] for k in keys], [x64, h64] + p64, [cots[k].double() for k in keys], allow_unused=True)
    grads = [g if g is not None else torch.zeros_like(v) for g, v in zip(grads, [x64, h64] + p64)]
    gz = torch.zeros_like(z)
    if cots.get("z") is not None:
        gz = gz + cots["z"].double()
    if cots.get("zrev") is not None:
        gz = gz + cots["zrev"].double().flip(1)
    grads[0] = grads[0] + jac.detach() * gz
    ref.update(zip(grad_names(n), grads))
    return ref


def make_cots(keys, B, d, device, seed):
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randn(*((B,) if k == "logdet" else (B, d)), generator=g).to(device) for k in keys}


def rel(got, ref, key=None, d=1):
    """Relative L2.  z, zrev and logdet are sums whose terms are O(1) even where the sum is near zero (fp32 carries an absolute
    error there, not a relative one), so their norm is floored at sqrt(number of terms): numel, times d for logdet."""
    ref = ref.double()
    den = ref.norm()
    if key in ("z", "zrev", "logdet"):
        den = den.clamp_min((ref.numel() * (d if key == "logdet" else 1)) ** .5)
    return float((got.double() - ref).norm() / den.clamp_min(1e-300))


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


# ---------------------------------------------------------------------------------------------------------------------
# GPU harness
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def poison():
    """Returns a function that NaN-fills free blocks in the small (<= 1 MB) and the large pool of the caching allocator and
    releases them again (no empty_cache): the next torch.empty calls -- workspaces, saved planes, outputs -- start non-finite."""
    def fill():
        held = [torch.full((n,), float("nan"), device="cuda") for n in [64, 1024, 16384, 65536, 262144] * 4]
        held += [torch.full((n,), float("nan"), device="cuda") for n in (1 << 20, 1 << 22, 1 << 24, 1 << 26, 1 << 28)]
        del held
    fill()
    yield fill
    G.ops.UMNN_ENGINE = "auto"
    G.ops.set_gemm_mode("ffma")


def run_umnn(params, x, h, S, train, cots, fast=False, poison=None):
    """One UmnnFn forward (+ backward of the given cotangents when training) with kernel timing on: (outputs + gradients, entry
    points called)."""
    xg, hg = x.detach().clone().requires_grad_(train), h.detach().clone().requires_grad_(train)
    ps = [p.detach().clone().requires_grad_(train) for p in params]
    if poison is not None:
        poison()
    G.ops.enable_kernel_timing(True)
    try:
        with torch.set_grad_enabled(train):
            outs = dict(zip(OUTS, G.ops.UmnnFn.apply(xg, hg, S, True, fast, *ps)))
            got = {k: v.detach() for k, v in outs.items()}
            keys = [k for k in OUTS if cots.get(k) is not None]
            if train:
                grads = torch.autograd.grad([outs[k] for k in keys], [xg, hg] + ps, [cots[k] for k in keys])
                got.update(zip(grad_names(len(ps) // 2), grads))
        used = set(G.ops.collect_kernel_timing())
    finally:
        G.ops.enable_kernel_timing(False)
    for k, v in got.items():
        assert torch.isfinite(v).all(), f"{k} is not finite"
    return got, used


def ffma_grad_bars(params, x, h, S, cots, ref, poison):
    """Gradient bars of a case: 10x the fused FFMA kernels' float64 error, floored at 5e-5, capped at 2e-4."""
    G.ops.UMNN_ENGINE = "fused"
    G.ops.set_gemm_mode("ffma")
    got, used = run_umnn(params, x, h, S, True, cots, poison=poison)
    assert {"gnf_umnn_fwd", "gnf_umnn_bwd"} <= used, used
    errs = {k: rel(got[k], ref[k]) for k in grad_names(len(params) // 2)}
    return {k: min(GRAD_CAP, max(GRAD_FLOOR, 10 * e)) for k, e in errs.items()}, errs


def report(tag, errs, bars):
    worst = max(errs, key=lambda k: errs[k] / bars[k])
    print(f"\n[{tag}] worst {worst}: {errs[worst]:.3g} (bar {bars[worst]:.3g}); "
          + " ".join(f"{k}={errs[k]:.2g}/{bars[k]:.2g}" for k in errs))


def check(errs, bars):
    bad = {k: (errs[k], bars[k]) for k in errs if not errs[k] < bars[k]}
    assert not bad, f"out of tolerance (error, bar): {bad}"


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
    fwd, bwd = {"tc3": ("gnf_umnn_fwd_tc3", "gnf_umnn_bwd_tc3"), "lw": ("gnf_umnn_fwd_lw", "gnf_umnn_bwd_lw"),
                "tc3_lw": ("gnf_umnn_fwd_tc3", "gnf_umnn_bwd_lw")}[expect]
    others = {"gnf_umnn_fwd_tc3", "gnf_umnn_bwd_tc3", "gnf_umnn_fwd_lw", "gnf_umnn_bwd_lw", "gnf_umnn_fwd", "gnf_umnn_bwd"}
    assert fwd in used and (bwd in used) == train, used
    assert not (used & others) - {fwd, bwd}, used
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
def test_fused_backward_rejection_runs_layerwise(poison):
    """Hidden 160 x 160 weights do not fit the resident weight-gradient kernel: gnf_umnn_bwd_tc3 declines the shape (zero workspace,
    error message), and UmnnFn's backward runs gnf_umnn_bwd_lw after the fused forward; against float64 at its 2e-4 bar."""
    import ctypes as C
    params = make_params([160, 160, 160], 6, 0, "cuda")
    net = G.ops._mlp_struct(params[0::2], params[1::2])
    assert G._lib.lib().gnf_umnn_bwd_tc3_workspace_bytes(C.byref(net), 240, 20) == 0
    assert b"resident weight-gradient" in G._lib.lib().gnf_last_error()
    errs, bars = tc3_case(poison, [160, 160, 160], 6, 40, 6, 20, True, seed=9, expect="tc3_lw")
    report("fused backward declined", errs, bars)
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
