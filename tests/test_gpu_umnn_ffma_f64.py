"""The strict FFMA UMNN kernels, the layer-wise engine and the bisection inverse against the quadrature evaluated in float64, at
the shape limits of their instances:

  * gnf_umnn_fwd + gnf_umnn_bwd (UMNN_ENGINE = 'fused', GEMM mode 'ffma'): the largest hidden width on both sides of every
    template width TN = 2, 4, 7, 10, 13, 16 (padded widths 32 / 64 / 112 / 160 / 208 / 256), mixed widths, 2 to 8 linear layers
    up to what the backward holds in shared memory, E = 1 and E at its limits (1 + E padded to 16 = the padded hidden width;
    1 + E padded to 32 = 256), S = 1, 62 / 63 and 126 / 127 (a row's S + 1 forward or S + 2 backward node-rows end exactly on
    a 64-row tile boundary or one past it) and 1000 (one row spans 16 tiles), fewer node-rows than one tile and more than
    2 x 148 tiles (the grid-stride loops), B = d = 1, the saved-activation and the recomputing backward, each
    cotangent alone, all four together and none;
  * the routing of UmnnFn: training on integrands whose tiles the FFMA backward cannot hold in 227 KB of shared memory
    ([256, 256, 256], [160] x 5, [256, 256] with E = 255), and integrands the FFMA forward refuses (1 + E wider than the
    padded hidden width), run on the layer-wise engine with the passes of the GEMM mode;
  * gnf_umnn_fwd_lw + gnf_umnn_bwd_lw (UMNN_ENGINE = 'layerwise') with passes 0 (FFMA), 1 (TF32) and 3 (3xTF32), at hidden
    widths 161 .. 256 where the fused tensor-core kernels decline, S = 256 and 1000, E = 1;
  * gnf_umnn_invert against a float64 bisection that restates MonotonicNormalizer.inverse_transform: every TN instance,
    S = 1, 20, 62 and 63 (one row per tile), R not a multiple of the rows per tile, iters = 0, 1, 20 and 30, asymmetric
    intervals and targets outside the reachable range; S = 64 is refused.

Every GPU case asserts which UMNN entry points ran and starts from a NaN-poisoned caching allocator (umnn_ref.poison).

Bars (relative L2; z, zrev and logdet floored as in umnn_ref.rel), with the worst errors measured on a B200:
  * FFMA kernels: forward 1e-6 (measured 5.3e-7, jac of depth7_w112), gradients 2e-5 (measured 5.8e-6, dx of b1_d1; every
    other gradient <= 3.0e-6).
  * layer-wise engine, passes 0 and 3: the engine's 1e-6 on the forward (measured 6.4e-7) and 2e-4 on gradients (measured
    1.6e-5, dW0 of w161_e1 with both passes).
  * layer-wise engine, passes 1 (single-pass TF32 GEMMs): 5e-3 on the forward and 6e-2 on gradients, about twice the measured
    2.7e-3 (logdet) and 2.9e-2 (db0), both of w160x5_s256.  The project's TF32 bar of 2e-3 holds for the 2-layer nets only:
    each hidden GEMM rounds its operands to 10 mantissa bits, and the dgrad chain through five layers and the cancelling sums
    of dW0 / db0 grow that to 1e-2 .. 3e-2.
  * inverse: f = ELU + 1.05 >= 0.05, so a forward error dz moves the crossing by at most 20 dz:
    |x - x64| <= (hi - lo) / 2^iters + 20 dz + 2 ulp(max(|lo|, |hi|)), where dz is the FFMA forward's largest absolute z error on
    the same case and the last term is the float32 spacing of the midpoints (the interval stops halving there).
  * a CPU test checks that these bars see a kernel that loses one node-row at a tile boundary: the float64 quadrature with
    that node left out misses the strict bars by >= 100x at every shape used here.  (The TF32 bars cannot see one node; they
    are not part of that check.)
"""
import ctypes as C

import pytest
import torch

import gnf_b200 as G
from umnn_ref import (GNF_ERR_UNSUPPORTED, O, OUTS, UMNN_ENTRY_POINTS, check, explicit_quadrature, grad_names,
                      make_cots, make_params, reference, rel, report, run_umnn)
from umnn_ref import poison  # noqa: F401  (pytest fixture)

FFMA_FWD_BAR, FFMA_GRAD_BAR = 1e-6, 2e-5
LW_FWD_BAR, LW_GRAD_BAR = 1e-6, 2e-4
LW_TF32_FWD_BAR, LW_TF32_GRAD_BAR = 5e-3, 6e-2
SMEM_LIMIT = 227 * 1024


def inputs(widths, E, B, d, seed, device="cuda"):
    params = make_params(widths, E, seed, device)
    g = torch.Generator().manual_seed(seed + 1)
    return params, torch.randn(B, d, generator=g).to(device), torch.randn(B, d, E, generator=g).to(device)


def bars_for(n, fwd, grad):
    return {**{k: fwd for k in OUTS}, **{k: grad for k in grad_names(n)}}


def expected_route(fwd, bwd, train):
    return {fwd, bwd} if train else {fwd}


def umnn_case(poison, widths, E, B, d, S, keys=OUTS, train=True, seed=0, engine="fused", gemm="ffma", save=True,
              expect=("gnf_umnn_fwd", "gnf_umnn_bwd"), fwd_bar=FFMA_FWD_BAR, grad_bar=FFMA_GRAD_BAR):
    """Errors of one UmnnFn call against float64, with its bars; asserts that exactly the UMNN entry points `expect` ran."""
    params, x, h = inputs(widths, E, B, d, seed)
    cots = make_cots(keys, B, d, "cuda", seed + 2) if train else {}
    ref = reference(params, x, h, S, cots)
    G.ops.UMNN_ENGINE = engine
    G.ops.set_gemm_mode(gemm)
    if not save:
        G.ops.SAVE_ACTIVATIONS_MAX_BYTES = 0
    got, used = run_umnn(params, x, h, S, train, cots, poison=poison)
    assert used & UMNN_ENTRY_POINTS == expected_route(*expect, train), used
    bars = bars_for(len(params) // 2, fwd_bar, grad_bar)
    errs = {k: rel(got[k], ref[k], k, d) for k in ref}
    return errs, {k: bars[k] for k in errs}


# ---------------------------------------------------------------------------------------------------------------------
# gnf_umnn_fwd + gnf_umnn_bwd
# ---------------------------------------------------------------------------------------------------------------------
def bwd_smem_bytes(hidden, E):
    """Shared memory of gnf_umnn_bwd (umnn.cu: bwd_smem_bytes): a 64-row tile (row stride 68) of the input, padded to 32
    columns, and of every hidden layer, padded to 16 TN, two 16-row weight panels and 384 floats of scratch."""
    TN = next(t for t in (2, 4, 7, 10, 13, 16) if 16 * t >= max(hidden))
    NP, KB0 = 16 * TN, -(-(1 + E) // 32) * 32
    return (KB0 * 68 + len(hidden) * NP * 68 + 32 * NP + 384) * 4, NP


def ffma_takes(hidden, E, train=True):
    """Do gnf_umnn_fwd (and, training, gnf_umnn_bwd) take this integrand?"""
    smem, NP = bwd_smem_bytes(hidden, E)
    return max(hidden) <= 256 and -(-(1 + E) // 16) * 16 <= NP and (not train or smem <= SMEM_LIMIT)


# (widths, E, B, d, S); forward node-rows Q = B d (S + 1), backward B d (S + 2), 64-row tiles
FFMA_SHAPES = {
    "w32_kp0_eq_np": ([32, 32], 31, 10, 7, 20),           # TN = 2; 1 + E = 32 = padded hidden width
    "w33": ([33, 20], 5, 9, 5, 20),                       # TN = 4
    "w64_kp0_eq_np": ([64, 64, 64], 63, 8, 5, 11),
    "w65": ([65, 30], 3, 7, 6, 20),                       # TN = 7
    "w112": ([112, 112], 12, 6, 5, 20),
    "w113": ([113, 60, 113], 8, 5, 4, 20),                # TN = 10
    "w160_depth5": ([160, 160, 160, 160], 30, 4, 5, 20),
    "w161": ([161, 161], 9, 5, 3, 20),                    # TN = 13
    "w208_e95": ([208, 208, 208], 95, 4, 3, 20),          # 1 + E = 96: the widest input 3 x 208 hidden layers leave room for
    "w209": ([209, 100], 40, 4, 3, 20),                   # TN = 16
    "w256_kb0_256": ([256], 255, 6, 4, 20),               # 1 + E = 256: eight 32-column blocks of the first-layer dgrad
    "w256x2_e191": ([256, 256], 191, 3, 3, 9),
    "mixed_narrow_wide": ([7, 200, 3], 2, 6, 5, 20),
    "depth7_w112": ([112] * 6, 95, 3, 4, 10),             # 56 KB under the limit
    "depth8": ([64] * 7, 6, 4, 5, 20),
    "e1": ([100, 100], 1, 10, 6, 20),
    "s1": ([64, 64], 4, 40, 5, 1),
    "s62": ([48, 48], 4, 5, 7, 62),                       # forward rows of 63, backward rows of 64 node-rows
    "s63": ([48, 48], 4, 5, 7, 63),                       # forward rows of 64, backward rows of 65
    "s126": ([80, 80], 6, 3, 5, 126),
    "s127": ([80, 80], 6, 3, 5, 127),
    "s1000": ([64, 64], 3, 1, 3, 1000),                   # a row spans 16 tiles
    "b1_d1": ([100, 100, 100], 10, 1, 1, 20),             # 21 / 22 node-rows: one partial tile
    "b1_d1_s1": ([32], 1, 1, 1, 1),
    "many_tiles": ([100, 100, 100], 30, 100, 10, 20),     # 329 forward / 344 backward tiles: grid-stride loops run
}
RECOMPUTE = ["w256x2_e191", "depth8", "s63", "s1000", "many_tiles", "w32_kp0_eq_np"]


def test_ffma_shapes_fit_the_ffma_kernels():
    """CPU: every shape above is one the FFMA kernels take (else UmnnFn would route it elsewhere)."""
    for name, (widths, E, *_rest) in FFMA_SHAPES.items():
        assert ffma_takes(widths, E), name


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(FFMA_SHAPES))
def test_ffma_vs_float64(poison, shape):
    widths, E, B, d, S = FFMA_SHAPES[shape]
    errs, bars = umnn_case(poison, widths, E, B, d, S, seed=len(shape))
    report(f"ffma {shape}", errs, bars)
    check(errs, bars)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", RECOMPUTE)
def test_ffma_recomputing_backward_vs_float64(poison, shape):
    """SAVE_ACTIVATIONS_MAX_BYTES = 0: the forward keeps nothing and gnf_umnn_bwd recomputes every hidden layer."""
    widths, E, B, d, S = FFMA_SHAPES[shape]
    errs, bars = umnn_case(poison, widths, E, B, d, S, seed=len(shape), save=False)
    report(f"ffma recompute {shape}", errs, bars)
    check(errs, bars)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["w113", "s63", "w256_kb0_256"])
def test_ffma_evaluation_vs_float64(poison, shape):
    widths, E, B, d, S = FFMA_SHAPES[shape]
    errs, bars = umnn_case(poison, widths, E, B, d, S, train=False, seed=len(shape))
    report(f"ffma eval {shape}", errs, bars)
    check(errs, bars)


@pytest.mark.gpu
@pytest.mark.parametrize("save", [True, False], ids=["saved", "recompute"])
@pytest.mark.parametrize("key", OUTS)
@pytest.mark.parametrize("shape", ["s63", "w209"])
def test_ffma_single_cotangent_vs_float64(poison, shape, key, save):
    """One output's cotangent, the other three None: the backward reads NULL for them."""
    widths, E, B, d, S = FFMA_SHAPES[shape]
    errs, bars = umnn_case(poison, widths, E, B, d, S, keys=(key,), seed=11, save=save)
    report(f"ffma {shape} only {key}", errs, bars)
    check(errs, bars)


@pytest.mark.gpu
def test_ffma_backward_without_cotangents_writes_zero_gradients(poison):
    """gnf_umnn_bwd with all four cotangents NULL: every gradient, NaN-filled before the call, comes back exactly zero."""
    widths, E, B, d, S = [113, 60], 8, 9, 7, 63
    params, x, h = inputs(widths, E, B, d, 3)
    R, lib, P = B * d, G._lib.lib(), G.ops.ptr
    net = G.ops._mlp_struct(params[0::2], params[1::2])
    nbytes = lib.gnf_umnn_bwd_workspace_bytes(C.byref(net))
    assert nbytes == lib.gnf_umnn_workspace_bytes(C.byref(net)) > 0
    ws = torch.full((nbytes // 4,), float("nan"), device="cuda")
    ccw, ccn = G.ops.cc_weights(S, "cuda")
    dx, dh = torch.full_like(x, float("nan")), torch.full_like(h, float("nan"))
    dps = [torch.full_like(p, float("nan")) for p in params]
    grads = G._lib.MlpGradT()
    for l in range(len(params) // 2):
        grads.dW[l], grads.db[l] = dps[2 * l].data_ptr(), dps[2 * l + 1].data_ptr()
    jac = torch.ones_like(x)
    rc = lib.gnf_umnn_bwd(P(x), P(h), C.byref(net), S, P(ccw), P(ccn), P(jac), None, None, None, None, None, P(dx), P(dh),
                          C.byref(grads), R, d, P(ws), nbytes, G._lib.stream_ptr())
    assert rc == 0, lib.gnf_last_error()
    torch.cuda.synchronize()
    for t in [dx, dh] + dps:
        assert bool((t == 0).all())


# ---------------------------------------------------------------------------------------------------------------------
# routing of integrands the FFMA kernels refuse
# ---------------------------------------------------------------------------------------------------------------------
# (widths, E, B, d, S)
REFUSED = {
    "w256x3": ([256, 256, 256], 7, 6, 5, 20),             # backward: 251,904 B + the input tile
    "w160x5": ([160] * 5, 5, 4, 5, 20),                   # backward: ~248 KB
    "w256x2_e255": ([256, 256], 255, 3, 3, 9),            # backward: 243,200 B
    "w16x2_e40": ([16, 16], 40, 5, 4, 20),                # forward: 1 + E = 41 > padded hidden width 32
}


def test_refused_shapes_are_refused():
    """CPU: the FFMA forward or backward refuses each of these (restated shared-memory formula)."""
    for name, (widths, E, *_rest) in REFUSED.items():
        assert not ffma_takes(widths, E), name


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(REFUSED))
def test_training_on_nets_the_ffma_kernels_refuse_runs_layerwise(poison, shape):
    """Default engine, GEMM mode 'ffma': the integrand trains on gnf_umnn_fwd_lw + gnf_umnn_bwd_lw with FFMA GEMMs (until this
    routing existed, the forward ran and loss.backward() raised from gnf_umnn_bwd)."""
    widths, E, B, d, S = REFUSED[shape]
    errs, bars = umnn_case(poison, widths, E, B, d, S, seed=len(shape), engine="auto", gemm="ffma",
                           expect=("gnf_umnn_fwd_lw", "gnf_umnn_bwd_lw"), fwd_bar=LW_FWD_BAR, grad_bar=LW_GRAD_BAR)
    report(f"routed {shape}", errs, bars)
    check(errs, bars)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["w256x3", "w16x2_e40"])
def test_evaluation_route_of_refused_nets(poison, shape):
    """Evaluation needs no backward: [256, 256, 256] stays on gnf_umnn_fwd, the net whose input the FFMA forward refuses runs
    gnf_umnn_fwd_lw."""
    widths, E, B, d, S = REFUSED[shape]
    fwd = "gnf_umnn_fwd" if ffma_takes(widths, E, train=False) else "gnf_umnn_fwd_lw"
    errs, bars = umnn_case(poison, widths, E, B, d, S, train=False, seed=len(shape), engine="auto", gemm="ffma",
                           expect=(fwd, None))
    report(f"routed eval {shape}", errs, bars)
    check(errs, bars)


# ---------------------------------------------------------------------------------------------------------------------
# gnf_umnn_fwd_lw + gnf_umnn_bwd_lw
# ---------------------------------------------------------------------------------------------------------------------
LW_SHAPES = {
    "w161_e1": ([161, 161, 161], 1, 20, 5, 20),
    "w256x3": ([256, 256, 256], 7, 10, 6, 20),            # FFMA backward refuses it
    "w160x5_s256": ([160] * 5, 5, 2, 3, 256),             # FFMA backward refuses it; S + 1 > 256: no fused tc3 kernels
    "w256x2_e255_s256": ([256, 256], 255, 2, 3, 256),     # FFMA backward refuses it
    "w230_s1000_e1": ([200, 230], 1, 2, 2, 1000),
}
LW_PASSES = {0: ("ffma", LW_FWD_BAR, LW_GRAD_BAR), 1: ("tf32", LW_TF32_FWD_BAR, LW_TF32_GRAD_BAR),
             3: ("tf32x3", LW_FWD_BAR, LW_GRAD_BAR)}


@pytest.mark.gpu
@pytest.mark.parametrize("passes", list(LW_PASSES))
@pytest.mark.parametrize("shape", list(LW_SHAPES))
def test_layerwise_vs_float64(poison, shape, passes):
    widths, E, B, d, S = LW_SHAPES[shape]
    gemm, fwd_bar, grad_bar = LW_PASSES[passes]
    errs, bars = umnn_case(poison, widths, E, B, d, S, seed=len(shape), engine="layerwise", gemm=gemm,
                           expect=("gnf_umnn_fwd_lw", "gnf_umnn_bwd_lw"), fwd_bar=fwd_bar, grad_bar=grad_bar)
    report(f"layerwise passes={passes} {shape}", errs, bars)
    check(errs, bars)


# ---------------------------------------------------------------------------------------------------------------------
# bars against a kernel that loses one node-row
# ---------------------------------------------------------------------------------------------------------------------
def dropped_node(R, S):
    """(row, node) of the first forward node-row that starts a 64-row tile and carries at least the mean Clenshaw-Curtis weight
    2 / (S + 1); the middle node of the middle row when no tile boundary does.  Nodes near the ends of the interval weigh
    O(1 / S^2): at large S losing one of them alone is below what a forward bar can see (a kernel that loses node 0 of a row
    leaves its jac unwritten instead)."""
    w, _ = O.cc_weights_nodes(S)
    nodes = S + 1
    for q in range(64, R * nodes, 64):
        if float(w[q % nodes]) >= 2 / nodes:
            return q // nodes, q % nodes
    return R // 2, S // 2


STRICT_CASES = [(f"ffma_{k}", *v, FFMA_FWD_BAR, FFMA_GRAD_BAR) for k, v in FFMA_SHAPES.items()] + \
               [(f"routed_{k}", *v, LW_FWD_BAR, LW_GRAD_BAR) for k, v in REFUSED.items()] + \
               [(f"lw_{k}", *v, LW_FWD_BAR, LW_GRAD_BAR) for k, v in LW_SHAPES.items()]


@pytest.mark.parametrize("case", STRICT_CASES, ids=[c[0] for c in STRICT_CASES])
def test_bars_reject_a_lost_node_row(case):
    """CPU: the float64 quadrature without one node of one row misses the strict bars of the shape by >= 100x."""
    name, widths, E, B, d, S, fwd_bar, grad_bar = case
    params, x, h = inputs(widths, E, B, d, 0, "cpu")
    cots = make_cots(OUTS, B, d, "cpu", 2)
    ref = explicit_quadrature(params, x, h, S, cots)
    bad = explicit_quadrature(params, x, h, S, cots, drop=dropped_node(B * d, S))
    bars = bars_for(len(params) // 2, fwd_bar, grad_bar)
    worst = max(rel(bad[k], ref[k], k, d) / bars[k] for k in ref)
    assert worst >= 100, (name, worst)


# ---------------------------------------------------------------------------------------------------------------------
# gnf_umnn_invert
# ---------------------------------------------------------------------------------------------------------------------
def forward64(params, x, h, S):
    return explicit_quadrature(params, x, h, S, {})["z"]


def bisect64(params, z, h, S, iters, lo, hi):
    """MonotonicNormalizer.inverse_transform (MonotonicNormalizer.py:69-83) in float64, on the interval [lo, hi]."""
    z = z.double().cpu()
    x_max, x_min = torch.full_like(z, hi), torch.full_like(z, lo)
    for _ in range(iters):
        x_mid = (x_max + x_min) / 2
        left = forward64(params, x_mid, h, S) > z
        x_max, x_min = torch.where(left, x_mid, x_max), torch.where(left, x_min, x_mid)
    return (x_max + x_min) / 2


# (widths, E, B, d, S, iters, lo, hi); rows per tile = 64 // (S + 1)
INVERT_SHAPES = {
    "tn2_s20": ([32, 20], 3, 7, 5, 20, 20, -20., 20.),          # 3 rows per tile, R = 35
    "tn4_s62": ([64, 64], 6, 11, 3, 62, 20, -5., 12.),          # one row per tile
    "tn7_s63_iters30": ([100, 112], 9, 5, 5, 63, 30, -20., 20.),
    "tn10_s1": ([160, 150], 30, 9, 7, 1, 20, -3., 9.),          # 32 rows per tile, R = 63
    "tn13_iters1": ([208], 12, 9, 7, 20, 1, -20., 20.),
    "tn16_iters0": ([256, 256], 4, 5, 13, 20, 0, -7., 3.),
}


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(INVERT_SHAPES))
def test_invert_vs_float64_bisection(poison, shape):
    widths, E, B, d, S, iters, lo, hi = INVERT_SHAPES[shape]
    params, _, h = inputs(widths, E, B, d, len(shape))
    p64 = [p.cpu() for p in params]
    g = torch.Generator().manual_seed(7)
    x_true = lo + (hi - lo) * (.02 + .96 * torch.rand(B, d, generator=g, dtype=torch.float64))
    z = forward64(p64, x_true, h.cpu(), S).float()
    z.view(-1)[::5] = 1e4                                   # out of reach: x lands on hi
    z.view(-1)[2::5] = -1e4                                 # and on lo
    z = z.cuda()
    x64 = bisect64(p64, z, h.cpu(), S, iters, lo, hi)
    poison()
    G.ops.enable_kernel_timing(True)
    try:
        x = G.ops.umnn_invert(z, h, S, params[0::2], params[1::2], iters, lo, hi)
        used = set(G.ops.collect_kernel_timing())
    finally:
        G.ops.enable_kernel_timing(False)
    assert used == {"gnf_umnn_invert"}, used
    assert torch.isfinite(x).all()
    # the FFMA forward's absolute z error on the same case, at the points the search converged to
    G.ops.UMNN_ENGINE = "fused"
    got, used = run_umnn(params, x, h, S, False, {}, poison=poison)
    assert used & UMNN_ENTRY_POINTS == {"gnf_umnn_fwd"}, used
    dz = float((got["z"].double().cpu() - forward64(p64, x.double().cpu(), h.cpu(), S)).abs().max())
    ulp = torch.finfo(torch.float32).eps * 2 ** torch.tensor(max(abs(lo), abs(hi))).log2().ceil().item()
    bar = (hi - lo) / 2 ** iters + 20 * dz + 2 * ulp
    err = (x.double().cpu() - x64).abs()
    print(f"\n[invert {shape}] max |x - x64| = {float(err.max()):.3g} (bar {bar:.3g}; dz = {dz:.3g})")
    assert float(err.max()) <= bar, (float(err.max()), bar)
    edge = (hi - lo) / 2 ** (iters + 1)
    assert float((x.view(-1)[::5].double().cpu() - (hi - edge)).abs().max()) <= 2 * ulp
    assert float((x.view(-1)[2::5].double().cpu() - (lo + edge)).abs().max()) <= 2 * ulp


@pytest.mark.gpu
def test_invert_refuses_65_nodes():
    """S = 64: the 65 quadrature nodes of a row do not fit one 64-row tile, a loud GNF_ERR_UNSUPPORTED."""
    params, x, h = inputs([32, 32], 3, 4, 3, 0)
    with pytest.raises(RuntimeError, match=f"libgnf error {GNF_ERR_UNSUPPORTED}: .*do not fit"):
        G.ops.umnn_invert(x, h, 64, params[0::2], params[1::2])


def test_float64_bisection_inverts_the_float64_forward():
    """CPU: the float64 bisection after 40 halvings lands on the x that produced z, and on the endpoints for z out of reach."""
    params, _, h = inputs([20, 20], 3, 3, 4, 1, "cpu")
    x_true = torch.rand(3, 4, generator=torch.Generator().manual_seed(0), dtype=torch.float64) * 6 - 4
    z = forward64(params, x_true, h, 20)
    z[0, 0], z[1, 1] = 1e4, -1e4
    x = bisect64(params, z, h, 20, 40, -5., 3.)
    ok = torch.ones_like(x, dtype=torch.bool)
    ok[0, 0] = ok[1, 1] = False
    assert float((x - x_true)[ok].abs().max()) < 1e-10
    assert abs(float(x[0, 0]) - 3.) < 1e-10 and abs(float(x[1, 1]) + 5.) < 1e-10
