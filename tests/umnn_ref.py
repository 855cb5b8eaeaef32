"""Float64 reference of the UMNN integral and the GPU harness shared by the float64 tests of every UMNN engine
(test_gpu_umnn_tc_f64.py, test_gpu_umnn_ffma_f64.py): parameters, the reference (oracle/gnf_oracle.monotonic_normalizer, UMNN's
gradient convention) and an explicit node sum that can drop one node, cotangents, the relative error, the NaN-poisoned
allocator, one UmnnFn call with the entry points it ran, and the bar helpers."""
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
UMNN_ENTRY_POINTS = {"gnf_umnn_fwd_tc3", "gnf_umnn_bwd_tc3", "gnf_umnn_fwd_lw", "gnf_umnn_bwd_lw", "gnf_umnn_fwd", "gnf_umnn_bwd"}


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


def explicit_quadrature(params, x, h, S, cots, drop=None):
    """The same quantities from plain autograd through an explicit float64 sum over the quadrature nodes.  The nodes are
    detached from x: UMNN differentiates the integral's upper limit by the Leibniz rule, dx += f(x) * (gz + gzrev flipped).
    drop = (row, node): that node of that row (row = b * d + i) is left out of the sum, as a kernel that loses one node-row
    at a tile boundary would."""
    n = len(params) // 2
    p64 = [p.detach().double().requires_grad_(True) for p in params]
    x64 = x.detach().double().requires_grad_(True)
    h64 = h.detach().double().requires_grad_(True)
    sd = _sd(p64)
    B, d = x.shape
    hr, xr = h64.reshape(B * d, -1), x64.reshape(B * d)
    xc = xr.detach()
    w, t = O.cc_weights_nodes(S)
    acc = 0
    for k in range(S + 1):
        wk = torch.full((B * d,), float(w[k]), dtype=torch.float64)
        if drop is not None and drop[1] == k:
            wk[drop[0]] = 0
        acc = acc + wk * O.integrand(xc * (t[k] + 1) / 2, hr, sd, "n", n)
    z = (acc * xc / 2).view(B, d) + h64[:, :, 0]
    jac = O.integrand(xr, hr, sd, "n", n).view(B, d)
    outs = {"z": z, "jac": jac, "logdet": torch.log(jac).sum(1), "zrev": z.flip(1)}
    ref = {k: v.detach() for k, v in outs.items()}
    keys = [k for k in OUTS if cots.get(k) is not None]
    if not keys:
        return ref
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


# ---------------------------------------------------------------------------------------------------------------------
# GPU harness
# ---------------------------------------------------------------------------------------------------------------------
def poison_allocator():
    """NaN-fill free blocks in the small (<= 1 MB) and the large pool of the caching allocator and release them again (no
    empty_cache): the next torch.empty calls -- workspaces, saved planes, outputs -- start non-finite."""
    held = [torch.full((n,), float("nan"), device="cuda") for n in [64, 1024, 16384, 65536, 262144] * 4]
    held += [torch.full((n,), float("nan"), device="cuda") for n in (1 << 20, 1 << 22, 1 << 24, 1 << 26, 1 << 28)]
    del held


@pytest.fixture
def poison():
    """Returns poison_allocator after a first fill; restores the library's UMNN engine, GEMM mode and activation budget."""
    budget = G.ops.SAVE_ACTIVATIONS_MAX_BYTES
    poison_allocator()
    yield poison_allocator
    G.ops.UMNN_ENGINE = "auto"
    G.ops.set_gemm_mode("ffma")
    G.ops.SAVE_ACTIVATIONS_MAX_BYTES = budget


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
