"""Conditional flows (cond_in > 0): the conditional DAG and coupling conditioners restated on the oracle's building blocks
(oracle/gnf_oracle.py: masked input, MLP, normalizers, MADE), and a seeded product model with a context compared against that
float64 reference on the same inputs, weights and gate noise.  Shared by the simulator and GPU tests of the conditional routes.

Semantics (the reference builds the wider first layers, DAGConditioner.py:7-20 and CouplingConditioner.py:6-18, but never feeds
the context in: quirk Q8):
  * DAG, cond_in = c > 0: the embedding net's input row for sample b, variable i is [e[b,i,:] | onehot(i) (hot_encoding) |
    context[b,:]], the in_net + cond_in columns of DAGMLP's first Linear;
  * coupling, c > 0: the embedding net takes cat(x[:, :indep], context);
  * c = 0: the oracle's own conditioners (a context is ignored, like the reference)."""
import math
import os
import sys

import torch

import gnf_b200 as G
from helpers import rel_err, rel_l2
import parity

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import gnf_oracle as O  # noqa: E402


def _check_context(context, B, c, who):
    if context is None or tuple(context.shape) != (B, c):
        raise ValueError(f"a conditional {who} conditioner needs a [B, {c}] context")


def dag_conditioner(x, sd, prefix, spec, mode=None, noise=None, context=None):
    """h [B, d, H] of a DAG conditioner with cond_in = c > 0."""
    B, d = x.shape
    c = spec["cond_in"]
    _check_context(context, B, c, "DAG")
    e = O.dag_masked_input(x, sd[f"{prefix}.A"], mode, spec.get("gumble_T", 1.), noise)
    if spec.get("hot_encoding", False):
        e = torch.cat((e, torch.eye(d, dtype=e.dtype).unsqueeze(0).expand(B, -1, -1).reshape(-1, d)), 1)
    e = torch.cat((e, context.unsqueeze(1).expand(B, d, c).reshape(B * d, c)), 1)
    return O.mlp(e, sd, f"{prefix}.embedding_net.net", len(spec["hidden"]) + 1).view(B, d, -1)


def coupling_conditioner(x, sd, prefix, spec, context=None):
    """h [B, d, H] of a coupling conditioner with cond_in = c > 0."""
    B, d = x.shape
    cond = int(d / 2)
    indep = d - cond
    _check_context(context, B, spec["cond_in"], "coupling")
    h1 = sd[f"{prefix}.constants"].unsqueeze(0).expand(B, -1, -1)
    h2 = O.mlp(torch.cat((x[:, :indep], context), 1), sd, f"{prefix}.embeding_net.net", len(spec["hidden"]) + 1)
    return torch.cat((h1, h2.view(B, cond, spec["out"])), 1)


def flow_forward(x, sd, spec, modes=None, noises=None, context=None):
    """O.flow_forward with the conditional conditioners above: (z, log-determinant)."""
    jac_tot = 0.
    inv_idx = torch.arange(x.shape[1] - 1, -1, -1).long()
    z = None
    c = spec.get("cond_in", 0)
    for k in range(spec["nb_flow"]):
        pc = f"steps.{k}.conditioner"
        mode = None if modes is None else modes[k]
        noise = None if noises is None else noises[k]
        if spec["cond"] == "DAG":
            h = dag_conditioner(x, sd, pc, spec, mode, noise, context) if c else O.dag_conditioner(x, sd, pc, spec, mode, noise)
        elif spec["cond"] == "Coupling":
            h = coupling_conditioner(x, sd, pc, spec, context) if c else O.coupling_conditioner(x, sd, pc, spec, context)
        else:
            h = O.made_conditioner(x, sd, pc, spec, context)
        if spec["norm"] == "affine":
            z, jac = O.affine_normalizer(x, h)
        else:
            z, jac = O.monotonic_normalizer(x, h, sd, f"steps.{k}.normalizer.integrand_net.net", len(spec["int_net"]) + 1,
                                            spec["nb_steps"])
        x = z[:, inv_idx]
        jac_tot = jac_tot + torch.log(jac).sum(1)
    return z, jac_tot


def init_state_dict(spec, seed=0):
    """O.init_state_dict of the unconditional flow, with cond_in more columns (nn.Linear's init bound for the wider layer) in the
    first layer of every DAG / coupling embedding net."""
    c = spec.get("cond_in", 0)
    sd = O.init_state_dict(dict(spec, cond_in=0), seed=seed)
    if c == 0:
        return sd
    if spec["cond"] not in ("DAG", "Coupling"):
        raise NotImplementedError("conditional MADE: take the state_dict of a product model")
    g = torch.Generator().manual_seed(seed + 1)
    net = "embedding_net" if spec["cond"] == "DAG" else "embeding_net"
    for k in range(spec["nb_flow"]):
        key = f"steps.{k}.conditioner.{net}.net.0.weight"
        W = sd[key]
        bound = 1. / math.sqrt(W.shape[1] + c)
        sd[key] = torch.cat((W, (torch.rand(W.shape[0], c, generator=g) * 2 - 1) * bound), 1)
    return sd


def spec_of(cond="DAG", d=5, c=3, hidden=(24, 24), out=2, hot=True, norm="affine", nb_flow=1, **kw):
    s = dict(nb_flow=nb_flow, d=d, cond=cond, hidden=list(hidden), out=out, cond_in=c, norm=norm, gumble_T=.5, l1=0.)
    if cond == "DAG":
        s["hot_encoding"] = hot
    if norm == "monotonic":
        s.update(int_net=[16, 16], nb_steps=10, solver="CC")
    s.update(kw)
    return s


def oracle_grads(x, ctx, sd, spec, modes, noises, keys):
    """float64 forward + autograd of sum(ll) through the oracle: (ll, z, {key: grad}, dcontext)."""
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    for k in keys:
        sd64[k] = sd64[k].detach().clone().requires_grad_(True)
    x64 = x.double().detach().clone().requires_grad_(True)
    c64 = ctx.double().detach().clone().requires_grad_(True) if ctx is not None else None
    nz = None if noises is None else [None if n is None else tuple(t.double() for t in n) for n in noises]
    z, jac = flow_forward(x64, sd64, spec, modes, nz, c64)
    ll = O.normal_log_density(z) + jac
    wrt = [sd64[k] for k in keys] + [x64] + ([c64] if c64 is not None else [])
    grads = torch.autograd.grad(ll.sum(), wrt, allow_unused=True)
    g = dict(zip(keys, grads[:len(keys)]))
    g["x"] = grads[len(keys)]
    if c64 is not None:
        g["context"] = grads[len(keys) + 1]
    return ll.detach(), z.detach(), g


def compare(spec, B, device, mode=None, seed=0, train=True, zero_context_weights=False):
    """Relative errors of a conditional flow against the float64 oracle: ll (max relative), z (max abs), and with train=True the
    relative L2 error of the gradient of sum(ll) w.r.t. every parameter, x and the context."""
    model = G.build_from_spec(spec, device, seed)
    parity.set_modes(model, mode)
    if zero_context_weights:
        zero_context_columns(model, spec)
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, spec["d"], generator=g).to(device)
    ctx = torch.randn(B, spec["cond_in"], generator=g).to(device)
    if train:
        x.requires_grad_(True)
        ctx.requires_grad_(True)
    model.zero_grad()
    with torch.set_grad_enabled(train):
        z, jac = model(x, ctx)
        ll = model.z_log_density(z) + jac
    noises = dag_noises(model, spec, B, x.device)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    ospec = {k: v for k, v in spec.items() if k != "A_prior"}
    modes = None if mode is None else [mode] * spec["nb_flow"]
    params = dict(model.named_parameters())
    keys = [k for k in O.trainable_keys(sd) if k in params and params[k].requires_grad]
    ll_o, z_o, g_o = oracle_grads(x.detach().cpu(), ctx.detach().cpu(), sd, ospec, modes, noises, keys)
    rep = {"ll": rel_err(ll.detach().cpu(), ll_o), "z_abs": float((z.detach().cpu().double() - z_o).abs().max())}
    if train:
        ll.sum().backward()
        for k in keys:
            if g_o[k] is None:
                continue
            assert params[k].grad is not None, k
            rep["grad." + k] = rel_l2(params[k].grad.detach().cpu(), g_o[k])
        rep["grad.x"] = rel_l2(x.grad.detach().cpu(), g_o["x"])
        rep["grad.context"] = rel_l2(ctx.grad.detach().cpu(), g_o["context"])
    return rep


def dag_noises(model, spec, B, device):
    """The gate noise each DAG step drew (replayed into the oracle), or None."""
    if spec["cond"] != "DAG":
        return None
    noises = [tuple(n.cpu() for n in G.ops.dag_dump_noise(c._last_gate, B, spec["d"], device)) if c._last_gate.mode != G._lib.GATE_TABLE
              else None for c in model.getConditioners()]
    return None if all(n is None for n in noises) else noises


def first_linear(cond):
    return cond.embedding_net.net[0] if hasattr(cond, "embedding_net") else cond.embeding_net.net[0]


def zero_context_columns(model, spec):
    """W1[:, in_net:] = 0 in every conditioner: the conditional flow then computes the unconditional one."""
    with torch.no_grad():
        for cond in model.getConditioners():
            lin = first_linear(cond)
            lin.weight[:, lin.weight.shape[1] - spec["cond_in"]:] = 0.


def assert_report(rep, ll_tol, grad_tol):
    bad = {k: v for k, v in rep.items() if (k == "ll" and v > ll_tol) or (k.startswith("grad.") and v > grad_tol)}
    assert not bad, f"{bad} (all: {rep})"
