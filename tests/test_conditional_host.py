"""Conditional flows (cond_in > 0) without a GPU: the conditional float64 reference of tests/cond_oracle.py, and the conditional
layer-1 kernels (csrc/mlp.cu) run by the host SIMT simulator (tests/emu) against it."""
import ctypes as C
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

import gnf_b200 as G
import cond_oracle as CO
from cond_oracle import O
import sim_hook

TABLE = dict(stoch_gate=False, noise_gate=False, s_thresh=True)      # deterministic soft-threshold gate


def _oracle_ll(spec, sd, x, ctx, noises=None):
    z, jac = CO.flow_forward(x, sd, spec, None, noises, ctx)
    return O.normal_log_density(z) + jac, z


# ---------------------------------------------------------------------------------------------------------------------------
# oracle
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cond,norm,nb_flow", [("DAG", "affine", 1), ("DAG", "monotonic", 2), ("Coupling", "affine", 2),
                                               ("Coupling", "monotonic", 1)])
def test_oracle_zero_context_weights_equal_unconditional(cond, norm, nb_flow):
    """Columns in_net.. of layer 1 set to zero: the conditional oracle flow computes the unconditional one, whatever the context."""
    spec = CO.spec_of(cond, d=4, c=3, norm=norm, nb_flow=nb_flow)
    uspec = dict(spec, cond_in=0)
    sd = CO.init_state_dict(spec, seed=3)
    usd = dict(sd)
    for k in range(nb_flow):
        net = "embedding_net" if cond == "DAG" else "embeding_net"
        key = f"steps.{k}.conditioner.{net}.net.0.weight"
        W = sd[key].clone()
        W[:, -3:] = 0.
        sd[key], usd[key] = W, W[:, :-3].contiguous()
    g = torch.Generator().manual_seed(5)
    x, ctx = torch.randn(6, 4, generator=g), torch.randn(6, 3, generator=g) * 10.
    noises = [(torch.rand(6, 4, 4, generator=g), torch.rand(6, 4, 4, generator=g)) for _ in range(nb_flow)] if cond == "DAG" else None
    ll, z = _oracle_ll(spec, sd, x, ctx, noises)
    ll0, z0 = _oracle_ll(uspec, usd, x, None, noises)
    assert torch.equal(ll, ll0) and torch.equal(z, z0)


@pytest.mark.parametrize("cond", ["DAG", "Coupling"])
def test_oracle_context_gradients_match_finite_differences(cond):
    """The oracle's conditional flow is differentiable in the context and in layer 1's context columns: float64 gradcheck."""
    spec = CO.spec_of(cond, d=3, c=2, hidden=(6,), nb_flow=2)
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in CO.init_state_dict(spec, seed=1).items()}
    net = "embedding_net" if cond == "DAG" else "embeding_net"
    key = f"steps.0.conditioner.{net}.net.0.weight"
    g = torch.Generator().manual_seed(2)
    x = torch.randn(4, 3, generator=g, dtype=torch.float64)
    ctx = torch.randn(4, 2, generator=g, dtype=torch.float64, requires_grad=True)
    W = sd[key].clone().requires_grad_(True)
    noises = [(torch.rand(4, 3, 3, generator=g, dtype=torch.float64), torch.rand(4, 3, 3, generator=g, dtype=torch.float64))] * 2 \
        if cond == "DAG" else None

    def f(c, w):
        s = dict(sd)
        s[key] = w
        return _oracle_ll(spec, s, x, c, noises)[0]
    assert torch.autograd.gradcheck(f, (ctx, W), eps=1e-6, atol=1e-6)


def test_oracle_rejects_missing_or_misshapen_context():
    for cond in ("DAG", "Coupling"):
        spec = CO.spec_of(cond, d=4, c=3)
        sd = CO.init_state_dict(spec, seed=0)
        x = torch.randn(2, 4)
        for ctx in (None, torch.randn(2, 2), torch.randn(3, 3)):
            with pytest.raises(ValueError):
                _oracle_ll(spec, sd, x, ctx, [(torch.rand(2, 4, 4), torch.rand(2, 4, 4))])


# ---------------------------------------------------------------------------------------------------------------------------
# simulator
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu():
    import build_emu
    path = build_emu.build()
    sim_hook.install(path)
    yield
    sim_hook.uninstall()


# (B, d, N1, c, hot): c = 1 and c > N1 / 4; B*d = 9, 65, 130, 195 not multiples of the 32-row tile; d = 64 (last resident-gate
# shape) and 65 (the tile GEMM's DAG loader)
SHAPES = [(3, 3, 20, 1, True), (13, 5, 40, 7, False), (2, 64, 36, 3, True), (3, 65, 20, 1, False), (2, 65, 33, 5, True)]


@pytest.mark.parametrize("B,d,N1,c,hot", SHAPES)
def test_conditional_layer1_training_in_simulator(emu, B, d, N1, c, hot):
    """Stochastic gate, training: gnf_dag_l1_fwd_cond with the gate planes (the resident-gate kernel with kSave) for d <= 64, the tile
    GEMM with the context epilogue for d > 64; backward through gnf_dag_l1_bias_sums and the context GEMMs.  ll, and the gradient of
    sum(ll) w.r.t. every parameter, x and the context, against the float64 oracle."""
    torch.set_num_threads(1)
    spec = CO.spec_of("DAG", d=d, c=c, hidden=(N1,), out=2, hot=hot)
    rep = CO.compare(spec, B, "cpu", seed=B + d + c)
    CO.assert_report(rep, 1e-4, 1e-3)


@pytest.mark.parametrize("B,d,N1,c,hot", SHAPES)
def test_conditional_layer1_evaluation_in_simulator(emu, B, d, N1, c, hot):
    """Deterministic gate, no gradient: gnf_dag_l1_fwd_cond without planes (resident-gate kernel, kSave off) for d <= 64, the tile GEMM
    for d > 64."""
    torch.set_num_threads(1)
    spec = CO.spec_of("DAG", d=d, c=c, hidden=(N1, 12), out=2, hot=hot)
    rep = CO.compare(spec, B, "cpu", mode=TABLE, seed=2 * B + d, train=False)
    CO.assert_report(rep, 1e-4, 1e-3)


@pytest.mark.parametrize("B,d,N,period,lds", [(1, 1, 1, 1, 4), (3, 5, 40, 5, 40), (9, 7, 300, 1, 304), (17, 65, 33, 65, 36),
                                              (2, 3, 257, 3, 260)])
def test_bias_sums_kernel_in_simulator(emu, B, d, N, period, lds):
    """gnf_dag_l1_bias_sums: dT[i % period] = sum_b delta[b*d+i], S[b] = sum_i delta[b*d+i], delta with a padded row stride,
    samples past a multiple of the kernel's batch chunk, and the padding columns of S left alone."""
    torch.set_num_threads(1)
    from gnf_b200.ops import _call, ptr, stream_ptr
    g = torch.Generator().manual_seed(B * N + d)
    ldd = N + 3
    full = torch.randn(B * d, ldd, generator=g)
    delta = full[:, :N]
    dT = torch.full((period, N), float("nan"))
    S = torch.full((B, lds), float("nan"))
    _call("gnf_dag_l1_bias_sums", ptr(full), ldd, ptr(dT), ptr(S), lds, B, d, N, period, stream_ptr())
    d64 = delta.double().view(B, d, N)
    want_T = d64.sum(0) if period == d else d64.sum((0, 1)).view(1, N)
    want_S = d64.sum(1)
    assert torch.allclose(dT.double(), want_T, rtol=1e-5, atol=1e-5)
    assert torch.allclose(S[:, :N].double(), want_S, rtol=1e-5, atol=1e-5)
    if lds > N:
        assert torch.isnan(S[:, N:]).all()


def test_bias_sums_rejects_bad_arguments_in_simulator(emu):
    from gnf_b200.ops import ptr, stream_ptr
    t = torch.zeros(64)
    lib = G._lib.lib()
    assert lib.gnf_dag_l1_bias_sums(ptr(t), 4, ptr(t), ptr(t), 4, 2, 3, 4, 2, stream_ptr()) != 0      # period neither 1 nor d
    assert lib.gnf_dag_l1_bias_sums(ptr(t), 3, ptr(t), ptr(t), 4, 2, 3, 4, 1, stream_ptr()) != 0      # ldd < N


@pytest.mark.parametrize("cond", ["DAG", "Coupling", "Autoregressive"])
def test_conditional_flows_in_simulator(emu, cond):
    """Two-step conditional flows of every conditioner against the oracle (the DAG one with the monotonic normalizer)."""
    torch.set_num_threads(1)
    if cond == "Autoregressive":
        spec = CO.spec_of(cond, d=3, c=3, hidden=(12,), out=4, nb_flow=2)      # ConditionnalMADE: out * d divisible by d + c
    else:
        spec = CO.spec_of(cond, d=4, c=2, hidden=(16,), out=3 if cond == "DAG" else 2, nb_flow=2,
                          norm="monotonic" if cond == "DAG" else "affine")
    rep = CO.compare(spec, 5, "cpu", seed=7)
    CO.assert_report(rep, 1e-4, 1e-3)


def test_conditional_errors_in_simulator(emu):
    torch.set_num_threads(1)
    for cond in ("DAG", "Coupling"):
        model = G.build_from_spec(CO.spec_of(cond, d=4, c=3), "cpu", seed=0)
        x = torch.randn(2, 4)
        with pytest.raises(ValueError):
            model(x)
        with pytest.raises(ValueError):
            model(x, torch.randn(2, 2))
        with pytest.raises(ValueError):
            model(x, torch.randn(3, 3))
        with pytest.raises(TypeError):
            model(x, torch.randn(3, 2).t())              # [2, 3], not contiguous
        with pytest.raises(TypeError):
            model(x, torch.randn(2, 3, dtype=torch.float64))
