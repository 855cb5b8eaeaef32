"""GPU parity tests added in round 2 (VERDICT r1 'parity gaps'):
  * the benchmark's evaluation mode AS A COMBINATION (TF32 UMNN forward + single-pass TF32 conditioner GEMMs + stochastic
    gate + S = 40 + GraphedEvalStep) against the CPU oracle, per-sample log-likelihood within north_star's TF32 bar 2e-3;
  * the large configs against the oracle at non-toy batches (cfg5 B = 16, cfg3 B = 512);
  * the fused strict UMNN forward (gnf_umnn_fwd_tc3) against the layer-wise engine and the oracle;
  * Monotonic invert(forward(x)) to the bisection resolution 40 / 2^20 = 3.8e-5 (MonotonicNormalizer.py:69-83);
  * DAG dual-ascent control (step / update_dual_param / post_process / constrainA(thr > 0)) replayed against the
    reference's recorded state trajectories (tests/golden/dag_control.npz).
"""
import os
import sys

import pytest
import torch

import gnf_b200 as G
import parity
from helpers import rel_err

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import gnf_oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture
def engine_reset():
    yield
    G.ops.UMNN_ENGINE = "auto"
    G.ops.UMNN_FWD_FUSED_TC3 = True
    G.ops.set_gemm_mode("ffma")


# ---------------------------------------------------------------------------------------------------------------------
# bench.py's eval headline mode, exactly, against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg,B", [("cfg2", 2500), ("cfg3", 256), ("cfg4", 100)])
def test_bench_eval_mode_vs_oracle(engine_reset, cfg, B):
    """precision='tf32' + set_gemm_mode('auto-fast') + stochastic gate (in-kernel Philox, dumped and replayed into the
    oracle) + S = 40 + GraphedEvalStep: what `bench.py` reports as log-lik eval samples/s.  Tolerance: 2e-3 relative per
    sample (north_star's bar for TF32 tensor cores with fp32 accumulation)."""
    import model_vs_oracle as M
    spec = M.CONFIGS[cfg]
    S = 40
    model = M.build(spec, "cuda")
    G.ops.set_gemm_mode("auto-fast")
    for n in model.getNormalizers():
        n.nb_steps = S
        n.precision = "tf32"
    x = torch.randn(B, spec["d"], generator=torch.Generator().manual_seed(5)).cuda()
    try:
        step = G.GraphedEvalStep(model, x, warmup=2)
    except RuntimeError as err:
        # bench.py's own fallback (cfg3: a 200-wide integrand does not fit the single-pass TF32 UMNN kernel): strict UMNN forward,
        # still with the single-pass TF32 conditioner GEMMs
        assert "umnn tc" in str(err)
        for n in model.getNormalizers():
            n.precision = "strict"
        step = G.GraphedEvalStep(model, x, warmup=2)
    ll, z = step(x)
    ll, z = ll.clone(), z.clone()
    noises = None
    if spec["cond"] == "DAG":
        # the gate noise of the LAST replay: the captured step bumped the device counter before the forward
        noises = [tuple(n.cpu() for n in G.ops.dag_dump_noise(c._last_gate, B, spec["d"], x.device)) for c in model.getConditioners()]
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    ospec = {k: v for k, v in spec.items() if k != "A_prior"}
    with torch.no_grad():
        ll_o, z_o = O.compute_ll(x.cpu(), sd, ospec, None, noises, S)
    rel = rel_err(ll.cpu(), ll_o)
    assert rel < 2e-3, f"{cfg}: per-sample ll relative error {rel} (TF32 bar 2e-3)"
    assert float((z.cpu() - z_o).abs().max()) < 2e-2


# ---------------------------------------------------------------------------------------------------------------------
# large configs against the oracle at non-toy batches
# ---------------------------------------------------------------------------------------------------------------------
def _strict_check(rep):
    bad = {k: v for k, v in rep.items() if (k.startswith("grad.") and not v < 1e-3) or (k in ("ll", "loss") and not v < 1e-4)}
    assert not bad, f"out of tolerance: {bad}\n{rep}"


def test_cfg5_vs_oracle_batch16(engine_reset):
    """MNIST shape (d = 784, DAG 1568 -> 1024^3 -> 2, Affine), B = 16: the oracle materialises 16 x 784 x 1568 (79 MB) rows."""
    import model_vs_oracle as M
    G.ops.set_gemm_mode("auto")
    _strict_check(M.compare(M.CONFIGS["cfg5"], 16, "cuda", train=True))


def test_cfg3_vs_oracle_batch512(engine_reset):
    """HEPMASS shape (d = 21, MADE 210^3, UMNN 200^3), B = 512: 11 k rows, 237 k node-rows through the layer-wise engine."""
    import model_vs_oracle as M
    G.ops.set_gemm_mode("auto")
    _strict_check(M.compare(M.CONFIGS["cfg3"], 512, "cuda", train=True))


def test_bench_eval_mode_cfg5_vs_oracle(engine_reset):
    """cfg5 (d = 784, Affine) in bench.py's eval mode: with a tensor-core GEMM mode layer 1 of the DAG conditioner runs as a
    single-pass TF32 GEMM against the masked-embedding plane too (gnf_dag_embed_fwd); ll within the TF32 bar at B = 16."""
    import model_vs_oracle as M
    spec = M.CONFIGS["cfg5"]
    B = 16
    model = M.build(spec, "cuda")
    G.ops.set_gemm_mode("auto-fast")
    x = torch.randn(B, spec["d"], generator=torch.Generator().manual_seed(5)).cuda()
    step = G.GraphedEvalStep(model, x, warmup=2)
    ll, z = step(x)
    ll, z = ll.clone(), z.clone()
    noises = [tuple(n.cpu() for n in G.ops.dag_dump_noise(c._last_gate, B, spec["d"], x.device)) for c in model.getConditioners()]
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    ospec = {k: v for k, v in spec.items() if k != "A_prior"}
    with torch.no_grad():
        ll_o, z_o = O.compute_ll(x.cpu(), sd, ospec, None, noises, 20)
    rel = rel_err(ll.cpu(), ll_o)
    assert rel < 2e-3, f"cfg5: per-sample ll relative error {rel} (TF32 bar 2e-3)"


@pytest.mark.parametrize("mode,imp", [("GATE_GUMBEL", "IMP_SOFT"), ("GATE_TABLE", "IMP_HARD_SOFT"), ("GATE_NOISER", "IMP_SOFT")])
@pytest.mark.parametrize("B,d,N1,hot", [(40, 96, 160, True), (7, 130, 136, False)])
@pytest.mark.parametrize("layers,keep", [(1, True), (1, False), (2, True)])
def test_dag_layer1_embedding_plane_matches_the_loader_kernels(engine_reset, mode, imp, B, d, N1, hot, layers, keep):
    """Wide-flow layer 1 (d > 64) on the tensor-core engine: embedding plane + 3xTF32 GEMMs + cotangent reduction
    (gnf_dag_embed_fwd / gnf_dag_embed_bwd) against the FFMA kernels that generate the gate in their operand loaders --
    same Philox counters, so the two paths see the same gates: h, dx, dA and every weight gradient agree to fp32 accuracy
    (1e-5) when layer 1 is the whole net.  With a ReLU and a second layer behind it the two summation orders may put a
    pre-activation that is zero to 1e-7 on different sides, which moves one row of dx by one unit's share: 5e-3 there."""
    torch.manual_seed(d + B)
    dev = "cuda"
    gate = G.ops.GateSpec(getattr(G._lib, mode), getattr(G._lib, imp), 0.05, .5, seed=77, offset=11)
    x0 = torch.randn(B, d, device=dev)
    A0 = torch.rand(d, d, device=dev) * 1.5
    W = [torch.randn(N1, 2 * d if hot else d, device=dev) / d ** .5, torch.randn(24, N1, device=dev) / N1 ** .5][:layers]
    b = [torch.randn(N1, device=dev) * .1, torch.randn(24, device=dev) * .1][:layers]
    gh = torch.randn(B, d, 24 if layers == 2 else N1, device=dev)
    outs = {}
    G.ops.set_gemm_mode("tf32x3")
    for plane in (True, False):
        G.ops.DAG_L1_PLANE = plane
        G.ops.DAG_L1_PLANE_KEEP_DERIVATIVES = keep     # the backward reduction streams the kept de/dx, de/dP planes / regenerates the gates
        try:
            x, A = x0.clone().requires_grad_(), A0.clone().requires_grad_()
            params = [t.clone().requires_grad_() for pair in zip(W, b) for t in pair]
            G.ops.enable_kernel_timing(True)
            h = G.ops.DagMlpFn.apply(x, A, gate, hot, *params)
            h.backward(gh)
            called = set(G.ops.collect_kernel_timing())
            G.ops.enable_kernel_timing(False)
        finally:
            G.ops.DAG_L1_PLANE = True
            G.ops.DAG_L1_PLANE_KEEP_DERIVATIVES = True
        assert ("gnf_dag_embed_fwd" in called) == plane and ("gnf_dag_embed_bwd" in called) == plane
        outs[plane] = [h.detach(), x.grad, A.grad] + [p.grad for p in params]
    for name, a, r in zip(["h", "dx", "dA", "dW1", "db1", "dW2", "db2"], outs[True], outs[False]):
        assert torch.isfinite(a).all()
        err = float((a.double() - r.double()).norm() / r.double().norm().clamp_min(1e-30))
        assert err < (1e-5 if layers == 1 or name == "h" else 5e-3), f"{name}: relative L2 {err}"


# ---------------------------------------------------------------------------------------------------------------------
# fused strict UMNN forward
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,d,S,widths,E", [(100, 63, 20, [150, 150, 150], 30), (37, 6, 29, [100, 100, 100], 30),
                                            (64, 21, 40, [64, 96], 12), (5, 3, 7, [160, 33, 150], 5), (300, 2, 1, [32, 32], 1),
                                            (40, 9, 12, [130, 140, 150, 160], 7)])
@pytest.mark.parametrize("train", [False, True])
def test_umnn_fused_tc3_forward_vs_float64(engine_reset, B, d, S, widths, E, train):
    """gnf_umnn_fwd_tc3 (3xTF32, TMEM-resident chain, streamed weights) through MonotonicNormalizer: z and jac against the
    quadrature evaluated in float64 (1e-6 relative L2), and -- in training -- gradients against the layer-wise forward's."""
    torch.manual_seed(B + d)
    norm = G.MonotonicNormalizer(widths, E, nb_steps=S, solver="CC").to("cuda")
    x, h = torch.randn(B, d, device="cuda"), torch.randn(B, d, E, device="cuda")
    G.ops.UMNN_ENGINE = "layerwise"
    G.ops.set_gemm_mode("tf32x3")
    sd64 = {"n." + k: v.detach().double() for k, v in norm.state_dict().items()}
    z64, j64 = O.monotonic_normalizer(x.double(), h.double(), sd64, "n.integrand_net.net", len(widths) + 1, S)
    outs = {}
    for fused in (True, False):
        G.ops.UMNN_FWD_FUSED_TC3 = fused
        G.ops.enable_kernel_timing(True)
        xg, hg = x.clone().requires_grad_(train), h.clone().requires_grad_(train)
        norm.zero_grad()
        with torch.enable_grad() if train else torch.no_grad():
            z, jac = norm(xg, hg)
            if train:
                ((z * z).sum() + torch.log(jac).sum()).backward()
        used = set(G.ops.collect_kernel_timing())
        G.ops.enable_kernel_timing(False)
        assert ("gnf_umnn_fwd_tc3" in used) == fused, used
        outs[fused] = (z.detach(), jac.detach(), {k: p.grad.clone() for k, p in norm.named_parameters()} if train else {},
                       xg.grad, hg.grad)
    for fused in outs:
        z, jac = outs[fused][:2]
        assert float((z.double() - z64).norm() / z64.norm()) < 1e-6
        assert float((jac.double() - j64).norm() / j64.norm()) < 1e-6
    if train:
        for k, g in outs[True][2].items():
            ref = outs[False][2][k]
            assert float((g - ref).norm() / ref.norm().clamp_min(1e-20)) < 2e-4, k
        assert float((outs[True][3] - outs[False][3]).norm() / outs[False][3].norm()) < 1e-5
        assert float((outs[True][4] - outs[False][4]).norm() / outs[False][4].norm()) < 1e-5


def test_umnn_fused_tc3_unsupported_shapes_are_loud():
    """Hidden width > 160 or fewer than 3 linear layers: GNF_ERR_UNSUPPORTED from the C-ABI, never a silent fallback inside it."""
    import ctypes as C
    for widths in ([200, 200, 200], [64]):
        norm = G.MonotonicNormalizer(widths, 4, nb_steps=8).to("cuda")
        ps = list(norm.integrand_net.parameters())
        net = G.ops._mlp_struct(ps[0::2], ps[1::2])
        assert G._lib.lib().gnf_umnn_tc3_workspace_bytes(C.byref(net), 10) == 0
        assert b"tc3" in G._lib.lib().gnf_last_error()


# ---------------------------------------------------------------------------------------------------------------------
# sampling path
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cond", ["DAG", "Autoregressive", "Coupling"])
def test_monotonic_invert_of_forward(cond):
    """1-step Monotonic flow: invert(forward(x)) == x to the bisection resolution of MonotonicNormalizer.inverse_transform
    (20 halvings of [-20, 20]: 40 / 2^20 = 3.8e-5), through NormalizingFlowStep.invert's depth + 1 fixed-point passes."""
    d = 5
    spec = dict(nb_flow=1, d=d, cond=cond, hidden=[40, 40], out=8, hot_encoding=True, gumble_T=.5, l1=0., norm="monotonic",
                int_net=[50, 50, 50], nb_steps=30, solver="CC")
    model = G.build_from_spec(spec, "cuda", seed=3)
    if cond == "DAG":
        # a binary strictly-triangular adjacency = the state after a successful post_process (deterministic gate, invertible)
        c = model.getConditioners()[0]
        with torch.no_grad():
            c.A.copy_(torch.tril(torch.ones(d, d), -1))
        c.stoch_gate, c.noise_gate, c.s_thresh, c.h_thresh, c.is_invertible = False, False, False, 0., True
    x = torch.randn(64, d, device="cuda") * 1.5
    with torch.no_grad():
        z, _ = model(x)
        x_rec = model.invert(z)
    err = float((x_rec - x).abs().max())
    assert err < 2 * 3.8e-5 + 1e-5, err


@pytest.mark.parametrize("B,d,S,widths,E", [(100, 63, 20, [150, 150, 150], 30), (33, 5, 30, [50, 50, 50], 8), (7, 3, 63, [16], 1),
                                            (50, 4, 9, [200, 100], 12)])
def test_fused_bisection_inverse_matches_the_reference_loop(B, d, S, widths, E):
    """gnf_umnn_invert (all 20 forward passes of MonotonicNormalizer.inverse_transform in one launch) against
    (a) the reference's own loop of 20 forward passes on the same CUDA forward kernel: same interval decisions, so the same x
        except where a z_middle lands within rounding of z (the two evaluate the quadrature in different tile layouts):
        then they differ by at most the last interval, 40 / 2^20;
    (b) the oracle's float64 integral: forward(x_found) reproduces z to the slope times the bisection resolution."""
    torch.manual_seed(S + d)
    norm = G.MonotonicNormalizer(widths, E, nb_steps=S, solver="CC").to("cuda")
    h = torch.randn(B, d, E, device="cuda") * .7
    x_true = torch.randn(B, d, device="cuda") * 3
    G.ops.set_gemm_mode("ffma")
    with torch.no_grad():
        z, jac = norm(x_true, h)
        G.ops.enable_kernel_timing(True)
        norm.fused_inverse = True
        x_fused = norm.inverse_transform(z, h)
        assert "gnf_umnn_invert" in G.ops.collect_kernel_timing()
        G.ops.enable_kernel_timing(False)
        norm.fused_inverse = False
        x_loop = norm.inverse_transform(z, h)
    res = 40. / 2 ** 20
    assert float((x_fused - x_loop).abs().max()) <= res * 1.01
    assert float((x_fused == x_loop).float().mean()) > .98
    assert float((x_fused - x_true).abs().max()) < 2 * res
    sd64 = {"n." + k: v.detach().double().cpu() for k, v in norm.state_dict().items()}
    z64, _ = O.monotonic_normalizer(x_fused.double().cpu(), h.double().cpu(), sd64, "n.integrand_net.net", len(widths) + 1, S)
    assert float(((z64 - z.double().cpu()).abs() / jac.double().cpu().clamp_min(1e-3)).max()) < 2 * res


# ---------------------------------------------------------------------------------------------------------------------
# DAG dual-ascent control against the reference's recorded trajectories
# ---------------------------------------------------------------------------------------------------------------------
def _control_state(c):
    return dict(lambd=float(c.lambd), c=float(c.c), dag_const=float(c.dag_const), l1_weight=float(c.l1_weight),
                exponent=int(c.exponent), prev_trace=float(c.prev_trace), alpha=float(c.alpha), no_update=int(c.no_update),
                stoch_gate=bool(c.stoch_gate), noise_gate=bool(c.noise_gate), s_thresh=bool(c.s_thresh), h_thresh=float(c.h_thresh),
                is_invertible=bool(c.is_invertible), requires_grad=bool(c.A.requires_grad))


def test_dag_control_trajectories_match_the_reference():
    """tests/golden/dag_control.npz: the reference's DAGConditioner driven through scripted sequences of step(epoch, loss_avg),
    update_dual_param(), post_process(), constrainA(thr) and direct edits of A; after every call its scalar state and A were
    recorded.  The product conditioner replays the same script on the GPU (power trace through the K2 kernel)."""
    import json
    import numpy as np
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dag_control.npz")
    data = np.load(path, allow_pickle=False)
    scripts = json.loads(str(data["scripts"]))
    for si, script in enumerate(scripts):
        d = script["d"]
        c = G.DAGConditioner(d, [8], 2, l1=script["l1"], nb_epoch_update=script["nb_epoch_update"], hot_encoding=True).to("cuda")
        with torch.no_grad():
            c.A.copy_(torch.from_numpy(data[f"s{si}_A0"]).cuda())
        c.prev_trace.copy_(torch.tensor(float(data[f"s{si}_prev_trace0"])))
        for k, (op, args) in enumerate(script["ops"]):
            if op == "step":
                c.step(args[0], torch.tensor(args[1]))
            elif op == "update_dual_param":
                c.update_dual_param()
            elif op == "post_process":
                c.post_process(*args)
            elif op == "constrainA":
                with torch.no_grad():
                    c.constrainA(*args)
            elif op == "setA":
                with torch.no_grad():
                    c.A.data.copy_(torch.from_numpy(data[f"s{si}_setA{k}"]).cuda())
            elif op == "set":
                setattr(c, args[0], args[1])
            elif op == "setdual":
                getattr(c, args[0]).fill_(args[1])
            elif op == "depth":
                assert c.depth() == script["states"][k]["depth"], (si, k)
            st, ref = _control_state(c), script["states"][k]
            for key, v in st.items():
                r = ref[key]
                if isinstance(v, float):
                    assert abs(v - r) <= 2e-5 * max(1., abs(r)) or (v != v and r != r), (si, k, op, key, v, r)
                else:
                    assert v == r, (si, k, op, key, v, r)
            A_ref = torch.from_numpy(data[f"s{si}_A{k + 1}"])
            assert float((c.A.detach().cpu() - A_ref).abs().max()) < 1e-6, (si, k, op)


# ---------------------------------------------------------------------------------------------------------------------
# optimizer
# ---------------------------------------------------------------------------------------------------------------------
def test_fused_adam_matches_torch_adam():
    """G.FusedAdam (one multi-tensor launch, device step counter) against torch.optim.Adam, the reference drivers' optimizer
    (UCIExperiments.py:100): same parameters after 5 steps with L2 weight decay, odd sizes, one tensor without gradient."""
    torch.manual_seed(0)
    shapes = [(630, 126), (630,), (7, 3), (1,), (150, 150), (4097,), (33, 5)]
    pa = [torch.randn(s, device="cuda").requires_grad_(True) for s in shapes]
    pb = [p.detach().clone().requires_grad_(True) for p in pa]
    oa = G.FusedAdam(pa, lr=1e-3, weight_decay=1e-4)
    ob = torch.optim.Adam(pb, lr=1e-3, weight_decay=1e-4)
    for it in range(5):
        for k, (a, b) in enumerate(zip(pa, pb)):
            if k == 3 and it < 2:
                a.grad = b.grad = None
                continue
            g = torch.randn_like(a) * (10. ** (k - 3))
            a.grad, b.grad = g.clone(), g.clone()
        oa.step()
        ob.step()
    for k, (a, b) in enumerate(zip(pa, pb)):
        if k == 3:
            continue            # its step count differs from the other tensors' (torch keeps one count per tensor, FusedAdam one per group)
        assert float((a - b).abs().max()) <= 1e-6 * float(b.abs().max()) + 1e-7, (k, float((a - b).abs().max()))


@pytest.mark.parametrize("M,N,K,period,relu", [(6300, 30, 630, 1, 0), (2048, 32, 1024, 1, 1), (4100, 2, 77, 1, 0), (6300, 30, 630, 63, 1)])
def test_skinny_forward_layer(M, N, K, period, relu):
    """gnf_linear_fwd on tall-and-skinny shapes (N <= 32: the conditioner's output layer, DAGConditioner.py:7-20), with a
    periodic bias table, against float64.  (A dedicated shuffle-broadcast kernel for this shape measured 43 us against the
    generic 32x32x64 tile's 35 us on B200 -- profiles/r02g_launches_cfg4_train_eager.csv -- and was dropped.)"""
    G.ops.set_gemm_mode("ffma")
    torch.manual_seed(M + N)
    X = torch.randn(M, K, device="cuda")
    W = torch.randn(N, K, device="cuda") / K ** .5
    b = torch.randn(period, N, device="cuda").contiguous()
    Y = G.ops.linear_fwd(X, W, b, relu, bias_period=period)
    ref = X.double() @ W.double().t() + b.double().repeat(M // period, 1)
    if relu:
        ref = ref.clamp_min(0)
    assert float((Y.double() - ref).abs().max()) < 2e-5


# ---------------------------------------------------------------------------------------------------------------------
# experiment plumbing: the reference driver's loop on the CUDA path
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("use_graph", [True, False])
def test_uci_training_loop_runs_and_checkpoints(tmp_path, engine_reset, use_graph):
    """G.experiments.train_uci = the loop of UCIExperiments.py:117-220 (constrainA, random S, Adam, model.step, validation at S + 20,
    checkpoints): three epochs on a standardised synthetic mixture; the loss must fall, the checkpoints must load back --
    also with the `module.` prefix of a DataParallel checkpoint."""
    import numpy as np
    rng = np.random.RandomState(0)
    mk = lambda n: (rng.randn(n, 4) * np.array([1., .3, 2., .7]) + np.array([0., 1., -1., 2.])).astype(np.float32)
    trn, val, tst = mk(2048), mk(512), mk(512)
    cfg = dict(G.experiments.DRIVER_DEFAULTS, conditioner="DAG", normalizer="monotonic", emb_net=[32, 32, 8], int_net=[40, 40, 40],
               b_size=256, nb_steps=10, nb_steps_dual=2, l1=.1, learning_rate=5e-3)
    G.ops.set_gemm_mode("auto")
    model, hist = G.experiments.train_uci(trn, val, tst, cfg, path=str(tmp_path), nb_epoch=3, use_graph=use_graph, log=lambda s: None, seed=0)
    assert len(hist) == 3 and all(np.isfinite(h["train_loss"]) and np.isfinite(h["valid_ll"]) for h in hist)
    assert hist[-1]["train_loss"] < hist[0]["train_loss"]
    for f in ("model.pt", "ADAM.pt", "model_2.pt"):
        assert (tmp_path / f).is_file()
    sd = torch.load(str(tmp_path / "model.pt"), map_location="cpu")
    fresh = G.experiments.build_uci_flow(4, cfg).to("cuda")
    G.load_checkpoint(fresh, {"module." + k: v for k, v in sd.items()})
    fresh.getNormalizers()[0].nb_steps = model.getNormalizers()[0].nb_steps
    for c_new, c_old in zip(fresh.getConditioners(), model.getConditioners()):
        c_new.stoch_gate = c_old.stoch_gate = False
        c_new.exponent = c_old.exponent
    x = torch.from_numpy(val[:64]).cuda()
    with torch.no_grad():
        assert torch.allclose(fresh.compute_ll(x)[0], model.compute_ll(x)[0], atol=1e-5)


# ---------------------------------------------------------------------------------------------------------------------
# image flows: DAGConditioner(hidden=<nn.Module>), CNN embedding nets, multi-scale CNNormalizingFlow (SURVEY 8f rank 3)
# ---------------------------------------------------------------------------------------------------------------------
def _build_image_flow():
    outer = []
    for img, fc, ntype in (([1, 14, 14], [400, 64], "affine"), ([1, 7, 7], [16, 16], "monotonic")):
        d = img[1] * img[2]
        emb = 2 if ntype == "affine" else 6
        cond = G.DAGConditioner(d, G.MNISTCNN(fc_l=fc, size_img=img, out_d=emb), emb, l1=.3, nb_epoch_update=10, hot_encoding=False,
                                A_prior=G.MNIST_A_prior(img[1], 2))
        norm = G.AffineNormalizer() if ntype == "affine" else G.MonotonicNormalizer(integrand_net=[20, 20], cond_size=emb, nb_steps=12, solver="CC")
        flow = G.FCNormalizingFlow([G.NormalizingFlowStep(cond, norm)], None)
        flow.img_sizes = img
        outer.append(flow)
    return G.CNNormalizingFlow(outer, G.NormalLogDensity(), [[1, 2, 2], [1, 1, 1]])


def test_image_cnn_flow_matches_the_reference():
    """tests/golden/image_cnn_flow.npz (reference run, make_image_golden.py): a two-scale CNNormalizingFlow of
    DAGConditioner(hidden=MNISTCNN) steps.  The reference's state_dict loads strictly; z, log-det, loss and every gradient agree."""
    import numpy as np
    f = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "image_cnn_flow.npz"))
    model = _build_image_flow().to("cuda")
    sd = {k[3:]: torch.from_numpy(f[k]).cuda() for k in f.files if k.startswith("sd.")}
    res = model.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    for c in model.getConditioners():
        c.stoch_gate = False
    G.ops.set_gemm_mode("ffma")
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False          # the CNN body is the user's module on cuDNN: keep its convolutions in fp32 here
    try:
        x = torch.from_numpy(f["x"]).cuda()
        z, jac = model(x)
        loss = model.loss(z, jac)
        loss.backward()
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    assert float((z.detach().cpu() - torch.from_numpy(f["z"])).abs().max()) < 5e-5
    assert float((jac.detach().cpu() - torch.from_numpy(f["logdet"])).abs().max()) < 1e-4
    assert abs(float(loss) - float(f["loss"])) < 1e-4 * abs(float(f["loss"]))
    for k, p in model.named_parameters():
        if "grad." + k in f.files:
            g = torch.from_numpy(f["grad." + k])
            assert p.grad is not None, k
            assert float((p.grad.cpu() - g).norm() / g.norm().clamp_min(1e-12)) < 1e-3, k
    # sampling through the multi-scale structure: invert(forward(x)) on a flow whose conditioners are exact DAGs
    for c in model.getConditioners():
        with torch.no_grad():
            c.A.copy_(torch.tril((c.A.detach() != 0).float(), -1))
        c.s_thresh, c.h_thresh, c.is_invertible = False, 0., True
    with torch.no_grad():
        z2, _ = model(x)
        x_rec = model.invert(z2)
    assert float((x_rec - x).abs().max()) < 2e-4


def test_mnist_and_cifar_factories_build_the_reference_structure():
    m = G.buildMNISTNormalizingFlow([1, 1, 1], G.AffineNormalizer, {}, prior_kernel=2)
    assert isinstance(m, G.CNNormalizingFlow) and [s.img_sizes for s in m.steps] == [[1, 28, 28], [1, 14, 14], [1, 7, 7]]
    assert m.steps[0].steps[0].conditioner.embedding_net.fc1.in_features == 2304
    assert G.buildMNISTNormalizingFlow([1, 1], G.AffineNormalizer, {}) is None
    c = G.buildCIFAR10NormalizingFlow([1], G.AffineNormalizer, {})
    assert isinstance(c, G.FCNormalizingFlow) and c.steps[0].conditioner.in_size == 3072


@pytest.mark.parametrize("B,d,with_constraint", [(1, 1, False), (100, 63, True), (6400, 784, True), (100000, 6, False)])
def test_fused_training_loss_vs_float64(B, d, with_constraint):
    """gnf_nll_loss_{fwd,bwd}: constraintsLoss() - mean(jac + log N(z)) (NormalizingFlow.py:144-146) as one kernel per direction,
    against float64 torch, repeatedly through the same work buffer (self-resetting block counter)."""
    from test_emu_kernels import _nll_loss_case
    for _ in range(3):
        _nll_loss_case("cuda", B, d, with_constraint)


@pytest.mark.parametrize("M_,N,K", [(6300, 632, 632), (2100, 300, 260), (5000, 1024, 520), (3000, 30, 630), (100, 64, 64)])
def test_weight_and_bias_gradient_in_one_launch(M_, N, K):
    """gnf_linear_wgrad_bias_tc: the weight-gradient engine sums the dY columns it streams (db); shapes it does not take fall back
    to the column-sum kernel inside the call.  Against float64."""
    g = torch.Generator().manual_seed(M_ + N)
    dY = _rows_pad(torch.randn(M_, N, generator=g).cuda())
    X = _rows_pad(torch.randn(M_, K, generator=g).cuda())
    G.ops.set_gemm_mode("tf32x3")
    try:
        for _ in range(2):
            dW, db = G.ops.linear_wgrad_bias(dY, dY.stride(0), X, X.stride(0), M_, N, K)
    finally:
        G.ops.set_gemm_mode("ffma")
    dY64, X64 = dY[:, :N].double(), X[:, :K].double()
    assert float((dW.double() - dY64.t() @ X64).norm() / (dY64.t() @ X64).norm()) < 2e-6
    want = dY64.sum(0)
    assert float((db.double() - want).abs().max()) < 1e-5 * float(dY64.abs().sum(0).max())


def _rows_pad(t):
    """[M, N] view of a buffer whose rows are padded to a multiple of 4 floats (what the engine's TMA maps need)."""
    M_, N = t.shape
    buf = torch.zeros(M_, (N + 3) // 4 * 4, device=t.device, dtype=t.dtype)
    buf[:, :N] = t
    return buf


@pytest.mark.parametrize("B,d", [(1, 1), (100, 63), (101, 64), (1000, 21)])
def test_narrow_layer1_plane_reduction(B, d):
    from test_emu_kernels import _narrow_reduce_case
    _narrow_reduce_case("cuda", B, d)


def test_narrow_layer1_backward_on_tensor_cores_matches_resident_kernels():
    """cfg4-shaped DAG conditioner, stochastic gate: the backward through the saved gate planes on the tensor-core engine
    (gnf_linear_wgrad_tc / gnf_linear_dgrad_tc_ps + gnf_dag_l1_reduce_saved) against the FFMA kernels that regenerate every gate."""
    torch.manual_seed(3)
    cond = G.DAGConditioner(63, [630, 630], 30, gumble_T=.5, hot_encoding=True, l1=0.).cuda()
    x = torch.randn(100, 63, device="cuda", requires_grad=True)
    w = torch.randn(100, 63, 30, device="cuda")
    grads = {}
    from gnf_b200.conditioners import _stack_params
    gate = cond._gate_spec(x)            # one Philox (seed, offset) for the three variants
    G.ops.DAG_L1_NARROW_TC_FWD = False   # same forward kernel in all three: this test is about the backward (the forward: next test)
    for tag, keep, tc, mode in (("regen", False, False, "auto"), ("saved", True, False, "auto"), ("tc", True, True, "auto")):   # same forward in all three
        G.ops.DAG_L1_KEEP_GATES, G.ops.DAG_L1_NARROW_TC = keep, tc
        G.ops.set_gemm_mode(mode)
        try:
            cond.zero_grad()
            x.grad = None
            h = G.ops.DagMlpFn.apply(x, cond.A, gate, True, *_stack_params(cond.embedding_net.net))
            (h * w).sum().backward()
            grads[tag] = [x.grad.clone(), cond.A.grad.clone()] + [p.grad.clone() for p in cond.embedding_net.parameters()]
        finally:
            G.ops.DAG_L1_KEEP_GATES = G.ops.DAG_L1_NARROW_TC = True
            G.ops.set_gemm_mode("ffma")
    G.ops.DAG_L1_NARROW_TC_FWD = True
    for tag in ("saved", "tc"):
        for a, b in zip(grads["regen"], grads[tag]):
            assert float((a - b).norm() / b.norm()) < (2e-6 if tag == "saved" else 2e-5), tag


@pytest.mark.parametrize("M_,N,K,relu", [(6300, 30, 630, False), (1024, 32, 128, True), (5000, 1, 1000, False)])
def test_skinny_split_k_forward(M_, N, K, relu):
    from test_emu_kernels import _splitk_case
    _splitk_case("cuda", M_, N, K, relu)


def test_branched_schedule_matches_the_in_line_schedule():
    """The late round-2 schedule of the captured step -- penalty chain on a side branch, layer-1 backward as three branches on the
    tensor-core engine against the saved gate planes, skinny layer wgrad next to dgrad, weight splits next to layer 1 -- against the
    in-line schedule with every one of those switches off: same first-step loss and gradients (the gate noise is the same Philox
    stream: counters start equal), parameters after six Adam steps equal up to summation-order noise."""
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import model_vs_oracle as M
    spec = M.CONFIGS["cfg4"]
    g = torch.Generator(device="cuda").manual_seed(5)
    xs = [torch.randn(100, 63, device="cuda", generator=g) for _ in range(6)]
    G.ops.set_gemm_mode("auto")
    results = {}
    try:
        for tag, on in (("in-line", False), ("branched", True)):
            G.ops.PARALLEL_BRANCHES = G.ops.DAG_L1_KEEP_GATES = G.ops.DAG_L1_NARROW_TC = G.ops.SPLITK_SKINNY = on
            model = M.build(spec, "cuda", seed=11)
            for c in model.getConditioners():
                c._noise_seed = 1234                       # same Philox key in both runs
            bucket = G.dist.GradBucket(model.parameters())
            opt = G.FusedAdam(model.parameters(), lr=1e-4, weight_decay=1e-5)
            step = G.GraphedTrainStep(model, opt, bucket, xs[0], allreduce=False, warmup=1, side_branch=on)
            losses = [float(step(x)) for x in xs]
            results[tag] = (losses, [p.detach().clone() for p in model.parameters()])
    finally:
        G.ops.PARALLEL_BRANCHES = G.ops.DAG_L1_KEEP_GATES = G.ops.DAG_L1_NARROW_TC = G.ops.SPLITK_SKINNY = True
        G.ops.set_gemm_mode("ffma")
    (la, pa), (lb, pb) = results["in-line"], results["branched"]
    assert abs(la[0] - lb[0]) <= 1e-5 * abs(la[0]), (la[0], lb[0])
    for a, b in zip(la, lb):
        assert abs(a - b) <= 2e-3 * abs(a), (la, lb)
    for a, b in zip(pa, pb):
        assert float((a - b).norm() / a.norm().clamp_min(1e-12)) < 2e-3


def test_narrow_layer1_forward_on_tensor_cores_matches_resident_kernel():
    """Layer 1 of a cfg4-shaped DAG conditioner, stochastic gate, training: gate-planes kernel + engine-v2 GEMM with the padded bias
    table (gnf_dag_gate_planes, gnf_dag_bias_table_ld, gnf_linear_fwd_tc_ps_tb) against the resident-gate FFMA kernel, same Philox
    stream: the conditioner output within 3xTF32 rounding."""
    from gnf_b200.conditioners import _stack_params
    torch.manual_seed(4)
    cond = G.DAGConditioner(63, [630, 630], 30, gumble_T=.5, hot_encoding=True, l1=0.).cuda()
    x = torch.randn(100, 63, device="cuda", requires_grad=True)
    gate = cond._gate_spec(x)
    out = {}
    G.ops.set_gemm_mode("auto")
    try:
        for tag, on in (("ffma", False), ("tc", True)):
            G.ops.DAG_L1_NARROW_TC_FWD = on
            l0 = G.ops.launch_count()
            out[tag] = G.ops.DagMlpFn.apply(x, cond.A, gate, True, *_stack_params(cond.embedding_net.net)).detach().clone()
    finally:
        G.ops.DAG_L1_NARROW_TC_FWD = True
        G.ops.set_gemm_mode("ffma")
    err = float((out["tc"] - out["ffma"]).abs().max() / out["ffma"].abs().max())
    assert err < 2e-5, err
