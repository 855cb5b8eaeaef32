"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/gnf.h declares,
argument contracts, state_dict compatibility with the reference's key names, and the data-parallel plumbing
(world_size 2, gloo) — kernels executed by the host SIMT simulator where arithmetic is needed."""
import os
import re
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import gnf_b200 as G
from helpers import load_golden, golden_names

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "gnf.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gnf_[A-Za-z0-9_]+)\s*\(", src)))


def test_product_library_has_no_measurement_knobs():
    """The process-global switches (traces, ablation bits, tiling / engine overrides) live in the -DGNF_DEVTOOLS build only
    (include/gnf_devtools.h): the product library neither declares nor exports them."""
    import __graft_entry__
    __graft_entry__.build()
    lib = G._lib.load_library()
    src = open(os.path.join(ROOT, "include", "gnf_devtools.h")).read()
    knobs = sorted(set(re.findall(r"\b(gnf_[A-Za-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", src, flags=re.S))))
    assert len(knobs) >= 10
    for name in knobs:
        assert not hasattr(lib, name), f"{name} is exported by the product library"
        assert name not in G._lib.EXPORTED_SYMBOLS


def test_library_exports_every_declared_symbol():
    import __graft_entry__
    __graft_entry__.build()
    lib = G._lib.load_library()          # dlopen + bind; no compute call, no GPU needed
    declared = _header_symbols()
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/gnf.h but not exported"
    assert set(declared) == set(G._lib.EXPORTED_SYMBOLS), set(declared) ^ set(G._lib.EXPORTED_SYMBOLS)
    assert lib.gnf_version() >= 100 and lib.gnf_has_device_code() == 1


def test_missing_library_is_a_loud_error(tmp_path):
    with pytest.raises(RuntimeError, match="no CPU"):
        G._lib.load_library(str(tmp_path / "libgnf_sm100.so"))


def test_cpu_tensors_are_rejected_by_the_product_path():
    assert not G._lib._SIMULATOR
    with pytest.raises(TypeError, match="CUDA"):
        G.AffineNormalizer()(torch.randn(2, 3), torch.randn(2, 3, 2))
    model = G.build_from_spec(G.CONFIGS["cfg2"])
    with pytest.raises(TypeError, match="CUDA"):
        model(torch.randn(4, 6))


@pytest.mark.parametrize("name", golden_names())
def test_state_dict_keys_match_the_reference(name):
    c = load_golden(name)
    model = G.build_from_spec(c["spec"])
    ours = model.state_dict()
    assert set(ours) == set(c["sd"]), set(ours) ^ set(c["sd"])
    for k, v in c["sd"].items():
        assert tuple(ours[k].shape) == tuple(v.shape), k
    model.load_state_dict(c["sd"], strict=True)


def test_reference_attribute_surface():
    m = G.build_from_spec(G.CONFIGS["cfg2"])
    c, n = m.getConditioners()[0], m.getNormalizers()[0]
    for attr in ("stoch_gate", "noise_gate", "s_thresh", "h_thresh", "gumble_T", "exponent", "A", "alpha", "is_invertible",
                 "nb_epoch_update", "no_update", "hot_encoding", "in_size"):
        assert hasattr(c, attr), attr
    assert c.exponent == 6 % 50 and c.stoch_gate and not c.noise_gate and c.s_thresh and not c.is_invertible
    assert n.nb_steps == 20 and n.solver == "CC"
    assert float(c.A.diag().abs().max()) == 0.                     # constrainA at construction
    assert not m.isInvertible()
    for meth in ("forward", "compute_ll", "loss", "constraintsLoss", "DAGness", "step", "invert", "getConditioners",
                 "getNormalizers", "isInvertible"):
        assert callable(getattr(m, meth))
    assert G.AutoregressiveConditioner(5, [8], 3).depth() == 4 and G.CouplingConditioner(5, [8], 3).depth() == 1


def test_made_masks_match_oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gnf_oracle as O
    c = G.AutoregressiveConditioner(7, [20, 13], 3)
    layers = [m for m in c.masked_autoregressive_net.net if isinstance(m, G.MaskedLinear)]
    for m, want in zip(layers, O.made_masks(7, [20, 13], 21)):
        assert torch.equal(m.mask, want)


def test_dag_graph_helpers():
    D = G.DAGConditioner
    chain = torch.tensor([[0, 0, 0], [1, 0, 0], [0, 1, 0]]).numpy() > 0
    assert D._is_dag(chain) and D._longest_path(chain) == 2
    cyc = torch.tensor([[0, 1], [1, 0]]).numpy() > 0
    assert not D._is_dag(cyc)


# ---------------- data-parallel plumbing, world_size 2 on gloo ----------------
def _dp_worker(rank, world, port, emu_path, ret):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    import sim_hook
    sim_hook.install(emu_path)
    spec = dict(nb_flow=1, d=4, cond="DAG", hidden=[8, 8], out=3, hot_encoding=True, gumble_T=.5, l1=.1, norm="monotonic",
                int_net=[6, 6], nb_steps=5, solver="CC")
    model = G.build_from_spec(spec, "cpu", seed=100 + rank)       # different init per rank on purpose
    G.dist.broadcast_parameters(model)
    for c in model.getConditioners():
        c.stoch_gate = False
    bucket = G.dist.GradBucket(model.parameters())
    x_full = torch.randn(6, 4, generator=torch.Generator().manual_seed(5))
    x = G.dist.shard_batch(x_full, rank, world).contiguous()
    bucket.zero()
    z, jac = model(x)
    model.loss(z, jac).backward()
    assert bucket.check_aliasing()
    bucket.allreduce_mean()
    flat_dp = bucket.flat.clone()
    # single-process reference: the full batch on this rank's (now identical) replica
    bucket.zero()
    z, jac = model(x_full)
    model.loss(z, jac).backward()
    err = float((flat_dp - bucket.flat).norm() / bucket.flat.norm())
    # the accumulation-free step protocol (what bench.py / GraphedTrainStep use) must give the same averaged gradients
    bucket.begin_step()
    z, jac = model(x)
    model.loss(z, jac).backward()
    assert not bucket.check_aliasing()            # autograd adopted the backward kernels' tensors
    bucket.finish_step()
    assert bucket.check_aliasing()                # p.grad points at the all-reduced slices again
    err = max(err, float((flat_dp - bucket.flat).norm() / flat_dp.norm()))
    sd = torch.cat([p.detach().flatten() for p in model.parameters()])
    gathered = [torch.zeros_like(sd) for _ in range(world)]
    dist.all_gather(gathered, sd)
    same = all(torch.equal(gathered[0], g) for g in gathered)
    ret[rank] = (err, same)
    dist.destroy_process_group()


def test_data_parallel_gradients_match_single_process():
    import build_emu
    emu_path = build_emu.build()
    world = 2
    port = 29500 + (os.getpid() % 2000)
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_dp_worker, args=(world, port, emu_path, ret), nprocs=world, join=True)
    for r in range(world):
        err, same = ret[r]
        assert same, "parameters differ across ranks after broadcast"
        assert err < 1e-5, f"rank {r}: sharded+averaged gradient differs from the full-batch gradient by {err}"


def test_shard_batch_covers_the_batch():
    x = torch.arange(12).view(12, 1)
    parts = [G.dist.shard_batch(x, r, 4) for r in range(4)]
    assert torch.equal(torch.cat(parts), x) and all(p.shape[0] == 3 for p in parts)
    # unequal / empty shards would bias the AVG all-reduce and poison it with the NaN mean of an empty shard: refused loudly
    with pytest.raises(ValueError):
        G.dist.shard_batch(torch.arange(10).view(10, 1), 0, 4)
    with pytest.raises(ValueError):
        G.dist.shard_batch(torch.arange(3).view(3, 1), 3, 4)


def test_tensor_core_gemm_plan_fills_the_last_round_of_work_items():
    """The persistent tcgen05 GEMM hands (tile x k-split) items round-robin to 148 CTAs: the planner must not leave a nearly
    empty last round (the first version ran cfg4's wgrad as 160 items = 2 rounds for 12 stragglers).  Host-only query."""
    import ctypes as C
    import __graft_entry__
    __graft_entry__.build()
    lib = G._lib.load_library()          # dlopen + bind; the query is host code, no GPU needed
    bn, sp = C.c_int(0), C.c_int(0)

    def plan(M, N, K, passes, wgrad):
        assert lib.gnf_tc_gemm_plan(M, N, K, passes, wgrad, C.byref(bn), C.byref(sp)) == 0
        tiles = -(-M // 128) * -(-N // bn.value)
        return bn.value, sp.value, tiles * sp.value

    # cfg4 conditioner hidden layer, 100 samples: forward / dgrad (no split), wgrad (split-K over the 6300 rows)
    b, s, items = plan(6300, 632, 632, 3, 0)
    assert s == 1 and b in (64, 96, 128, 160) and items <= 2 * 148 and items / (-(-items // 148) * 148) > 0.8, (b, s, items)
    b, s, items = plan(632, 632, 6300, 3, 1)
    assert b <= 160 and s >= 1 and items <= 148 and items >= 120, (b, s, items)
    # big batch: many rounds, the widest 3xTF32 tile wins; single pass may use up to 256 columns
    assert plan(64512, 632, 632, 3, 0)[0] == 160
    assert plan(78400, 1024, 1024, 1, 0)[0] == 256
    # every plan is a legal tile
    for (M, N, K, p, w) in [(100, 30, 630, 3, 0), (15000, 60, 60, 1, 0), (210, 210, 10000, 3, 1), (1, 1, 1, 1, 1)]:
        b, s, _ = plan(M, N, K, p, w)
        assert b % 32 == 0 and 64 <= b <= (160 if p == 3 else 256) and s >= 1
    assert lib.gnf_tc_gemm_plan(0, 1, 1, 3, 0, C.byref(bn), C.byref(sp)) != 0


def test_fused_umnn_backward_takes_every_net_the_fused_forward_takes():
    """A training forward on gnf_umnn_fwd_tc3 is always followed by gnf_umnn_bwd_tc3, so at S + 1 <= 256 nodes the two workspace
    queries accept the same integrands: 3- and 4-layer nets over hidden widths on both sides of every 32-column padding step,
    up to 160 and one past it.  Host-only queries (the weight pointers are never read)."""
    import ctypes as C
    import itertools
    import __graft_entry__
    __graft_entry__.build()
    lib = G._lib.load_library()
    E, R = 5, 240
    widths = (1, 31, 32, 33, 64, 128, 129, 152, 153, 160, 161)
    accepted = 0
    for hidden in itertools.chain(itertools.product(widths, repeat=2), itertools.product(widths, repeat=3)):
        net = G._lib.MlpT()
        dims = [1 + E, *hidden, 1]
        net.n_layers = len(dims) - 1
        for i, v in enumerate(dims):
            net.dims[i] = v
        fwd = lib.gnf_umnn_tc3_workspace_bytes(C.byref(net), R)
        assert (fwd != 0) == (max(hidden) <= 160), hidden
        for S in (20, 255):
            bwd = lib.gnf_umnn_bwd_tc3_workspace_bytes(C.byref(net), R, S)
            assert (bwd != 0) == (fwd != 0), (hidden, S, lib.gnf_last_error())
        accepted += fwd != 0
    assert accepted == 10 ** 2 + 10 ** 3


def test_ffma_umnn_backward_query_matches_its_shared_memory_limit():
    """gnf_umnn_bwd_workspace_bytes is non-zero exactly when gnf_umnn_bwd takes the integrand: the forward's plan (1 + E padded
    to 16 within the padded hidden width 16 TN) and the backward's tiles, (KB0 68 + L NP 68 + 32 NP + 384) floats <= 227 KB,
    over 2..8 linear layers, the largest hidden width on both sides of every TN step, and E at 1, 31, 32, 223, 255.
    Host-only query (the weight pointers are never read)."""
    import ctypes as C
    import __graft_entry__
    __graft_entry__.build()
    lib = G._lib.load_library()
    widths = (1, 16, 32, 33, 64, 65, 112, 113, 160, 161, 208, 209, 255, 256)
    seen = set()
    for n_layers in range(2, 9):
        for w in widths:
            for hidden in {(w,) * (n_layers - 1), (1,) * (n_layers - 2) + (w,)}:
                for E in (1, 31, 32, 223, 255):
                    TN = next(t for t in (2, 4, 7, 10, 13, 16) if 16 * t >= w)
                    NP, KP0, KB0 = 16 * TN, -(-(1 + E) // 16) * 16, -(-(1 + E) // 32) * 32
                    fits = KP0 <= NP and (KB0 * 68 + len(hidden) * NP * 68 + 32 * NP + 384) * 4 <= 227 * 1024
                    net = G._lib.MlpT()
                    dims = [1 + E, *hidden, 1]
                    net.n_layers = len(dims) - 1
                    for i, v in enumerate(dims):
                        net.dims[i] = v
                    got = lib.gnf_umnn_bwd_workspace_bytes(C.byref(net))
                    assert (got != 0) == fits, (hidden, E, got, lib.gnf_last_error())
                    if fits:
                        assert got == lib.gnf_umnn_workspace_bytes(C.byref(net))
                    seen.add(fits)
    assert seen == {True, False}
    net = G._lib.MlpT()
    for i, v in enumerate([8, 256, 256, 256, 1]):
        net.dims[i] = v
    net.n_layers = 4
    assert lib.gnf_umnn_workspace_bytes(C.byref(net)) > 0 and lib.gnf_umnn_bwd_workspace_bytes(C.byref(net)) == 0
    assert b"shared memory" in lib.gnf_last_error()


# ---------------- experiment plumbing (SURVEY 8f rank 4) ----------------
def test_reference_yaml_preset_and_driver_defaults(tmp_path):
    """A preset in the reference's YAML format (UCIExperimentsConfigurations.yml:1-14) merged over the driver's argparse defaults;
    the flow it builds has the reference's parameter count (SURVEY 8e: cfg2 = 33 467)."""
    y = tmp_path / "cfg.yml"
    y.write_text("power-mono-DAG:\n  dataset: 'power'\n  nb_flow: 1\n  b_size: 2500\n  nb_epoch: 10000\n  conditioner: 'DAG'\n"
                 "  emb_net: [60, 60, 60, 30]\n  nb_steps_dual: 30\n  l1: 0.\n  gumble_T: .5\n  normalizer: 'monotonic'\n"
                 "  int_net: [100, 100, 100]\n  nb_steps: 20\n  solver: 'CC'\n  weight_decay: 1e-5\n")
    cfg = G.experiments.load_preset(str(y), "power-mono-DAG")
    assert cfg["b_size"] == 2500 and cfg["emb_net"] == [60, 60, 60, 30] and cfg["weight_decay"] == 1e-5 and cfg["learning_rate"] == 1e-3
    model = G.experiments.build_uci_flow(6, cfg)
    assert sum(p.numel() for p in model.parameters()) == 33467
    c = model.getConditioners()[0]
    assert c.nb_epoch_update == 30 and c.hot_encoding and c.gumble_T == .5
    with pytest.raises(KeyError):
        G.experiments.load_preset(str(y), "nope")


def test_data_parallel_checkpoint_prefix_and_bpp():
    model = G.build_from_spec(G.CONFIGS["cfg2"])
    sd = {"module." + k: v.clone() + 1 for k, v in model.state_dict().items()}          # what nn.DataParallel(model).state_dict() saves
    G.load_checkpoint(model, sd)
    for k, v in model.state_dict().items():
        assert torch.equal(v, sd["module." + k]), k
    # bits per pixel (ImageExperiments.py:33-37) against the formula written out in float64
    x, ll = torch.randn(5, 12), torch.randn(5) * 10 - 50
    ref = (-ll.double() / (12 * np.log(2)) - np.log2(1 - 2e-6) + 8 +
           (torch.log2(torch.sigmoid(x.double())) + torch.log2(1 - torch.sigmoid(x.double()))).sum(1) / 12)
    assert torch.allclose(G.compute_bpp(ll, x).double(), ref, atol=1e-5)
