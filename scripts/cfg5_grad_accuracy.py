"""Where do the gradient differences of the wide DAG flow (cfg5, d = 784) come from?  One training step at batch B through
  * the CPU oracle in float64 (the yardstick) and in float32 (what the parity tests compare with),
  * the CUDA path with layer 1 on the embedding plane + tensor-core GEMMs, with layer 1 on the FFMA loader kernels, and all-FFMA,
every gradient as relative L2 against the float64 oracle.  usage: cfg5_grad_accuracy.py [B]"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gnf_b200 as G  # noqa: E402
import gnf_oracle as O  # noqa: E402


def l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def main(B=16, cfg="cfg5"):
    spec = G.CONFIGS[cfg]
    ospec = {k: v for k, v in spec.items() if k != "A_prior"}
    x = torch.randn(B, spec["d"], generator=torch.Generator().manual_seed(1)).cuda()
    runs = {}
    noises = None
    sd = None
    fold = os.environ.get("GNF_FOLD")
    if fold:                                                   # dev build: k-chunks per in-core accumulation group of the GEMM engine
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import devlib
        devlib.install().gnf_tc_gemm_set_fold(int(fold))
        print(f"fold = {fold}")
    for name, gemm, plane in (("plane+tc", "auto", True), ("ffma-l1+tc", "auto", False), ("all-ffma", "ffma", True)):
        G.ops.set_gemm_mode(gemm)
        G.ops.DAG_L1_PLANE = plane
        model = G.build_from_spec(spec, "cuda", 0)
        model.zero_grad()
        z, jac = model(x)
        loss = model.loss(z, jac)
        loss.backward()
        if noises is None:
            noises = [tuple(n.cpu() for n in G.ops.dag_dump_noise(c._last_gate, B, spec["d"], x.device)) for c in model.getConditioners()]
            sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        runs[name] = {k: p.grad.detach().cpu() for k, p in model.named_parameters() if p.grad is not None}
    G.ops.DAG_L1_PLANE = True
    _, _, _, g32 = O.train_step_grads(x.cpu(), sd, ospec, None, noises, None)
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    n64 = [tuple(n.double() for n in t) for t in noises]
    _, _, _, g64 = O.train_step_grads(x.cpu().double(), sd64, ospec, None, n64, None)
    print(f"{cfg} B={B}: relative L2 error of every gradient against the float64 oracle")
    print(f"{'tensor':60s} {'oracle fp32':>12s} " + " ".join(f"{n:>12s}" for n in runs))
    for k, g in g64.items():
        if g is None:
            continue
        print(f"{k:60s} {l2(g32[k], g):12.2e} " + " ".join(f"{l2(r[k], g):12.2e}" for r in runs.values()))


if __name__ == "__main__":
    main(*[int(v) for v in sys.argv[1:2]])
