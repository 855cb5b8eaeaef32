"""Cost of the context in a conditional DAG flow: the cfg4 shape (d = 63, DAG [630, 630, 630] + UMNN [150, 150, 150], S = 20,
batch 100, GEMM mode 'auto') with cond_in = 0, 8 and 64, as a captured training step (GraphedTrainStep) and a captured evaluation
step (GraphedEvalStep).  The variants are timed in alternation (round r times every variant once), with CUDA events around
`--replays` replays per sample; the median over `--rounds` rounds is reported per variant, with its overhead against cond_in = 0.
A second, eager pass per variant brackets every C-ABI call with CUDA events (ops.enable_kernel_timing) and prints the per-call
times that differ from the unconditional step.  One GPU.  usage: conditional_bench.py [--rounds R] [--replays K] [--batch B]"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gnf_b200 as G  # noqa: E402

CONDS = (0, 8, 64)


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit not readable"
    return f"{name} ({q})"


def build(c, B, seed=0):
    spec = dict(G.CONFIGS["cfg4"], cond_in=c)
    model = G.build_from_spec(spec, "cuda", seed=seed)
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(B, spec["d"], device="cuda", generator=g)
    ctx = torch.randn(B, c, device="cuda", generator=g) if c else None
    return spec, model, x, ctx


def make_steps(c, B):
    _, model, x, ctx = build(c, B)
    bucket = G.dist.GradBucket(model.parameters())
    opt = G.FusedAdam(model.parameters(), lr=1e-4)
    train = G.GraphedTrainStep(model, opt, bucket, x, allreduce=False, warmup=3, example_context=ctx)
    _, emodel, ex, ectx = build(c, B, seed=1)
    ev = G.GraphedEvalStep(emodel, ex, example_context=ectx)
    return {"train": lambda: train(x, ctx), "eval": lambda: ev(ex, ectx)}


def time_ms(fn, replays):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / replays


def per_call(c, B):
    """{entry point: total ms per eager training step} (mean of 5 steps after 3 warm-up steps)."""
    _, model, x, ctx = build(c, B)
    for _ in range(3):
        model.zero_grad()
        z, jac = model(x, ctx)
        model.loss(z, jac).backward()
    G.ops.enable_kernel_timing(True)
    for _ in range(5):
        model.zero_grad()
        z, jac = model(x, ctx)
        model.loss(z, jac).backward()
    t = G.ops.collect_kernel_timing()
    G.ops.enable_kernel_timing(False)
    return {k: (sum(v) / 5, len(v) // 5) for k, v in t.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--replays", type=int, default=50)
    ap.add_argument("--batch", type=int, default=100)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "conditional_bench.py needs a GPU"
    G.ops.set_gemm_mode("auto")
    print(f"card: {card()}")
    steps = {c: make_steps(c, args.batch) for c in CONDS}
    for c in CONDS:                                   # warm every graph
        for fn in steps[c].values():
            time_ms(fn, 5)
    samples = {(c, k): [] for c in CONDS for k in ("train", "eval")}
    for _ in range(args.rounds):
        for k in ("train", "eval"):
            for c in CONDS:
                samples[(c, k)].append(time_ms(steps[c][k], args.replays))
    print(f"cfg4 shape, batch {args.batch}, gemm auto; median [min, max] of {args.rounds} rounds x {args.replays} replays, ms per step")
    for k in ("train", "eval"):
        base = statistics.median(samples[(0, k)])
        for c in CONDS:
            s = samples[(c, k)]
            med = statistics.median(s)
            print(f"  {k:5s} cond_in={c:3d}: {med:8.4f} [{min(s):.4f}, {max(s):.4f}]  overhead {100. * (med / base - 1.):+6.2f} %")
    calls = {c: per_call(c, args.batch) for c in CONDS}
    print("eager training step, per-call times that differ from cond_in = 0 (ms per step, calls per step):")
    for c in CONDS[1:]:
        for name in sorted(set(calls[0]) | set(calls[c])):
            a, na = calls[0].get(name, (0., 0))
            b, nb = calls[c].get(name, (0., 0))
            if na != nb or abs(b - a) > 0.002:
                print(f"  cond_in={c:3d} {name:28s} {a:8.4f} ({na}) -> {b:8.4f} ({nb})")


if __name__ == "__main__":
    main()
