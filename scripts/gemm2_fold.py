"""Engine v2 of the conditioner GEMMs: duration against the fold interval (k-chunks per in-core accumulation group) and against the
first engine; dev build.  usage: gemm2_fold.py [M N K]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import devlib  # noqa: E402

lib = devlib.install()
import gnf_b200 as G  # noqa: E402

M, N, K = (int(v) for v in sys.argv[1:4]) if len(sys.argv) > 3 else (6300, 630, 630)
G.ops.set_gemm_mode("tf32x3")
like = torch.empty(1, device="cuda")
X = G.ops._rows(M, K, like); X.normal_()
dY = G.ops._rows(M, N, like); dY.normal_()
W = torch.randn(N, K, device="cuda") / K ** .5
b = torch.randn(N, device="cuda")
ref = (X[:, :K].double() @ W.double().t() + b.double()).clamp_min(0)


def timed(fn, n=30):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1000


for v2 in (1, 0):
    lib.gnf_tc_gemm_set_v2(v2)
    for fold in (1, 2, 4, 1000):
        lib.gnf_tc_gemm_set_fold(fold)
        f = timed(lambda: G.ops.linear_fwd(X, W, b, relu=True))
        d = timed(lambda: G.ops.linear_dgrad(dY, dY.stride(0), W, X, M))
        Y = G.ops.linear_fwd(X, W, b, relu=True)
        err = float((Y.double() - ref).norm() / ref.norm())
        bias = float((Y.double() - ref).mean() / ref.abs().mean())
        worst = float((Y.double() - ref).abs().max() / ref.abs().mean())
        print(f"engine v{('1', '2')[v2]} fold={fold:4d}: fwd {f:6.1f} us  dgrad {d:6.1f} us   fwd rel L2 err {err:.2e}  mean signed err / mean |y| {bias:+.2e}"
              f"  max |err| / mean |y| {worst:.2e}")
lib.gnf_tc_gemm_set_fold(2)
lib.gnf_tc_gemm_set_v2(1)
