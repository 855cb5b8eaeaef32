"""Micro-benchmark of the conditioner GEMM engines (run on the GPU box)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gnf_b200 as G

def t(fn, n=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n

for (M, N, K) in [(138600, 160, 160), (138600, 152, 152), (6300, 632, 632), (6300, 630, 630), (64512, 632, 632), (78400, 1024, 1024), (10000, 212, 212)]:
    X = torch.randn(M, K, device="cuda"); W = torch.randn(N, K, device="cuda") / K ** .5; b = torch.randn(N, device="cuda")
    dY = torch.randn(M, N, device="cuda")
    fl = 2. * M * N * K
    row = f"M={M} N={N} K={K}:"
    for mode in ("ffma", "tf32", "tf32x3"):
        G.ops.set_gemm_mode(mode)
        a = t(lambda: G.ops.linear_fwd(X, W, b, relu=True))
        c = t(lambda: G.ops.linear_dgrad(dY, N, W, X, M))
        d = t(lambda: G.ops.linear_wgrad(dY, N, X, K, M, N, K))
        row += f"  {mode}: fwd {a*1e3:.0f}us {fl/a/1e9:.0f}TF  dgrad {c*1e3:.0f}us {fl/c/1e9:.0f}TF  wgrad {d*1e3:.0f}us {fl/d/1e9:.0f}TF |"
    print(row)
    tt = t(lambda: torch.relu(X @ W.t() + b))
    print(f"      torch fp32 (cuBLAS) fwd {tt*1e3:.0f}us {fl/tt/1e9:.0f}TF")

print("resident wgrad kernel (tc_rw_wgrad.cu)")
for (M, N, K) in [(138600, 150, 150), (1419264, 150, 150), (150000, 100, 100)]:
    NPn, KP = (N + 31) // 32 * 32, (K + 31) // 32 * 32
    X = torch.zeros(M, KP, device="cuda"); X[:, :K] = torch.randn(M, K, device="cuda")
    dY = torch.zeros(M, NPn, device="cuda"); dY[:, :N] = torch.randn(M, N, device="cuda")
    fl = 2. * M * N * K
    row = f"M={M} N={N} K={K}:"
    for passes in (1, 3):
        a = t(lambda: G.ops.linear_wgrad_rw(dY, X, N, K, passes=passes))
        row += f"  passes={passes}: wgrad {a*1e3:.0f}us {fl/a/1e9:.0f}TF {M*(NPn+KP)*4/a/1e6:.0f}GB/s |"
    print(row)
