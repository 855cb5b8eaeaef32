"""The fp32 CUDA-core GEMM engine (csrc/gemm.cuh, csrc/thin.cuh, the linear entry points of csrc/mlp.cu) and the power-trace chain
(csrc/power_trace.cu) against float64, route by route, at the limits of their selection code.

This engine runs under the default GEMM mode and, under 'auto', every layer below the tensor-core thresholds, the 630 -> 30 output
layer (split-K), the 1024 -> 2 output dgrad (thin kernel), the small weight gradients, the context GEMMs and the d > 64 power trace.

Every case calls the C-ABI directly with explicit leading dimensions and base offsets; operand padding holds NaN (a kernel that reads
it fails), every output element the call must not write holds the sentinel -777 (padding columns, dW columns [K, lddw), the row after
the last one).  On the GPU each case asserts, with torch.profiler, which kernels ran:
  * gemm_kernel<TileCfg<BM, BN, BK, TM, TN>, ...> -- told apart by the template arguments of the demangled name: Tiny (32x32x64),
    Skinny (128x32x16), Short (32x128x16), Mid (128x64x16), Big (128x128x16);
  * thin_red_kernel, splitk_sum_kernel, colsum_kernel, power_trace_small_fwd / _small_bwd / _small_fwd_save, trace_bwd_kernel,
    build_B_kernel.
The expected route of every case is written in its table, on both sides of every threshold of launch_gemm_auto, thin_launch_red,
sk_splits and gnf_colsum, so that a moved threshold fails a route assertion.  The development library's gnf_linear_set_thin(0)
puts the calls the thin kernel would take on the tile GEMM, and both routes are held to float64.

Checks of every case:
  * integer operands in [-4, 4] (every GEMM, split-K and colsum case): every product and partial sum is exact in fp32, so every
    route must reproduce float64 bit for bit, whatever the rounding and the order of the atomics (periodic bias rows m % period,
    partial k tiles, split-K slices, period sums);
  * normal operands against float64, componentwise: max |C - ref| / (|A| |B|^T + |bias|); the power trace: |t - ref| / (d + |ref|)
    and the relative L2 error of dA, against torch.linalg.matrix_power in float64 and dA = gt 2 alpha p A o (B^(p-1))^T;
  * test_bars_reject_a_missing_term_block (CPU): at every normal-operand case the bar rejects, by 10x at least, a result that misses
    one k tile (16 terms, 64 on Tiny) or one split-K slice, or a power trace one power short.

Bars (componentwise errors of normal operands), measured on a B200 at its 1000 W power limit over the whole table:
  route                                  worst measured            bar
  forward, tile GEMM                     3.5e-7 (Skinny, K = 64)    1e-6
  dgrad, tile GEMM                       2.8e-7                     1e-6
  thin kernel, forward and dgrad         2.8e-7                     1e-6
  split-K forward                        1.5e-7                     1e-6
  weight gradient (split-K atomics)      2.3e-7                     7e-7
  gnf_colsum                             1.7e-7 (7-term sums)       4e-7 (a 7-term sum in order is bounded by 6 x 2^-24 = 3.6e-7)
  power trace t and dA                   2.8e-9 x max(p, 2) max(d, 64)    1e-8 x max(p, 2) max(d, 64)
The power trace's error grows with p and with d: every product of the chain sums d positive terms in order, and B^p carries the
rounding of B = I + alpha A o A and of every product p-fold.  Largest: 6.7e-5 at d = 784, p = 34 (torch's own fp32
matrix_power, with its blocked sums, is off by 3.2e-5 there), 4.6e-5 at d = p = 129; the simulator build gives the same bits.

The same case table, at its small shapes, runs in the host SIMT-simulator build of the kernels (tests/emu) on a machine without a
GPU.  test_simulator_matches_gpu_bitwise runs the simulator next to the GPU library in one process: tile forward / dgrad, thin and
split-K forward are deterministic (explicit fmaf chains, epilogues that only add), so both must give the same bits.
"""
import ctypes as C
import os
import re
import sys

import pytest
import torch

import gnf_b200 as G
from gemm_ref import NAN, SENT, Mat, check_sentinels, cw_err, launched, pad4

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

BAR = {"fwd": 1e-6, "dgrad": 1e-6, "thin": 1e-6, "splitk": 1e-6, "wgrad": 7e-7, "colsum": 4e-7, "pt": 1e-8}

TINY, SKINNY, SHORT, MID, BIG = "Tiny", "Skinny", "Short", "Mid", "Big"
TILES = {(32, 32, 64, 4, 4): TINY, (128, 32, 16, 4, 4): SKINNY, (32, 128, 16, 4, 8): SHORT, (128, 64, 16, 8, 4): MID,
         (128, 128, 16, 8, 8): BIG}
BK = {TINY: 64, SKINNY: 16, SHORT: 16, MID: 16, BIG: 16}
THIN, SKSUM, COLSUM = "thin_red_kernel", "splitk_sum_kernel", "colsum_kernel"
PT_FWD, PT_BWD, PT_SAVE, PT_BWD_SAVED, BUILD_B = ("power_trace_small_fwd", "power_trace_small_bwd", "power_trace_small_fwd_save",
                                                 "trace_bwd_kernel", "build_B_kernel")
KERNELS = (THIN, SKSUM, COLSUM, PT_FWD, PT_BWD, PT_SAVE, PT_BWD_SAVED, BUILD_B)
TILE_RE = re.compile(r"\bgemm_kernel<\s*(?:gnf::)?TileCfg<\s*(\d+),\s*(\d+),\s*(\d+),\s*(\d+),\s*(\d+)\s*>")


def routes(names):
    """The engine's kernels among the launched kernel names: tile names for gemm_kernel, the kernel name otherwise."""
    out = set()
    for n in names:
        m = TILE_RE.search(n)
        if m:
            out.add(TILES.get(tuple(map(int, m.groups())), n))
        elif re.search(r"\bgemm_kernel\b", n):
            out.add("unparsed: " + n)
        out |= {k for k in KERNELS if re.search(rf"\b{k}\b", n)}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# where a case runs: the product library on the GPU, the development library, or the simulator on the CPU
# ---------------------------------------------------------------------------------------------------------------------
class Dev:
    def __init__(self, lib, device):
        self.lib, self.device = lib, device

    def stream(self):
        return C.c_void_p(torch.cuda.current_stream().cuda_stream) if self.device == "cuda" else None

    def rc(self, name, *args):
        if self.device == "cuda":
            torch.cuda.synchronize()
        return getattr(self.lib, name)(*args, self.stream())

    def call(self, name, *args):
        rc = self.rc(name, *args)
        assert rc == 0, f"{name}: {rc} {self.lib.gnf_last_error()}"

    def mat(self, rows, cols, ld, fill, off=0):
        return Mat(rows, cols, ld, fill, off, device=self.device)


@pytest.fixture(scope="module")
def gpu():
    return Dev(G._lib.load_library(), "cuda")


@pytest.fixture
def no_thin():
    """The development library with gnf_linear_set_thin(0): the calls the thin kernel takes run on the tile GEMM."""
    dev_so = os.path.join(os.path.dirname(G._lib.LIB_PATH), "libgnf_sm100_dev.so")
    assert os.path.isfile(dev_so), "engine switches are development-build knobs: __graft_entry__.build() builds libgnf_sm100_dev.so"
    lib = G._lib._bind(C.CDLL(dev_so))
    lib.gnf_linear_set_thin.argtypes, lib.gnf_linear_set_thin.restype = [C.c_int], C.c_int
    lib.gnf_linear_set_thin(0)
    try:
        yield Dev(lib, "cuda")
    finally:
        lib.gnf_linear_set_thin(1)


@pytest.fixture(scope="module")
def sim():
    """The host SIMT-simulator build of the same sources, loaded next to (not in place of) the package's library."""
    import build_emu
    return Dev(G._lib._bind(C.CDLL(build_emu.build())), "cpu")


def operands(kind, seed, device):
    """Drawn on the CPU, so that the GPU, the simulator and the sensitivity test see the same values."""
    g = torch.Generator().manual_seed(seed)
    if kind == "int":
        return lambda *s: torch.randint(-4, 5, s, generator=g).float().to(device)
    return lambda *s: torch.randn(*s, generator=g).to(device)


def lay(dim, layout):
    """(leading dimension, base offset): 'A' = 16-byte aligned rows with 4 padding columns, 'U' = one padding column (odd ld
    for even dim) and a base one float off: 4-byte aligned rows, 'D' = dense (ld = dim)."""
    return {"A": (pad4(dim) + 4, 0), "U": (dim + 1, 1), "D": (dim, 0)}[layout]


# ---------------------------------------------------------------------------------------------------------------------
# the operations: operands, the call, the float64 reference, and the reduction as (A, B) for the sensitivity test
# ---------------------------------------------------------------------------------------------------------------------
class Fwd:
    """Y = act(X W^T + bias[m % period]) through gnf_linear_fwd; bias None (NULL), 1 (plain) or a period."""
    op = "fwd"

    def __init__(self, M, N, K, bias=1, relu=True, layout="A"):
        self.M, self.N, self.K, self.bias, self.relu, self.layout = M, N, K, bias, relu, layout

    def fill(self, dev, kind, seed):
        r = operands(kind, seed, dev.device)
        M, N, K = self.M, self.N, self.K
        (ldx, off), (ldw, _) = lay(K, self.layout), lay(K, self.layout)
        self.X = dev.mat(M, K, ldx, NAN, off).set(r(M, K))
        self.W = dev.mat(N, K, ldw, NAN, off).set(r(N, K))
        self.B = dev.mat(self.bias, N, N, NAN).set(r(self.bias, N)) if self.bias else None

    def run(self, dev):
        M, N, K = self.M, self.N, self.K
        ldy, off = lay(N, self.layout)
        self.Y = dev.mat(M, N, ldy, SENT, off)
        dev.call("gnf_linear_fwd", self.X.p, self.X.ld, self.W.p, self.W.ld, self.B.p if self.B else None, self.bias or 0, self.Y.p, ldy,
                 M, N, K, int(self.relu))
        return [self.Y]

    def parts(self, rows=None):
        rows = rows or self.M
        A, B = self.X.t[:rows].double(), self.W.t.double().t()
        add = self.B.t.double()[torch.arange(rows, device=A.device) % self.bias] if self.B else None
        return A, B, add, (lambda y: y.clamp_min(0)) if self.relu else (lambda y: y)


class Dgrad:
    """dX = (dY W) * (act > 0) through gnf_linear_dgrad; act None (NULL) or the number of extra ldact columns."""
    op = "dgrad"

    def __init__(self, M, N, K, act=None, layout="A"):
        self.M, self.N, self.K, self.act, self.layout = M, N, K, act, layout

    def fill(self, dev, kind, seed):
        r = operands(kind, seed, dev.device)
        M, N, K = self.M, self.N, self.K
        (lddy, off), (ldw, _) = lay(N, self.layout), lay(K, self.layout)
        self.dY = dev.mat(M, N, lddy, NAN, off).set(r(M, N))
        self.W = dev.mat(N, K, ldw, NAN, off).set(r(N, K))
        self.A = dev.mat(M, K, K + self.act, NAN, off).set(r(M, K)) if self.act is not None else None

    def run(self, dev):
        lddx, off = lay(self.K, self.layout)
        self.dX = dev.mat(self.M, self.K, lddx, SENT, off)
        ap, lda = (self.A.p, self.A.ld) if self.A is not None else (None, 0)
        dev.call("gnf_linear_dgrad", self.dY.p, self.dY.ld, self.W.p, self.W.ld, ap, lda, self.dX.p, lddx, self.M, self.N, self.K)
        return [self.dX]

    def parts(self, rows=None):
        rows = rows or self.M
        A, B = self.dY.t[:rows].double(), self.W.t.double()
        if self.A is None:
            return A, B, None, lambda y: y
        mask = (self.A.t[:rows] > 0).double()
        return A, B, None, lambda y: y * mask


class Wgrad:
    """dW = dY^T X through gnf_linear_wgrad (split-K, atomics into a zeroed dW) into the first K columns of [N, K + extra]."""
    op = "wgrad"

    def __init__(self, M, N, K, extra=0):
        self.M, self.N, self.K, self.extra = M, N, K, extra

    def fill(self, dev, kind, seed):
        r = operands(kind, seed, dev.device)
        self.dY = dev.mat(self.M, self.N, self.N + 3, NAN, 1).set(r(self.M, self.N))
        self.X = dev.mat(self.M, self.K, pad4(self.K) + 4, NAN).set(r(self.M, self.K))

    def run(self, dev):
        self.dW = dev.mat(self.N, self.K, self.K + self.extra, SENT)
        dev.call("gnf_linear_wgrad", self.dY.p, self.dY.ld, self.X.p, self.X.ld, self.dW.p, self.dW.ld, self.M, self.N, self.K)
        return [self.dW]

    def parts(self, rows=None):
        rows = rows or self.N
        return self.dY.t.double().t()[:rows], self.X.t.double(), None, lambda y: y


class SplitK:
    """gnf_linear_fwd_splitk: Y = act(X W^T + bias), partial tiles of the slices in a NaN-filled workspace, fixed-order sum."""
    op = "splitk"

    def __init__(self, M, N, K, bias=True, relu=True, extra=0):
        self.M, self.N, self.K, self.bias, self.relu, self.extra = M, N, K, bias, relu, extra

    def fill(self, dev, kind, seed):
        r = operands(kind, seed, dev.device)
        M, N, K = self.M, self.N, self.K
        self.X = dev.mat(M, K, K + 1, NAN, 1).set(r(M, K))
        self.W = dev.mat(N, K, K + 2, NAN).set(r(N, K))
        self.B = dev.mat(1, N, N, NAN).set(r(1, N)) if self.bias else None

    def slice_len(self):
        """launch_gemm's slice: sk_splits(K) slices rounded to whole k tiles of 16."""
        K = self.K
        splits = 6 if K // 6 >= 64 else (K // 64 if K >= 128 else 1)
        return -(-(-(-K // 16)) // splits) * 16

    def run(self, dev):
        M, N, K = self.M, self.N, self.K
        need = dev.lib.gnf_linear_fwd_splitk_workspace_bytes(M, N, K)
        assert need > 0
        work = torch.full((need // 4,), NAN, device=dev.device)
        self.Y = dev.mat(M, N, N + self.extra, SENT)
        dev.call("gnf_linear_fwd_splitk", self.X.p, self.X.ld, self.W.p, self.W.ld, self.B.p if self.B else None, self.Y.p, self.Y.ld,
                 M, N, K, int(self.relu), C.c_void_p(work.data_ptr()), need)
        return [self.Y]

    def parts(self, rows=None):
        rows = rows or self.M
        A, B = self.X.t[:rows].double(), self.W.t.double().t()
        add = self.B.t.double().expand(rows, -1) if self.B else None
        return A, B, add, (lambda y: y.clamp_min(0)) if self.relu else (lambda y: y)


class Colsum:
    """out[p, n] = sum_{m % period == p} Y[m, n] through gnf_colsum; Y of row stride N + extra with NaN in the padding."""
    op = "colsum"

    def __init__(self, M, N, period, extra=0):
        self.M, self.N, self.period, self.extra = M, N, period, extra

    def fill(self, dev, kind, seed):
        r = operands(kind, seed, dev.device)
        self.Y = dev.mat(self.M, self.N, self.N + self.extra, NAN).set(r(self.M, self.N))

    def run(self, dev):
        self.out = dev.mat(self.period, self.N, self.N, SENT)
        dev.call("gnf_colsum", self.Y.p, self.Y.ld, self.out.p, self.M, self.N, self.period)
        return [self.out]

    def parts(self, rows=None):
        """out = A B with A [period, M] the indicator of m % period == p."""
        m = torch.arange(self.M, device=self.Y.t.device)
        A = (m[None, :] % self.period == torch.arange(self.period, device=m.device)[:, None]).double()
        return A, self.Y.t.double(), None, lambda y: y


def reference(case, rows=None, drop=None):
    """float64 result and componentwise denominator; drop = (k0, k1): the result without reduction terms [k0, k1)."""
    A, B, add, post = case.parts(rows)
    if drop is not None:
        keep = torch.ones(A.shape[1], dtype=torch.bool, device=A.device)
        keep[drop[0]:drop[1]] = False
        A, B = A[:, keep], B[keep]
    ref, den = A @ B, A.abs() @ B.abs()
    if add is not None:
        ref, den = ref + add, den + add.abs()
    return post(ref), den


# ---------------------------------------------------------------------------------------------------------------------
# the case table: name -> (case, expected kernels)
# ---------------------------------------------------------------------------------------------------------------------
CASES = {}


def case(name, c, expect, sim=False):
    assert name not in CASES, name
    c.expect, c.sim, c.name = set(expect), sim, name
    CASES[name] = c


# gnf_linear_fwd, tile GEMM.  launch_gemm_auto: N <= 32 and ceil(M / 128) < 148 -> Tiny; N <= 32 -> Skinny; M <= 32 and N > 64 ->
# Short; N <= 64 -> Mid; else Big.  (M >= 512, K <= 8, N <= 4096 and period <= 1 go to the thin kernel instead.)
for L in "AU":
    for N, t in ((32, TINY), (33, MID), (64, MID), (65, BIG)):
        case(f"fwd_n{N}_{L}", Fwd(300, N, 40, bias=1, layout=L), {t}, sim=True)
    case(f"fwd_m32_n65_{L}", Fwd(32, 65, 40, layout=L), {SHORT}, sim=True)
    case(f"fwd_m33_n65_{L}", Fwd(33, 65, 40, layout=L), {BIG}, sim=True)
    case(f"fwd_m32_n64_{L}", Fwd(32, 64, 40, layout=L), {MID}, sim=True)
    case(f"fwd_m32_n200_{L}", Fwd(32, 200, 40, layout=L), {SHORT})
    case(f"fwd_m18816_{L}", Fwd(18816, 30, 20, layout=L), {TINY})      # 147 row tiles of 128
    case(f"fwd_m18817_{L}", Fwd(18817, 30, 20, layout=L), {SKINNY})    # 148
for K in (15, 16, 17, 63, 64, 65):
    case(f"fwd_tiny_k{K}", Fwd(200, 20, K, bias=1, layout="U"), {TINY}, sim=True)
    case(f"fwd_big_k{K}", Fwd(200, 100, K, bias=1), {BIG}, sim=K < 32)
    case(f"fwd_mid_k{K}", Fwd(200, 48, K, bias=None, relu=False), {MID})
    case(f"fwd_skinny_k{K}", Fwd(18817, 24, K, bias=7, layout="U"), {SKINNY})
    case(f"fwd_short_k{K}", Fwd(20, 130, K, bias=1, relu=False), {SHORT})
case("fwd_111", Fwd(1, 1, 1), {TINY}, sim=True)
case("fwd_111_nobias", Fwd(1, 1, 1, bias=None, relu=False), {TINY}, sim=True)
for bias in (None, 1, 2, 63, 252):                                      # periodic bias rows m % period (period = M: 252)
    for relu in (False, True):
        for N, t in ((65, BIG), (30, TINY), (40, MID)):
            case(f"fwd_bias{bias}_relu{int(relu)}_n{N}", Fwd(252, N, 33, bias=bias, relu=relu, layout="U" if relu else "A"), {t},
                 sim=N == 65 or bias in (2, 252))
case("fwd_period2_k8_m600", Fwd(600, 100, 8, bias=2), {BIG}, sim=True)  # a periodic bias keeps the thin shape on the tile GEMM

# gnf_linear_fwd, thin kernel: M >= 512, K <= kThinT = 8, N <= 4096
THIN_FWD = {"m511": (Fwd(511, 100, 8), {BIG}), "m512": (Fwd(512, 100, 8), {THIN}),
            "k8": (Fwd(600, 100, 8, bias=None), {THIN}), "k9": (Fwd(600, 100, 9, bias=None), {BIG}),
            "n4096": (Fwd(600, 4096, 8, relu=False), {THIN}), "n4097": (Fwd(600, 4097, 8, relu=False), {BIG}),
            "k1_dense": (Fwd(600, 70, 1, layout="D"), {THIN}), "k1_u": (Fwd(600, 70, 1, layout="U"), {THIN}),
            "n30_k2": (Fwd(515, 30, 2, layout="U"), {THIN}),
            "rows40000": (Fwd(40000, 4096, 8), {THIN})}    # one CTA per SM: 4736 rows per pass, the warps loop
for name, (c, e) in THIN_FWD.items():
    case(f"thin_fwd_{name}", c, e, sim=c.M * c.N <= 700 * 128)

# gnf_linear_dgrad: output [M, K], reduction over N.  Tile choice as above with the output width K; thin: M >= 512, N <= 8, K <= 4096
for L in "AU":
    for K, t in ((32, TINY), (33, MID), (64, MID), (65, BIG)):
        case(f"dgrad_k{K}_act_{L}", Dgrad(300, 40, K, act=5, layout=L), {t}, sim=True)
        case(f"dgrad_k{K}_none_{L}", Dgrad(300, 40, K, layout=L), {t})
    case(f"dgrad_m32_k65_{L}", Dgrad(32, 40, 65, act=0, layout=L), {SHORT}, sim=True)
    case(f"dgrad_m33_k65_{L}", Dgrad(33, 40, 65, act=0, layout=L), {BIG})
    case(f"dgrad_m18816_{L}", Dgrad(18816, 20, 30, act=3, layout=L), {TINY})
    case(f"dgrad_m18817_{L}", Dgrad(18817, 20, 30, act=3, layout=L), {SKINNY})
for N in (15, 16, 17, 63, 64, 65):
    case(f"dgrad_tiny_n{N}", Dgrad(200, N, 20, act=4), {TINY}, sim=True)
    case(f"dgrad_big_n{N}", Dgrad(200, N, 100, act=1, layout="U"), {BIG}, sim=N < 32)
case("dgrad_1_1_6_act", Dgrad(1, 1, 6, act=0), {TINY}, sim=True)
case("dgrad_111_none", Dgrad(1, 1, 1), {TINY}, sim=True)
THIN_DGRAD = {"m511": (Dgrad(511, 8, 100, act=3), {BIG}), "m512": (Dgrad(512, 8, 100, act=3), {THIN}),
              "n8_act": (Dgrad(600, 8, 100, act=5), {THIN}), "n8_none": (Dgrad(600, 8, 100), {THIN}),
              "n9_act": (Dgrad(600, 9, 100, act=5), {BIG}), "n9_none": (Dgrad(600, 9, 100), {BIG}),
              "n1": (Dgrad(600, 1, 70, act=1, layout="D"), {THIN}), "n2_cfg5": (Dgrad(4096, 2, 1024, act=0), {THIN}),
              "k4096": (Dgrad(600, 8, 4096, act=2), {THIN}), "k4097": (Dgrad(600, 8, 4097, act=2), {BIG})}
for name, (c, e) in THIN_DGRAD.items():
    case(f"thin_dgrad_{name}", c, e, sim=c.M * c.K <= 700 * 128)

# gnf_linear_wgrad: launch_gemm_auto(N, K, M, split-K): output width K <= 32 -> Skinny; N <= 32 and K > 64 -> Short; K <= 64 -> Mid;
# else Big.  Reduction rows M: one tile, 63 / 64 / 65 (partial tiles), ~20000 (split over slices)
WG_TILES = {"skinny": (40, 32, SKINNY), "mid33": (40, 33, MID), "mid64": (40, 64, MID), "big": (40, 65, BIG),
            "short": (32, 65, SHORT), "n33_big": (33, 65, BIG), "n32_mid": (32, 64, MID)}
for tname, (N, K, t) in WG_TILES.items():
    for M in (1, 63, 64, 65, 20000):
        case(f"wgrad_{tname}_m{M}", Wgrad(M, N, K, extra=3 if M % 2 else 0), {t}, sim=M <= 65)
case("wgrad_m0", Wgrad(0, 40, 65, extra=3), set(), sim=True)
case("wgrad_m0_dense", Wgrad(0, 40, 65), set(), sim=True)
case("wgrad_111", Wgrad(1, 1, 1), {SKINNY}, sim=True)

# gnf_linear_fwd_splitk: sk_splits(K) = 6 if K / 6 >= 64, K / 64 if K >= 128, else 1 (refused); launch_gemm rounds the slices to
# whole k tiles (K = 400: 5 slices of 80, not 6)
for K in (128, 191, 192, 383, 384, 400, 630):
    case(f"splitk_k{K}", SplitK(1024, 30, K), {SKINNY, SKSUM}, sim=K in (128, 192, 400))
case("splitk_nobias_relu0", SplitK(1500, 32, 630, bias=False, relu=False, extra=5), {SKINNY, SKSUM}, sim=False)
case("splitk_relu0_ldy", SplitK(6300, 30, 630, relu=False, extra=2), {SKINNY, SKSUM})
case("splitk_n1", SplitK(1024, 1, 200, extra=1), {SKINNY, SKSUM}, sim=True)

# gnf_colsum: Q = M / period rows per column; 8 rows per iteration, then the remainder
for period in (1, 2, 63):
    for Q in (1, 7, 8, 9, 8 * 5 + 3, 3000):
        M = Q * period
        case(f"colsum_p{period}_q{Q}", Colsum(M, 37, period, extra=3), {COLSUM}, sim=M <= 400)
case("colsum_p_eq_m", Colsum(500, 37, 500, extra=1), {COLSUM}, sim=True)
case("colsum_wide", Colsum(20000, 630, 1, extra=2), {COLSUM})
case("colsum_m0", Colsum(0, 37, 3, extra=3), set(), sim=True)


def run_case(c, dev, seed, kind):
    c.fill(dev, kind, seed)
    if dev.device != "cuda":
        return c.run(dev)
    outs = []
    got = routes(launched(lambda: outs.extend(c.run(dev))))
    assert got == c.expect, f"{c.name}: expected {sorted(c.expect)}, launched {sorted(got)}"
    return outs


def check_case(c, dev, seed=0):
    """Integer operands: bit-exact against float64, sentinels intact (and on the GPU: the expected kernels).  Normal operands:
    componentwise error within the bar.  Returns the componentwise error."""
    out, = run_case(c, dev, seed, "int")
    ref, _ = reference(c)
    assert torch.equal(out.t.double(), ref), f"{c.name}: integer operands, max err {float((out.t.double() - ref).abs().max())}"
    check_sentinels(out, False)
    if c.M == 0:
        return 0.
    out, = run_case(c, dev, seed + 1, "randn")
    ref, den = reference(c)
    assert bool(torch.isfinite(out.t).all()), f"{c.name}: non-finite output"
    check_sentinels(out, False)
    e = cw_err(out.t, ref, den)
    op = "thin" if THIN in c.expect else c.op
    print(f"ERR {op} {c.name} {e:.3g}")
    assert e < BAR[op], f"{c.name}: error {e:.3g} over the bar {BAR[op]:.3g}"
    return e


def seed_of(name):
    return sum(map(ord, name))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_gpu(gpu, name):
    check_case(CASES[name], gpu, seed_of(name))


def tile_of(c):
    w = c.N if c.op == "fwd" else c.K
    if w <= 32:
        return TINY if -(-c.M // 128) < 148 else SKINNY
    if c.M <= 32 and w > 64:
        return SHORT
    return MID if w <= 64 else BIG


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n, c in CASES.items() if THIN in c.expect])
def test_gpu_thin_shapes_on_tile_gemm(no_thin, name):
    c = CASES[name]
    saved = c.expect
    c.expect = {tile_of(c)}
    try:
        check_case(c, no_thin, seed_of(name) + 7)
    finally:
        c.expect = saved


@pytest.mark.parametrize("name", [n for n, c in CASES.items() if c.sim])
def test_simulator(sim, name):
    torch.set_num_threads(1)
    check_case(CASES[name], sim, seed_of(name))


# ---------------------------------------------------------------------------------------------------------------------
# refusals and determinism
# ---------------------------------------------------------------------------------------------------------------------
def _refusals(dev):
    ws = dev.lib.gnf_linear_fwd_splitk_workspace_bytes
    assert ws(1023, 30, 630) == 0 and ws(1024, 33, 630) == 0 and ws(1024, 30, 127) == 0
    assert ws(1024, 32, 128) == 2 * 1024 * 32 * 4 and ws(1024, 30, 384) == 6 * 1024 * 32 * 4
    for M, N, K in ((1023, 30, 630), (1024, 33, 630), (1024, 30, 127)):
        X, W, Y = dev.mat(M, K, K, 1.), dev.mat(N, K, K, 1.), dev.mat(M, N, N, SENT)
        work = torch.zeros(6 * M * 32 + 64, device=dev.device)
        assert dev.rc("gnf_linear_fwd_splitk", X.p, K, W.p, K, None, Y.p, N, M, N, K, 0, C.c_void_p(work.data_ptr()), work.numel() * 4) != 0
        assert bool((Y.full == SENT).all())
    M, N, K = 1024, 30, 630
    X, W, Y = dev.mat(M, K, K, 1.), dev.mat(N, K, K, 1.), dev.mat(M, N, N, SENT)
    need = ws(M, N, K)
    work = torch.zeros(need // 4, device=dev.device)
    assert dev.rc("gnf_linear_fwd_splitk", X.p, K, W.p, K, None, Y.p, N, M, N, K, 0, C.c_void_p(work.data_ptr()), need - 1) != 0
    assert bool((Y.full == SENT).all())
    Yc, out = dev.mat(50, 8, 8, 1.), dev.mat(7, 8, 8, SENT)
    assert dev.rc("gnf_colsum", Yc.p, 8, out.p, 50, 8, 7) != 0                  # M % period != 0
    assert bool((out.full == SENT).all())


@pytest.mark.gpu
def test_gpu_refusals(gpu):
    _refusals(gpu)


def test_simulator_refusals(sim):
    _refusals(sim)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n in CASES if n.startswith("splitk")])
def test_gpu_splitk_is_deterministic(gpu, name):
    """Partial tiles summed in a fixed order: two calls on the same operands give the same bits."""
    c = CASES[name]
    c.fill(gpu, "randn", 5)
    a = c.run(gpu)[0].full.clone()
    b = c.run(gpu)[0].full
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))


# ---------------------------------------------------------------------------------------------------------------------
# gnf_pack_rows / gnf_unpack_rows / gnf_unpack_vec: bit equality with a torch gather / scatter
# ---------------------------------------------------------------------------------------------------------------------
def _pack_case(dev, with_mask, with_perm):
    R, N, K = 37, 50, 29
    g = torch.Generator().manual_seed(R + 2 * with_mask + with_perm)
    W, dWp, src = torch.randn(N, K, generator=g), torch.randn(R, K, generator=g), torch.randn(R, generator=g)
    mask = (torch.rand(N, K, generator=g) < .6).float() * torch.randn(N, K, generator=g) if with_mask else None
    perm = torch.randperm(N, generator=g)[:R].int() if with_perm else None
    rows = perm.long() if with_perm else torch.arange(R)
    on = (lambda t: None if t is None else t.to(dev.device))
    Wd, dWpd, srcd, maskd, permd = (on(t) for t in (W, dWp, src, mask, perm))
    ptr = (lambda t: None if t is None else C.c_void_p(t.data_ptr()))

    out = torch.full((R * K + 1,), SENT, device=dev.device)
    dev.call("gnf_pack_rows", ptr(Wd), ptr(maskd), ptr(permd), ptr(out), R, K)
    want = W[rows] * mask[rows] if with_mask else W[rows]
    dW = torch.full((N * K + 1,), SENT, device=dev.device)
    dev.call("gnf_unpack_rows", ptr(dWpd), ptr(maskd), ptr(permd), ptr(dW), R, N, K)
    want_dW = torch.zeros(N, K)
    want_dW[rows] = dWp * mask[rows] if with_mask else dWp
    dst = torch.full((N + 1,), SENT, device=dev.device)
    dev.call("gnf_unpack_vec", ptr(srcd), ptr(permd), ptr(dst), R, N)
    want_v = torch.zeros(N)
    want_v[rows] = src
    for got, ref, n in ((out, want, R * K), (dW, want_dW, N * K), (dst, want_v, N)):
        got = got.cpu()
        assert torch.equal(got[:n].view(torch.int32), ref.reshape(-1).view(torch.int32)), "differs from the torch gather / scatter"
        assert float(got[n]) == SENT, "element past the end written"


@pytest.mark.gpu
@pytest.mark.parametrize("with_perm", [False, True], ids=["no_perm", "perm"])
@pytest.mark.parametrize("with_mask", [False, True], ids=["no_mask", "mask"])
def test_gpu_pack_unpack(gpu, with_mask, with_perm):
    _pack_case(gpu, with_mask, with_perm)


@pytest.mark.parametrize("with_perm", [False, True], ids=["no_perm", "perm"])
@pytest.mark.parametrize("with_mask", [False, True], ids=["no_mask", "mask"])
def test_simulator_pack_unpack(sim, with_mask, with_perm):
    _pack_case(sim, with_mask, with_perm)


# ---------------------------------------------------------------------------------------------------------------------
# power trace: t = tr((I + alpha A o A)^p) - d and dA = gt 2 alpha p A o (B^(p-1))^T, both sides of the d = 64 switch
# ---------------------------------------------------------------------------------------------------------------------
ALPHA, GT = .5, .75
PT_CASES = [(d, p) for d in (1, 2, 63, 64, 65, 128, 129) for p in (0, 1, 2, 3, 4, 5, 7, 8, 13, d) if p != d or d > 13]
PT_GPU = PT_CASES + [(784, 34)]
PT_SIM = PT_CASES


def pt_A(d, p, device):
    """Row sums of alpha A o A near 4 / p: the entries of B^p stay below ~e^4 whatever p, and one power more or less moves t by
    about 4 / p of itself."""
    g = torch.Generator().manual_seed(1000 * d + p)
    return (torch.randn(d, d, generator=g) * (4. / (ALPHA * d * max(p, 1))) ** .5).to(device)


def pt_reference(A, p, short=0):
    """float64 t and dA, the chain `short` powers short."""
    A = A.double()
    d = A.shape[0]
    B = torch.eye(d, dtype=torch.float64, device=A.device) + ALPHA * A * A
    t = float(torch.linalg.matrix_power(B, p - short).diagonal().sum()) - d
    q = p - 1 - short
    dA = GT * 2 * ALPHA * p * A * torch.linalg.matrix_power(B, q).t() if p >= 1 and q >= 0 else torch.zeros_like(A)
    return t, dA


def pt_bar(d, p):
    """Per power (at least two) and per term of the products' sums (at least 64): see the module docstring."""
    return BAR["pt"] * max(p, 2) * max(d, 64)


def pt_expect(d, p, bwd):
    if d <= 64:
        return {PT_BWD if bwd else PT_FWD}
    chain = p - 1 if bwd else p
    if bwd and p == 0:
        return set()
    return {BUILD_B} | ({PT_BWD_SAVED} if bwd else set()) | ({BIG} if chain >= 2 else set())


def pt_errors(t, dA, d, p):
    t_ref, dA_ref = pt_reference(pt_A(d, p, "cpu"), p)
    e_t = abs(t - t_ref) / (d + abs(t_ref))
    if p == 0:
        assert bool((dA == 0).all()), "p = 0: dA must be zero"
        return e_t, 0.
    return e_t, float((dA.cpu().double() - dA_ref).norm() / dA_ref.norm())


def run_pt(dev, name, expect, *args):
    if dev.device != "cuda":
        return dev.call(name, *args)
    got = routes(launched(lambda: dev.call(name, *args)))
    assert got == expect, f"{name}: expected {sorted(expect)}, launched {sorted(got)}"


def _power_trace(dev, d, p, saved):
    A = pt_A(d, p, dev.device)
    ptr = (lambda t: C.c_void_p(t.data_ptr()))
    t = torch.full((2,), SENT, device=dev.device)
    dA = torch.full((d * d + 1,), SENT, device=dev.device)
    gt = torch.tensor([GT], device=dev.device)
    if saved:
        Gm = torch.full((d * d + 1,), SENT, device=dev.device)
        run_pt(dev, "gnf_power_trace_fwd_save", {PT_SAVE}, ptr(A), d, ALPHA, p, ptr(t), ptr(Gm))
        run_pt(dev, "gnf_power_trace_bwd_saved", {PT_BWD_SAVED}, ptr(A), ptr(Gm), d, ALPHA, p, ptr(gt), ptr(dA))
        assert float(Gm[d * d]) == SENT
    else:
        need = dev.lib.gnf_power_trace_workspace_bytes(d)
        work = torch.full((need // 4,), NAN, device=dev.device)
        run_pt(dev, "gnf_power_trace_fwd", pt_expect(d, p, False), ptr(A), d, ALPHA, p, ptr(t), ptr(work), need)
        work.fill_(NAN)
        run_pt(dev, "gnf_power_trace_bwd", pt_expect(d, p, True), ptr(A), d, ALPHA, p, ptr(gt), ptr(dA), ptr(work), need)
    assert float(t[1]) == SENT and float(dA[d * d]) == SENT, "element past the end written"
    e_t, e_dA = pt_errors(float(t[0]), dA[:d * d].view(d, d), d, p)
    print(f"ERR pt{'_saved' if saved else ''} d{d}_p{p} t {e_t:.3g} dA {e_dA:.3g}")
    bar = pt_bar(d, p)
    assert e_t < bar and e_dA < bar, f"d {d} p {p}: t error {e_t:.3g}, dA error {e_dA:.3g} (bar {bar:.3g})"


def _power_trace_refusals(dev):
    A = torch.zeros(65 * 65, device=dev.device)
    t, dA, gt = (torch.zeros(65 * 65, device=dev.device) for _ in range(3))
    ptr = (lambda x: C.c_void_p(x.data_ptr()))
    assert dev.rc("gnf_power_trace_fwd_save", ptr(A), 65, ALPHA, 3, ptr(t), ptr(dA)) != 0
    for d in (65, 129):
        need = dev.lib.gnf_power_trace_workspace_bytes(d)
        assert need == 5 * d * d * 4
        work = torch.zeros(need // 4, device=dev.device)
        assert dev.rc("gnf_power_trace_fwd", ptr(A), d, ALPHA, 3, ptr(t), ptr(work), need - 1) != 0
        assert dev.rc("gnf_power_trace_bwd", ptr(A), d, ALPHA, 3, ptr(gt), ptr(dA), ptr(work), need - 1) != 0


@pytest.mark.gpu
@pytest.mark.parametrize("d,p", PT_GPU)
def test_gpu_power_trace(gpu, d, p):
    _power_trace(gpu, d, p, saved=False)


@pytest.mark.gpu
@pytest.mark.parametrize("d,p", [(d, p) for d, p in PT_CASES if d <= 64])
def test_gpu_power_trace_saved(gpu, d, p):
    _power_trace(gpu, d, p, saved=True)


@pytest.mark.gpu
def test_gpu_power_trace_refusals(gpu):
    _power_trace_refusals(gpu)


@pytest.mark.parametrize("d,p", PT_SIM)
def test_simulator_power_trace(sim, d, p):
    torch.set_num_threads(1)
    _power_trace(sim, d, p, saved=False)
    if d <= 64:
        _power_trace(sim, d, p, saved=True)


def test_simulator_power_trace_refusals(sim):
    _power_trace_refusals(sim)


# ---------------------------------------------------------------------------------------------------------------------
# the bars against a result that misses a block of terms (CPU, float64)
# ---------------------------------------------------------------------------------------------------------------------
def dropped_block(c):
    """The reduction terms of one k tile of the case's route (split-K: one slice; colsum: one unrolled step of 8 rows per column)."""
    if c.op == "splitk":
        return 0, c.slice_len()
    if c.op == "colsum":
        return 0, 8 * c.period
    tile = next((t for t in c.expect if t in BK), SKINNY)
    return 0, BK[tile]


@pytest.mark.parametrize("name", [n for n, c in CASES.items() if c.M > 0])
def test_bars_reject_a_missing_term_block(name):
    c = CASES[name]
    dev = Dev(None, "cpu")
    c.fill(dev, "randn", seed_of(name) + 1)
    rows = min(c.M, 2048) if c.op in ("fwd", "dgrad", "splitk") else None
    ref, den = reference(c, rows)
    short, _ = reference(c, rows, dropped_block(c))
    op = "thin" if THIN in c.expect else c.op
    e = cw_err(short.float(), ref, den)
    assert e > 10 * BAR[op], f"{name}: a result without terms {dropped_block(c)} is off by {e:.3g}, the bar is {BAR[op]:.3g}"


@pytest.mark.parametrize("d,p", [(d, p) for d, p in PT_GPU if p >= 1])
def test_bars_reject_a_power_trace_one_power_short(d, p):
    A = pt_A(d, p, "cpu")
    t, dA = pt_reference(A, p)
    t1, dA1 = pt_reference(A, p, short=1)
    assert abs(t1 - t) / (d + abs(t)) > 10 * pt_bar(d, p)
    if p >= 2:
        assert float((dA1 - dA).norm() / dA.norm()) > 10 * pt_bar(d, p)


# ---------------------------------------------------------------------------------------------------------------------
# the simulator against the GPU, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
BITWISE = ["fwd_n65_U", "fwd_n32_A", "fwd_m32_n65_A", "fwd_tiny_k65", "fwd_bias63_relu1_n65", "fwd_bias2_relu0_n40",
           "dgrad_k33_act_A", "dgrad_tiny_n17", "dgrad_m32_k65_U", "dgrad_big_n17",
           "thin_fwd_m512", "thin_fwd_k1_dense", "thin_dgrad_n8_act", "thin_dgrad_n1", "splitk_k400", "splitk_n1"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", BITWISE)
def test_simulator_matches_gpu_bitwise(gpu, sim, name):
    """The same operands through the GPU library and the simulator build in one process: every output element and sentinel
    identical (-0 and +0 count as equal: the sign of a zero from fmaxf is not specified)."""
    torch.set_num_threads(1)
    c = CASES[name]
    outs = []
    for dev in (gpu, sim):
        c.fill(dev, "randn", seed_of(name) + 3)
        outs.append((c.run(dev)[0].full.cpu() + 0.).view(torch.int32))
    diff = (outs[0] != outs[1]).nonzero()
    assert diff.numel() == 0, f"{name}: {diff.shape[0]} elements differ, first at {diff[:4].tolist()}"
