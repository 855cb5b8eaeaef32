"""The conditioner's tensor-core GEMM engine (csrc/tc_gemm.cu) against float64, route by route, at its shape limits.

Every case calls the C-ABI directly with explicit leading dimensions and asserts, with torch.profiler, which kernel ran:
  * tc_gemm_kernel   -- the planned-tile engine: operand layouts that the host code stages by TMA or by cp.async of 16, 8 or 4
                        bytes (the kernel name does not show which), every tile width and split-K factor of the weight gradient;
  * tc_gemm2_kernel  -- engine v2 of the pre-split forward / dgrad, on both sides of every band of g2_eligible, with a plain, a
                        periodic (fold 1) and a strided-table bias and with / without the dgrad ReLU mask;
  * tc_wgrad2_kernel -- the weight-gradient engine on both sides of every threshold of w2_eligible, into a wider dW (lddw > K), and
                        its in-kernel bias-gradient row sum;
  * colsum_kernel    -- the bias-gradient fallback of gnf_linear_wgrad_bias_tc;
  * split_tf32_kernel -- bit for bit against a numpy emulation of round-to-nearest TF32.
The development library's switches (gnf_tc_gemm_set_v2 / _set_tma / _set_tile) force the routes the product never picks by itself.

Checks of every case:
  * integer operands in [-4, 4]: every product and partial sum is exact in TF32 and fp32, so every route must reproduce float64
    bit for bit (indexing: periodic bias row m % period, table stride, straddling 16-byte pieces, split-K accumulation);
  * normal operands against float64, componentwise: max |C - ref| / (|A| |B|^T + |bias|) (a relative norm hides the cancellation
    of the long weight-gradient reductions).  3xTF32 bar: max(4 x the same error of the FFMA engine on the same case, floor);
    single-pass TF32: 2e-3 relative L2 (the project's TF32 bar);
  * output columns [N, round_up(N, 4)) are unchanged or exactly 0, every column past them and the row after the last one are
    unchanged (sentinel -777); dW columns [K, lddw) are unchanged.  Operand padding holds NaN, so a kernel that reads it fails.

Bars, measured on a B200 at its 1000 W power limit (componentwise errors of normal operands):
  * FFMA engine (the multiplier's baseline): up to 4e-7 on forward and dgrad, up to 1.2e-7 on the weight gradients, up to 4.2e-8
    on db (gnf_colsum);
  * 3xTF32 at the default fold: largest 5.6e-7 (forward, v1 at K = 64 with a bias table); at most 2.2x the FFMA error wherever
    the FFMA error exceeds 1e-7.  With one product per output (K = 1, N = 1, M = 1) the error is that of one 3xTF32 product
    through the truncating accumulator: up to 3.6e-7 measured (the bound is ~1.1e-6), while the FFMA engine rounds once;
  * FLOOR = 8e-7 on the three GEMMs (1.4x the largest 3xTF32 error measured), 1e-7 on db (the engine sums dY in plain fp32:
    largest 4.4e-8);
  * single-pass TF32: 1.2e-3 relative L2 at most, bar 2e-3.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import gnf_b200 as G

SENT = -777.0                      # outputs: every element the kernel must not write
GARBAGE = 1234.5                   # padding columns of a bias table: finite, so a read shows up as a wrong value
NAN = float("nan")                 # operand padding: a read shows up as NaN
V1, V2, W2, CS, SPLIT = "tc_gemm_kernel", "tc_gemm2_kernel", "tc_wgrad2_kernel", "colsum_kernel", "split_tf32_kernel"
ENGINES = (V1, V2, W2, CS, SPLIT)
FLOOR = {"fwd": 8e-7, "dgrad": 8e-7, "wgrad": 8e-7, "db": 1e-7}
TF32_BAR = 2e-3


def pad4(n):
    return (n + 3) // 4 * 4


# ---------------------------------------------------------------------------------------------------------------------
# harness
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def poison():
    """Returns a function that NaN-fills free blocks in the small (<= 1 MB) and the large pool of the caching allocator and
    releases them again (no empty_cache): the next torch.empty calls -- workspaces, saved planes, outputs -- start non-finite."""
    def fill():
        held = [torch.full((n,), float("nan"), device="cuda") for n in [64, 1024, 16384, 65536, 262144] * 4]
        held += [torch.full((n,), float("nan"), device="cuda") for n in (1 << 20, 1 << 22, 1 << 24, 1 << 26, 1 << 28)]
        del held
    fill()
    yield fill
    G.ops.set_gemm_mode("ffma")


@pytest.fixture
def devlib():
    """The package routed through libgnf_sm100_dev.so, whose process-global switches force a kernel; reset on the way out."""
    dev_so = os.path.join(os.path.dirname(G._lib.LIB_PATH), "libgnf_sm100_dev.so")
    assert os.path.isfile(dev_so), "engine overrides are development-build knobs: __graft_entry__.build() builds libgnf_sm100_dev.so"
    lib = C.CDLL(dev_so)
    for name, args in (("gnf_tc_gemm_set_v2", [C.c_int]), ("gnf_tc_gemm_set_tma", [C.c_int]), ("gnf_tc_gemm_set_tile", [C.c_int, C.c_int])):
        getattr(lib, name).argtypes = args
        getattr(lib, name).restype = C.c_int
    product = G._lib.lib()
    G._lib._lib = G._lib._bind(lib)
    try:
        yield lib
    finally:
        lib.gnf_tc_gemm_set_v2(1)
        lib.gnf_tc_gemm_set_tma(1)
        lib.gnf_tc_gemm_set_tile(0, 0)
        G._lib._lib = product


def call(name, *args):
    lib = G._lib.lib()
    rc = getattr(lib, name)(*args, G._lib.stream_ptr())
    assert rc == 0, f"{name}: {rc} {lib.gnf_last_error()}"


def launched(fn):
    """Names of the CUDA kernels fn launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events()]


def assert_engines(names, expect):
    found = {k for k in ENGINES if any(k in n for n in names)}
    assert found == set(expect), f"expected {sorted(expect)}, launched {sorted(found)}: {names}"


class Mat:
    """A [rows, cols] matrix of row stride ld inside a flat buffer filled with `fill`, its first element `off` floats past a
    256-byte aligned base, one spare row after the last: padding columns and the spare row keep `fill` unless written."""

    def __init__(self, rows, cols, ld, fill, off=0):
        self.rows, self.cols, self.ld = rows, cols, ld
        self.buf = torch.full((off + (rows + 1) * ld,), fill, device="cuda")
        self.full = self.buf[off:].view(rows + 1, ld)
        self.t = self.full[:rows, :cols]

    @property
    def p(self):
        return C.c_void_p(self.full.data_ptr())

    def set(self, v):
        self.t.copy_(v)
        return self


def check_sentinels(out, zero_ok):
    """Columns [cols, round_up(cols, 4)) unchanged or exactly 0 (zero_ok: forward / dgrad store 16-byte pieces), every column
    past them and the spare row unchanged."""
    c4 = pad4(out.cols) if zero_ok else out.cols
    tail = out.full[:out.rows, out.cols:c4]
    assert bool(((tail == SENT) | (tail == 0)).all()), f"columns [{out.cols}, {c4}): {tail[(tail != SENT) & (tail != 0)][:8].tolist()}"
    rest = out.full[:out.rows, c4:]
    assert bool((rest == SENT).all()), f"columns >= {c4} written: {rest[rest != SENT][:8].tolist()}"
    assert bool((out.full[out.rows:] == SENT).all()), "row past the last one written"


def cw_err(got, ref, den):
    """max |got - ref| / den (0 where both are 0; a non-zero difference over a zero denominator is infinite)."""
    d = (got.double() - ref).abs()
    return float(torch.where(d == 0, torch.zeros_like(d), d / den).max()) if d.numel() else 0.


def rel_l2(got, ref):
    return float((got.double() - ref).norm() / ref.norm().clamp_min(1e-300))


def operands(kind, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "int":
        return lambda *s: torch.randint(-4, 5, s, device="cuda", generator=g).float()
    return lambda *s: torch.randn(*s, device="cuda", generator=g)


def split_weight(W, ld=None):
    """gnf_split_tf32 of W.t into [N, ld] hi / lo (ld: K rounded up to 4 floats by default)."""
    N, K = W.rows, W.cols
    ld = ld or pad4(K)
    hi, lo = Mat(N, ld, ld, NAN), Mat(N, ld, ld, NAN)
    call("gnf_split_tf32", W.p, W.ld, hi.p, lo.p, ld, N, K)
    return hi, lo


# ---------------------------------------------------------------------------------------------------------------------
# the three operations: operands, the tensor-core call, the FFMA call, the float64 reference
# ---------------------------------------------------------------------------------------------------------------------
class Fwd:
    """Y = act(X W^T + bias[m % period]) through gnf_linear_fwd_tc (entry 'tc', passes 1 / 3), gnf_linear_fwd_tc_ps ('ps') or
    gnf_linear_fwd_tc_ps_tb ('tb': bias table of row stride ldt with GARBAGE in its padding columns)."""
    op = "fwd"

    def __init__(self, M, N, K, entry="ps", passes=3, bias=True, period=1, relu=True, ldx=None, ldw=None, ldy=None, ldt=None, off=0):
        self.M, self.N, self.K, self.entry, self.passes, self.bias, self.period, self.relu = M, N, K, entry, passes, bias, period, relu
        self.ldx, self.ldw, self.ldy = ldx or pad4(K), ldw or pad4(K), ldy or pad4(N)
        self.ldt, self.off = ldt or N, off
        if entry != "tc":
            assert passes == 3

    def fill(self, kind, seed):
        r = operands(kind, seed)
        M, N, K = self.M, self.N, self.K
        self.X = Mat(M, K, self.ldx, NAN, self.off).set(r(M, K))
        self.W = Mat(N, K, self.ldw, NAN, self.off).set(r(N, K))
        self.B = None
        if self.bias:
            self.B = Mat(self.period, N, self.ldt, GARBAGE if self.entry == "tb" else NAN).set(r(self.period, N))
        if self.entry != "tc":
            self.hi, self.lo = split_weight(self.W)

    def run(self):
        M, N, K = self.M, self.N, self.K
        self.Y = Mat(M, N, self.ldy, SENT, self.off)
        bp = self.B.p if self.B is not None else None
        if self.entry == "tc":
            call("gnf_linear_fwd_tc", self.X.p, self.ldx, self.W.p, self.ldw, bp, self.period, self.Y.p, self.ldy, M, N, K, int(self.relu), self.passes)
        elif self.entry == "ps":
            assert self.ldt == N
            call("gnf_linear_fwd_tc_ps", self.X.p, self.ldx, self.hi.p, self.lo.p, self.hi.ld, bp, self.period, self.Y.p, self.ldy, M, N, K, int(self.relu))
        else:
            call("gnf_linear_fwd_tc_ps_tb", self.X.p, self.ldx, self.hi.p, self.lo.p, self.hi.ld, bp, self.ldt, self.period, self.Y.p, self.ldy,
                 M, N, K, int(self.relu))
        return [self.Y]

    def ffma(self):
        Y = Mat(self.M, self.N, self.N, SENT)
        b = Mat(self.period, self.N, self.N, NAN).set(self.B.t) if self.B is not None else None
        call("gnf_linear_fwd", self.X.p, self.ldx, self.W.p, self.ldw, b.p if b else None, self.period, Y.p, self.N, self.M, self.N, self.K, int(self.relu))
        return [Y]

    def reference(self):
        X, W = self.X.t.double(), self.W.t.double()
        ref, den = X @ W.t(), X.abs() @ W.abs().t()
        if self.B is not None:
            rows = self.B.t.double()[torch.arange(self.M, device="cuda") % self.period]
            ref, den = ref + rows, den + rows.abs()
        return [(ref.clamp_min(0) if self.relu else ref, den)]


class Dgrad:
    """dX = (dY W) * (act > 0) through gnf_linear_dgrad_tc (entry 'tc', passes 1 / 3) or gnf_linear_dgrad_tc_ps ('ps');
    act = None: the plain product."""
    op = "dgrad"

    def __init__(self, M, N, K, entry="ps", passes=3, act=True, lddy=None, ldw=None, ldact=None, lddx=None, off=0):
        self.M, self.N, self.K, self.entry, self.passes, self.act = M, N, K, entry, passes, act
        self.lddy, self.ldw, self.ldact, self.lddx, self.off = lddy or pad4(N), ldw or pad4(K), ldact or pad4(K), lddx or pad4(K), off

    def fill(self, kind, seed):
        r = operands(kind, seed)
        M, N, K = self.M, self.N, self.K
        self.dY = Mat(M, N, self.lddy, NAN, self.off).set(r(M, N))
        self.W = Mat(N, K, self.ldw, NAN, self.off).set(r(N, K))
        self.A = Mat(M, K, self.ldact, NAN, self.off).set(r(M, K)) if self.act else None
        if self.entry == "ps":
            self.hi, self.lo = split_weight(self.W)

    def run(self):
        M, N, K = self.M, self.N, self.K
        self.dX = Mat(M, K, self.lddx, SENT, self.off)
        ap, lda = (self.A.p, self.ldact) if self.A is not None else (None, 0)
        if self.entry == "tc":
            call("gnf_linear_dgrad_tc", self.dY.p, self.lddy, self.W.p, self.ldw, ap, lda, self.dX.p, self.lddx, M, N, K, self.passes)
        else:
            call("gnf_linear_dgrad_tc_ps", self.dY.p, self.lddy, self.hi.p, self.lo.p, self.hi.ld, ap, lda, self.dX.p, self.lddx, M, N, K)
        return [self.dX]

    def ffma(self):
        dX = Mat(self.M, self.K, self.K, SENT)
        ap, lda = (self.A.p, self.ldact) if self.A is not None else (None, 0)
        call("gnf_linear_dgrad", self.dY.p, self.lddy, self.W.p, self.ldw, ap, lda, dX.p, self.K, self.M, self.N, self.K)
        return [dX]

    def reference(self):
        dY, W = self.dY.t.double(), self.W.t.double()
        ref, den = dY @ W, dY.abs() @ W.abs()
        if self.A is not None:
            mask = (self.A.t > 0).double()
            ref, den = ref * mask, den * mask
        return [(ref, den)]


class Wgrad:
    """dW = dY^T X (gnf_linear_wgrad_tc, passes 1 / 3) into the first K columns of [N, lddw]; bias=True: gnf_linear_wgrad_bias_tc,
    db = the column sums of dY too."""
    op = "wgrad"

    def __init__(self, M, N, K, passes=3, bias=False, lddy=None, ldx=None, lddw=None, off=0):
        self.M, self.N, self.K, self.passes, self.bias = M, N, K, passes, bias
        self.lddy, self.ldx, self.lddw, self.off = lddy or pad4(N), ldx or pad4(K), lddw or K, off
        assert not bias or passes == 3

    def fill(self, kind, seed):
        r = operands(kind, seed)
        self.dY = Mat(self.M, self.N, self.lddy, NAN, self.off).set(r(self.M, self.N))
        self.X = Mat(self.M, self.K, self.ldx, NAN, self.off).set(r(self.M, self.K))

    def run(self):
        M, N, K = self.M, self.N, self.K
        self.dW = Mat(N, K, self.lddw, SENT)
        if not self.bias:
            call("gnf_linear_wgrad_tc", self.dY.p, self.lddy, self.X.p, self.ldx, self.dW.p, self.lddw, M, N, K, self.passes)
            return [self.dW]
        self.db = Mat(1, N, N, SENT)
        call("gnf_linear_wgrad_bias_tc", self.dY.p, self.lddy, self.X.p, self.ldx, self.dW.p, self.lddw, self.db.p, M, N, K)
        return [self.dW, self.db]

    def ffma(self):
        dW = Mat(self.N, self.K, self.K, SENT)
        call("gnf_linear_wgrad", self.dY.p, self.lddy, self.X.p, self.ldx, dW.p, self.K, self.M, self.N, self.K)
        if not self.bias:
            return [dW]
        db = Mat(1, self.N, self.N, SENT)
        call("gnf_colsum", self.dY.p, self.lddy, db.p, self.M, self.N, 1)
        return [dW, db]

    def reference(self):
        dY, X = self.dY.t.double(), self.X.t.double()
        out = [(dY.t() @ X, dY.abs().t() @ X.abs())]
        if self.bias:
            out.append((dY.sum(0, keepdim=True), dY.abs().sum(0, keepdim=True)))
        return out


def check_case(case, expect, poison, seed=0, tag=""):
    """Integer operands: bit-exact, the expected kernel (and no other engine) launched, sentinels intact.  Normal operands:
    componentwise error against float64 within the bar.  Returns the errors and bars of the normal-operand run."""
    zero_ok = case.op != "wgrad"
    case.fill("int", seed)
    poison()
    outs = []
    assert_engines(launched(lambda: outs.extend(case.run())), expect)
    for out, (ref, _) in zip(outs, case.reference()):
        assert torch.equal(out.t.double(), ref), f"{tag}: integer operands, max err {float((out.t.double() - ref).abs().max())}"
        check_sentinels(out, zero_ok and out is outs[0])
    if case.M == 0:
        return None
    case.fill("randn", seed + 1)
    refs = case.reference()
    ffma = [cw_err(o.t, r, d) for o, (r, d) in zip(case.ffma(), refs)]
    poison()
    outs = case.run()
    names = [case.op, "db"][:len(outs)]
    for name, out, (ref, den), ef in zip(names, outs, refs, ffma):
        assert bool(torch.isfinite(out.t).all()), f"{tag} {name}: non-finite output"
        check_sentinels(out, zero_ok and name != "db")
        if getattr(case, "passes", 3) == 3:
            e, bar = cw_err(out.t, ref, den), max(4 * ef, FLOOR[name])
        else:
            e, bar = rel_l2(out.t, ref), TF32_BAR
        assert e < bar, f"{tag} {name} on {sorted(expect)}: error {e:.3g} over the bar {bar:.3g} (FFMA engine: {ef:.3g})"


# ---------------------------------------------------------------------------------------------------------------------
# 1. gnf_linear_fwd_tc: the planned-tile engine, TMA and cp.async staging
# ---------------------------------------------------------------------------------------------------------------------
# route -> (leading-dimension padding, base offset in floats).  The staging path is not observable from outside the kernel: the
# test asserts tc_gemm_kernel ran, and the layouts are chosen by the host code's rules (make_operand_map, vec_width): TMA needs
# 16-byte aligned bases and rows; ldx odd or a base one float off stages with 4-byte cp.async, two floats off with 8-byte cp.async
FWD_LAYOUTS = {"tma": (4, 0), "cp_async_knob": (4, 0), "ldx_odd": (None, 0), "off2": (2, 2), "off1": (4, 1)}


@pytest.mark.gpu
@pytest.mark.parametrize("bias,relu", [(True, True), (True, False), (False, True), (False, False)], ids=["bias_relu", "bias", "relu", "plain"])
@pytest.mark.parametrize("passes", [1, 3])
@pytest.mark.parametrize("route", list(FWD_LAYOUTS))
def test_fwd_tc_routes(poison, request, route, passes, bias, relu):
    M, N, K = 777, 150, 97
    pad, off = FWD_LAYOUTS[route]
    if pad is None:
        lay = dict(ldx=99, ldw=pad4(K), ldy=pad4(N))
    else:
        lay = dict(ldx=pad4(K) + pad, ldw=pad4(K) + pad, ldy=pad4(N) + pad, off=off)
    if route == "cp_async_knob":
        request.getfixturevalue("devlib").gnf_tc_gemm_set_tma(0)
    check_case(Fwd(M, N, K, entry="tc", passes=passes, bias=bias, relu=relu, **lay), {V1}, poison, seed=passes, tag=f"fwd_tc {route}")


# ---------------------------------------------------------------------------------------------------------------------
# 2. gnf_linear_fwd_tc_ps: both sides of g2_eligible, the same shapes on v1, periodic biases
# ---------------------------------------------------------------------------------------------------------------------
FWD_PS = {                                  # (M, N, K, kernel of the default route, ReLU)
    "m1023": (1023, 256, 128, V1, True), "m1024": (1024, 256, 128, V2, True),
    "n255": (1100, 255, 128, V1, True), "n256": (1100, 256, 128, V2, True),
    "k31": (1100, 256, 31, V1, True), "k32": (1100, 256, 32, V2, True), "k64": (1100, 256, 64, V2, True), "k65": (1100, 256, 65, V1, True),
    "n64_k256": (1100, 64, 256, V2, True), "n65_k256": (1100, 65, 256, V1, True), "n32_k255": (1100, 32, 255, V1, True),
    # N % 4 != 0 into a [M, 632] buffer: the last piece of a row straddles N (without ReLU a bias leaking into the padding
    # columns shows whatever its sign)
    "cfg4_hidden": (6300, 630, 630, V2, True), "cfg4_linear": (6300, 630, 630, V2, False),
}
FWD_PS_CASES = [(s, "default") for s in FWD_PS] + [(s, "v2_off") for s in FWD_PS if FWD_PS[s][3] == V2]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,v2", FWD_PS_CASES)
def test_fwd_tc_ps_routes(poison, request, shape, v2):
    M, N, K, kern, relu = FWD_PS[shape]
    if v2 == "v2_off":
        request.getfixturevalue("devlib").gnf_tc_gemm_set_v2(0)
        kern = V1
    check_case(Fwd(M, N, K, relu=relu), {kern}, poison, seed=M + N + K, tag=f"fwd_tc_ps {shape} {v2}")


@pytest.mark.gpu
@pytest.mark.parametrize("period", [2, 63, 784, 1001, 2100])
@pytest.mark.parametrize("N", [256, 258])
def test_fwd_tc_ps_periodic_bias(poison, N, period):
    """bias [period, N] with bias_ld = N: N % 4 == 0 runs engine v2's table path (folding every k-chunk), N % 4 != 0 the first
    engine's per-element bias tile.  Periods dividing M, not dividing it (1001) and period = M."""
    check_case(Fwd(2100, N, 128, period=period), {V2 if N % 4 == 0 else V1}, poison, seed=period, tag=f"fwd_tc_ps period {period} N {N}")


# ---------------------------------------------------------------------------------------------------------------------
# 3. gnf_linear_fwd_tc_ps_tb: layer 1 of a narrow DAG flow (X = the [B d, 64] plane, bias table [d, ldt > N])
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("v2", ["default", "v2_off"])
@pytest.mark.parametrize("d", [63, 32, 64])
def test_fwd_tc_ps_table(poison, request, d, v2):
    kern = V2
    if v2 == "v2_off":
        request.getfixturevalue("devlib").gnf_tc_gemm_set_v2(0)
        kern = V1
    case = Fwd(100 * d, 630, d, entry="tb", period=d, ldx=64, ldt=632, ldy=632)
    check_case(case, {kern}, poison, seed=d, tag=f"fwd_tc_ps_tb d {d} {v2}")


# ---------------------------------------------------------------------------------------------------------------------
# 4. gnf_linear_dgrad_tc / _tc_ps
# ---------------------------------------------------------------------------------------------------------------------
DGRAD_PS = {                                # (M, N, K) in layer terms: output dX is [M, K], the reduction runs over N
    "wide": (2048, 256, 630, V2), "m1023": (1023, 256, 256, V1),
    "n127": (1100, 127, 256, V1), "n128": (1100, 128, 256, V2),
    "n64": (1100, 64, 256, V2), "n65": (1100, 65, 256, V1),
    "k31": (1100, 256, 31, V1), "k32": (1100, 256, 32, V2), "k64": (1100, 256, 64, V2), "k65": (1100, 256, 65, V1),
    "narrow_dag": (6300, 630, 63, V2),      # input cotangent of DAG layer 1 into the [B d, 64] plane
}
DGRAD_ACTS = {"act": 0, "act_wide": 8, "none": None}     # extra ldact columns past round_up(K, 4)
DGRAD_CASES = [(s, a, "default") for s in DGRAD_PS for a in DGRAD_ACTS] + \
              [(s, a, "v2_off") for s in DGRAD_PS for a in DGRAD_ACTS if DGRAD_PS[s][3] == V2]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,act,v2", DGRAD_CASES)
def test_dgrad_tc_ps_routes(poison, request, shape, act, v2):
    M, N, K, kern = DGRAD_PS[shape]
    if v2 == "v2_off":
        request.getfixturevalue("devlib").gnf_tc_gemm_set_v2(0)
        kern = V1
    extra = DGRAD_ACTS[act]
    case = Dgrad(M, N, K, act=extra is not None, ldact=pad4(K) + (extra or 0), lddx=64 if shape == "narrow_dag" else None)
    check_case(case, {kern}, poison, seed=M + N + K, tag=f"dgrad_tc_ps {shape} {act} {v2}")


@pytest.mark.gpu
@pytest.mark.parametrize("act", [True, False], ids=["act", "none"])
@pytest.mark.parametrize("passes", [1, 3])
@pytest.mark.parametrize("layout", ["tma", "off1"])
def test_dgrad_tc_routes(poison, layout, passes, act):
    M, N, K = 777, 150, 97
    lay = dict(lddy=pad4(N) + 4, ldw=pad4(K) + 4, ldact=pad4(K) + 4, lddx=pad4(K) + 4, off=1 if layout == "off1" else 0)
    check_case(Dgrad(M, N, K, entry="tc", passes=passes, act=act, **lay), {V1}, poison, seed=passes, tag=f"dgrad_tc {layout}")


# ---------------------------------------------------------------------------------------------------------------------
# 5. gnf_linear_wgrad_tc
# ---------------------------------------------------------------------------------------------------------------------
WGRAD = {                                   # (M rows, N weight rows, K input width, 3xTF32 kernel, base offset)
    "small": (1500, 200, 150, V1, 0), "small_off1": (1500, 200, 150, V1, 1),
    "m2047": (2047, 256, 256, V1, 0), "m2048": (2048, 256, 256, W2, 0), "m2048_off1": (2048, 256, 256, V1, 1),
    "n255": (2048, 255, 256, V1, 0),
    "k31": (2048, 256, 31, V1, 0), "k32": (2048, 256, 32, W2, 0), "k64": (2048, 256, 64, W2, 0), "k65": (2048, 256, 65, V1, 0),
    "k255": (2048, 256, 255, V1, 0),
}


@pytest.mark.gpu
@pytest.mark.parametrize("passes", [1, 3])
@pytest.mark.parametrize("shape", list(WGRAD))
def test_wgrad_tc_planned(poison, shape, passes):
    M, N, K, kern, off = WGRAD[shape]
    check_case(Wgrad(M, N, K, passes=passes, off=off), {kern if passes == 3 else V1}, poison, seed=M + N + K,
               tag=f"wgrad_tc {shape} passes {passes}")


WGRAD_TILES = [(3, bn) for bn in (64, 96, 128, 160)] + [(1, bn) for bn in (64, 96, 128, 160, 192, 224, 256)]


@pytest.mark.gpu
@pytest.mark.parametrize("splits", [1, 2, "max"])
@pytest.mark.parametrize("passes,bn", WGRAD_TILES)
def test_wgrad_tc_forced_tiles(poison, devlib, passes, bn, splits):
    """Every tile width and split-K factor 1, 2 and the largest (one split per 8 k-chunks of the 1500-row reduction: 6), read
    back through gnf_tc_gemm_plan."""
    M, N, K = 1500, 200, 150
    devlib.gnf_tc_gemm_set_tile(bn, 1 << 20 if splits == "max" else splits)
    got_bn, got_sp = C.c_int(), C.c_int()
    assert G._lib.lib().gnf_tc_gemm_plan(N, K, M, passes, 1, C.byref(got_bn), C.byref(got_sp)) == 0
    assert (got_bn.value, got_sp.value) == (bn, 6 if splits == "max" else splits)
    check_case(Wgrad(M, N, K, passes=passes), {V1}, poison, seed=bn, tag=f"wgrad_tc bn {bn} splits {splits} passes {passes}")


@pytest.mark.gpu
@pytest.mark.parametrize("v2", ["default", "v2_off"])
def test_wgrad_tc_into_wider_matrix(poison, request, v2):
    """cfg5's layer-1 weight gradient scaled down: dW1[:, :d] written into the [N1, 2d] gradient (lddw > K)."""
    kern = W2
    if v2 == "v2_off":
        request.getfixturevalue("devlib").gnf_tc_gemm_set_v2(0)
        kern = V1
    check_case(Wgrad(4096, 1024, 784, lddw=1568), {kern}, poison, seed=5, tag=f"wgrad_tc lddw 1568 {v2}")


# ---------------------------------------------------------------------------------------------------------------------
# 6. gnf_linear_wgrad_bias_tc
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["rowsum", "colsum", "m0"])
def test_wgrad_bias_tc(poison, shape):
    """db from tc_wgrad2_kernel's row sums (split-K atomics, N = 300: three tile rows), from the colsum fallback, and M = 0:
    dW and db come back as zeros."""
    M, N, K, kern = {"rowsum": (4096, 300, 256, {W2}), "colsum": (1500, 200, 150, {CS, V1}), "m0": (0, 300, 256, set())}[shape]
    check_case(Wgrad(M, N, K, bias=True), kern, poison, seed=N, tag=f"wgrad_bias_tc {shape}")


# ---------------------------------------------------------------------------------------------------------------------
# 7. gnf_split_tf32 against a numpy emulation
# ---------------------------------------------------------------------------------------------------------------------
def rn_tf32(x):
    """float32 -> TF32 grid (10 explicit mantissa bits), round to nearest, ties away from zero; computed in float64."""
    x = np.asarray(x, np.float32).astype(np.float64)
    _, e = np.frexp(np.abs(x))
    ulp = np.ldexp(1.0, e - 11)
    return (np.sign(x) * np.floor(np.abs(x) / ulp + 0.5) * ulp).astype(np.float32)


def split_inputs(N, K, seed):
    """Normal float32 values over 2^-27 .. 2^23 with every rounding case of the 13 dropped bits: ties, one below / above a tie,
    all ones (rounds into the next binade), exact TF32 values and zeros."""
    rng = np.random.default_rng(seed)
    bits = (rng.integers(100, 150, (N, K)).astype(np.uint32) << 23) | rng.integers(0, 1 << 23, (N, K)).astype(np.uint32)
    bits |= rng.integers(0, 2, (N, K)).astype(np.uint32) << 31
    low = rng.choice(np.array([0x1000, 0x0fff, 0x1001, 0x1fff, 0x0000], np.uint32), (N, K))
    pick = rng.random((N, K)) < .5
    bits[pick] = (bits[pick] & ~np.uint32(0x1fff)) | low[pick]
    w = bits.view(np.float32)
    w[rng.random((N, K)) < .02] = 0.
    return w


def test_tf32_emulation():
    """CPU: the emulation itself on hand-made cases."""
    one = np.float32(1.)
    ulp = np.float32(2. ** -10)
    assert rn_tf32(one + ulp / 2) == one + ulp                          # tie: away from zero
    assert rn_tf32(-(one + ulp / 2)) == -(one + ulp)
    assert rn_tf32(np.nextafter(one + ulp / 2, one)) == one             # just below the tie
    assert rn_tf32(np.float32(2.) - np.float32(2. ** -23)) == 2.        # all dropped bits set: next binade
    assert rn_tf32(np.float32(0.)) == 0.
    w = split_inputs(5, 7, 0)
    assert ((rn_tf32(w).view(np.uint32) & 0x1fff) == 0).all()
    assert (np.abs(rn_tf32(w).astype(np.float64) - w) <= np.abs(w) * 2. ** -11).all()


@pytest.mark.gpu
@pytest.mark.parametrize("N,K,ldw,ld", [(37, 33, 33, 36), (37, 33, 40, 44), (1, 1, 1, 4), (300, 256, 260, 256)])
def test_split_tf32_bits(poison, N, K, ldw, ld):
    w = split_inputs(N, K, N + K)
    W = Mat(N, K, ldw, NAN).set(torch.from_numpy(w).cuda())
    poison()
    out = []
    assert_engines(launched(lambda: out.extend(split_weight(W, ld))), {SPLIT})
    hi, lo = out
    hi_ref = rn_tf32(w)
    lo_ref = rn_tf32(w.astype(np.float64) - hi_ref.astype(np.float64))
    for got, ref, name in ((hi, hi_ref, "hi"), (lo, lo_ref, "lo")):
        g = got.t[:, :K].cpu().numpy()
        assert ((g.view(np.uint32) & 0x1fff) == 0).all(), f"{name}: low 13 bits set"
        bad = g.view(np.uint32) != ref.view(np.uint32)
        assert not bad.any(), f"{name}: {bad.sum()} elements differ, e.g. w={w[bad][:4]} got={g[bad][:4]} want={ref[bad][:4]}"
        assert bool((got.full[:N, K:] == 0).all()), f"{name}: padding columns not zero"
        assert bool(torch.isnan(got.full[N]).all()), f"{name}: row past the last one written"


# ---------------------------------------------------------------------------------------------------------------------
# 8. ops._split_weight: an in-place weight update invalidates the cached split
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_split_cache_follows_in_place_update(poison):
    G.ops.set_gemm_mode("tf32x3")
    g = torch.Generator(device="cuda").manual_seed(3)
    X, W = torch.randn(1024, 128, device="cuda", generator=g), torch.randn(256, 128, device="cuda", generator=g)
    b = torch.randn(256, device="cuda", generator=g)
    G.ops.linear_fwd(X, W, b, relu=False)
    W.add_(1)
    Y = G.ops.linear_fwd(X, W, b, relu=False)
    X64, W64 = X.double(), W.double()
    err = cw_err(Y, X64 @ W64.t() + b.double(), X64.abs() @ W64.abs().t() + b.double().abs())
    assert err < FLOOR["fwd"], f"error {err:.3g}: the second call used the split of the old W"


# ---------------------------------------------------------------------------------------------------------------------
# 9. degenerate shapes on every entry point
# ---------------------------------------------------------------------------------------------------------------------
DEGENERATE = {"m0": (0, 40, 36), "m1": (1, 40, 36), "n1": (70, 1, 36), "k1": (70, 40, 1), "k33": (70, 40, 33)}
ENTRIES = {
    "fwd_tc1": lambda M, N, K: (Fwd(M, N, K, entry="tc", passes=1), {V1}),
    "fwd_tc3": lambda M, N, K: (Fwd(M, N, K, entry="tc", passes=3), {V1}),
    "fwd_tc_ps": lambda M, N, K: (Fwd(M, N, K, period=3), {V1}),
    "fwd_tc_ps_tb": lambda M, N, K: (Fwd(M, N, K, entry="tb", period=3, ldt=pad4(N) + 4), {V1}),
    "dgrad_tc1": lambda M, N, K: (Dgrad(M, N, K, entry="tc", passes=1), {V1}),
    "dgrad_tc3": lambda M, N, K: (Dgrad(M, N, K, entry="tc", passes=3), {V1}),
    "dgrad_tc_ps": lambda M, N, K: (Dgrad(M, N, K), {V1}),
    "wgrad_tc1": lambda M, N, K: (Wgrad(M, N, K, passes=1), {V1}),
    "wgrad_tc3": lambda M, N, K: (Wgrad(M, N, K, passes=3), {V1}),
    "wgrad_bias_tc": lambda M, N, K: (Wgrad(M, N, K, bias=True), {CS, V1}),
}


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(DEGENERATE))
@pytest.mark.parametrize("entry", list(ENTRIES))
def test_degenerate_shapes(poison, entry, shape):
    """M = 0 launches nothing and leaves every output untouched, except dW and db, which are documented to come back zero."""
    M, N, K = DEGENERATE[shape]
    case, kern = ENTRIES[entry](M, N, K)
    check_case(case, kern if M > 0 else set(), poison, seed=M + N + K, tag=f"{entry} {shape}")
