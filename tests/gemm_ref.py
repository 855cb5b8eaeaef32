"""Shared harness of the GEMM tests against float64 (test_gpu_tc_gemm_f64.py, test_ffma_gemm_f64.py): strided operands inside
sentinel-filled buffers, the sentinel check, the kernels a call launched, and the componentwise error metric.  Every helper
takes CPU tensors too, so that the same cases run through the host SIMT-simulator build of the kernels (tests/emu)."""
import ctypes as C

import pytest
import torch

import gnf_b200 as G

SENT = -777.0                      # outputs: every element the kernel must not write
NAN = float("nan")                 # operand padding: a read shows up as NaN


def pad4(n):
    return (n + 3) // 4 * 4


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


def launched(fn):
    """Names of the CUDA kernels fn launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events()]


def assert_engines(names, expect, engines):
    """The kernels of `engines` (substrings of kernel names) that ran are exactly `expect`."""
    found = {k for k in engines if any(k in n for n in names)}
    assert found == set(expect), f"expected {sorted(expect)}, launched {sorted(found)}: {names}"


class Mat:
    """A [rows, cols] matrix of row stride ld inside a flat buffer filled with `fill`, its first element `off` floats past a
    256-byte aligned base, one spare row after the last: padding columns and the spare row keep `fill` unless written."""

    def __init__(self, rows, cols, ld, fill, off=0, device="cuda"):
        self.rows, self.cols, self.ld = rows, cols, ld
        self.buf = torch.full((off + (rows + 1) * ld,), fill, device=device)
        self.full = self.buf[off:].view(rows + 1, ld)
        self.t = self.full[:rows, :cols]

    @property
    def p(self):
        return C.c_void_p(self.full.data_ptr())

    def set(self, v):
        self.t.copy_(v)
        return self


def check_sentinels(out, zero_ok):
    """Columns [cols, round_up(cols, 4)) unchanged or exactly 0 (zero_ok: kernels that store 16-byte pieces), every column
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
