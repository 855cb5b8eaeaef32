"""ctypes binding of libgnf_sm100.so (C-ABI declared in include/gnf.h).

The product path has exactly one backend: the sm_100a CUDA library built in-tree by
``build.py`` / ``__graft_entry__.build()``.  If it is missing, every op raises — there is no
CPU or eager-PyTorch fallback.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libgnf_sm100.so"
LIB_PATH = os.path.join(_HERE, LIB_NAME)

GNF_MAX_LAYERS = 8
GATE_TABLE, GATE_GUMBEL, GATE_NOISER = 0, 1, 2
IMP_RAW, IMP_SOFT, IMP_HARD_SOFT, IMP_HARD_SQ = 0, 1, 2, 3

_lib = None
# True only while tests/emu/sim_hook.py has swapped in the host SIMT-simulator build of the same kernels (CPU tensors): the
# argument checks then accept CPU tensors.  Nothing in the product sets it.
_SIMULATOR = False


class GateT(C.Structure):
    _fields_ = [("mode", C.c_int32), ("temperature", C.c_float), ("seed", C.c_uint64), ("offset", C.c_uint64),
                ("noise1", C.c_void_p), ("noise2", C.c_void_p), ("offset_dev", C.c_void_p)]


class MlpT(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("dims", C.c_int32 * (GNF_MAX_LAYERS + 1)),
                ("W", C.c_void_p * GNF_MAX_LAYERS), ("b", C.c_void_p * GNF_MAX_LAYERS)]


class AdamTensorT(C.Structure):
    _fields_ = [("param", C.c_void_p), ("grad", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
                ("numel", C.c_int64)]


class MlpGradT(C.Structure):
    _fields_ = [("dW", C.c_void_p * GNF_MAX_LAYERS), ("db", C.c_void_p * GNF_MAX_LAYERS)]


_P, _I, _F, _SZ = C.c_void_p, C.c_int, C.c_float, C.c_size_t

_PROTOS = {
    "gnf_version": ([], C.c_int),
    "gnf_last_error": ([], C.c_char_p),
    "gnf_has_device_code": ([], C.c_int),
    "gnf_affine_fwd": ([_P, _P, _I, _P, _P, _P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_affine_bwd": ([_P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_normal_ll_fwd": ([_P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_normal_ll_bwd": ([_P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_power_trace_workspace_bytes": ([_I], _SZ),
    "gnf_power_trace_fwd": ([_P, _I, _F, _I, _P, _P, _SZ, _P], C.c_int),
    "gnf_power_trace_bwd": ([_P, _I, _F, _I, _P, _P, _P, _SZ, _P], C.c_int),
    "gnf_power_trace_fwd_save": ([_P, _I, _F, _I, _P, _P, _P], C.c_int),
    "gnf_power_trace_bwd_saved": ([_P, _P, _I, _F, _I, _P, _P, _P], C.c_int),
    "gnf_linear_fwd": ([_P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _P], C.c_int),
    "gnf_linear_dgrad": ([_P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _P], C.c_int),
    "gnf_linear_wgrad": ([_P, _I, _P, _I, _P, _I, _I, _I, _I, _P], C.c_int),
    "gnf_linear_fwd_tc": ([_P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _I, _P], C.c_int),
    "gnf_linear_dgrad_tc": ([_P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _P], C.c_int),
    "gnf_linear_wgrad_tc": ([_P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _P], C.c_int),
    "gnf_linear_wgrad_bias_tc": ([_P, _I, _P, _I, _P, _I, _P, _I, _I, _I, _P], C.c_int),
    "gnf_split_tf32": ([_P, _I, _P, _P, _I, _I, _I, _P], C.c_int),
    "gnf_linear_fwd_tc_ps": ([_P, _I, _P, _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _P], C.c_int),
    "gnf_linear_dgrad_tc_ps": ([_P, _I, _P, _P, _I, _P, _I, _P, _I, _I, _I, _I, _P], C.c_int),
    "gnf_colsum": ([_P, _I, _P, _I, _I, _I, _P], C.c_int),
    "gnf_pack_rows": ([_P, _P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_unpack_rows": ([_P, _P, _P, _P, _I, _I, _I, _P], C.c_int),
    "gnf_unpack_vec": ([_P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_dag_importance": ([_P, _I, _I, _F, _P, _P, _P], C.c_int),
    "gnf_dag_bias_table": ([_P, _I, _P, _P, _I, _I, _I, _P], C.c_int),
    "gnf_dag_bias_table_bwd": ([_P, _P, _I, _P, _I, _I, _I, _P], C.c_int),
    "gnf_dag_l1_fwd": ([_P, _P, C.POINTER(GateT), _P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _P], C.c_int),
    "gnf_dag_l1_wgrad": ([_P, _I, _P, _P, C.POINTER(GateT), _P, _I, _I, _I, _I, _P], C.c_int),
    "gnf_dag_l1_dgrad": ([_P, _I, _P, _I, _P, _P, C.POINTER(GateT), _P, _P, _I, _I, _I, _P], C.c_int),
    "gnf_dag_l1_fwd_save": ([_P, _P, C.POINTER(GateT), _P, _I, _P, _I, _P, _I, _P, _P, _P, _I, _I, _I, _I, _P], C.c_int),
    "gnf_dag_l1_fwd_cond": ([_P, _P, C.POINTER(GateT), _P, _I, _P, _I, _I, _P, _I, _P, _I, _P, _P, _P, _I, _I, _I, _I, _P], C.c_int),
    "gnf_dag_l1_bias_sums": ([_P, _I, _P, _P, _I, _I, _I, _I, _I, _P], C.c_int),
    "gnf_dag_l1_wgrad_saved": ([_P, _I, _P, _P, _I, _I, _I, _I, _P], C.c_int),
    "gnf_dag_l1_dgrad_saved": ([_P, _I, _P, _I, _P, _P, _P, _P, _I, _I, _I, _P], C.c_int),
    "gnf_linear_fwd_splitk_workspace_bytes": ([_I, _I, _I], _SZ),
    "gnf_linear_fwd_splitk": ([_P, _I, _P, _I, _P, _P, _I, _I, _I, _I, _I, _P, _SZ, _P], C.c_int),
    "gnf_dag_bias_table_ld": ([_P, _I, _P, _P, _I, _I, _I, _I, _P], C.c_int),
    "gnf_linear_fwd_tc_ps_tb": ([_P, _I, _P, _P, _I, _P, _I, _I, _P, _I, _I, _I, _I, _I, _P], C.c_int),
    "gnf_linear_fwd_tc_cond": ([_P, _I, _P, _P, _I, _P, _I, _I, _P, _I, _I, _P, _I, _I, _I, _I, _I, _I, _P], C.c_int),
    "gnf_dag_gate_planes": ([_P, _P, C.POINTER(GateT), _P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_dag_l1_reduce_saved": ([_P, _P, _P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_nll_loss_work_floats": ([_I], _SZ),
    "gnf_nll_loss_fwd": ([_P, _P, _P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_nll_loss_bwd": ([_P, _P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_peer_alloc": ([_SZ, C.POINTER(C.c_void_p)], C.c_int),
    "gnf_peer_free": ([_P], C.c_int),
    "gnf_peer_export": ([_P, C.c_char_p], C.c_int),
    "gnf_peer_import": ([C.c_char_p, C.POINTER(C.c_void_p)], C.c_int),
    "gnf_peer_close": ([_P], C.c_int),
    "gnf_peer_flag_bytes": ([], _SZ),
    "gnf_peer_allreduce_avg": ([C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _I, _I, C.c_longlong, _P], C.c_int),
    "gnf_dag_embed_fwd": ([_P, _P, C.POINTER(GateT), _P, _P, _P, _I, _I, _I, _P], C.c_int),
    "gnf_dag_embed_bwd": ([_P, _I, _P, _P, C.POINTER(GateT), _P, _P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_dag_finish_dA": ([_P, _P, _P, _I, _I, _P], C.c_int),
    "gnf_dag_dump_noise": ([C.POINTER(GateT), _P, _P, _I, _I, _P], C.c_int),
    "gnf_umnn_workspace_bytes": ([C.POINTER(MlpT)], _SZ),
    "gnf_umnn_saved_floats_per_node_row": ([C.POINTER(MlpT)], _SZ),
    "gnf_umnn_fwd": ([_P, _P, C.POINTER(MlpT), _I, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P, _SZ, _P], C.c_int),
    "gnf_umnn_invert": ([_P, _P, C.POINTER(MlpT), _I, _P, _P, _P, _I, _F, _F, _I, _P, _SZ, _P], C.c_int),
    "gnf_umnn_bwd_workspace_bytes": ([C.POINTER(MlpT)], _SZ),
    "gnf_umnn_bwd": ([_P, _P, C.POINTER(MlpT), _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(MlpGradT), _I, _I,
                      _P, _SZ, _P], C.c_int),
    "gnf_umnn_tc_workspace_bytes": ([C.POINTER(MlpT)], _SZ),
    "gnf_umnn_fwd_tc": ([_P, _P, C.POINTER(MlpT), _I, _P, _P, _P, _P, _P, _P, _I, _I, _P, _SZ, _P], C.c_int),
    "gnf_umnn_lw_saved_floats": ([C.POINTER(MlpT), _I, _I, _I], _SZ),
    "gnf_umnn_lw_workspace_bytes": ([C.POINTER(MlpT), _I, _I, _I], _SZ),
    "gnf_umnn_fwd_lw": ([_P, _P, C.POINTER(MlpT), _I, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _SZ, _P], C.c_int),
    "gnf_umnn_bwd_lw": ([_P, _P, C.POINTER(MlpT), _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(MlpGradT), _I, _I, _I,
                         _P, _SZ, _P], C.c_int),
    "gnf_umnn_tc3_workspace_bytes": ([C.POINTER(MlpT), _I], _SZ),
    "gnf_umnn_tc3_saved_floats": ([C.POINTER(MlpT), _I, _I], _SZ),
    "gnf_umnn_bwd_tc3_workspace_bytes": ([C.POINTER(MlpT), _I, _I], _SZ),
    "gnf_umnn_bwd_tc3": ([_P, _P, C.POINTER(MlpT), _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(MlpGradT), _I, _I,
                          _P, _SZ, _P], C.c_int),
    "gnf_umnn_fwd_tc3": ([_P, _P, C.POINTER(MlpT), _I, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _SZ, _P], C.c_int),
    "gnf_linear_wgrad_rw_workspace_bytes": ([_I, _I], _SZ),
    "gnf_linear_wgrad_rw": ([_P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _P, _SZ, _P], C.c_int),
    "gnf_tc_gemm_plan": ([_I, _I, _I, _I, _I, _P, _P], C.c_int),
    "gnf_tc_selftest": ([_P, _P, _P, _I, _I, _I, _P], C.c_int),
    "gnf_reverse_cols": ([_P, _P, _I, _I, _P], C.c_int),
    "gnf_broadcast_rows": ([_P, _P, _I, _I, _I, _I, _P], C.c_int),
    "gnf_counter_add": ([_P, C.c_uint64, _P], C.c_int),
    "gnf_adam_step": ([C.POINTER(AdamTensorT), _I, _P, _F, _F, _F, _F, _F, _P], C.c_int),
    "gnf_dag_loss_fwd": ([_P, _I, _P, _P, _P, _P, _P, _P, _P], C.c_int),
    "gnf_dag_loss_bwd": ([_P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P], C.c_int),
}

EXPORTED_SYMBOLS = tuple(_PROTOS)


def _bind(lib):
    for name, (argtypes, restype) in _PROTOS.items():
        fn = getattr(lib, name)          # AttributeError if the library lacks a declared symbol
        fn.argtypes = argtypes
        fn.restype = restype
    return lib


def load_library(path=LIB_PATH):
    """dlopen + bind every symbol of include/gnf.h.  Does not touch the GPU."""
    if not os.path.isfile(path):
        raise RuntimeError(
            f"{LIB_NAME} not found at {path}: the CUDA library is the only backend of this package "
            f"(no CPU / eager fallback). Build it with `python -c 'import __graft_entry__ as g; g.build()'`.")
    return _bind(C.CDLL(path))


def lib():
    global _lib
    if _lib is None:
        _lib = load_library()
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().gnf_last_error()
        raise RuntimeError(f"libgnf error {rc}: {msg.decode() if msg else '?'}")


def stream_ptr():
    if _SIMULATOR:
        return None
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def require(t, name, dtype=torch.float32):
    """Argument contract of every op: CUDA, contiguous, fp32 (SURVEY.md §8b error convention)."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not _SIMULATOR and not t.is_cuda:
        raise TypeError(f"{name}: expected a CUDA tensor (this package has no CPU path)")
    if not t.is_contiguous():
        raise TypeError(f"{name}: expected a contiguous tensor")
    return t
