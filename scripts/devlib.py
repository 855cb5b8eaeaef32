"""scripts/ only: load the GNF_DEVTOOLS build (libgnf_sm100_dev.so: traces, ablation switches, tiling overrides) in place of
the product library.  The package itself never loads it."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gnf_b200 as G  # noqa: E402

_P, _I = C.c_void_p, C.c_int
_F, _SZ = C.c_float, C.c_size_t
DEV_PROTOS = {
    "gnf_tc_gemm_set_tma": ([_I], C.c_int),
    "gnf_tc_gemm_set_tile": ([_I, _I], C.c_int),
    "gnf_tc_gemm_set_fold": ([_I], C.c_int),
    "gnf_tc_gemm_set_trace": ([_P], C.c_int),
    "gnf_dag_l1_set_resident": ([_I], C.c_int),
    "gnf_linear_wgrad_rw_set_trace": ([_P], C.c_int),
    "gnf_tc_probe": ([_I, _I, _P, _P], C.c_int),
    "gnf_tc_set_trace": ([_P], C.c_int),
    "gnf_tc_gemm_set_v2": ([_I], C.c_int),
    "gnf_umnn_tc3_set_trace": ([_P], C.c_int),
    "gnf_umnn_tc3_set_debug": ([_I], C.c_int),
    "gnf_linear_set_thin": ([_I], C.c_int),
}


def install():
    path = os.path.join(ROOT, "graphical-normalizing-flows_b200", "libgnf_sm100_dev.so")
    if not os.path.isfile(path):
        raise RuntimeError("build the dev library first: python graphical-normalizing-flows_b200/build.py --dev")
    lib = G._lib._bind(C.CDLL(path))
    for name, (argtypes, restype) in DEV_PROTOS.items():
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = argtypes, restype
    G._lib._lib = lib
    return lib
