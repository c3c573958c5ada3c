"""ctypes binding of libhipgp_b200.so (C ABI declared in include/hipgp_b200.h).

The library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is no CPU fallback and
no alternative backend: if the library is missing or a CUDA device is not present, the product raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libhipgp_b200.so")

F32, F64 = 0, 1
MV_K, MV_CINV, MV_RT, MV_R = 0, 1, 2, 3
SPEC_D, SPEC_D_SQRT, SPEC_DI, SPEC_DI_SQRT = 0, 1, 2, 3
K_SQEXP, K_MATERN12, K_MATERN32, K_MATERN52, K_GNEITING = 0, 1, 2, 3, 4
KXU_POINT, KXU_SEMI_ANALYTIC, KXU_SEMI_MC, KXU_DERIV, KXU_DERIV2 = 0, 1, 2, 3, 4

ITER_CB = C.CFUNCTYPE(None, C.c_int, C.c_void_p, C.c_void_p)

_vp, _i, _i64, _d, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_size_t
_pi64, _pd, _pi = C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int)

# name -> (restype, argtypes); every symbol include/hipgp_b200.h declares
SIGNATURES = {
    "hipgp_last_error": (C.c_char_p, []),
    "hipgp_version": (_i, []),
    "hipgp_plan_create": (_i, [_i, _pi64, _i, _i, C.POINTER(_vp)]),
    "hipgp_plan_destroy": (_i, [_vp]),
    "hipgp_plan_sizes": (_i, [_vp, _pi64, _pi64]),
    "hipgp_plan_embedding": (_i, [_vp, _pi64, _pi64]),
    "hipgp_plan_set_first_row": (_i, [_vp, _vp, _d, _pi64, _vp]),
    "hipgp_plan_spectrum": (_i, [_vp, _i, _vp, _vp]),
    "hipgp_matvec": (_i, [_vp, _i, _vp, _vp, _i64, _vp]),
    "hipgp_matvec_host": (_i, [_vp, _i, _vp, _vp, _i64, _vp]),
    "hipgp_pcg": (_i, [_vp, _vp, _vp, _i64, _i, _d, _i, _pi, _pi, _pd, ITER_CB, _vp, _vp]),
    "hipgp_pcg_begin": (_i, [_vp, _vp, _vp, _i64, _d, _i, _vp]),
    "hipgp_pcg_step": (_i, [_vp, _i, _pi, _pi, _pd, _vp]),
    "hipgp_pcg_host": (_i, [_vp, _vp, _vp, _i64, _i, _d, _i, _pi, _pi, _pd, _vp]),
    "hipgp_pcg_host_pipelined": (_i, [_vp, _vp, _vp, _i64, _i, _d, _i, _i64, _pi, _vp]),
    "hipgp_pcg_host_submit": (_i, [_vp, _vp, _vp, _i64, _i, _d, _i, _i, _vp]),
    "hipgp_pcg_host_wait": (_i, [_vp, _i, _pi]),
    "hipgp_compute_kn": (_i, [_vp, _vp, _vp, _i64, _i, _d, _pi, _vp]),
    "hipgp_vec_dot": (_i, [_i, _vp, _vp, _vp, _i64, _i64, _vp]),
    "hipgp_vec_xr_update": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "hipgp_vec_p_update": (_i, [_i, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "hipgp_kxu": (_i, [_i, _i, _i, _d, _pd, _i, _d, _vp, _i64, _i, _pi64, _vp, _vp, _i, _vp, _vp]),
    "hipgp_kernel_pairwise": (_i, [_i, _i, _i, _d, _pd, _i, _d, _vp, _i64, _vp, _i64, _i, _vp, _i, _vp, _vp]),
    "hipgp_kxu_param_grad": (_i, [_i, _i, _i, _d, _pd, _i, _vp, _i64, _i, _pi64, _vp, _vp, _i64, _vp, _i, _vp, _vp, _vp]),
    "hipgp_doubly_diag": (_i, [_i, _vp, _i64, _i, _d, _pd, _i, _vp, _vp, _vp, _i, _vp, _vp]),
    "hipgp_doubly_diag_param_grad": (_i, [_i, _vp, _i64, _i, _d, _pd, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "hipgp_meanfield_rowstats": (_i, [_i, _vp, _vp, _vp, _i64, _i64, _vp, _vp]),
    "hipgp_meanfield_colstats": (_i, [_i, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    "hipgp_block_lam": (_i, [_i, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _d, _d, _vp, _vp]),
    "hipgp_block_diag_multiply": (_i, [_i, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    "hipgp_block_quadform_grad": (_i, [_i, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp]),
    "hipgp_toeplitz_quadform": (_i, [_vp, _vp, _vp, _i64, _d, _vp, _vp]),
    "hipgp_rt_column_grad": (_i, [_vp, _vp, _vp, _i64, _d, _vp, _vp]),
    "hipgp_plan_set_slab": (_i, [_vp, _i, _i]),
    "hipgp_slab2_sizes": (_i, [_vp, _pi64, _pi64]),
    "hipgp_slab2_stage_a": (_i, [_vp, _vp, _vp, _vp]),
    "hipgp_slab2_stage_b": (_i, [_vp, _i, _vp, _vp]),
    "hipgp_slab2_stage_b_chunk": (_i, [_vp, _i, _vp, _i, _vp]),
    "hipgp_plan_set_slab_chunks": (_i, [_vp, _i]),
    "hipgp_slab2_peer_alloc": (_i, [_vp, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), _vp, _vp]),
    "hipgp_slab2_peer_open": (_i, [_vp, _vp, _vp]),
    "hipgp_slab2_peer_set": (_i, [_vp, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "hipgp_slab2_push_a": (_i, [_vp, _vp, _vp]),
    "hipgp_slab2_push_b": (_i, [_vp, _i, _i, _vp]),
    "hipgp_slab2_finish": (_i, [_vp, _vp, _vp]),
    "hipgp_slab2_push_only": (_i, [_vp, _i, _vp]),
    "hipgp_slab2_stage_c": (_i, [_vp, _vp, _vp, _vp]),
    "hipgp_plan_device_bytes": (_i, [_vp, C.POINTER(_sz)]),
    "hipgp_plan_launch_count": (_i, [_vp, _pi64]),
    "hipgp_plan_profile": (_i, [_vp, _i]),
    "hipgp_plan_profile_read": (_i, [_vp, _i, _pd, _pi64, _i]),
}


def declare(lib):
    """Attach prototypes; raises AttributeError if a declared symbol is not exported."""
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libhipgp_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "from the repo root; there is no CPU fallback." % LIB_PATH)
        _lib = declare(C.CDLL(LIB_PATH))
    return _lib


def check(lib, status):
    if status != 0:
        raise RuntimeError("hipgp_b200: " + lib.hipgp_last_error().decode())
