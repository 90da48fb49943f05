"""ctypes binding of the C-ABI declared in include/sparsh_b200.h (lib/libsparsh_b200.so).

This is plumbing only: every call goes straight to the CUDA library.  There is no CPU fallback anywhere in this
package — if the shared library is missing or no GPU is present the calls raise.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsparsh_b200.so")

c_int_p = C.POINTER(C.c_int)
c_dbl_p = C.POINTER(C.c_double)

SPARSH_OK = 0
SPARSH_ERR_NOT_CONVERGED = 3
KIND_SCALAR, KIND_STREAM, KIND_VECTOR, KIND_DICT, KIND_PATTERN = 0, 1, 2, 3, 4


class SparshError(RuntimeError):
    pass


class LevelDesc(C.Structure):
    _fields_ = [("nrow", C.c_int), ("nnz", C.c_int), ("rowptr", c_int_p), ("colindex", c_int_p), ("val", c_dbl_p),
                ("diag", c_dbl_p), ("p_ncol", C.c_int), ("p_nnz", C.c_int), ("p_rowptr", c_int_p),
                ("p_colindex", c_int_p), ("p_val", c_dbl_p), ("total_colors", C.c_int), ("color_count", c_int_p)]


class Params(C.Structure):
    _fields_ = [("omega", C.c_double), ("pre_sweeps", C.c_int), ("post_sweeps", C.c_int), ("use_graph", C.c_int),
                ("coarse_mode", C.c_int), ("smoother", C.c_int), ("halo_mode", C.c_int)]


# every symbol include/sparsh_b200.h declares: (restype, argtypes)
_vp, _vpp, _sz, _i, _d = C.c_void_p, C.POINTER(C.c_void_p), C.c_size_t, C.c_int, C.c_double
SIGNATURES = {
    "sparsh_init": (_i, [_i]),
    "sparsh_shutdown": (_i, []),
    "sparsh_last_error": (C.c_char_p, []),
    "sparsh_set_stream": (_i, [_vp]),
    "sparsh_get_stream": (_i, [_vpp]),
    "sparsh_sync": (_i, []),
    "sparsh_device_name": (_i, [C.c_char_p, _sz, c_int_p]),
    "sparsh_launch_count": (C.c_longlong, []),
    "sparsh_launch_count_reset": (None, []),
    "sparsh_launch_count_add": (None, [C.c_longlong]),
    "sparsh_malloc": (_i, [_sz, _vpp]),
    "sparsh_free": (_i, [_vp]),
    "sparsh_host_alloc": (_i, [_sz, _vpp]),
    "sparsh_host_free": (_i, [_vp]),
    "sparsh_memcpy_h2d": (_i, [_vp, _vp, _sz]),
    "sparsh_memcpy_d2h": (_i, [_vp, _vp, _sz]),
    "sparsh_memcpy_d2d": (_i, [_vp, _vp, _sz]),
    "sparsh_fill": (_i, [_vp, _sz, _d]),
    "sparsh_matrix_create": (_i, [_i, _i, _i, c_int_p, c_int_p, c_dbl_p, c_dbl_p, _vpp]),
    "sparsh_matrix_create_transpose": (_i, [_i, _i, _i, c_int_p, c_int_p, c_dbl_p, _vpp]),
    "sparsh_matrix_update_values": (_i, [_vp, _vp, _vp]),
    "sparsh_matrix_fetch": (_i, [_vp, c_int_p, c_int_p, c_dbl_p, c_dbl_p]),
    "sparsh_matrix_destroy": (_i, [_vp]),
    "sparsh_matrix_dims": (_i, [_vp, c_int_p, c_int_p, c_int_p]),
    "sparsh_matrix_kernel": (_i, [_vp, c_int_p, c_int_p, c_int_p]),
    "sparsh_matrix_force_kernel": (_i, [_vp, _i, _i]),
    "sparsh_matrix_kernel_name": (_i, [_vp, _i, C.c_char_p, _sz]),
    "sparsh_matrix_pattern_stats": (_i, [_vp, c_int_p, c_int_p, c_int_p, c_dbl_p]),
    "sparsh_matrix_pattern_mask_stats": (_i, [_vp, c_int_p, c_dbl_p]),
    "sparsh_matrix_transfer_info": (_i, [_vp, c_int_p, c_int_p, c_dbl_p]),
    "sparsh_pattern_masks": (_i, [_i, c_int_p, c_dbl_p, c_int_p, _vp]),
    "sparsh_pattern_encode": (_i, [_i, _i, _i, c_int_p, c_int_p, c_dbl_p, c_dbl_p, _vp, c_dbl_p, c_int_p, c_int_p, c_int_p,
                                   c_int_p]),
    "sparsh_dict_encode": (_i, [_i, _i, _i, c_int_p, c_int_p, c_dbl_p, _vp, c_dbl_p, c_int_p, c_int_p, c_int_p]),
    "sparsh_galerkin_rap": (_i, [_i, c_int_p, c_int_p, c_dbl_p, _i, c_int_p, c_int_p, c_dbl_p, _vpp, c_int_p]),
    "sparsh_galerkin_rap_next": (_i, [_vp, _i, c_int_p, c_int_p, c_dbl_p, _vpp, c_int_p]),
    "sparsh_rap_fetch": (_i, [_vp, c_int_p, c_int_p, c_dbl_p]),
    "sparsh_rap_destroy": (_i, [_vp]),
    "sparsh_spmv": (_i, [_vp, _vp, _vp]),
    "sparsh_spmv_dot": (_i, [_vp, _vp, _vp, _vp]),
    "sparsh_residual": (_i, [_vp, _vp, _vp, _vp]),
    "sparsh_residual_norm": (_i, [_vp, _vp, _vp, c_dbl_p]),
    "sparsh_jacobi": (_i, [_vp, _vp, _vp, _vp, _d, _i]),
    "sparsh_mc_sor": (_i, [_vp, c_int_p, _i, _vp, _vp, _d, _i]),
    "sparsh_restrict": (_i, [_vp, _vp, _vp]),
    "sparsh_prolong_add": (_i, [_vp, _vp, _vp]),
    "sparsh_residual_restrict": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "sparsh_jacobi_zero": (_i, [_vp, _vp, _d, _vp]),
    "sparsh_dot": (_i, [_sz, _vp, _vp, c_dbl_p]),
    "sparsh_nrm2": (_i, [_sz, _vp, c_dbl_p]),
    "sparsh_dot_device": (_i, [_sz, _vp, _vp, _vp]),
    "sparsh_axpy": (_i, [_sz, _d, _vp, _vp]),
    "sparsh_axpby": (_i, [_sz, _d, _vp, _d, _vp]),
    "sparsh_axpbypcz": (_i, [_sz, _d, _vp, _d, _vp, _d, _vp]),
    "sparsh_params_default": (None, [C.POINTER(Params)]),
    "sparsh_hierarchy_create": (_i, [_i, C.POINTER(LevelDesc), C.POINTER(Params), _vpp]),
    "sparsh_hierarchy_destroy": (_i, [_vp]),
    "sparsh_hierarchy_refresh": (_i, [_vp, _vp, _vp]),
    "sparsh_hierarchy_nlevels": (_i, [_vp]),
    "sparsh_hierarchy_level": (_i, [_vp, _i, _vpp, _vpp, _vpp]),
    "sparsh_hierarchy_coarse_solve": (_i, [_vp, _vp, _vp]),
    "sparsh_hierarchy_vcycle": (_i, [_vp, _vp, _vp, _i, _i]),
    "sparsh_hierarchy_amg_solve": (_i, [_vp, _vp, _vp, _d, _i, c_dbl_p, c_int_p]),
    "sparsh_hierarchy_pcg": (_i, [_vp, _vp, _vp, _d, _i, c_dbl_p, c_int_p]),
    "sparsh_hierarchy_pbicgstab": (_i, [_vp, _vp, _vp, _d, _i, c_dbl_p, c_int_p]),
    "sparsh_cg": (_i, [_vp, _vp, _vp, _d, _i, c_dbl_p, c_int_p]),
    "sparsh_bicgstab": (_i, [_vp, _vp, _vp, _d, _i, c_dbl_p, c_int_p]),
    "sparsh_hierarchy_pgmres": (_i, [_vp, _vp, _vp, _d, _i, _i, c_dbl_p, c_int_p]),
    "sparsh_gmres": (_i, [_vp, _vp, _vp, _d, _i, _i, c_dbl_p, c_int_p]),
    "sparsh_hierarchy_solve_host": (_i, [_vp, _i, _vp, _vp, _d, _i, c_dbl_p, c_int_p]),
    "sparsh_hierarchy_vcycle_bytes": (_d, [_vp, _i]),
    "sparsh_hierarchy_pcg_enqueue": (_i, [_vp, _vp, _vp, _d, _i, _vp, _vp]),
    "sparsh_hierarchy_pbicgstab_enqueue": (_i, [_vp, _vp, _vp, _d, _i, _vp, _vp]),
    "sparsh_hierarchy_amg_solve_enqueue": (_i, [_vp, _vp, _vp, _d, _i, _vp, _vp]),
    # multi-GPU
    "sparsh_dist_get_unique_id": (_i, [C.c_char_p]),
    "sparsh_dist_init": (_i, [C.c_char_p, _i, _i]),
    "sparsh_dist_finalize": (_i, []),
    "sparsh_dist_info": (_i, [c_int_p, c_int_p]),
    "sparsh_dist_hierarchy_create": (_i, [_i, _vp, _i, _vp, c_int_p, c_int_p, _vp, _vpp]),
    "sparsh_dist_hierarchy_destroy": (_i, [_vp]),
    "sparsh_dist_local_rows": (_i, [_vp, _i, c_int_p]),
    "sparsh_dist_level_matrix": (_i, [_vp, _i, _vpp]),
    "sparsh_dist_spmv": (_i, [_vp, _i, _vp, _vp]),
    "sparsh_dist_vcycle": (_i, [_vp, _vp, _vp, _i, _i]),
    "sparsh_dist_pcg": (_i, [_vp, _vp, _vp, _d, _i, c_dbl_p, c_int_p]),
    "sparsh_dist_allgather_rows": (_i, [c_dbl_p, c_int_p, _i, c_dbl_p, _i]),
    "sparsh_dist_amg_solve": (_i, [_vp, _vp, _vp, _d, _i, c_dbl_p, c_int_p]),
    "sparsh_dist_pbicgstab": (_i, [_vp, _vp, _vp, _d, _i, c_dbl_p, c_int_p]),
}


class DistOpDesc(C.Structure):
    """sparsh_dist_op_desc (include/sparsh_b200.h)"""
    _fields_ = [("nrow", C.c_int), ("ncol_local", C.c_int), ("nhalo", C.c_int), ("nnz", C.c_int),
                ("rowptr", c_int_p), ("colindex", c_int_p), ("val", c_dbl_p), ("diag", c_dbl_p),
                ("n_send", C.c_int), ("send_rank", c_int_p), ("send_ptr", c_int_p), ("send_idx", c_int_p),
                ("n_recv", C.c_int), ("recv_rank", c_int_p), ("recv_ptr", c_int_p),
                ("interior_begin", C.c_int), ("interior_end", C.c_int)]

_lib = None


def load():
    """dlopen the CUDA library (no GPU needed for this step) and type every entry point."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SparshError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export what the header declares
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, allow_not_converged=False):
    if rc == SPARSH_OK or (allow_not_converged and rc == SPARSH_ERR_NOT_CONVERGED):
        return rc
    raise SparshError(f"sparsh_b200 error {rc}: {load().sparsh_last_error().decode(errors='replace')}")


def ip(a):
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_int_p)


def dp(a):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_dbl_p)
