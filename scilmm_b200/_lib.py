"""ctypes binding of libscilmm_b200.so (the C-ABI declared in include/scilmm_b200.h).

There is deliberately no fallback: if the library is missing or a call fails, the caller gets an
exception, never a CPU result.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libscilmm_b200.so")

i32, i64, f64 = C.c_int32, C.c_int64, C.c_double
vp = C.c_void_p
pp = C.POINTER(C.c_void_p)


class SlmmError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "scilmm_b200 error %d: %s" % (code, msg))
        self.code = code


class NotPositiveDefiniteError(SlmmError):
    """Raised where sksparse would raise CholmodNotPositiveDefiniteError."""

    def __init__(self, code, msg, column=-1):
        SlmmError.__init__(self, code, msg)
        self.column = column


SIGNATURES = {
    "slmm_last_error": (C.c_char_p, []),
    "slmm_version": (C.c_int, []),
    "slmm_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "slmm_matset_create": (C.c_int, [i32, i32, pp]),
    "slmm_matset_destroy": (C.c_int, [vp]),
    "slmm_matset_upload": (C.c_int, [vp, i32, vp, vp, vp]),
    "slmm_matset_bind_device": (C.c_int, [vp, i32, vp, vp, vp, i64, i32]),
    "slmm_matset_build_tiles": (C.c_int, [vp, i32, vp, vp]),
    "slmm_matset_tile_stats": (C.c_int, [vp, i32, vp]),
    "slmm_matset_tile_cta_profile": (C.c_int, [vp, i32, vp, i32]),
    "slmm_quadform_tiled": (C.c_int, [vp, i32, vp, vp, i32, i32, vp, vp]),
    "slmm_chol_device_perm": (C.c_int, [vp, pp, pp]),
    "slmm_matset_set_row_range": (C.c_int, [vp, i32, i32]),
    "slmm_matset_symmetry_hash": (C.c_int, [vp, i32, vp]),
    "slmm_matset_set_symmetric": (C.c_int, [vp, i32, i32]),
    "slmm_upload_h2d": (C.c_int, [vp, vp, i64, i32]),
    "slmm_upload_h2d_2d": (C.c_int, [vp, i64, vp, i64, i64, i64]),
    "slmm_upload_h2d_on": (C.c_int, [vp, vp, i64, i32, vp]),
    "slmm_upload_h2d_2d_on": (C.c_int, [vp, i64, vp, i64, i64, i64, vp]),
    "slmm_assoc_genotypes": (C.c_int, [vp, i64, i32, i64, i64, vp, i32, vp, vp, vp, vp]),
    "slmm_assoc_colsumsq": (C.c_int, [vp, i64, i32, vp]),
    "slmm_assoc_region_gram": (C.c_int, [vp, i64, i32, i32, vp, vp]),
    "slmm_glmm_working": (C.c_int, [vp, vp, vp, vp, i64, vp, vp]),
    "slmm_assoc_spa": (C.c_int, [vp, i64, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "slmm_blup_spmm": (C.c_int, [vp, i32, vp, vp, vp, vp, i64, i32, vp]),
    "slmm_blup_rowsumsq": (C.c_int, [vp, i32, vp, vp, vp, vp, i64, i32, vp, vp]),
    "slmm_matset_nnz": (C.c_int, [vp, i32, C.POINTER(i64)]),
    "slmm_matset_values": (C.c_int, [vp, i32, pp]),
    "slmm_he_moments": (C.c_int, [vp, vp, i32, i32, vp]),
    "slmm_he_moments_host": (C.c_int, [vp, vp, vp]),
    "slmm_spmm": (C.c_int, [vp, i32, vp, i32, vp]),
    "slmm_spmm_coldot": (C.c_int, [vp, i32, vp, i32, i32, i32, vp]),
    "slmm_spmm_coldot_multi": (C.c_int, [vp, i32, vp, vp, i32, i32, vp, i32, i32, vp]),
    "slmm_matset_pattern_id": (C.c_int, [vp, i32, C.POINTER(i32)]),
    "slmm_quadform_multi": (C.c_int, [vp, i32, vp, vp, i32, i32, i32, vp]),
    "slmm_matset_is_symmetric": (C.c_int, [vp, i32, C.POINTER(i32)]),
    "slmm_matset_validate": (C.c_int, [vp, i32, C.POINTER(i32)]),
    "slmm_device_arrays_equal_i32": (C.c_int, [vp, vp, i64, C.POINTER(i32)]),
    "slmm_quadform_gram_multi": (C.c_int, [vp, i32, vp, vp, i32, vp, i32, i32, i32, vp, vp]),
    "slmm_chol_analyze": (C.c_int, [i32, vp, vp, i32, vp, pp]),
    "slmm_chol_destroy": (C.c_int, [vp]),
    "slmm_chol_stats": (C.c_int, [vp, vp, vp]),
    "slmm_chol_perm": (C.c_int, [vp, vp]),
    "slmm_chol_register_pattern": (C.c_int, [vp, vp, vp, C.POINTER(i32)]),
    "slmm_chol_register_pattern_tri": (C.c_int, [vp, vp, vp, i32, C.POINTER(i32)]),
    "slmm_chol_register_pattern_device": (C.c_int, [vp, vp, vp, i64, i32, C.POINTER(i32)]),
    "slmm_device_csr_is_symmetric": (C.c_int, [vp, vp, vp, i32, C.POINTER(i32)]),
    "slmm_device_pattern_subset": (C.c_int, [vp, vp, vp, vp, i32, C.POINTER(i32)]),
    "slmm_symbolic_entry_map_tri": (C.c_int, [vp, vp, vp, i32, vp]),
    "slmm_chol_add_values": (C.c_int, [vp, i32, vp, f64, i32]),
    "slmm_chol_add_values2": (C.c_int, [vp, i32, vp, f64, vp, f64, i32]),
    "slmm_chol_factorize": (C.c_int, [vp, C.POINTER(i32)]),
    "slmm_chol_logdet": (C.c_int, [vp, C.POINTER(f64)]),
    "slmm_chol_solve": (C.c_int, [vp, vp, i32, i32]),
    "slmm_chol_lmul": (C.c_int, [vp, vp, vp, i32]),
    "slmm_probe_normals": (C.c_int, [vp, i64, i32, i32, C.c_uint64, C.c_uint64]),
    "slmm_chol_export_L": (C.c_int, [vp, vp, vp, vp]),
    "slmm_chol_copy_panels": (C.c_int, [vp, vp]),
    "slmm_chol_aux_begin": (C.c_int, [vp]),
    "slmm_chol_aux_end": (C.c_int, [vp]),
    "slmm_chol_aux_join": (C.c_int, [vp]),
    "slmm_launch_count": (C.c_int, [C.POINTER(i64), i32]),
    "slmm_chol_set_profiling": (C.c_int, [vp, i32]),
    "slmm_chol_set_timeline": (C.c_int, [vp, i32]),
    "slmm_chol_get_timeline": (C.c_int, [vp, i32, C.POINTER(i32), vp, vp]),
    "slmm_chol_get_profile_ex": (C.c_int, [vp, i32, vp, vp, vp]),
    "slmm_chol_get_launch_timeline": (C.c_int, [vp, i32, C.POINTER(i32), vp, vp, vp, vp, vp]),
    "slmm_chol_get_profile": (C.c_int, [vp, vp, vp, vp]),
    "slmm_chol_get_launch_profile": (C.c_int, [vp, i64, C.POINTER(i64), vp, vp, vp, vp]),
    "slmm_symbolic_create": (C.c_int, [i32, vp, vp, i32, vp, pp]),
    "slmm_symbolic_destroy": (C.c_int, [vp]),
    "slmm_symbolic_stats": (C.c_int, [vp, vp, vp]),
    "slmm_symbolic_arrays": (C.c_int, [vp] + [vp] * 12),
    "slmm_symbolic_entry_map": (C.c_int, [vp, vp, vp, vp]),
    "slmm_ibd_build": (C.c_int, [i32, vp, vp, pp]),
    "slmm_ibd_sizes": (C.c_int, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i32)]),
    "slmm_ibd_copy_L": (C.c_int, [vp, vp, vp, vp]),
    "slmm_ibd_copy_DF": (C.c_int, [vp, vp, vp]),
    "slmm_ibd_copy_A": (C.c_int, [vp, vp, vp, vp]),
    "slmm_ibd_destroy": (C.c_int, [vp]),
    "slmm_gemm_selftest_ex": (C.c_int, [i32, i32, i32, vp, i64, vp, i64, vp, i64, i32, i32]),
    "slmm_gemm_selftest": (C.c_int, [i32, i32, i32, vp, vp, vp, i32, i32, C.POINTER(C.c_float)]),
}

_lib = None


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def check(code, column=None):
    if code == 0:
        return
    msg = lib().slmm_last_error().decode("utf-8", "replace")
    if code == 3:
        raise NotPositiveDefiniteError(code, msg, -1 if column is None else column)
    raise SlmmError(code, msg)


def np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)
