"""ctypes binding of librri_b200.so -- the C-ABI declared in include/rri_b200.h.

There is NO CPU fallback: if the shared library is missing, or no sm_100 device is present when an
engine is created, the call raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'librri_b200.so')

RRI_F32, RRI_F64 = 0, 1
RRI_MATH_IEEE, RRI_MATH_TF32 = 0, 1
RRI_ORDER_RRI, RRI_ORDER_HALS = 0, 1
RRI_MASK_NONE, RRI_MASK_REAL, RRI_MASK_U8 = 0, 1, 2
FLAG_ZERO_T, FLAG_ZERO_W, FLAG_UNBOUNDED, FLAG_NONFINITE = 1, 2, 4, 8
FLAG_NOT_IMPLEMENTED = 16


class RriParams(C.Structure):
    """rri_params_t (include/rri_b200.h)"""
    _fields_ = [('reg_w_l1', C.c_double), ('reg_w_l2', C.c_double), ('reg_t_l1', C.c_double),
                ('reg_t_l2', C.c_double), ('ub_w', C.c_double), ('ub_t', C.c_double), ('eps', C.c_double),
                ('fix_W', C.c_int32), ('fix_T', C.c_int32), ('simplex_T', C.c_int32), ('sp_refresh_every', C.c_int32)]


# every symbol include/rri_b200.h declares: name -> (restype, argtypes)
_vp, _i32, _i64, _cp = C.c_void_p, C.c_int32, C.c_int64, C.c_char_p
SYMBOLS = {
    'rri_version': (_cp, []),
    'rri_last_error': (_cp, []),
    'rri_create': (C.c_int, [C.POINTER(_vp), _i64, _i64, _i32, _i32, _i32, _i32, _i32]),
    'rri_destroy': (C.c_int, [_vp]),
    'rri_set_comm': (C.c_int, [_vp, _vp, _i32, _i32, _cp]),
    'rri_nccl_unique_id': (C.c_int, [C.c_char * 128, _cp]),
    'rri_nccl_comm_create': (C.c_int, [C.POINTER(_vp), C.c_char * 128, _i32, _i32, _i32, _cp]),
    'rri_nccl_comm_destroy': (C.c_int, [_vp]),
    'rri_peer_export': (C.c_int, [_vp, C.c_char * 64]),
    'rri_peer_import': (C.c_int, [_vp, _cp, _i32, _i32]),
    'rri_peer_enable': (C.c_int, [_vp, _i32]),
    'rri_peer_close': (C.c_int, [_vp]),
    'rri_set_transpose_storage': (C.c_int, [_vp, _vp, _i64]),
    'rri_bind': (C.c_int, [_vp, _vp, _i64, _vp, _i32, _i64, _vp]),
    'rri_x_operand_bits': (C.c_int, [_vp, C.POINTER(_i32)]),
    'rri_bind_csr': (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    'rri_bind_csr_zero': (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp]),
    'rri_spmm': (C.c_int, [_vp, _i32, _vp, _i64, _vp, _i64, _i32, _vp]),
    'rri_sweeps': (C.c_int, [_vp, _vp, _vp, _i32, C.POINTER(RriParams), C.POINTER(_i32), _vp]),
    'rri_topics': (C.c_int, [_vp, _vp, _vp, _i32, _i32, C.POINTER(RriParams), C.POINTER(_i32), _vp]),
    'rri_topic_sums': (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double), _vp]),
    'rri_objective': (C.c_int, [_vp, _vp, _vp, C.POINTER(C.c_double), _vp]),
    'rri_objective_contraction': (C.c_int, [_vp, _vp, _vp, _i32, C.POINTER(C.c_double), _vp]),
    'rri_partials_T': (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    'rri_project_rows_simplex': (C.c_int, [_vp, _vp, _i64, _i64, C.c_double, _vp]),
    'rri_cache_trim': (C.c_int, [_i32]),
    'rri_stats': (C.c_int, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    'rri_profile_kernel': (C.c_int, [_vp, _i32, _vp, _vp, _i32, C.POINTER(C.c_float), _vp]),
    'rri_contract_x': (C.c_int, [_vp, _i32, _vp, _i64, _i32, _vp, _vp]),
    'rri_gemm_nt': (C.c_int, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i32, _i64, _vp]),
}

_lib = None


class RriError(RuntimeError):
    pass


def load():
    """Load librri_b200.so (built in-tree by `__graft_entry__.build()` / `make -C rri_nmf_b200/csrc`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RriError('%s not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                       '(there is no CPU fallback)' % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)            # AttributeError if the ABI and the header diverge
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RriError(load().rri_last_error().decode('utf-8', 'replace'))


def nccl_library_path():
    """Path of the NCCL that torch bundles (so the engine and torch share one libnccl.so.2)."""
    try:
        import nvidia.nccl
        for base in nvidia.nccl.__path__:
            p = os.path.join(base, 'lib', 'libnccl.so.2')
            if os.path.isfile(p):
                return p
    except Exception:
        pass
    return None
