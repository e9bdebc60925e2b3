"""ctypes binding of liblmcma_b200.so (include/lmcma_b200.h).  Fails loudly when the library is
missing or a call returns an error: there is no CPU / PyTorch fallback anywhere in this package."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblmcma_b200.so")

OK, ERR_ARG, ERR_CUDA, ERR_STATE, ERR_NOMEM = 0, -1, -2, -3, -4
RNG_PHILOX, RNG_HANSEN, RNG_INJECT = 0, 1, 2
MAP_F32, MAP_U8 = 0, 1

F64 = {"xmean": 0, "sigma": 1, "s": 2, "best_f": 3, "consts": 4, "weights": 5, "Nj": 6, "Lj": 7}
F32 = {"X": 0, "pc": 1, "V": 2, "P": 3, "fit": 4, "fit_sorted": 5, "prev_fit": 6, "Z": 7}
I32 = {"t": 0, "vec": 1, "arindex": 2, "rank": 3, "itr": 4, "live": 5, "counteval": 6, "ncoll": 7, "nsamp": 8}
I32_LAUNCH = 9
# the fields of LMCMA_B200_I32_LAUNCH in order (LMCMA_B200_LAUNCH_*)
LAUNCH_FIELDS = ("sampler", "smp_nv", "smp_spec", "smp_threads", "smp_RBW", "smp_CW", "smp_R", "smp_rows_qw", "smp_rows_rl",
                 "smp_kc", "smp_stages", "upd_nvb", "upd_rmax", "upd_rows_in_smem", "upd_gram", "upd_warps",
                 "upd_sweep_warps", "coef_elems", "rank_threads", "rank_ftile", "rank_tile_sorted", "progressive", "overlap")
SAMPLERS = ("narrow", "wide", "rows")


class LmcmaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("lmcma_b200 error %d: %s" % (code, msg))
        self.code = code


class Config(C.Structure):
    _fields_ = [("n", C.c_int32), ("lambda_", C.c_int32), ("m", C.c_int32), ("batch", C.c_int32),
                ("sigma0", C.c_double), ("seed", C.c_int64), ("rng", C.c_int32), ("device", C.c_int32),
                ("record_z", C.c_int32), ("pop_offset", C.c_int32), ("pop_count", C.c_int32),
                ("reserved", C.c_int32 * 5)]


class Endpoints(C.Structure):
    _fields_ = [("start", C.c_float * 3), ("goal", C.c_float * 3)]


class Objective(C.Structure):
    _fields_ = [("waypoints", C.c_int32), ("w_len", C.c_float), ("w_clr", C.c_float), ("w_col", C.c_float)]


_vp, _i32, _i64 = C.c_void_p, C.c_int32, C.c_int64
_pf, _pd, _pi, _pl = C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_int64)

# every symbol include/lmcma_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "lmcma_b200_abi_version": (C.c_int, []),
    "lmcma_b200_last_error": (C.c_char_p, []),
    "lmcma_b200_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "lmcma_b200_device_info": (C.c_int, [C.c_int, C.POINTER(C.c_int), _pl, _pl, C.POINTER(C.c_int)]),
    "lmcma_b200_map_create": (C.c_int, [C.c_int, C.c_int, _pi, _pf, C.c_int, C.c_float, C.c_float, C.POINTER(_vp)]),
    "lmcma_b200_edt": (C.c_int, [C.c_int, C.c_int, _pi, C.POINTER(C.c_uint8), C.c_float, _pf]),
    "lmcma_b200_map_create_from_occupancy": (C.c_int, [C.c_int, C.c_int, _pi, C.POINTER(C.c_uint8), C.c_float, C.c_int, C.c_float,
                                                     C.c_float, C.POINTER(_vp)]),
    "lmcma_b200_load_bmp": (C.c_int, [C.c_char_p, C.POINTER(C.c_uint8), _i64, _pi, _pi]),
    "lmcma_b200_load_binvox": (C.c_int, [C.c_char_p, C.POINTER(C.c_uint8), _i64, _pi, _pd, _pd]),
    "lmcma_b200_load_bt": (C.c_int, [C.c_char_p, C.POINTER(C.c_uint8), _i64, _pi, _pi, _pd]),
    "lmcma_b200_load_text_matrix": (C.c_int, [C.c_char_p, _pd, _i64, _pi, _pi]),
    "lmcma_b200_map_destroy": (C.c_int, [_vp]),
    "lmcma_b200_map_dequantized": (C.c_int, [_vp, _pf]),
    "lmcma_b200_map_set_l2_persist": (C.c_int, [_vp, C.c_int]),
    "lmcma_b200_cost_evaluate": (C.c_int, [_vp, C.POINTER(Objective), C.POINTER(Endpoints), _pf, _i32, _pf, _pi, _pi]),
    "lmcma_b200_cost_evaluate_dev": (C.c_int, [_vp, C.POINTER(Objective), C.POINTER(Endpoints), _vp, _i64, _i32, _vp, _vp, _vp, _vp]),
    "lmcma_b200_cost_trace": (C.c_int, [_vp, C.POINTER(Objective), C.POINTER(Endpoints), _pf, _pl, _i64, _pl]),
    "lmcma_b200_create": (C.c_int, [C.POINTER(Config), _pd, _pd, _pd, C.POINTER(_vp)]),
    "lmcma_b200_create_with_prior": (C.c_int, [C.POINTER(Config), _pd, _pd, _pd, _pd, C.POINTER(_vp)]),
    "lmcma_b200_destroy": (C.c_int, [_vp]),
    "lmcma_b200_set_stream": (C.c_int, [_vp, _vp]),
    "lmcma_b200_shape": (C.c_int, [_vp, _pi]),
    "lmcma_b200_ask_one": (C.c_int, [_vp, _pd, _i32]),
    "lmcma_b200_tell_one": (C.c_int, [_vp, _pd, _i32]),
    "lmcma_b200_ask_all": (C.c_int, [_vp, _pf]),
    "lmcma_b200_tell_all": (C.c_int, [_vp, _pf]),
    "lmcma_b200_ask_all_view": (C.c_int, [_vp, C.POINTER(_pf), _pl]),
    "lmcma_b200_inject_z": (C.c_int, [_vp, _pf]),
    "lmcma_b200_resample": (C.c_int, [_vp]),
    "lmcma_b200_is_done": (C.c_int, [_vp, _pi]),
    "lmcma_b200_attach_cost": (C.c_int, [_vp, _vp, C.POINTER(Objective), C.POINTER(Endpoints)]),
    "lmcma_b200_run": (C.c_int, [_vp, _i32]),
    "lmcma_b200_sync": (C.c_int, [_vp]),
    "lmcma_b200_launch_count": (C.c_int64, []),
    "lmcma_b200_last_run_ms": (C.c_int, [_vp, _pf]),
    "lmcma_b200_profile_kernels": (C.c_int, [_vp, _i32, _pf]),
    "lmcma_b200_best": (C.c_int, [_vp, _pf, _pf]),
    "lmcma_b200_get_f64": (C.c_int, [_vp, _i32, _pd, _i64]),
    "lmcma_b200_get_f32": (C.c_int, [_vp, _i32, _pf, _i64]),
    "lmcma_b200_get_i32": (C.c_int, [_vp, _i32, _pi, _i64]),
    "lmcma_b200_set_f64": (C.c_int, [_vp, _i32, _pd, _i64]),
    "lmcma_b200_set_f32": (C.c_int, [_vp, _i32, _pf, _i64]),
    "lmcma_b200_set_i32": (C.c_int, [_vp, _i32, _pi, _i64]),
    "lmcma_b200_mg_payload_floats": (C.c_int, [_vp, _pi]),
    "lmcma_b200_mg_evaluate": (C.c_int, [_vp, _vp, _vp]),
    "lmcma_b200_mg_rank": (C.c_int, [_vp, _vp, _vp, _vp]),
    "lmcma_b200_mg_update": (C.c_int, [_vp, _vp, _i32, _vp]),
    "lmcma_b200_hansen_gauss": (C.c_int, [_i64, _i64, _i64, _pd]),
    "lmcma_b200_hansen_uniform": (C.c_int, [_i64, _i64, _pd]),
    "lmcma_b200_covariance": (C.c_int, [_i32, _i32, _pd]),
    "lmcma_b200_cholesky": (C.c_int, [_i32, _pd, _pd]),
    "lmcma_b200_differentiation_matrix": (C.c_int, [_i32, _i32, C.c_double, _pd, _i32]),
    "lmcma_b200_invert": (C.c_int, [_pd, _pd, _i32]),
    "lmcma_b200_apply_cov_l": (C.c_int, [_pd, _pd, _i32]),
    "lmcma_b200_myqsort": (C.c_int, [_i32, _pd, _pi]),
    "lmcma_b200_rng_create": (C.c_int, [_i64, C.POINTER(_vp)]),
    "lmcma_b200_rng_destroy": (C.c_int, [_vp]),
    "lmcma_b200_rng_uniform": (C.c_double, [_vp]),
    "lmcma_b200_rng_gauss": (C.c_double, [_vp]),
}

_lib = None


def lib():
    """Load the native library; raise if it was not built (python __graft_entry__.py / make -C csrc)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("liblmcma_b200.so is missing at %s: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != OK:
        raise LmcmaError(rc, lib().lmcma_b200_last_error().decode("utf-8", "replace"))


def fptr(a):
    return a.ctypes.data_as(_pf)


def dptr(a):
    return a.ctypes.data_as(_pd)


def iptr(a):
    return a.ctypes.data_as(_pi)


def lptr(a):
    return a.ctypes.data_as(_pl)


def f32c(a):
    return np.ascontiguousarray(a, np.float32)


def f64c(a):
    return np.ascontiguousarray(a, np.float64)
