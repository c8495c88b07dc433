"""ctypes binding of libtsb200.so (include/tsb200.h).  Fails loudly if the CUDA extension is missing:
there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("TSB200_LIB") or os.path.join(PKG_DIR, "libtsb200.so")  # (TSB200_LIB: A/B builds)

MAX_JOBS = 20
MAX_MACHINES = 20
MAX_PAIRS = 190

OK, EINVAL, ECUDA, ENOMEM, ENODEV, EALIGN, EUNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
LB1_D, LB1, LB2 = 0, 1, 2
XFER_AUTO, XFER_MEMCPY, XFER_ZEROCOPY = 0, 1, 2


class TsbError(RuntimeError):
    def __init__(self, code: int, where: str):
        L = lib()
        msg = L.tsb_strerror(code).decode()
        if code == ECUDA:
            msg += " — " + L.tsb_last_cuda_error().decode()
        super().__init__(f"{where}: {msg} ({code})")
        self.code = code


class PfspTables(C.Structure):
    """tsb_pfsp_tables"""
    _fields_ = [
        ("jobs", C.c_int32), ("machines", C.c_int32), ("pairs", C.c_int32),
        ("p_times", C.c_int32 * (MAX_MACHINES * MAX_JOBS)),
        ("min_heads", C.c_int32 * MAX_MACHINES), ("min_tails", C.c_int32 * MAX_MACHINES),
        ("johnson", C.c_int32 * (MAX_PAIRS * MAX_JOBS)), ("lags", C.c_int32 * (MAX_PAIRS * MAX_JOBS)),
        ("mp0", C.c_int32 * MAX_PAIRS), ("mp1", C.c_int32 * MAX_PAIRS), ("mp_order", C.c_int32 * MAX_PAIRS),
    ]


class PfspTables50(C.Structure):
    """tsb_pfsp_tables50 (MAX_JOBS = 50 build)"""
    _fields_ = [
        ("jobs", C.c_int32), ("machines", C.c_int32), ("pairs", C.c_int32),
        ("p_times", C.c_int32 * (MAX_MACHINES * 50)),
        ("min_heads", C.c_int32 * MAX_MACHINES), ("min_tails", C.c_int32 * MAX_MACHINES),
        ("johnson", C.c_int32 * (MAX_PAIRS * 50)), ("lags", C.c_int32 * (MAX_PAIRS * 50)),
        ("mp0", C.c_int32 * MAX_PAIRS), ("mp1", C.c_int32 * MAX_PAIRS), ("mp_order", C.c_int32 * MAX_PAIRS),
    ]


class SearchStats(C.Structure):
    """tsb_search_stats"""
    _fields_ = [
        ("explored_tree", C.c_uint64), ("explored_sol", C.c_uint64), ("best", C.c_int64),
        ("t_step1", C.c_double), ("t_step2", C.c_double), ("t_step3", C.c_double),
        ("offloads", C.c_uint64), ("offloaded_parents", C.c_uint64), ("kernel_launches", C.c_uint64),
        ("per_gpu_tree", C.c_uint64 * 8), ("steals", C.c_uint64),
    ]


# every symbol include/tsb200.h declares: name -> (restype, argtypes)
_vp, _i, _i64, _u64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64
_pi32 = C.c_void_p
SYMBOLS = {
    "tsb_strerror": (C.c_char_p, [_i]),
    "tsb_last_cuda_error": (C.c_char_p, []),
    "tsb_device_count": (_i, []),
    "tsb_init_devices": (_i, [_i]),
    "tsb_bind_thread_to_device": (_i, [_i]),
    "tsb_version": (C.c_char_p, []),
    "tsb_nq_create": (_i, [C.POINTER(_vp), _i, _i, _i, _i]),
    "tsb_nq_destroy": (None, [_vp]),
    "tsb_nq_evaluate": (_i, [_vp, _vp, _i, _vp]),
    "tsb_nq_evaluate_device": (_i, [_vp, _vp, _i, _vp, _vp]),
    "tsb_nq_expand": (_i, [_vp, _vp, _i, _vp, _u64, C.POINTER(_u64), C.POINTER(_u64)]),
    "tsb_nq_expand_device": (_i, [_vp, _vp, _i, _vp, C.POINTER(_u64), C.POINTER(_u64), _vp]),
    "tsb_nq_pool_push": (_i, [_vp, _vp, _i64]),
    "tsb_nq_pool_size": (_i64, [_vp]),
    "tsb_nq_pool_step": (_i, [_vp, _i, _i, C.POINTER(_i64), C.POINTER(_u64), C.POINTER(_u64)]),
    "tsb_nq_pool_drain": (_i, [_vp, _vp, _i64, C.POINTER(_i64)]),
    "tsb_nq_pool_steal": (_i, [_vp, _vp, _i, C.POINTER(_i64)]),
    "tsb_pfsp_pool_steal": (_i, [_vp, _vp, _i, C.POINTER(_i64)]),
    "tsb_nq_pool_run": (_i, [_vp, _i, _i, _i64, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64)]),
    "tsb_nq_pool_run_multi": (_i, [C.POINTER(_vp), _i, _i, _i, _i64, C.POINTER(_u64)]),
    "tsb_release_cached_handles": (None, []),
    "tsb_nq_sibling": (_i, [_vp, _i, C.POINTER(_vp)]),
    "tsb_nq_pools_per_launch": (_i, [_vp, _i]),
    "tsb_nq_register_host": (_i, [_vp, _vp, C.c_size_t]),
    "tsb_nq_unregister_host": (_i, [_vp, _vp]),
    "tsb_debug_flag_exchange": (_i, [_i, _i, _i, _i, C.POINTER(C.c_double)]),
    "tsb_nq_set_xfer": (_i, [_vp, _i]),
    "tsb_nq_kernel_launches": (_u64, [_vp]),
    "tsb_pfsp_create": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _pi32, _pi32, _pi32, _i, _pi32, _pi32, _pi32, _pi32, _pi32]),
    "tsb_pfsp_create_wide": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _i, _pi32, _pi32, _pi32, _i, _pi32, _pi32, _pi32, _pi32, _pi32]),
    "tsb_pfsp_tables50_build": (_i, [C.POINTER(PfspTables50), _i, _i]),
    "tsb_pfsp_create50_from_tables": (_i, [C.POINTER(_vp), _i, _i, C.POINTER(PfspTables50)]),
    "tsb_pfsp_destroy": (None, [_vp]),
    "tsb_pfsp_evaluate": (_i, [_vp, _i, _vp, _i, _i64, _vp]),
    "tsb_pfsp_evaluate_device": (_i, [_vp, _i, _vp, _i, _i64, _vp, _vp]),
    "tsb_pfsp_expand": (_i, [_vp, _i, _vp, _i, C.POINTER(_i64), _vp, _u64, C.POINTER(_u64), C.POINTER(_u64)]),
    "tsb_pfsp_expand_device": (_i, [_vp, _i, _vp, _i, C.POINTER(_i64), _vp, C.POINTER(_u64), C.POINTER(_u64), _vp]),
    "tsb_pfsp_pool_push": (_i, [_vp, _vp, _i64]),
    "tsb_pfsp_pool_size": (_i64, [_vp]),
    "tsb_pfsp_pool_step": (_i, [_vp, _i, _i, _i, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_u64), C.POINTER(_u64)]),
    "tsb_pfsp_pool_drain": (_i, [_vp, _vp, _i64, C.POINTER(_i64)]),
    "tsb_pfsp_slow_rounds": (_u64, [_vp]),
    "tsb_pfsp_register_host": (_i, [_vp, _vp, C.c_size_t]),
    "tsb_pfsp_unregister_host": (_i, [_vp, _vp]),
    "tsb_pfsp_set_xfer": (_i, [_vp, _i]),
    "tsb_pfsp_kernel_launches": (_u64, [_vp]),
    "tsb_taillard_nb_jobs": (_i, [_i]),
    "tsb_taillard_nb_machines": (_i, [_i]),
    "tsb_taillard_best_ub": (_i64, [_i]),
    "tsb_pfsp_tables_build": (_i, [C.POINTER(PfspTables), _i]),
    "tsb_pfsp_tables_build_variant": (_i, [C.POINTER(PfspTables), _i, _i]),
    "tsb_pfsp_create_from_tables": (_i, [C.POINTER(_vp), _i, _i, C.POINTER(PfspTables)]),
    "tsb_nq_warmup": (_i, [_i, _i, _vp, _i64, C.POINTER(_i64), C.POINTER(_u64), C.POINTER(_u64)]),
    "tsb_nq_stream": (_vp, [_vp]),
    "tsb_pfsp_stream": (_vp, [_vp]),
    "tsb_nq_search": (_i, [_i, _i, _i, _i, _i, C.POINTER(SearchStats)]),
    "tsb_nq_search_device": (_i, [_i, _i, _i, _i, _i, C.POINTER(SearchStats)]),
    "tsb_pfsp_search": (_i, [_i, _i, _i, _i, _i, _i, C.POINTER(SearchStats)]),
    "tsb_pfsp_search_device": (_i, [_i, _i, _i, _i, _i, _i, C.POINTER(SearchStats)]),
    "tsb_pfsp_search_wide": (_i, [_i, _i, _i, _i, _i, _i, _i, C.POINTER(SearchStats)]),
    "tsb_pfsp_search_device_wide": (_i, [_i, _i, _i, _i, _i, _i, _i, C.POINTER(SearchStats)]),
    "tsb_nq_search_on": (_i, [_vp, _i, _i, _i, C.POINTER(SearchStats)]),
    "tsb_pfsp_search_on": (_i, [_vp, _i, _i, _i, _i, _i, C.POINTER(SearchStats)]),
    "tsb_nq_search_device_part": (_i, [_i, _i, _i, _i, _i, _i, _i, C.POINTER(SearchStats)]),
    "tsb_pfsp_search_device_part": (_i, [_i, _i, _i, _i, _i, _i, _i, _i, C.POINTER(SearchStats)]),
}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              f"or `make -C {PKG_DIR}` — tsb200 has no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code: int, where: str) -> None:
    if code != OK:
        raise TsbError(code, where)
