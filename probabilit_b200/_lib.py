"""ctypes binding of libprobabilit_b200.so (the C ABI declared in include/probabilit_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is visible, the
calls raise.  Importing this module does not touch the GPU (the CPU-only test suite loads the
library and checks its exports without making a compute call).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libprobabilit_b200.so")
# developer aid: A/B a differently compiled build of the same sources (tools/ only; the product path is LIB_PATH)
LIB_PATH = os.environ.get("PBL_LIB", LIB_PATH)

STATUS_OK, STATUS_NOT_PD, STATUS_NON_FINITE, STATUS_BAD_SHAPE, STATUS_CUDA, STATUS_INTERNAL = range(6)
STATUS_OUT_OF_TABLE = 7  # pbl_stats_histogram: a bin index left the edge table (NumPy raises there)


class PblError(RuntimeError):
    """CUDA / internal failure inside libprobabilit_b200 (no reference equivalent)."""


_lib = None

_vp, _i32, _i64, _u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
_pd = C.c_void_p  # double* (host or device): passed as raw addresses

# name -> (restype, argtypes); must list every PBL_API symbol of include/probabilit_b200.h
SIGNATURES = {
    "pbl_version": (C.c_int, []),
    "pbl_last_error": (C.c_char_p, []),
    "pbl_device_count": (C.c_int, []),
    "pbl_set_device": (C.c_int, [C.c_int]),
    "pbl_get_device": (C.c_int, [C.POINTER(C.c_int)]),
    "pbl_kernel_launches": (_i64, []),
    "pbl_sort_profile_enable": (C.c_int, [C.c_int]),
    "pbl_sort_profile_read": (C.c_int, [C.POINTER(_i64), C.POINTER(C.c_double), C.POINTER(_i64)]),
    "pbl_device_malloc": (C.c_int, [C.POINTER(_vp), _u64]),
    "pbl_device_free": (C.c_int, [_vp]),
    "pbl_host_malloc_pinned": (C.c_int, [C.POINTER(_vp), _u64]),
    "pbl_host_free_pinned": (C.c_int, [_vp]),
    "pbl_memcpy_h2d": (C.c_int, [_vp, _vp, _u64, _vp]),
    "pbl_memcpy_d2h": (C.c_int, [_vp, _vp, _u64, _vp]),
    "pbl_stream_synchronize": (C.c_int, [_vp]),
    "pbl_ipc_export": (C.c_int, [_vp, _vp]),
    "pbl_ipc_open": (C.c_int, [_vp, C.POINTER(_vp)]),
    "pbl_ipc_close": (C.c_int, [_vp]),
    "pbl_peer_copy_streams": (C.c_int, [_i32]),
    "pbl_peer_copy_many": (C.c_int, [_i32, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_u64), _vp]),
    "pbl_ic_plan_create": (C.c_int, [_i64, _i32, _i32, C.POINTER(_vp)]),
    "pbl_ic_plan_create_ex": (C.c_int, [_i64, _i32, _i32, _i32, C.POINTER(_vp)]),
    "pbl_ic_plan_destroy": (C.c_int, [_vp]),
    "pbl_ic_plan_bytes": (_u64, [_vp]),
    "pbl_ic_plan_set_target": (C.c_int, [_vp, _pd]),
    "pbl_ic_plan_run": (C.c_int, [_vp, _pd, _i64, _i64, _pd, _i64, _i64, _vp]),
    "pbl_cholesky_plan_run": (C.c_int, [_vp, _pd, _i64, _i64, _pd, _i64, _i64, _vp]),
    "pbl_permcorr_begin": (C.c_int, [_vp, _pd, _i64, _i64, _pd, _i32, _pd, _pd, _vp]),
    "pbl_permcorr_steps": (C.c_int, [_vp, _pd, _vp, _vp, _vp, _vp, _i64, _i64, C.c_double, C.POINTER(_i64),
                                     C.POINTER(_i32), _pd, _i64, C.POINTER(_i64), _vp]),
    "pbl_permcorr_corr": (C.c_int, [_vp, _pd]),
    "pbl_ic_plan_run_host": (C.c_int, [_vp, _pd, _i64, _i64, _pd, _i64, _i64, _pd, _pd, _vp]),
    "pbl_corrcoef_f64": (C.c_int, [_vp, _pd, _i64, _i64, _i32, _pd, _vp]),
    "pbl_copy_strided_f64": (C.c_int, [_pd, _i64, _i64, _pd, _i64, _i64, _i64, _i32, _vp]),
    "pbl_iman_conover_f64": (C.c_int, [_pd, _i64, _i32, _i64, _i64, _pd, _pd, _i64, _i64]),
    "pbl_ic_stage_begin": (C.c_int, [_vp, _vp]),
    "pbl_ic_stage_rank_scores": (C.c_int, [_vp, _pd, _i64, _i64, _i32, _i32, _vp]),
    "pbl_ic_stage_gram": (C.c_int, [_vp, _vp]),
    "pbl_ic_stage_solve": (C.c_int, [_vp, _i64, _vp]),
    "pbl_ic_stage_transform": (C.c_int, [_vp, _vp]),
    "pbl_ic_stage_rank_gather": (C.c_int, [_vp, _pd, _i64, _i64, _i32, _i32, _vp]),
    "pbl_ic_stage_status": (C.c_int, [_vp, _vp]),
    "pbl_ic_plan_set_chunk_hook": (C.c_int, [_vp, _i64, _i32, _vp, _vp]),
    "pbl_ic_plan_buffer": (C.c_int, [_vp, _i32, C.POINTER(_vp), C.POINTER(_u64)]),
    "pbl_uniform_f64": (C.c_int, [_u64, _u64, _i64, _i32, _pd, _i64, _i64, _vp]),
    "pbl_sobol_direction_numbers": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "pbl_sobol_scramble": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "pbl_sobol_f64": (C.c_int, [_vp, _vp, _i32, _i32, _u64, _i64, _pd, _i64, _i64, _vp]),
    "pbl_halton_f64": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _u64, _i64, _pd, _i64, _i64, _vp]),
    "pbl_lhs_f64": (C.c_int, [_u64, _i64, _i32, _i32, _pd, _i64, _i64, _vp]),
    "pbl_graph_eval_f64": (C.c_int, [_vp, _i32, _i32, _i64, _u64, _vp, _i32, _vp, _i32, C.POINTER(_i32), _vp]),
    "pbl_ppf_f64": (C.c_int, [_i32, _pd, _i64, C.c_double, C.c_double, C.c_double, _pd, _vp]),
    "pbl_stats_moments": (C.c_int, [C.POINTER(_vp), C.POINTER(_i32), _i32, _i64, _i64, _i32, C.c_double, _pd, _vp]),
    "pbl_stats_quantiles": (C.c_int, [C.POINTER(_vp), C.POINTER(_i32), _i32, _i64, C.POINTER(C.c_double), _i32, _i32,
                                      _vp, _vp]),
    "pbl_stats_minmax": (C.c_int, [C.POINTER(_vp), C.POINTER(_i32), _i32, _i64, _vp, _vp]),
    "pbl_stats_histogram": (C.c_int, [C.POINTER(_vp), C.POINTER(_i32), _i32, _i64, _vp, _vp, _i64, _vp, _vp]),
    "pbl_stats_compact": (C.c_int, [C.POINTER(_vp), C.POINTER(_i32), _i32, _i64, _vp, C.POINTER(_vp), _vp, _vp]),
}


CHUNK_FN = C.CFUNCTYPE(None, _i32, _i32, _vp)  # pbl_chunk_fn


class StatsRange(C.Structure):
    """pbl_stats_range of include/probabilit_b200.h"""
    _fields_ = [("lo_cmp", _i32), ("hi_cmp", _i32), ("lo_f", C.c_double), ("hi_f", C.c_double), ("lo_i", _i64),
                ("hi_i", _i64)]


class HistSpec(C.Structure):
    """pbl_stats_hist_spec of include/probabilit_b200.h"""
    _fields_ = [("mode", _i32), ("cmp", _i32), ("keep", StatsRange), ("first", C.c_double), ("denom", C.c_double),
                ("nbins", _i64), ("table", _vp), ("offset", _i64)]


class GraphInstr(C.Structure):
    """pbl_graph_instr of include/probabilit_b200.h"""
    _fields_ = [("op", _i32), ("dst", _i32), ("src", _i32 * 4), ("imm", C.c_double * 4)]


def load():
    """Load the shared library (once) and declare the prototypes.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PblError(
            f"{LIB_PATH} is missing: build it with `python -m probabilit_b200.build` "
            "(there is no CPU fallback)"
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    msg = load().pbl_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status, what="libprobabilit_b200 call"):
    """Map CUDA/internal failures to PblError; reference-visible statuses are returned."""
    if status in (STATUS_CUDA, STATUS_INTERNAL):
        raise PblError(f"{what} failed: {last_error()}")
    return status


def require_gpu():
    lib = load()
    if lib.pbl_device_count() < 1:
        raise PblError("no CUDA device visible: probabilit_b200 has no CPU fallback")
    return lib


class device_guard:
    """Make `device` the calling thread's current CUDA device for the duration of a library call and restore
    the previous one afterwards: a cached plan stays usable after the caller (or another correlator) has
    switched devices, and the caller's later torch work keeps the device it had."""

    def __init__(self, device):
        self.device = int(device)

    def __enter__(self):
        lib = load()
        prev = C.c_int(-1)
        check(lib.pbl_get_device(C.byref(prev)), "pbl_get_device")
        self.prev = prev.value
        if self.prev != self.device:
            check(lib.pbl_set_device(self.device), "pbl_set_device")
        return self

    def __exit__(self, *exc):
        if self.prev >= 0 and self.prev != self.device:
            load().pbl_set_device(self.prev)
        return False


def kernel_launches():
    return int(load().pbl_kernel_launches())
