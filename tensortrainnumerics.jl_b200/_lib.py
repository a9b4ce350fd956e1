"""ctypes binding of libttn_b200.so (the C ABI declared in include/ttn_b200.h).

There is no fallback of any kind: if the shared library is missing, or no CUDA device can be bound,
importing/initialising fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libttn_b200.so")

TTN_F64, TTN_C128 = 0, 1

STATUS_EXC = {
    1: AssertionError,      # TTN_EDIM     -> AssertionError("Incompatible dimensions")  tt_operations.jl:11,102
    2: AssertionError,      # TTN_EARG     -> AssertionError                              tt_tools.jl:744,773
    3: ValueError,          # TTN_ECENTER  -> DimensionMismatch                           tt_tools.jl:513
    4: AssertionError,      # TTN_ESCHED   -> AssertionError("Sweep schedule error")      dmrg.jl:513
    5: RuntimeError,        # TTN_ENOTCONV
    6: RuntimeError,        # TTN_ECUDA    -> ErrorException
    7: RuntimeError,        # TTN_EINTERNAL
}


class SolverParams(C.Structure):
    _fields_ = [
        ("N", C.c_int), ("tol", C.c_double),
        ("sweep_schedule", C.POINTER(C.c_int64)), ("n_sweep_schedule", C.c_int),
        ("rmax_schedule", C.POINTER(C.c_int64)), ("n_rmax_schedule", C.c_int),
        ("rmax", C.c_int64), ("sweep_count", C.c_int), ("it_solver", C.c_int),
        ("linsolv_maxiter", C.c_int), ("linsolv_tol", C.c_double), ("itslv_thresh", C.c_int),
        ("krylovdim", C.c_int), ("symmetrize", C.c_int),
    ]


class TdvpParams(C.Structure):
    _fields_ = [
        ("two_site", C.c_int), ("steps", C.POINTER(C.c_double)), ("n_steps", C.c_int),
        ("normalize", C.c_int), ("sweeps", C.c_int), ("imaginary_time", C.c_int),
        ("max_bond", C.c_int64), ("truncerr", C.c_double),
        ("krylovdim", C.c_int), ("krylov_tol", C.c_double), ("krylov_maxiter", C.c_int),
    ]


import threading

_lib = None
_signatures = {}
_inited_device = None
_tls = threading.local()       # the library keeps one context (streams, allocation cache) per host thread


def load():
    """dlopen the library (no GPU needed: used by the CPU test that checks the exported symbols)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  tensortrainnumerics.jl_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i64p, dp, ip = C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int)
    vpp = C.POINTER(C.c_void_p)
    sig = {
        "ttn_init": [C.c_int], "ttn_shutdown": [], "ttn_version": [], "ttn_synchronize": [], "ttn_last_jacobi_sweeps": [],
        "ttn_reset_launch_count": [], "ttn_profile": [C.c_int],
        "ttn_profile_read": [C.POINTER(C.c_double), C.POINTER(C.c_longlong)],
        "ttn_ttv_upload": [C.c_int, C.c_int, i64p, i64p, i64p, vpp, C.c_int, vpp],
        "ttn_ttv_upload_async": [C.c_int, C.c_int, i64p, i64p, i64p, vpp, C.c_int, vpp],
        "ttn_ttv_download_async": [vp, vpp], "ttn_copy_synchronize": [],
        "ttn_ttv_info": [vp, ip, ip, ip], "ttn_ttv_ranks": [vp, i64p], "ttn_ttv_dims": [vp, i64p],
        "ttn_ttv_ot": [vp, i64p], "ttn_ttv_download": [vp, vpp], "ttn_ttv_copy": [vp, vpp],
        "ttn_ttv_complex": [vp, vpp], "ttn_ttv_free": [vp],
        "ttn_tto_upload": [C.c_int, C.c_int, i64p, i64p, vpp, vpp], "ttn_tto_complex": [vp, vpp], "ttn_tto_free": [vp],
        "ttn_tto_info": [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)], "ttn_tto_ranks": [vp, i64p], "ttn_tto_dims": [vp, i64p],
        "ttn_tto_download": [vp, vpp],
        "ttn_apply": [vp, vp, vpp], "ttn_dot": [vp, vp, dp], "ttn_norm": [vp, dp], "ttn_add": [vp, vp, vpp],
        "ttn_scale": [vp, C.c_double, C.c_double, vpp], "ttn_orthogonalize": [vp, C.c_int, vpp],
        "ttn_compress": [vp, C.c_int64, C.c_double, C.c_int, dp, C.c_int64],
        "ttn_apply_compress": [vp, vp, C.c_int64, C.c_double, C.c_int, dp, C.c_int64, vpp],
        "ttn_bond_truncate": [vp, C.c_int, C.c_int64, C.c_double, vpp],
        "ttn_swap_sites": [vp, C.c_int, C.c_int, C.c_int64, C.c_double],
        "ttn_merge_sites_diag": [vp, C.c_int],
        "ttn_split_site": [vp, C.c_int, C.c_int64, C.c_int, C.c_int64, C.c_double],
        "ttn_solver_params_default": [C.POINTER(SolverParams)], "ttn_tdvp_params_default": [C.POINTER(TdvpParams)],
        "ttn_als_linsolve": [vp, vp, vp, C.POINTER(SolverParams), vpp, dp],
        "ttn_als_eigsolve": [vp, vp, C.POINTER(SolverParams), vpp, dp, C.c_int, ip],
        "ttn_als_gen_eigsolv": [vp, vp, vp, C.POINTER(SolverParams), vpp, dp, C.c_int, ip],
        "ttn_mals_linsolve": [vp, vp, vp, C.POINTER(SolverParams), vpp, dp],
        "ttn_mals_eigsolve": [vp, vp, C.POINTER(SolverParams), vpp, dp, i64p, C.c_int, ip],
        "ttn_dmrg_linsolve": [vp, vp, vp, C.POINTER(SolverParams), vpp, dp],
        "ttn_dmrg_eigsolve": [vp, vp, C.POINTER(SolverParams), vpp, dp, i64p, C.c_int, ip],
        "ttn_dmrg_eigsolve_sharded": [vp, vp, C.POINTER(SolverParams), vp, vpp, dp, i64p, C.c_int, ip],
        "ttn_shard_ctx_create": [C.c_int, C.c_int64, C.c_int, C.c_int, vpp], "ttn_shard_ctx_handles": [vp, vp],
        "ttn_shard_ctx_bind": [vp, vp], "ttn_shard_ctx_free": [vp],
        "ttn_tdvp": [vp, vp, C.POINTER(TdvpParams), vpp],
        "ttn_gemm": [C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int64, C.c_int64, C.c_int, vp, C.c_int64, C.c_int64,
                     C.c_int, vp, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_int, C.c_int64, C.c_int64, C.c_int64],
        "ttn_matvec2_host": [C.c_int] * 6 + [vp, vp, vp, vp, vp, C.c_int],
        "ttn_matvec2_create": [C.c_int] * 6 + [vp, vp, vp, vpp],
        "ttn_matvec2_apply": [vp, vp, vp], "ttn_matvec2_free": [vp],
        "ttn_shard_range": [C.c_int, C.c_int, C.c_int, ip, ip],
        "ttn_shard_matvec_create": [C.c_int] * 6 + [vp, vp, vp, C.c_int, C.c_int, vpp],
        "ttn_shard_matvec_handles": [vp, vp], "ttn_shard_matvec_bind": [vp, vp],
        "ttn_shard_matvec_apply": [vp, vp, vpp],
        "ttn_shard_eigsolve": [vp, vp, C.c_int, C.c_int, C.c_double, dp, ip],
        "ttn_shard_matvec_slice": [vp, ip, ip], "ttn_shard_matvec_error": [vp, ip], "ttn_shard_matvec_free": [vp],
        "ttn_env_left_host": [C.c_int] * 6 + [vp, vp, vp, vp],
        "ttn_env_right_host": [C.c_int] * 6 + [vp, vp, vp, vp],
        "ttn_set_option": [C.c_char_p, C.c_double],
        "ttn_get_option": [C.c_char_p, dp],
        "ttn_heig_host": [C.c_int, C.c_int, C.c_int, C.c_int, vp, dp, vp, ip],
        "ttn_svdtrunc_host": [C.c_int, C.c_int, C.c_int, vp, C.c_int64, C.c_double, vp, dp, vp, ip],
        "ttn_qr_host": [C.c_int, C.c_int, C.c_int, vp, vp, vp],
        "ttn_rank_rule": [C.c_int, dp, C.c_int, C.c_double, C.c_int64, ip],
        "ttn_r_and_d_to_rks": [i64p, i64p, C.c_int, C.c_int64, i64p],
        "ttn_dev_alloc": [C.c_size_t, vpp], "ttn_dev_free": [vp], "ttn_h2d": [vp, vp, C.c_size_t],
        "ttn_d2h": [vp, vp, C.c_size_t],
    }
    for name, argtypes in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    global _signatures
    _signatures = {k: list(v) for k, v in sig.items()}
    lib.ttn_last_error.restype = C.c_char_p
    lib.ttn_last_error.argtypes = []
    lib.ttn_launch_count.restype = C.c_longlong
    lib.ttn_launch_count.argtypes = []
    lib.ttn_stream.restype = C.c_void_p
    lib.ttn_stream.argtypes = []
    _lib = lib
    return lib


def signatures():
    """name -> ctypes argument list of every bound entry point (tests compare the arities with include/ttn_b200.h)."""
    load()
    return dict(_signatures)


def check(status: int):
    if status != 0:
        msg = load().ttn_last_error().decode("utf-8", "replace")
        raise STATUS_EXC.get(status, RuntimeError)(msg)


def lib(device: int | None = None):
    """The initialised library bound to a CUDA device (LOCAL_RANK by default).  Raises without a GPU."""
    global _inited_device
    l = load()
    if _inited_device is None:
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        check(l.ttn_init(int(device)))
        _inited_device = int(device)
        _tls.inited = True
    elif not getattr(_tls, "inited", False):
        check(l.ttn_init(_inited_device))     # first call from this thread: its own context on the same device
        _tls.inited = True
    return l
