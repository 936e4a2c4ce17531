"""ctypes binding of libcpi_b200.so (the C ABI declared in include/cpi_b200.h).

The library is loaded lazily and LOUDLY: if the shared object is missing, or an entry point is absent, ``load()``
raises -- there is no CPU fallback anywhere in this package.  Build it with ``python __graft_entry__.py`` (or
``make -C cpi_b200/csrc``).
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CPI_B200_LIB") or os.path.join(_HERE, "libcpi_b200.so")     # the override is for A/B kernel experiments only

c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_vp = ctypes.c_void_p

# every symbol include/cpi_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "cpi_preintegrate_batch": (c_int, [c_int, c_int, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_int, c_vp, c_vp]),
    "cpi_preintegrate_batch_continue": (c_int, [c_int, c_int, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_int, c_vp, c_vp]),
    "cpi_preintegrate_batch_host": (c_int, [c_int, c_int, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_int, c_vp]),
    "cpi_imu_factor_eval_batch": (c_int, [c_int, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "cpi_imu_factor_eval_batch_host": (c_int, [c_int, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "cpi_imu_factor_hessian_batch": (c_int, [c_int, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "cpi_imu_factor_whiten_batch": (c_int, [c_int, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "cpi_imu_chain_assemble": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.c_double, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "cpi_imu_chain_solve_workspace": (c_i64, [c_i64]),
    "cpi_imu_chain_solve": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "cpi_imu_chain_marginals_workspace": (c_i64, [c_i64]),
    "cpi_imu_chain_marginals": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "cpi_predict_state_batch": (c_int, [c_int, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "cpi_retract_batch": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp]),
    "cpi_host_last_timing": (c_int, [c_vp, c_vp]),
    "cpi_host_register": (c_int, [c_vp, ctypes.c_size_t]),
    "cpi_host_unregister": (c_int, [c_vp]),
    "cpi_cut_windows": (c_i64, [c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "cpi_comm_unique_id": (c_int, [c_vp]),
    "cpi_comm_create": (c_int, [c_vp, c_int, c_int, ctypes.POINTER(c_vp)]),
    "cpi_comm_destroy": (c_int, [c_vp]),
    "cpi_comm_rank": (c_int, [c_vp]),
    "cpi_comm_world": (c_int, [c_vp]),
    "cpi_preintegrate_batch_sharded": (c_int, [c_vp, c_int, c_int, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_int, c_vp, c_vp]),
    "cpi_comm_sm_free_barriers": (c_int, [c_vp]),
    "cpi_comm_register": (c_int, [c_vp, c_vp, ctypes.c_size_t, c_vp]),
    "cpi_comm_unregister": (c_int, [c_vp, c_vp]),
    "cpi_comm_wait": (c_int, [c_vp, c_vp]),
    "cpi_last_error": (ctypes.c_char_p, []),
    "cpi_version": (ctypes.c_char_p, []),
    "cpi_record_doubles": (c_int, [c_int]),
    "cpi_device_count": (c_int, []),
    "cpi_launch_count": (c_i64, []),
}

REC_DOUBLES = {1: 290, 2: 308}
SAMPLE_DOUBLES, LIN_DOUBLES, STATE_DOUBLES = 7, 13, 16
FLAG_IMU_AVG, FLAG_ANALYTIC_JACOBIANS = 1, 2
# record field slices (include/cpi_b200.h)
REC = dict(q=(0, 4), R=(4, 13), alpha=(13, 16), beta=(16, 19), DT=(19, 20), J_q=(20, 29), J_a=(29, 38), J_b=(38, 47),
           H_a=(47, 56), H_b=(56, 65), P=(65, 290), O_a=(290, 299), O_b=(299, 308))

_lib = None


class CpiError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"cpi_b200 error {code}: {msg}")
        self.code = code


def load():
    """Load libcpi_b200.so and bind every declared symbol.  Raises if the library or a symbol is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built (run `python __graft_entry__.py` or "
            f"`make -C cpi_b200/csrc`).  cpi_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise CpiError(rc, load().cpi_last_error().decode())


def launch_count() -> int:
    return int(load().cpi_launch_count())
