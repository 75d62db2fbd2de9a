"""ctypes binding of the C ABI in include/cave_b200.h.  There is no CPU fallback: if the CUDA
library has not been built the import of the product path fails loudly."""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# CAVE_B200_LIB: an alternative build of the same library (e.g. the -DCAVE_DENSE_PROFILE build of tools/dense_profile.py)
LIB_PATH = os.environ.get("CAVE_B200_LIB") or os.path.join(HERE, "_C", "libcave_b200.so")

CAVE_OK = 0
MODE_EXACT, MODE_INNER, MODE_HEURISTIC = 0, 1, 2
REDUCE = {"mean": 0, "sum": 1, "none": 2}
F32, F64 = 0, 1
ST_CONVERGED, ST_ITER_CAP, ST_STALLED, ST_NOSPACE, ST_SKIPPED, ST_BADINPUT, ST_PATH_LH, ST_PATH_GRAM = 0, 1, 2, 3, 4, 5, 0x100, 0x200
ST_WARM = 0x400     # flag: the (structured or dense) Newton solve started from the pack's warm-start state

EXPORTS = ("cave_abi_version", "cave_last_error", "cave_get_limits", "cave_pack_bytes",
           "cave_scratch_bytes", "cave_pack", "cave_forward_backward", "cave_plan_offset", "cave_plan_choice",
           "cave_dense_gram", "cave_launch_count", "cave_dense_ctrl_offset", "cave_pack_sparse",
           "cave_tsp_scratch_bytes", "cave_tsp_solve", "cave_pack_ex", "cave_warm_bytes", "cave_forward_backward_warm",
           "cave_dense_warm_bytes", "cave_forward_backward_warm_ex")


class SolverOpts(ctypes.Structure):
    _fields_ = [("max_iter", ctypes.c_int32), ("max_linesearch", ctypes.c_int32), ("tol", ctypes.c_double),
                ("cap_rows", ctypes.c_int64), ("cap_nnz", ctypes.c_int64), ("warm_pack", ctypes.c_int32),
                ("dense_mode", ctypes.c_int32), ("inst_index", ctypes.c_void_p), ("n_packed", ctypes.c_int64),
                ("dense_slots", ctypes.c_int64)]


class Limits(ctypes.Structure):
    _fields_ = [("max_d", ctypes.c_int64), ("max_m", ctypes.c_int64), ("max_batch", ctypes.c_int64)]


class CaveLibraryError(RuntimeError):
    pass


_lib = None


def load() -> ctypes.CDLL:
    """Load cave_b200/_C/libcave_b200.so; raise if it is missing (build it with
    ``python -m cave_b200.build`` or ``__graft_entry__.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CaveLibraryError(
            f"{LIB_PATH} not found: the CUDA backend is not built. Run `python cave_b200/build.py` "
            "(needs nvcc). There is deliberately no CPU fallback for solver='cuda'.")
    lib = ctypes.CDLL(LIB_PATH)
    P, I64, I32, F, SZP = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_double, ctypes.POINTER(ctypes.c_size_t)
    lib.cave_abi_version.restype = I32
    lib.cave_launch_count.restype = ctypes.c_uint64
    lib.cave_last_error.restype = ctypes.c_char_p
    lib.cave_get_limits.argtypes = [ctypes.POINTER(Limits)]
    lib.cave_pack_bytes.argtypes = [I64, I64, I64, SZP]
    lib.cave_scratch_bytes.argtypes = [I64, I64, I64, I32, ctypes.POINTER(SolverOpts), SZP]
    lib.cave_pack.argtypes = [P, P, I64, I64, I64, P, ctypes.c_size_t, P]
    lib.cave_pack_ex.argtypes = [P, P, I64, I64, I64, I32, P, ctypes.c_size_t, P]
    lib.cave_forward_backward.argtypes = [P, P, P, I64, I64, I64, F, I32, F, I32, I32, I32,
                                          ctypes.POINTER(SolverOpts), P, P, P, P, P, P, P,
                                          P, ctypes.c_size_t, P, ctypes.c_size_t, P]
    lib.cave_forward_backward_warm.argtypes = [P, P, P, I64, I64, I64, F, I32, F, I32, I32, I32,
                                               ctypes.POINTER(SolverOpts), P, P, P, P, P, P, P,
                                               P, ctypes.c_size_t, P, ctypes.c_size_t, P, ctypes.c_size_t, P]
    lib.cave_forward_backward_warm_ex.argtypes = [P, P, P, I64, I64, I64, F, I32, F, I32, I32, I32,
                                                  ctypes.POINTER(SolverOpts), P, P, P, P, P, P, P,
                                                  P, ctypes.c_size_t, P, ctypes.c_size_t, P, ctypes.c_size_t,
                                                  P, ctypes.c_size_t, P]
    lib.cave_warm_bytes.argtypes = [I64, I64, I64, SZP]
    lib.cave_dense_warm_bytes.argtypes = [I64, I64, I64, SZP]
    lib.cave_dense_gram.argtypes = [P, I64, I64, I64, ctypes.POINTER(SolverOpts), P, P, P, ctypes.c_size_t, P, ctypes.c_size_t, P]
    lib.cave_tsp_scratch_bytes.argtypes = [I64, I32, SZP]
    lib.cave_tsp_solve.argtypes = [P, I64, I32, P, P, P, ctypes.c_size_t, P]
    lib.cave_pack_sparse.argtypes = [P, P, P, P, I64, I64, I64, I32, P, ctypes.c_size_t, P]
    lib.cave_dense_ctrl_offset.argtypes = [I64, I64, I64, ctypes.POINTER(SolverOpts), SZP]
    lib.cave_plan_offset.argtypes = [I64, I64, I64, SZP]
    IP = ctypes.POINTER(ctypes.c_int)
    lib.cave_plan_choice.argtypes = [ctypes.POINTER(ctypes.c_uint64), I64, I32, I32, IP, IP, IP]
    for name in ("cave_get_limits", "cave_pack_bytes", "cave_scratch_bytes", "cave_pack", "cave_forward_backward",
                 "cave_plan_offset", "cave_plan_choice", "cave_dense_gram", "cave_dense_ctrl_offset", "cave_pack_sparse",
                 "cave_tsp_scratch_bytes", "cave_tsp_solve", "cave_pack_ex", "cave_warm_bytes", "cave_forward_backward_warm",
                 "cave_dense_warm_bytes", "cave_forward_backward_warm_ex"):
        getattr(lib, name).restype = I32
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != CAVE_OK:
        msg = load().cave_last_error().decode("utf-8", "replace")
        raise CaveLibraryError(f"cave_b200 C ABI error {code}: {msg}")
