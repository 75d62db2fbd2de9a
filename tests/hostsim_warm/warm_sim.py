"""ctypes wrapper around the CPU simulation of the solver core with the warm-start state (test infrastructure, see
warm_hostsim.cpp)."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_build", "libcave_hostsim_warm.so")
_CSRC = os.path.join(HERE, "..", "..", "cave_b200", "csrc")

_lib = None


def build(force=False):
    src = os.path.join(HERE, "warm_hostsim.cpp")
    deps = [src, os.path.join(HERE, "..", "hostsim", "hostsim.cpp")] + \
        [os.path.join(_CSRC, f) for f in ("solver_core.cuh", "ctx.cuh", "layout.cuh")]
    if not force and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(p) for p in deps):
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", OUT])
    return OUT


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.hostsim_warm_slot_bytes.restype = ctypes.c_size_t
    return _lib


def warm_slot_bytes(m):
    return int(lib().hostsim_warm_slot_bytes(int(m)))


def forward_backward(pred, ctrs, minimize=True, mode=0, inner_ratio=0.2, reduction="mean", compute_f32=False,
                     force_path=0, index=None, warm=None, max_iter=0):
    """As tests/hostsim/sim.py's forward_backward, plus: index, optional int [B], batch row -> instance of ctrs
    ([N, m, d]); warm, optional uint8 numpy buffer of N * warm_slot_bytes(m) bytes, the warm-start state, updated in
    place; max_iter, the Newton iteration cap (0: default)."""
    A = np.ascontiguousarray(ctrs, dtype=np.float32)
    N, m, d = A.shape
    p = np.ascontiguousarray(pred, dtype=np.float64)
    B = p.shape[0]
    idx = None if index is None else np.ascontiguousarray(index, dtype=np.int32)
    assert (idx is None and B == N) or (idx is not None and idx.shape == (B,) and idx.min() >= 0 and idx.max() < N)
    if warm is not None:
        assert warm.dtype == np.uint8 and warm.flags.c_contiguous and warm.nbytes >= N * warm_slot_bytes(m)
    sign = -1.0 if minimize else 1.0
    gscale = 1.0 / B if reduction == "mean" else 1.0
    loss_i = np.zeros(B); grad = np.zeros((B, d)); proj = np.zeros((B, d)); rnorm = np.zeros(B)
    status = np.zeros(B, np.int32); iters = np.zeros(B, np.int32)
    P = ctypes.c_void_p
    lib().hostsim_forward_backward_warm(
        A.ctypes.data_as(P), B, m, d, p.ctypes.data_as(P), ctypes.c_double(sign), mode, ctypes.c_double(inner_ratio),
        ctypes.c_double(gscale), int(compute_f32), int(force_path), int(max_iter),
        idx.ctypes.data_as(P) if idx is not None else None, warm.ctypes.data_as(P) if warm is not None else None,
        loss_i.ctypes.data_as(P), grad.ctypes.data_as(P), proj.ctypes.data_as(P), rnorm.ctypes.data_as(P),
        status.ctypes.data_as(P), iters.ctypes.data_as(P))
    loss = loss_i.mean() if reduction == "mean" else loss_i.sum() if reduction == "sum" else loss_i
    return dict(loss=loss, loss_i=loss_i, grad=grad, proj=proj, rnorm=rnorm, status=status, iters=iters)
