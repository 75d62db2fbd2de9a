"""Chunked calls on the CPU: the new entry points are declared, bound and exported, their argument checks return the right
codes and messages before anything is launched, the accumulator size, the chunk boundaries and the Python-side `chunk`
checks (no device needed)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("cave_chunk_acc_bytes", "cave_forward_backward_chunk", "cave_chunk_finalize", "cave_csr_rebase")
FAKE = 1 << 20      # an aligned dummy device address: every failing check below returns before a launch


@pytest.fixture(scope="module")
def lib():
    from cave_b200 import _lib, build
    build.build()
    return _lib.load()


def _align(x, a):
    return (x + a - 1) // a * a


def test_new_entry_points_are_declared_listed_and_exported(lib):
    from cave_b200 import _lib
    with open(os.path.join(ROOT, "include", "cave_b200.h")) as f:
        declared = set(re.findall(r"\b(cave_[a-z_]+)\s*\(", re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)))
    for name in NEW:
        assert name in _lib.EXPORTS and name in declared
        assert getattr(lib, name).restype == ctypes.c_int
    assert lib.cave_abi_version() == 4


def _acc_bytes(B):
    # float64 loss, float64 rnorm, int32 status, int32 iters, each array 256-byte aligned
    return _align(8 * B, 256) * 2 + _align(4 * B, 256) * 2


@pytest.mark.parametrize("B", [1, 31, 32, 64, 65, 1000, 65536])
def test_chunk_acc_bytes(lib, B):
    n = ctypes.c_size_t()
    assert lib.cave_chunk_acc_bytes(B, ctypes.byref(n)) == 0 and n.value == _acc_bytes(B)


def test_chunk_acc_bytes_errors(lib):
    n = ctypes.c_size_t()
    assert lib.cave_chunk_acc_bytes(0, ctypes.byref(n)) == -1 and b"positive" in lib.cave_last_error()
    assert lib.cave_chunk_acc_bytes(-5, ctypes.byref(n)) == -1
    assert lib.cave_chunk_acc_bytes(1 << 31, ctypes.byref(n)) == -2 and b"maximum" in lib.cave_last_error()
    assert lib.cave_chunk_acc_bytes(8, None) == -1 and b"null" in lib.cave_last_error()


def _sizes(lib, B, m, d):
    from cave_b200 import _lib
    n = ctypes.c_size_t()
    assert lib.cave_pack_bytes(B, m, d, ctypes.byref(n)) == 0
    pack_bytes = n.value
    assert lib.cave_scratch_bytes(B, m, d, _lib.F64, ctypes.byref(_lib.SolverOpts()), ctypes.byref(n)) == 0
    return pack_bytes, n.value


def test_forward_backward_chunk_argument_errors(lib):
    from cave_b200 import _lib
    B, m, d, total = 8, 40, 30, 100
    pack_bytes, scratch_bytes = _sizes(lib, B, m, d)
    acc_bytes = _acc_bytes(total)

    def call(offset=0, batch_total=total, acc=FAKE, abytes=acc_bytes, opts=None, warm=None, wbytes=0, gram=None, gbytes=0,
             nb=B):
        return lib.cave_forward_backward_chunk(FAKE, None, FAKE, nb, m, d, -1.0, 1, 0.2, 0, _lib.F32, _lib.F64,
                                               ctypes.byref(opts) if opts is not None else None, None, None, FAKE, None, None,
                                               None, None, FAKE, pack_bytes, FAKE, scratch_bytes, warm, wbytes, None, 0,
                                               gram, gbytes, offset, batch_total, acc, abytes, None)

    assert call(offset=-1) == -1 and b"not inside the batch" in lib.cave_last_error()
    assert call(offset=93) == -1 and b"not inside the batch" in lib.cave_last_error()        # 93 + 8 > 100
    assert call(batch_total=7, abytes=_acc_bytes(7)) == -1 and b"not inside the batch" in lib.cave_last_error()
    assert call(batch_total=0) == -1 and b"batch_total must be positive" in lib.cave_last_error()
    assert call(batch_total=1 << 31) == -2 and b"batch_total" in lib.cave_last_error()
    assert call(acc=None) == -1 and b"acc must not be null" in lib.cave_last_error()
    assert call(acc=FAKE + 128) == -1 and b"256-byte aligned" in lib.cave_last_error()
    assert call(abytes=acc_bytes - 1) == -3 and b"cave_chunk_acc_bytes" in lib.cave_last_error()
    # an accumulator sized for the chunk is too small for the batch
    assert call(abytes=_acc_bytes(B)) == -3
    # warm-start state and a Gram cache belong to a pack built beforehand
    assert call(warm=FAKE, wbytes=1 << 20) == -1 and b"warm_pack" in lib.cave_last_error()
    assert call(gram=FAKE, gbytes=1 << 20) == -1 and b"warm_pack" in lib.cave_last_error()
    # the checks of cave_forward_backward still apply (B <= 0, shapes, scratch size)
    assert call(nb=0) == -1 and b"positive" in lib.cave_last_error()
    assert lib.cave_forward_backward_chunk(FAKE, None, FAKE, B, m, d, -1.0, 1, 0.2, 0, _lib.F32, _lib.F64, None, None, None,
                                           FAKE, None, None, None, None, FAKE, pack_bytes, FAKE, scratch_bytes - 1, None, 0,
                                           None, 0, None, 0, 0, total, FAKE, acc_bytes, None) == -3
    assert b"scratch buffer" in lib.cave_last_error()


def test_chunk_finalize_argument_errors(lib):
    from cave_b200 import _lib
    total = 20
    ab = _acc_bytes(total)

    def fin(acc=FAKE, abytes=ab, batch_total=total, reduction=0, io=_lib.F32, loss=FAKE, loss_i=FAKE):
        return lib.cave_chunk_finalize(acc, abytes, batch_total, reduction, io, loss, loss_i, None, None, None, None)

    assert fin(acc=None) == -1 and b"acc must not be null" in lib.cave_last_error()
    assert fin(acc=FAKE + 8) == -1 and b"256-byte aligned" in lib.cave_last_error()
    assert fin(abytes=ab - 1) == -3 and b"cave_chunk_acc_bytes" in lib.cave_last_error()
    assert fin(batch_total=0) == -1 and b"positive" in lib.cave_last_error()
    assert fin(batch_total=1 << 31) == -2
    assert fin(reduction=3) == -1 and b"bad reduction" in lib.cave_last_error()
    assert fin(io=7) == -1 and b"bad io_dtype" in lib.cave_last_error()
    assert fin(loss_i=None) == -1 and b"loss_i" in lib.cave_last_error()
    assert fin(loss=None) == -1 and b"loss must not be null" in lib.cave_last_error()


def test_csr_rebase_argument_errors(lib):
    assert lib.cave_csr_rebase(FAKE, -1, 0, FAKE, 3, 0, None) == -1 and b"negative" in lib.cave_last_error()
    assert lib.cave_csr_rebase(None, 3, 0, FAKE, 3, 0, None) == -1 and b"null" in lib.cave_last_error()
    assert lib.cave_csr_rebase(FAKE, 3, 0, None, 3, 0, None) == -1
    assert lib.cave_csr_rebase(None, 0, 0, None, 0, 0, None) == 0          # nothing to do: no launch


@pytest.mark.parametrize("B,chunk", [(10, 3), (10, 1), (10, 9), (10, 10), (10, 11), (64, 7), (1, 1), (1024, 128)])
def test_chunk_bounds(B, chunk):
    from cave_b200.qpsolver import chunk_bounds
    bounds = chunk_bounds(B, chunk)
    assert bounds[0][0] == 0 and bounds[-1][1] == B
    assert all(hi0 == lo1 for (_, hi0), (lo1, _) in zip(bounds, bounds[1:]))
    assert all(hi - lo == chunk for lo, hi in bounds[:-1]) and 0 < bounds[-1][1] - bounds[-1][0] <= chunk
    assert len(bounds) == -(-B // chunk)


@pytest.mark.parametrize("chunk", [0, -3, 2.0, "8", True, 1.5])
def test_bad_chunk_raises(chunk):
    from cave_b200 import cave_forward_backward
    with pytest.raises(ValueError, match="chunk"):
        cave_forward_backward(torch.zeros((4, 3)), torch.zeros((4, 2, 3)), -1.0, 0, chunk=chunk)


def test_chunk_is_a_module_solver_kwarg():
    from cave_b200 import EPO, innerConeAlignedCosine

    class Model:
        modelSense = EPO.MINIMIZE

    mod = innerConeAlignedCosine(Model(), solver="cuda", solver_kwargs={"chunk": 64})
    assert mod._kernel_kwargs() == {"chunk": 64}
