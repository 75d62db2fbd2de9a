"""Warm start of the dense Gram-space Newton solve, on the CPU: the size of the dense warm-start buffer, the argument checks of
cave_forward_backward_warm_ex, the exports and the Python-side options (no device needed)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("cave_dense_warm_bytes", "cave_forward_backward_warm_ex")


@pytest.fixture(scope="module")
def lib():
    from cave_b200 import _lib, build
    build.build()
    return _lib.load()


def test_dense_warm_bytes(lib):
    n = ctypes.c_size_t()
    assert lib.cave_dense_warm_bytes(10, 100, 50, ctypes.byref(n)) == 0 and n.value == 10 * (16 + 100 * 8)
    assert lib.cave_dense_warm_bytes(4, 7, 50, ctypes.byref(n)) == 0 and n.value == 4 * 80        # 16 + 56, 16-byte slots
    assert lib.cave_dense_warm_bytes(3, 1024, 1225, ctypes.byref(n)) == 0 and n.value == 3 * (16 + 1024 * 8)
    assert lib.cave_dense_warm_bytes(3, 2048, 1225, ctypes.byref(n)) == 0 and n.value == 3 * (16 + 2048 * 8)
    assert lib.cave_dense_warm_bytes(3, 5000, 1225, ctypes.byref(n)) == 0 and n.value == 3 * (16 + 2048 * 8)  # at most 2048
    assert lib.cave_dense_warm_bytes(0, 10, 10, ctypes.byref(n)) == -1 and b"positive" in lib.cave_last_error()
    assert lib.cave_dense_warm_bytes(2, -1, 10, ctypes.byref(n)) == -1
    assert lib.cave_dense_warm_bytes(1, 10, 10 ** 6, ctypes.byref(n)) == -2
    assert lib.cave_dense_warm_bytes(1, 10 ** 6, 10, ctypes.byref(n)) == -2
    assert lib.cave_dense_warm_bytes(1, 10, 10, None) == -1


def test_forward_backward_warm_ex_argument_errors(lib):
    from cave_b200 import _lib
    B, m, d = 8, 40, 20
    fake = 1 << 20                 # aligned dummy device addresses: every check below fails before anything is launched
    n = ctypes.c_size_t()
    assert lib.cave_pack_bytes(B, m, d, ctypes.byref(n)) == 0
    pack_bytes = n.value
    assert lib.cave_scratch_bytes(B, m, d, _lib.F64, ctypes.byref(_lib.SolverOpts()), ctypes.byref(n)) == 0
    scratch_bytes = n.value
    assert lib.cave_warm_bytes(B, m, d, ctypes.byref(n)) == 0
    warm_bytes = n.value
    assert lib.cave_dense_warm_bytes(B, m, d, ctypes.byref(n)) == 0
    dense_bytes = n.value

    def call(opts, warm, wbytes, dense, dbytes):
        return lib.cave_forward_backward_warm_ex(fake, None, fake, B, m, d, -1.0, 1, 0.2, 0, _lib.F32, _lib.F64,
                                                 ctypes.byref(opts) if opts is not None else None, fake, fake, fake, None,
                                                 None, None, None, fake, pack_bytes, fake, scratch_bytes, warm, wbytes,
                                                 dense, dbytes, None)

    ok = _lib.SolverOpts()
    ok.warm_pack = 1
    assert call(ok, None, 0, None, 0) == -1
    assert b"must not both be null" in lib.cave_last_error()
    assert call(_lib.SolverOpts(), fake, warm_bytes, fake, dense_bytes) == -1
    assert b"warm_pack" in lib.cave_last_error()
    assert call(None, None, 0, fake, dense_bytes) == -1
    assert b"warm_pack" in lib.cave_last_error()
    assert call(ok, fake, warm_bytes, fake + 8, dense_bytes) == -1
    assert b"dense warm-start buffer must be 16-byte aligned" in lib.cave_last_error()
    assert call(ok, fake + 8, warm_bytes, fake, dense_bytes) == -1
    assert b"warm-start buffer must be 16-byte aligned" in lib.cave_last_error()
    assert call(ok, fake, warm_bytes, fake, dense_bytes - 1) == -3
    assert b"dense warm-start buffer" in lib.cave_last_error()
    assert call(ok, None, 0, fake, dense_bytes - 1) == -3
    assert b"cave_dense_warm_bytes" in lib.cave_last_error()
    assert call(ok, fake, warm_bytes - 1, fake, dense_bytes) == -3
    assert b"cave_warm_bytes" in lib.cave_last_error()
    # with an index both buffers are sized for the whole pack, not for the batch
    ok.inst_index = fake
    ok.n_packed = 4 * B
    assert lib.cave_pack_bytes(4 * B, m, d, ctypes.byref(n)) == 0
    pack_bytes = n.value
    assert lib.cave_warm_bytes(4 * B, m, d, ctypes.byref(n)) == 0
    assert call(ok, fake, n.value, fake, dense_bytes) == -3
    assert b"dense warm-start buffer" in lib.cave_last_error() and str(4 * B).encode() in lib.cave_last_error()


def test_new_entry_points_are_declared_listed_and_exported(lib):
    from cave_b200 import _lib
    with open(os.path.join(ROOT, "include", "cave_b200.h")) as f:
        declared = set(re.findall(r"\b(cave_[a-z_]+)\s*\(", f.read()))
    for name in NEW:
        assert name in _lib.EXPORTS and name in declared
        assert getattr(lib, name).restype == ctypes.c_int
    assert lib.cave_abi_version() == 4


def test_warm_dense_needs_warm_start():
    from cave_b200 import pack_constraints
    with pytest.raises(ValueError, match="warm_start"):
        pack_constraints(torch.zeros((2, 130, 8)), warm_dense=True)


def test_pack_dataclass_keeps_positional_fields_and_resets_both_buffers():
    from cave_b200.qpsolver import CavePack
    p = CavePack(None, (1, 2, 3), 0, None, 0, None)
    assert p.warm_dense is None
    p.reset_warm_start()
    p = CavePack(None, (1, 2, 3), 0, None, 0, torch.ones(32, dtype=torch.uint8), torch.ones(48, dtype=torch.uint8))
    p.reset_warm_start()
    assert int(p.warm.count_nonzero()) == 0 and int(p.warm_dense.count_nonzero()) == 0
