"""Gram cache of a resident dense dataset, on the CPU: the size of the cache, the argument checks of the new entry points,
the exports and the Python-side options (no device needed)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("cave_gram_cache_count", "cave_gram_cache_bytes", "cave_gram_cache_build", "cave_forward_backward_resident")


@pytest.fixture(scope="module")
def lib():
    from cave_b200 import _lib, build
    build.build()
    return _lib.load()


def _align(x, a):
    return (x + a - 1) // a * a


def test_gram_cache_bytes(lib):
    n = ctypes.c_size_t()
    # header (16) + map (4 N), padded to 1024, then m_pad^2 float32 per cached slot
    assert lib.cave_gram_cache_bytes(10, 3, 128, 190, ctypes.byref(n)) == 0 and n.value == 1024 + 3 * 128 * 128 * 4
    assert lib.cave_gram_cache_bytes(10, 0, 128, 190, ctypes.byref(n)) == 0 and n.value == 1024
    assert lib.cave_gram_cache_bytes(252, 0, 130, 190, ctypes.byref(n)) == 0 and n.value == 1024       # 16 + 1008
    assert lib.cave_gram_cache_bytes(253, 0, 130, 190, ctypes.byref(n)) == 0 and n.value == 2048       # 16 + 1012
    assert lib.cave_gram_cache_bytes(1184, 1184, 1024, 1225, ctypes.byref(n)) == 0
    assert n.value == _align(16 + 4 * 1184, 1024) + 1184 * 1024 * 1024 * 4
    assert lib.cave_gram_cache_bytes(5, 2, 300, 64, ctypes.byref(n)) == 0 and n.value == 1024 + 2 * 384 * 384 * 4
    assert lib.cave_gram_cache_bytes(5, 6, 300, 64, ctypes.byref(n)) == -1 and b"n_cached" in lib.cave_last_error()
    assert lib.cave_gram_cache_bytes(5, -1, 300, 64, ctypes.byref(n)) == -1
    assert lib.cave_gram_cache_bytes(0, 0, 300, 64, ctypes.byref(n)) == -1 and b"positive" in lib.cave_last_error()
    assert lib.cave_gram_cache_bytes(1, 0, 10, 10 ** 6, ctypes.byref(n)) == -2
    assert lib.cave_gram_cache_bytes(1, 0, 10, 10, None) == -1


def _sizes(lib, B, m, d, n_packed=None):
    from cave_b200 import _lib
    n = ctypes.c_size_t()
    N = n_packed or B
    assert lib.cave_pack_bytes(N, m, d, ctypes.byref(n)) == 0
    pack_bytes = n.value
    o = _lib.SolverOpts()
    o.dense_mode = 1
    assert lib.cave_scratch_bytes(B, m, d, _lib.F64, ctypes.byref(o), ctypes.byref(n)) == 0
    scratch_bytes = n.value
    assert lib.cave_gram_cache_bytes(N, 0, m, d, ctypes.byref(n)) == 0
    return pack_bytes, scratch_bytes, n.value


def test_forward_backward_resident_argument_errors(lib):
    from cave_b200 import _lib
    B, m, d = 8, 256, 300
    fake = 1 << 20                 # aligned dummy device addresses: every check below fails before anything is launched
    pack_bytes, scratch_bytes, gram_min = _sizes(lib, B, m, d)
    n = ctypes.c_size_t()
    assert lib.cave_warm_bytes(B, m, d, ctypes.byref(n)) == 0
    warm_bytes = n.value
    assert lib.cave_dense_warm_bytes(B, m, d, ctypes.byref(n)) == 0
    dense_bytes = n.value

    def call(opts, gram, gbytes, A=fake, warm=None, wbytes=0, dense=None, dbytes=0):
        return lib.cave_forward_backward_resident(A, None, fake, B, m, d, -1.0, 1, 0.2, 0, _lib.F32, _lib.F64,
                                                  ctypes.byref(opts) if opts is not None else None, fake, fake, fake, None,
                                                  None, None, None, fake, pack_bytes, fake, scratch_bytes, warm, wbytes,
                                                  dense, dbytes, gram, gbytes, None)

    ok = _lib.SolverOpts()
    ok.warm_pack = 1
    ok.dense_mode = 1
    assert call(ok, None, 0) == -1
    assert b"must not all be null" in lib.cave_last_error()
    assert call(_lib.SolverOpts(), fake, gram_min) == -1
    assert b"warm_pack" in lib.cave_last_error()
    assert call(None, fake, gram_min) == -1
    assert b"warm_pack" in lib.cave_last_error()
    assert call(ok, fake + 8, gram_min) == -1
    assert b"Gram cache must be 16-byte aligned" in lib.cave_last_error()
    assert call(ok, fake, gram_min - 1) == -3
    assert b"cave_gram_cache_bytes" in lib.cave_last_error()
    # the other buffers are still checked as for cave_forward_backward_warm_ex
    assert call(ok, fake, gram_min, dense=fake + 8, dbytes=dense_bytes) == -1
    assert b"dense warm-start buffer must be 16-byte aligned" in lib.cave_last_error()
    assert call(ok, fake, gram_min, warm=fake, wbytes=warm_bytes - 1) == -3
    assert b"cave_warm_bytes" in lib.cave_last_error()
    # a cache needs A; without A an indexed call is valid only without one
    ok.inst_index = fake
    ok.n_packed = 4 * B
    pack_bytes, _, gram_min = _sizes(lib, B, m, d, 4 * B)
    assert call(ok, fake, gram_min, A=None) == -1
    assert b"needs A" in lib.cave_last_error()
    # with an index the cache is sized for the whole pack, not for the batch
    assert call(ok, fake, gram_min - 1) == -3
    assert b"Gram cache" in lib.cave_last_error() and str(4 * B).encode() in lib.cave_last_error()


def test_gram_cache_count_and_build_argument_errors(lib):
    from cave_b200 import _lib
    N, m, d = 8, 256, 300
    fake = 1 << 20
    pack_bytes, scratch_bytes, gram_min = _sizes(lib, N, m, d)
    assert lib.cave_gram_cache_count(None, pack_bytes, N, m, d, fake, None) == -1
    assert lib.cave_gram_cache_count(fake, pack_bytes, N, m, d, None, None) == -1
    assert lib.cave_gram_cache_count(fake, pack_bytes - 1, N, m, d, fake, None) == -3
    assert lib.cave_gram_cache_count(fake + 16, pack_bytes, N, m, d, fake, None) == -1
    assert b"256-byte aligned" in lib.cave_last_error()
    assert lib.cave_gram_cache_count(fake, pack_bytes, 0, m, d, fake, None) == -1

    def build(A=fake, cache=fake, cbytes=gram_min, pack=fake, pbytes=pack_bytes, scratch=fake, sbytes=scratch_bytes,
              mm=m, opts=None):
        return lib.cave_gram_cache_build(A, N, mm, d, ctypes.byref(opts) if opts is not None else None, cache, cbytes,
                                         pack, pbytes, scratch, sbytes, None)

    assert build(A=None) == -1 and b"must not be null" in lib.cave_last_error()
    assert build(cache=None) == -1
    assert build(mm=100) == -2 and b"dense path" in lib.cave_last_error()          # m < 128
    assert build(mm=2100) == -2                                                     # m_pad > 2048
    assert build(cache=fake + 8) == -1 and b"16-byte aligned" in lib.cave_last_error()
    assert build(scratch=fake + 16) == -1 and b"256-byte aligned" in lib.cave_last_error()
    assert build(cbytes=gram_min - 1) == -3 and b"cave_gram_cache_bytes" in lib.cave_last_error()
    assert build(pbytes=pack_bytes - 1) == -3 and b"pack buffer" in lib.cave_last_error()
    assert build(sbytes=scratch_bytes - 1) == -3 and b"scratch buffer" in lib.cave_last_error()
    few = _lib.SolverOpts()
    few.dense_slots = 2                     # a smaller scratch suffices for fewer instances per round
    n = ctypes.c_size_t()
    few.dense_mode = 1
    assert lib.cave_scratch_bytes(N, m, d, _lib.F64, ctypes.byref(few), ctypes.byref(n)) == 0
    assert n.value < scratch_bytes
    assert build(opts=few, sbytes=n.value - 1) == -3


def test_new_entry_points_are_declared_listed_and_exported(lib):
    from cave_b200 import _lib
    with open(os.path.join(ROOT, "include", "cave_b200.h")) as f:
        declared = set(re.findall(r"\b(cave_[a-z_]+)\s*\(", f.read()))
    for name in NEW:
        assert name in _lib.EXPORTS and name in declared
        assert getattr(lib, name).restype == ctypes.c_int
    assert lib.cave_abi_version() == 4


def test_cache_gram_needs_keep_dense():
    from cave_b200 import pack_constraints
    with pytest.raises(ValueError, match="keep_dense"):
        pack_constraints(torch.zeros((2, 130, 8)), keep_dense=False, cache_gram=True)


def test_pack_dataclass_keeps_positional_fields_and_reset_keeps_the_cache():
    from cave_b200.qpsolver import CavePack
    p = CavePack(None, (1, 2, 3), 0, None, 0, None, None)
    assert p.gram is None
    p.reset_warm_start()
    p = CavePack(None, (1, 2, 3), 0, None, 0, torch.ones(32, dtype=torch.uint8), torch.ones(48, dtype=torch.uint8),
                 torch.ones(64, dtype=torch.uint8))
    p.reset_warm_start()
    assert int(p.warm.count_nonzero()) == 0 and int(p.warm_dense.count_nonzero()) == 0
    assert int(p.gram.count_nonzero()) == 64
