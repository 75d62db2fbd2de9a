"""Pack content of the warp-streaming scan (scan_rows_kernel) against the tile scan (CAVE_SCAN_KERNEL=tile) and, for
integer-valued rows, against the sparse ingestion (cave_pack_sparse), instance by instance."""
import ctypes
import importlib.util
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("scan_probe", os.path.join(ROOT, "tools", "scan_probe.py"))
scan_probe = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(scan_probe)


def _pack(A):
    from cave_b200 import _lib
    lib = _lib.load()
    B, m, d = A.shape
    nb = ctypes.c_size_t()
    _lib.check(lib.cave_pack_bytes(B, m, d, ctypes.byref(nb)))
    buf = torch.empty(nb.value, dtype=torch.uint8, device=A.device)
    _lib.check(lib.cave_pack_ex(ctypes.c_void_p(A.data_ptr()), None, B, m, d, 0, ctypes.c_void_p(buf.data_ptr()), nb.value,
                                ctypes.c_void_p(torch.cuda.current_stream(A.device).cuda_stream)))
    torch.cuda.synchronize()
    return scan_probe.pack_content(buf, B, m, d)


def _pack_sparse(A):
    from cave_b200 import SparseConstraints, pack_constraints_sparse
    B, m, d = A.shape
    pk = pack_constraints_sparse(SparseConstraints.from_dense(A), cache_setup=False)
    torch.cuda.synchronize()
    return scan_probe.pack_content(pk.buf, B, m, d)


def _special_dense(dev):
    """Dense N(0,1) rows that overflow the packed CSR, plus -0.0 entries, values on both sides of the 1e-7 thresholds,
    singleton rows and empty rows; d odd, so the rows start at every offset inside a 16-byte word."""
    rng = np.random.default_rng(5)
    B, m, d = 3, 120, 1225
    A = np.zeros((B, m, d), np.float32)
    A[:, :40] = rng.standard_normal((B, 40, d))
    A[:, 40:80] = np.where(rng.random((B, 40, d)) < 0.02, rng.standard_normal((B, 40, d)), 0.0)
    A[:, 5, ::7] = -0.0
    for b in range(B):
        for r in range(80, 115):
            A[b, r, rng.integers(d)] = rng.choice([-1.0, 2.5, 0.9e-7, -0.9e-7, 1.1e-7, -1.1e-7, -0.0])
        A[b, 115, [3, 900]] = [0.6e-7, -0.5e-7]          # general row below the threshold
        A[b, 116, [0, 1224]] = [1.1e-7, 1.0]               # first and last column
        A[b, 117, :4] = [1.0, -0.0, 2.0, 0.0]
    return torch.tensor(A, device=dev)


def _assert_same(a, b, tol_avg_l2):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        if tol_avg_l2:      # the tile kernel sums the average in float and squares the norm: compare those two loosely
            assert x[0] == y[0] and x[1] == y[1] and x[3] == y[3] and x[4] == y[4], i
            fa, fb = np.frombuffer(x[5], np.float32), np.frombuffer(y[5], np.float32)
            np.testing.assert_allclose(fa, fb, rtol=1e-5, atol=1e-6)
            l2a, l2b = np.array([x[2]], np.uint32).view(np.float32), np.array([y[2]], np.uint32).view(np.float32)
            np.testing.assert_allclose(l2a, l2b, rtol=1e-6)
        else:
            assert x == y, i


@pytest.mark.parametrize("kind,B", [("tsp50", 4), ("vrp20", 16), ("sp5", 16), ("dense", 0), ("tiny_d", 0)])
def test_rows_kernel_pack_matches_tile_kernel_and_sparse_ingestion(kind, B, monkeypatch):
    from cave_b200 import synth
    dev = torch.device("cuda:0")
    if kind == "dense":
        A = _special_dense(dev)
    elif kind == "tiny_d":
        rng = np.random.default_rng(2)
        An = rng.choice([0.0, 0.0, 1.0, -2.0], size=(5, 33, 3)).astype(np.float32)
        An[:, np.arange(33), np.arange(33) % 3] = 1.0      # no all-zero row: the sparse ingestion drops those
        A = torch.tensor(An, device=dev)
    else:
        A = synth.densify(synth.make_batch(kind, B, seed=21), device=dev)
    rows = _pack(A)
    monkeypatch.setenv("CAVE_SCAN_KERNEL", "tile")
    tile = _pack(A)
    monkeypatch.delenv("CAVE_SCAN_KERNEL")
    _assert_same(rows, tile, tol_avg_l2=True)
    integer = bool((A == A.round()).all())
    if integer:
        _assert_same(rows, _pack_sparse(A), tol_avg_l2=False)
    assert integer == (kind != "dense")
