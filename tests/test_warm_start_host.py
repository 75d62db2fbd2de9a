"""Warm start of the structured Newton solve from a pack's stored multipliers, on the CPU: the kernel source compiled for
the host (tests/hostsim_warm) reads, writes and falls back exactly as the solve kernel does, and the C ABI checks the
arguments of the warm entry points."""
import ctypes
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, golden_names
from oracle import cave_oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim_warm"))
import warm_sim as sim  # noqa: E402
from test_hostsim import _cmp  # noqa: E402

ST_WARM, ST_ITER_CAP, ST_STALLED = 0x400, 1, 2


def _structured(kind, n, seed, regime="near"):
    from cave_b200 import synth
    insts = synth.make_batch(kind, n, seed=seed)
    return synth.densify(insts).numpy(), synth.predictions(insts, seed, regime)


def _buffer(ctrs):
    return np.zeros(ctrs.shape[0] * sim.warm_slot_bytes(ctrs.shape[1]), np.uint8)


def _slots(warm, m):
    """(valid, nv, tag) per slot and a float64 view of the multipliers [N, cap]."""
    sb = sim.warm_slot_bytes(m)
    s = warm.reshape(-1, sb)
    hdr = s[:, :16].copy().view(np.int32)
    return hdr[:, 0], hdr[:, 1], hdr[:, 2], s[:, 16:]


def _nu(warm, m):
    return _slots(warm, m)[3].view(np.float64)


@pytest.mark.parametrize("kind", ["sp5", "tsp20", "vrp20"])
def test_same_predictions_restart_at_the_stored_solution(kind):
    ctrs, pred = _structured(kind, 16, 31)
    warm = _buffer(ctrs)
    cold = sim.forward_backward(pred, ctrs, mode=1, warm=warm)
    assert not (cold["status"] & ST_WARM).any()
    valid, nv, _, _ = _slots(warm, ctrs.shape[1])
    assert (valid == 1).all() and (nv > 0).all()               # every instance converged and was stored
    again = sim.forward_backward(pred, ctrs, mode=1, warm=warm)
    assert (again["status"] & ST_WARM).all()
    zero = again["iters"] == 0
    assert zero.sum() >= len(zero) // 2, again["iters"]
    for k in ("loss_i", "proj", "rnorm"):
        assert np.array_equal(again[k][zero], cold[k][zero])
    assert np.array_equal(again["grad"][zero], cold["grad"][zero])
    # a plain (cold) solve without a buffer is unchanged by all this
    plain = sim.forward_backward(pred, ctrs, mode=1)
    for k in ("loss_i", "grad", "proj", "status", "iters"):
        assert np.array_equal(plain[k], cold[k])


@pytest.mark.parametrize("kind", ["sp5", "tsp20", "vrp20"])
@pytest.mark.parametrize("f32", [False, True])
def test_perturbed_epochs_match_the_oracle_with_fewer_iterations(kind, f32):
    ctrs, pred = _structured(kind, 12, 7)
    rng = np.random.default_rng(3)
    warm = _buffer(ctrs)
    cold_iters, warm_iters = [], []
    p = pred.copy()
    for epoch in range(4):
        ref = O.forward_backward(p, ctrs, mode=1, fp64=True)
        out = sim.forward_backward(p, ctrs, mode=1, compute_f32=f32, warm=warm)
        _cmp(out, ref, 1)
        plain = sim.forward_backward(p, ctrs, mode=1, compute_f32=f32)
        cold_iters.append(plain["iters"].mean())
        if epoch > 0:
            assert (out["status"] & ST_WARM).all()
            warm_iters.append(out["iters"].mean())
        p = p * (1.0 + 1e-2 * rng.standard_normal(p.shape))
    assert np.mean(warm_iters) < np.mean(cold_iters[1:])


@pytest.mark.parametrize("fill", ["perturbed", "random", "negative", "nan", "torn"])
def test_any_slot_contents_are_only_a_starting_guess(fill):
    ctrs, pred = _structured("tsp20", 10, 13)
    m = ctrs.shape[1]
    warm = _buffer(ctrs)
    sim.forward_backward(pred, ctrs, mode=0, warm=warm)
    _, nv, _, _ = _slots(warm, m)
    nu = _nu(warm, m)
    rng = np.random.default_rng(5)
    for i, n in enumerate(nv):
        if fill == "perturbed":
            nu[i, :n] *= 1.0 + 0.3 * rng.standard_normal(n)
        elif fill == "random":
            nu[i, :n] = rng.random(n) * 10.0
        elif fill == "negative":
            nu[i, :n] = -1.0 - rng.random(n)
        elif fill == "nan":
            nu[i, :n] = np.where(rng.random(n) < 0.5, np.nan, np.inf)
        else:       # half of the values from another instance's solution, as when two writers of one slot interleave
            j = (i + 1) % len(nv)
            h = n // 2
            nu[i, :h] = nu[j, :h]
    ref = O.forward_backward(pred, ctrs, mode=0, fp64=True)
    out = sim.forward_backward(pred, ctrs, mode=0, warm=warm)
    _cmp(out, ref, 0)
    assert (out["status"] & ST_WARM).all()


@pytest.mark.parametrize("field", ["tag", "nv", "valid"])
def test_a_slot_of_other_variables_is_not_used(field):
    ctrs, pred = _structured("vrp20", 8, 17)
    m = ctrs.shape[1]
    warm = _buffer(ctrs)
    cold = sim.forward_backward(pred, ctrs, mode=1, warm=warm)
    sb = sim.warm_slot_bytes(m)
    s = warm.reshape(-1, sb)
    hdr = s[:, :16].view(np.int32)
    col = {"valid": 0, "nv": 1, "tag": 2}[field]
    hdr[:, col] += 1
    out = sim.forward_backward(pred, ctrs, mode=1, warm=warm)
    assert not (out["status"] & ST_WARM).any()
    assert np.array_equal(out["iters"], cold["iters"])           # started from zero
    for k in ("loss_i", "grad", "proj"):
        assert np.array_equal(out[k], cold[k])
    assert (s[:, :16].view(np.int32)[:, 0] == 1).all()           # ... and stored afresh


def test_failed_warm_start_falls_back_to_a_cold_solve():
    """max_iter = 1: a warm start from a poor guess cannot converge in one iteration; the instance is solved once more
    from zero in the same call, its iterations are the sum and the warm flag is clear."""
    ctrs, pred = _structured("tsp20", 6, 19)
    m = ctrs.shape[1]
    warm = _buffer(ctrs)
    sim.forward_backward(pred, ctrs, mode=0, warm=warm)
    _, nv, _, _ = _slots(warm, m)
    nu = _nu(warm, m)
    for i, n in enumerate(nv):
        nu[i, :n] = 5.0
    before = warm.copy()
    capped = sim.forward_backward(pred, ctrs, mode=0, max_iter=1)
    out = sim.forward_backward(pred, ctrs, mode=0, max_iter=1, warm=warm)
    failed = (capped["status"] & 0xff) != 0
    assert failed.any()
    assert not (out["status"][failed] & ST_WARM).any()
    assert np.array_equal(out["status"][failed], capped["status"][failed])
    assert (out["iters"][failed] == 1 + capped["iters"][failed]).all()
    assert np.array_equal(out["loss_i"][failed], capped["loss_i"][failed])
    sb = sim.warm_slot_bytes(m)
    for i in np.flatnonzero(failed):                             # not converged: the slot is left as it was
        assert np.array_equal(warm[i * sb:(i + 1) * sb], before[i * sb:(i + 1) * sb])


def test_index_with_duplicates_and_untouched_slots():
    ctrs, pred = _structured("sp5", 6, 23)
    m = ctrs.shape[1]
    warm = _buffer(ctrs)
    idx = np.array([0, 1, 2, 3, 4, 5, 5, 2, 0], np.int32)
    rng = np.random.default_rng(9)
    p = pred[idx] * (1.0 + 0.05 * rng.standard_normal((len(idx), pred.shape[1])))
    sim.forward_backward(p, ctrs, mode=1, index=idx, warm=warm)
    p = p * (1.0 + 0.01 * rng.standard_normal(p.shape))
    out = sim.forward_backward(p, ctrs, mode=1, index=idx, warm=warm)
    ref = O.forward_backward(p, ctrs[idx], mode=1, fp64=True)
    _cmp(out, ref, 1)
    assert (out["status"] & ST_WARM).all()
    # NaN prediction and heuristic mode leave the buffer byte for byte as it was
    before = warm.copy()
    bad = p.copy()
    bad[:, 0] = np.nan
    st = sim.forward_backward(bad, ctrs, mode=1, index=idx, warm=warm)["status"]
    assert ((st & 0xff) == 5).all() and np.array_equal(warm, before)
    st = sim.forward_backward(p, ctrs, mode=2, index=idx, warm=warm)["status"]
    assert ((st & 0xff) == 4).all() and not (st & ST_WARM).any() and np.array_equal(warm, before)


def test_lawson_hanson_instances_neither_read_nor_write():
    rng = np.random.default_rng(17)
    A = rng.standard_normal((6, 15, 10)).astype(np.float32)
    c = rng.standard_normal((6, 10)).astype(np.float32)
    warm = _buffer(A)
    warm[:] = 0xff                                              # garbage everywhere: must not matter, must not change
    before = warm.copy()
    out = sim.forward_backward(c, A, mode=0, warm=warm)
    _cmp(out, O.forward_backward(c, A, mode=0, fp64=True), 0)
    assert (out["status"] & 0x100).all() and not (out["status"] & ST_WARM).any()
    assert np.array_equal(warm, before)


@pytest.mark.parametrize("name", golden_names())
def test_golden_cases_warm(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    kw = dict(minimize=bool(z["minimize"]), mode=int(z["mode"]), inner_ratio=float(z["inner_ratio"]),
              reduction=str(z["reduction"]))
    ctrs = z["ctrs"]
    ref = O.forward_backward(z["pred"], ctrs, fp64=True, **kw)
    warm = _buffer(ctrs)
    for _ in range(2):
        out = sim.forward_backward(z["pred"], ctrs, warm=warm, **kw)
        _cmp(out, ref, kw["mode"])


# ---------------------------------------------------------------- C ABI argument checks (no device needed)
@pytest.fixture(scope="module")
def lib():
    from cave_b200 import _lib, build
    build.build()
    return _lib.load()


def test_warm_bytes(lib):
    n = ctypes.c_size_t()
    assert lib.cave_warm_bytes(10, 100, 50, ctypes.byref(n)) == 0 and n.value == 10 * (16 + 100 * 8)
    assert lib.cave_warm_bytes(3, 1000, 50, ctypes.byref(n)) == 0 and n.value == 3 * (16 + 256 * 8)      # at most 256 values
    assert lib.cave_warm_bytes(0, 10, 10, ctypes.byref(n)) == -1 and b"positive" in lib.cave_last_error()
    assert lib.cave_warm_bytes(1, 10, 10 ** 6, ctypes.byref(n)) == -2
    assert lib.cave_warm_bytes(1, 10, 10, None) == -1


def test_forward_backward_warm_argument_errors(lib):
    from cave_b200 import _lib
    B, m, d = 8, 40, 20
    fake = 1 << 20                 # aligned dummy device addresses: every check below fails before anything is launched
    n = ctypes.c_size_t()
    assert lib.cave_pack_bytes(B, m, d, ctypes.byref(n)) == 0
    pack_bytes = n.value
    opts = _lib.SolverOpts()
    assert lib.cave_scratch_bytes(B, m, d, _lib.F64, ctypes.byref(opts), ctypes.byref(n)) == 0
    scratch_bytes = n.value
    assert lib.cave_warm_bytes(B, m, d, ctypes.byref(n)) == 0
    warm_bytes = n.value

    def call(opts, warm, wbytes):
        return lib.cave_forward_backward_warm(fake, None, fake, B, m, d, -1.0, 1, 0.2, 0, _lib.F32, _lib.F64,
                                              ctypes.byref(opts) if opts is not None else None, fake, fake, fake, None,
                                              None, None, None, fake, pack_bytes, fake, scratch_bytes, warm, wbytes, None)

    assert call(_lib.SolverOpts(), fake, warm_bytes) == -1
    assert b"warm_pack" in lib.cave_last_error()
    assert call(None, fake, warm_bytes) == -1
    assert b"warm_pack" in lib.cave_last_error()
    ok = _lib.SolverOpts()
    ok.warm_pack = 1
    assert call(ok, None, warm_bytes) == -1
    assert b"warm must not be null" in lib.cave_last_error()
    assert call(ok, fake, warm_bytes - 1) == -3
    assert b"warm-start buffer" in lib.cave_last_error()
    assert call(ok, fake + 8, warm_bytes) == -1
    assert b"16-byte aligned" in lib.cave_last_error()
    # with an index the buffer is sized for the whole pack, not for the batch
    ok.inst_index = fake
    ok.n_packed = 4 * B
    assert lib.cave_pack_bytes(4 * B, m, d, ctypes.byref(n)) == 0
    pack_bytes = n.value
    assert call(ok, fake, warm_bytes) == -3
    assert str(4 * B).encode() in lib.cave_last_error()


def test_pack_dataclass_keeps_positional_fields():
    from cave_b200.qpsolver import CavePack
    p = CavePack(None, (1, 2, 3), 0, None, 0)
    assert p.warm is None
    p.reset_warm_start()                                        # nothing to reset
