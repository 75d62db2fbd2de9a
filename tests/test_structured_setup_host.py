"""The kernel source (tests/hostsim: solver_core.cuh compiled for the CPU, one thread) on the adversarial families of
tests/adversarial.py against the float64 oracle.  This checks the generator, the references and the algorithm of the
Newton setup (+- merge, int8 / float rows, CSR read back from A, cone types) without a GPU.  One thread fills every CSC
column in variable order, so the order-dependent defects of the GPU setup are the business of
test_structured_setup_gpu.py."""
import os
import sys

import numpy as np
import pytest

import adversarial as adv
from oracle import cave_oracle as O
from test_hostsim import _cmp

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim"))
import sim  # noqa: E402

POLAR = adv.REGIMES.index("polar")


def clear_of_inside_threshold(ref, pred):
    """Instances whose reference rnorm is further from the inside-the-cone threshold (rnorm < 1e-7, absolute) than the
    solver's stopping residual (relative to ||c||) reaches: only there is the push-inside decision of the inner loss
    defined to the solver's tolerance (an instance inside the cone with ||c|| = 340 stops at rnorm ~2e-7)."""
    band = 1e-9 * np.linalg.norm(pred.astype(np.float64), axis=1)
    return np.abs(np.asarray(ref["rnorm"], np.float64) - O.INSIDE_TOL) > band


def check_against_oracle(out, ref, regime, pred, mode, cmp=_cmp, skip=None):
    """`cmp` against the oracle on every instance whose projection is defined to a relative tolerance (in inner mode,
    clear of the inside threshold: see clear_of_inside_threshold).  A polar-cone
    prediction projects to 0, and that is what its projection and rnorm are checked against (where the cone is all of
    R^d the polar point is 0 up to rounding: hence the absolute floor).  Its loss and gradient are left out: they are
    the cosine with the direction of a projection of rounding size, which no tolerance pins down."""
    keep = regime != POLAR
    if skip is not None:
        keep &= ~skip
    if mode == 1:
        keep &= clear_of_inside_threshold(ref, pred)
    sub = lambda o: {k: (v[keep] if isinstance(v, np.ndarray) and v.ndim else v) for k, v in o.items()}
    cmp(sub(out), sub(ref), mode)
    polar = regime == POLAR
    c = np.linalg.norm(pred[polar].astype(np.float64), axis=1)
    assert (np.linalg.norm(np.asarray(out["proj"][polar], np.float64), axis=1) <= 1e-7 * c + 1e-12).all()
    np.testing.assert_allclose(np.asarray(out["rnorm"][polar], np.float64), c, rtol=1e-6, atol=1e-12)


def fp32_stall(name, A, regime):
    """The two instances the float32 factor cannot finish: int8_edges #2 (float rows of +-1 beside +-127 and a -128)
    with costs scaled by 1e4, and int8_edges #3 (the same with a 0.5) with costs inside the cone.  The Tikhonov term of
    the float32 factor (2e-6 max_i ||b_i||^2) swamps the diagonal of the short rows there, and the Newton steps crawl;
    the solver reports ITER_CAP for these, and only these (asserted; an open defect of the float32 factor)."""
    if name != "int8_edges":
        return np.zeros(len(A), bool)
    v = np.arange(len(A)) % (len(A) // len(adv.REGIMES))
    return ((v == 2) & (regime == adv.REGIMES.index("huge"))) | ((v == 3) & (regime == adv.REGIMES.index("inside")))


def check_stalled(out, ref, stall, mode):
    """A stalled instance is flagged (status ITER_CAP, asserted by the callers) and returns finite numbers; its
    projection is not the reference's (several per cent off), which is what the flag tells the caller."""
    for k in ("loss_i", "proj", "rnorm"):
        assert np.isfinite(np.asarray(out[k][stall], np.float64)).all(), k


@pytest.mark.parametrize("f32", [False, True])
@pytest.mark.parametrize("name", adv.FAMILIES)
def test_kernel_source_on_adversarial_families(name, f32):
    A, pred, regime = adv.batch(name)
    # the CPU pack holds every general row; force_path bit 1 makes the solver read its rows back from A, as the GPU
    # solver does for the instances this family overflows the packed CSR with
    force = 2 if name == "csr_overflow" else 0
    stall = fp32_stall(name, A, regime) if f32 else np.zeros(len(A), bool)
    for mode in (0, 1):
        ref = O.forward_backward(pred, A, mode=mode, reduction="none", fp64=True, certify=True)
        out = sim.forward_backward(pred, A, mode=mode, reduction="none", compute_f32=f32, force_path=force)
        assert ((out["status"] & 0xff) == 1).tolist() == stall.tolist()
        # rtol: the float64 tolerance of the GPU tests.  _cmp's 1e-6 assumes costs of order one: at 1e-4 the gradient
        # scales like 1/||c||, at 1e4 a long_column projection ends 2e-7 from the reference, and _cmp's absolute
        # floors follow the largest rnorm of the batch, which these regimes spread over eight decades
        check_against_oracle(out, ref, regime, pred, mode, cmp=lambda o, r, md: _cmp(o, r, md, rtol=1e-5), skip=stall)
        check_stalled(out, ref, stall, mode)
        lh = np.array([not adv.has_singletons(a) for a in A])
        assert ((out["status"] & 0x100) != 0).tolist() == (lh & (np.abs(A).sum(axis=(1, 2)) > 0)).tolist()


def test_generator_is_seeded_and_keeps_its_promises():
    for name in adv.FAMILIES:
        A, pred, regime = adv.batch(name)
        A2, pred2, _ = adv.batch(name)
        assert np.array_equal(A, A2) and np.array_equal(pred, pred2)
        assert A.dtype == np.float32 and pred.dtype == np.float32 and A.shape[2] <= 400 and A.shape[1] <= 700
        if name != "mixed_batch":
            assert all(adv.has_singletons(a) for a in A), name
    # the branches the families aim at are reached
    m = adv.family("long_column").shape[1]
    for a in adv.family("long_column")[:2]:
        g = adv.general_rows(a)
        assert sorted((g != 0).sum(axis=0))[-3:] == [65, 100, 250] and (g != 0).sum(axis=1).max() > 256
        assert adv.is_int8(a, m) and len(g) <= 256
    A = adv.family("setup_cap")
    assert [len(adv.general_rows(a)) for a in A] == [192, 193, 256, 257, 257]
    A = adv.family("csr_overflow")
    assert [adv.is_int8(a, A.shape[1]) for a in A] == [False, False, True]
    assert (A[0] != 0).sum() - ((A[0] != 0).sum(axis=1) == 1).sum() > adv.pack_cap_nnz(A.shape[1], A.shape[2])
    A = adv.family("int8_edges")
    assert [adv.is_int8(a, A.shape[1]) for a in A] == [True, False, False, False, True, True]
    assert np.signbit(A[4][A[4] == 0]).any()
    A = adv.family("mixed_batch")
    assert sum(not adv.has_singletons(a) for a in A) == 2
