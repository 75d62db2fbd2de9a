"""The oracle against the golden vectors produced by the unmodified reference
(tests/golden/make_golden.py) and against the reference's known-answer cases (SURVEY.md §8c)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_names
from oracle import cave_oracle as O


def _load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: z[k] for k in z.files}


@pytest.mark.parametrize("name", golden_names())
def test_oracle_matches_reference_golden(name):
    g = _load(name)
    out = O.forward_backward(g["pred"], g["ctrs"], minimize=bool(g["minimize"]), mode=int(g["mode"]),
                             inner_ratio=float(g["inner_ratio"]), reduction=str(g["reduction"]), fp64=False)
    # float32 reference arithmetic: torch vs numpy summation order only
    np.testing.assert_allclose(out["loss"], g["loss"], rtol=2e-5, atol=3e-7)
    np.testing.assert_allclose(out["grad"], g["grad"], rtol=2e-4, atol=2e-7 * max(1.0, np.abs(g["grad"]).max()))
    if int(g["mode"]) != O.MODE_HEURISTIC:
        np.testing.assert_allclose(out["proj"], g["proj"], rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(out["rnorm"], g["rnorm"], rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("name", ["tf_randn_exact", "sp5_exact_near", "tsp20_inner_near", "vrp20_inner_near"])
def test_oracle_fp64_mode_close_to_fp32_reference(name):
    g = _load(name)
    out = O.forward_backward(g["pred"], g["ctrs"], minimize=bool(g["minimize"]), mode=int(g["mode"]),
                             inner_ratio=float(g["inner_ratio"]), reduction=str(g["reduction"]), fp64=True)
    np.testing.assert_allclose(out["loss"], g["loss"], rtol=1e-3, atol=1e-6)
    np.testing.assert_allclose(out["proj"], g["proj"], rtol=1e-5, atol=1e-5)


def test_lawson_hanson_restatement_matches_scipy():
    from scipy.optimize import nnls
    rng = np.random.default_rng(0)
    for (m, d) in [(15, 10), (5, 8), (40, 12), (64, 190)]:
        for _ in range(5):
            A = rng.standard_normal((m, d))
            c = rng.standard_normal(d)
            x_ref, rn_ref = nnls(A.T, c)
            x, rn = O.lawson_hanson(A.T, c)
            np.testing.assert_allclose(x @ A, x_ref @ A, rtol=1e-9, atol=1e-10)
            assert abs(rn - rn_ref) <= 1e-9 * max(1.0, rn_ref)


def test_kat_rand_data_gives_unit_loss_zero_grad():
    # test/test_func.py:34-43 data: c <= 0, A >= 0 -> lambda = 0 -> loss 1, grad 0
    g = _load("tf_rand_exact")
    out = O.forward_backward(g["pred"], g["ctrs"], fp64=True)
    assert out["loss"] == pytest.approx(1.0, abs=1e-12)
    assert np.abs(out["grad"]).max() == 0.0


def test_kat_identity_cone_is_positive_part():
    rng = np.random.default_rng(1)
    c = rng.standard_normal((3, 7))
    A = np.broadcast_to(np.eye(7), (3, 7, 7)).copy()
    proj, rnorm = O.batch_project(c, A, fp64=True)
    np.testing.assert_allclose(proj, np.maximum(c, 0.0), atol=1e-14)


def test_kat_empty_cone_returns_cost():
    c = np.arange(1.0, 6.0)[None]
    proj, rnorm = O.batch_project(c, np.zeros((1, 4, 5)), fp64=True)
    np.testing.assert_array_equal(proj, c)
    assert rnorm[0] == 0.0


def test_kat_moreau_kkt():
    rng = np.random.default_rng(2)
    A = rng.standard_normal((1, 12, 9))
    c = rng.standard_normal((1, 9))
    proj, rnorm = O.batch_project(c, A, fp64=True)
    q = c[0] - proj[0]
    assert (A[0] @ q).max() <= 1e-10
    assert abs(proj[0] @ q) <= 1e-10


def test_padded_rows_do_not_change_anything():
    rng = np.random.default_rng(3)
    A = rng.standard_normal((2, 5, 6)).astype(np.float32)
    c = rng.standard_normal((2, 6)).astype(np.float32)
    Ap = np.concatenate([A, np.zeros((2, 10, 6), np.float32)], axis=1)
    for mode in (O.MODE_EXACT, O.MODE_INNER, O.MODE_HEURISTIC):
        a = O.forward_backward(c, A, mode=mode, fp64=True)
        b = O.forward_backward(c, Ap, mode=mode, fp64=True)
        np.testing.assert_allclose(a["loss"], b["loss"], atol=1e-14)
        np.testing.assert_allclose(a["grad"], b["grad"], atol=1e-14)


def test_analytic_gradient_matches_autograd():
    import torch
    import torch.nn.functional as F
    rng = np.random.default_rng(4)
    c = rng.standard_normal((5, 9))
    t = rng.standard_normal((5, 9))
    c[3] *= 1e-10          # below the eps clamp
    loss, grad = O.cosine_loss_and_grad(c, t)
    ct = torch.tensor(c, requires_grad=True)
    lt = 1.0 - F.cosine_similarity(ct, torch.tensor(t), dim=1)
    lt.sum().backward()
    np.testing.assert_allclose(loss, lt.detach().numpy(), rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(grad, ct.grad.numpy(), rtol=1e-9, atol=1e-12)


def test_certified_projection_meets_the_optimality_conditions_on_degenerate_cones():
    """certify=True: on cones with duplicated and opposite rows (tests/adversarial.py pm_pairs) every projection meets
    is_projection and equals the independent Lawson-Hanson restatement, whatever scipy's nnls returned."""
    import adversarial as adv
    A, pred, _ = adv.batch("pm_pairs")
    for b in range(0, len(A), 3):
        a = A[b][np.abs(A[b]).sum(axis=1) > 0].astype(np.float64)
        c = -pred[b].astype(np.float64)
        p, r = O.project_nnls(c, a, fp64_out=True, certify=True)
        assert O.is_projection(c, a, p)
        lam, r_lh = O.lawson_hanson(a.T, c)
        np.testing.assert_allclose(p, lam @ a, rtol=1e-9, atol=1e-10 * np.linalg.norm(c))
        np.testing.assert_allclose(r, r_lh, rtol=1e-9, atol=1e-12)
