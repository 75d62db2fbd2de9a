"""
CPU ORACLE for the CaVE cone-projection hot path.  TEST INFRASTRUCTURE ONLY.

This file is the checker, never the product: only tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline / ``--impl reference`` legs may import it.  Nothing
under cave_b200/ imports it, and the product path raises if its CUDA library is
missing instead of falling back to this code.

It restates, in numpy, the reference algorithm of khalil-research/CaVE
(/root/reference, read-only) for the path BASELINE.json names.  Every function
cites the reference lines it follows.

Where the arithmetic lives: the reference's NNLS projection calls the third-party
``scipy.optimize.nnls`` (src/cave.py:307; README.md:47 pins SciPy 1.11.2, this image
has SciPy 1.18.1 — both are Lawson-Hanson active-set solvers; the projection
A^T lambda is unique so the version does not matter at 1e-5).  ``project_nnls``
calls the same SciPy routine the reference calls; ``lawson_hanson`` is an
independent restatement of the published algorithm (Lawson & Hanson, "Solving
Least Squares Problems", 1974, ch. 23) used to cross-check SciPy and as the
solver when SciPy is absent.

Parity pinning: the reference's own tests hold no golden vectors for this path
(SURVEY.md §8c).  The oracle is pinned instead against outputs of the UNMODIFIED
reference executed in the build container (tests/golden/make_golden.py imports
/root/reference/src/cave.py with a 3-symbol PyEPO stand-in and stores its
loss / gradient / projection for fixed seeds in tests/golden/*.npz);
tests/test_oracle.py replays them.  The Clarabel (``max_iter=3``) backend cannot
be executed here (cvxpy/clarabel absent): parity for that backend is UNPINNED.
"""
from __future__ import annotations

import numpy as np

try:  # the reference's own dependency (src/cave.py:14)
    from scipy.optimize import nnls as _scipy_nnls
except Exception:  # pragma: no cover
    _scipy_nnls = None

EPS_COS = 1e-8      # torch.nn.functional.cosine_similarity default eps (src/cave.py:72)
ROW_TOL = 1e-7      # zero-row threshold (src/cave.py:303) and norm threshold (src/cave.py:225)
INSIDE_TOL = 1e-7   # rnorm < 1e-7 -> projection already inside the cone (src/cave.py:218)

MODE_EXACT, MODE_INNER, MODE_HEURISTIC = 0, 1, 2


# --------------------------------------------------------------------------- NNLS
def lawson_hanson(E: np.ndarray, f: np.ndarray, max_iter: int | None = None, tol: float | None = None):
    """min ||E x - f||_2 s.t. x >= 0 by the Lawson-Hanson active-set method (published
    algorithm NNLS, Lawson & Hanson 1974, ch. 23, steps 1-12).  Returns (x, rnorm)."""
    E = np.asarray(E, dtype=np.float64)
    f = np.asarray(f, dtype=np.float64)
    n = E.shape[1]
    max_iter = 3 * n if max_iter is None else max_iter
    tol = 10 * max(E.shape) * np.finfo(np.float64).eps * max(np.abs(E.T @ f).max(initial=0.0), 1e-300) \
        if tol is None else tol
    x = np.zeros(n)
    passive = np.zeros(n, dtype=bool)
    w = E.T @ (f - E @ x)
    it = 0
    while (not passive.all()) and w[~passive].max(initial=-np.inf) > tol:
        cand = np.where(~passive, w, -np.inf)
        j = int(np.argmax(cand))
        passive[j] = True
        s = np.zeros(n)
        s[passive] = np.linalg.lstsq(E[:, passive], f, rcond=None)[0]
        if s[j] <= 0:           # step 6 guard: numerically dependent column
            passive[j] = False
            w[j] = 0.0
            continue
        while s[passive].min() <= 0:
            it += 1
            if it > max_iter:
                raise RuntimeError("Maximum number of iterations reached.")
            mask = passive & (s <= 0)
            alpha = np.min(x[mask] / (x[mask] - s[mask]))
            x = x + alpha * (s - x)
            passive &= x > 1e-15 * max(np.abs(x).max(), 1e-300)
            x[~passive] = 0.0
            s = np.zeros(n)
            if passive.any():
                s[passive] = np.linalg.lstsq(E[:, passive], f, rcond=None)[0]
        x = s
        w = E.T @ (f - E @ x)
    return x, float(np.linalg.norm(E @ x - f))


def is_projection(c: np.ndarray, ctr: np.ndarray, p: np.ndarray, tol: float = 1e-9) -> bool:
    """Optimality conditions of p = lam @ ctr (lam >= 0) as the projection of c onto cone(ctr), in float64:
    q = c - p lies in the polar cone (ctr q <= tol ||c|| max ||a_i||) and is orthogonal to p (|<p, q>| <= tol ||c||^2)."""
    c, ctr, p = (np.asarray(x, np.float64) for x in (c, ctr, p))
    q = c - p
    cn = float(np.linalg.norm(c))
    an = float(np.linalg.norm(ctr, axis=1).max(initial=0.0))
    return float((ctr @ q).max(initial=0.0)) <= tol * cn * an and abs(float(p @ q)) <= tol * cn * cn


def project_nnls(cp: np.ndarray, ctr: np.ndarray, fp64_out: bool = False, use_scipy: bool = True, certify: bool = False):
    """src/cave.py:298-309 `_project_nnls`: drop zero rows (303); empty -> (cp, 0.0) (304-305);
    nnls(ctr.T, cp) (306-307); p = lam @ ctr, cast float32 (308-309).
    fp64_out=True returns the float64 projection *before* the float32 cast.
    certify=True: a SciPy result that fails `is_projection` is replaced by `lawson_hanson`'s, which must pass it (the
    installed SciPy's nnls can stop at a non-optimal point on degenerate cones, e.g. rows a, a, -a, -a)."""
    ctr = ctr[np.abs(ctr).sum(axis=1) > ROW_TOL]
    if len(ctr) == 0:
        return (cp.astype(np.float64) if fp64_out else cp.astype(np.float32)), 0.0
    if use_scipy and _scipy_nnls is not None:
        lam, rnorm = _scipy_nnls(np.asfortranarray(ctr.T), cp)
        if certify and not is_projection(cp, ctr, lam @ ctr):
            lam, rnorm = lawson_hanson(ctr.T, cp)
            if not is_projection(cp, ctr, lam @ ctr):
                raise RuntimeError("neither nnls nor lawson_hanson meets the optimality conditions")
    else:
        lam, rnorm = lawson_hanson(ctr.T, cp)
    p = lam @ ctr
    return (np.asarray(p, dtype=np.float64) if fp64_out else p.astype(np.float32)), float(rnorm)


def batch_project(signed_cost: np.ndarray, tight_ctrs: np.ndarray, fp64: bool = False, certify: bool = False):
    """src/cave.py:231-264 `_batch_project`, solver='nnls', processes=1 (line 257):
    stack per-instance results; rnorm goes through float32 (line 261) unless fp64.  certify: see project_nnls."""
    res = [project_nnls(signed_cost[i], tight_ctrs[i], fp64_out=fp64, certify=certify) for i in range(len(signed_cost))]
    proj = np.stack([r[0] for r in res])
    rnorm = np.asarray([r[1] for r in res], dtype=np.float64 if fp64 else np.float32)
    dt = np.float64 if fp64 else signed_cost.dtype
    return proj.astype(dt), rnorm.astype(dt)


# --------------------------------------------------------------------------- targets
def average_ctrs(tight_ctrs: np.ndarray) -> np.ndarray:
    """src/cave.py:222-228 `_average_ctrs`: mean of unit-normalised rows; rows with norm <= 1e-7
    (padding) excluded; count clamped >= 1.  Computed in the dtype of `tight_ctrs`."""
    norms = np.sqrt((tight_ctrs * tight_ctrs).sum(axis=2, keepdims=True))
    valid = (norms > ROW_TOL).astype(tight_ctrs.dtype)
    unit = tight_ctrs / np.maximum(norms, 1e-8) * valid
    n_valid = np.maximum(valid.sum(axis=1), 1.0)
    return unit.sum(axis=1) / n_valid


def _normalise(v: np.ndarray) -> np.ndarray:
    return v / np.maximum(np.linalg.norm(v, axis=1, keepdims=True), 1e-8)


def exact_target(signed_cost, tight_ctrs, fp64=False, certify=False):
    """src/cave.py:121-129: proj / ||proj||.clamp(1e-8)."""
    proj, rnorm = batch_project(signed_cost, tight_ctrs, fp64, certify)
    return _normalise(proj), proj, rnorm


def heuristic_target(signed_cost, tight_ctrs, inner_ratio):
    """src/cave.py:202-204: (1-r) * c/||c|| + r * avg."""
    avg = average_ctrs(tight_ctrs).astype(signed_cost.dtype)
    return (1 - inner_ratio) * _normalise(signed_cost) + inner_ratio * avg


def inner_target(signed_cost, tight_ctrs, inner_ratio, fp64=False, certify=False):
    """src/cave.py:206-219, solver='nnls' branch: where(rnorm < 1e-7, proj_norm, (1-r) proj_norm + r avg)."""
    proj, rnorm = batch_project(signed_cost, tight_ctrs, fp64, certify)
    proj_norm = _normalise(proj)
    avg = average_ctrs(tight_ctrs).astype(proj.dtype)
    pushed = (1 - inner_ratio) * proj_norm + inner_ratio * avg
    inside = (rnorm < INSIDE_TOL)[:, None]
    return np.where(inside, proj_norm, pushed), proj, rnorm


# --------------------------------------------------------------------------- loss + backward
def cosine_loss_and_grad(c: np.ndarray, t: np.ndarray):
    """loss_i = 1 - cosine_similarity(c_i, t_i) (src/cave.py:72) and d loss_i / d c_i with t constant
    (src/cave.py:70-71).  torch semantics (ATen cosine_similarity): both norms are clamped at eps on a
    clone outside the graph, so the division uses n = max(||c||, eps) while the norm's own backward
    uses the true norm (0 where ||c|| == 0).  With u = c/n, v = t/max(||t||, eps), w = c/||c||:
        cos = u.v ,  dloss/dc = -(v - cos*w) / n      (== SURVEY.md App. A.3 whenever ||c|| >= eps)."""
    nrm = np.linalg.norm(c, axis=1, keepdims=True)
    n_c = np.maximum(nrm, EPS_COS)
    n_t = np.maximum(np.linalg.norm(t, axis=1, keepdims=True), EPS_COS)
    u, v = c / n_c, t / n_t
    w = np.divide(c, nrm, out=np.zeros_like(c), where=nrm > 0)
    cos = (u * v).sum(axis=1)
    grad_c = -(v - cos[:, None] * w) / n_c
    return 1.0 - cos, grad_c


def forward_backward(pred_cost: np.ndarray, tight_ctrs: np.ndarray, minimize: bool = True,
                     mode: int = MODE_EXACT, inner_ratio: float = 0.2, reduction: str = "mean",
                     fp64: bool = False, certify: bool = False):
    """src/cave.py:55-73 `forward` + autograd backward of the reduced loss w.r.t. pred_cost.

    mode: MODE_EXACT (exactConeAlignedCosine), MODE_INNER (innerConeAlignedCosine QP branch,
    solver='nnls'), MODE_HEURISTIC (innerConeAlignedCosine heuristic branch, src/cave.py:201-204).
    fp64=True: all arithmetic in float64 without the reference's float32 casts (parity target for
    the CUDA path's fp64 mode); fp64=False: follows the reference's dtypes (float32 in / out).
    certify=True: every projection meets its optimality conditions (see project_nnls).
    Returns dict(loss, loss_i, grad, proj, rnorm, target)."""
    dt = np.float64 if fp64 else pred_cost.dtype
    pred = pred_cost.astype(dt)
    ctrs = tight_ctrs.astype(np.float64) if fp64 else tight_ctrs
    sign = -1.0 if minimize else 1.0                       # src/cave.py:62-68
    c = (sign * pred).astype(dt)
    proj = rnorm = None
    if mode == MODE_HEURISTIC:
        t = heuristic_target(c, ctrs, inner_ratio)
    elif mode == MODE_INNER:
        t, proj, rnorm = inner_target(c, ctrs, inner_ratio, fp64, certify)
    else:
        t, proj, rnorm = exact_target(c, ctrs, fp64, certify)
    t = t.astype(dt)
    loss_i, grad_c = cosine_loss_and_grad(c, t)
    B = len(pred)
    if reduction == "mean":                                # optModule._reduce (src/cave.py:73)
        loss, scale = loss_i.mean(), 1.0 / B
    elif reduction == "sum":
        loss, scale = loss_i.sum(), 1.0
    elif reduction == "none":
        loss, scale = loss_i, 1.0
    else:
        raise ValueError(f"invalid reduction {reduction!r}")
    grad = (sign * scale * grad_c).astype(dt)              # upstream gradient of ones
    return dict(loss=loss, loss_i=loss_i.astype(dt), grad=grad, proj=proj, rnorm=rnorm, target=t)
