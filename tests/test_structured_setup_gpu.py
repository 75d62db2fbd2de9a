"""The structured (Newton) setup on the adversarial families of tests/adversarial.py, through every route that builds it:
the one-shot dense call (setup inside the solver), a resident pack with ``index=`` (the cached setup of setup_kernel
where the instance is eligible), the same pack with the cache switched off (CAVE_SETUP_CACHE=0), and a pack built from
the non-zeros alone (pack_constraints_sparse).  Every route is checked against the float64 oracle (certified
projection), against the optimality conditions of the projection on the device result, and, where the code promises
it, bit for bit against the other routes:

* int8 rows (every general value an integer in [-127, 127], packed CSR complete): exact int32 Hessian, CSC columns in
  variable order on every route => identical bits across routes and repeated calls;
* float rows: the Hessian is accumulated with float shared-memory atomics, so only a tolerance holds (1e-10 relative
  with the float64 factor; with the float32 factor the routes agree to the oracle tolerance)."""
import functools

import numpy as np
import pytest
import torch

import adversarial as adv
from oracle import cave_oracle as O
from test_cuda_parity import RTOL, _check
from test_structured_setup_host import check_stalled, clear_of_inside_threshold, fp32_stall

pytestmark = pytest.mark.gpu

ST_LH, ST_NOSPACE, ST_ITER_CAP = 0x100, 3, 1
POLAR = adv.REGIMES.index("polar")
KEYS = ("loss_i", "grad", "proj", "rnorm")


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@functools.lru_cache(maxsize=None)
def _data(name):
    A, pred, regime = adv.batch(name)
    m = A.shape[1]
    info = dict(
        newton=np.array([adv.has_singletons(a) for a in A]),
        int8=np.array([adv.is_int8(a, m) for a in A]),
        overflow=np.array([len(adv.general_rows(a)[adv.general_rows(a) != 0]) > adv.pack_cap_nnz(m, A.shape[2]) for a in A]))
    info["lh"] = ~info["newton"]
    info["bits"] = info["newton"] & info["int8"]
    return A, pred, regime, info


@functools.lru_cache(maxsize=None)
def _ref(name, mode):
    A, pred, _, _ = _data(name)
    return O.forward_backward(pred, A, mode=mode, reduction="none", fp64=True, certify=True)


def _np(o):
    return {k: v.detach().double().cpu().numpy() if v.dtype.is_floating_point else v.cpu().numpy() for k, v in o.items()}


def _routes(name, precision, io64, mode, monkeypatch):
    from cave_b200 import SparseConstraints, cave_forward_backward, pack_constraints, pack_constraints_sparse
    dev = _dev()
    A, pred, _, _ = _data(name)
    At = torch.tensor(A, device=dev)
    p = torch.tensor(pred, device=dev, dtype=torch.float64 if io64 else torch.float32)
    idx = torch.arange(len(A), dtype=torch.int32, device=dev)
    kw = dict(precision=precision, want_proj=True, want_status=True)
    call = lambda ctrs, **k: _np(cave_forward_backward(p, ctrs, -1.0, mode, 0.2, "none", **kw, **k))
    out = {"one_shot": [call(At) for _ in range(3)]}
    pk = pack_constraints(At)
    out["pack"] = call(At, pack=pk, index=idx)
    monkeypatch.setenv("CAVE_SETUP_CACHE", "0")
    out["pack_no_cache"] = call(At, pack=pk, index=idx)
    monkeypatch.delenv("CAVE_SETUP_CACHE")
    out["sparse"] = call(None, pack=pack_constraints_sparse(SparseConstraints.from_dense(At)), index=idx)
    return At, p, out


def _sub(o, keep):
    return {k: v[keep] for k, v in o.items()}


def _check_against_reference(o, ref, regime, pred, info, precision, mode, keep):
    """_check of test_cuda_parity on the instances `keep`, polar-cone predictions against 0 (see
    test_structured_setup_host.check_against_oracle), and the inside-the-cone classification of the inner loss."""
    rtol = RTOL[precision]
    sel = keep & (regime != POLAR)
    if mode == 1:
        clear = clear_of_inside_threshold(ref, pred)
        inside = O.INSIDE_TOL
        assert ((o["rnorm"] < inside) == (ref["rnorm"] < inside))[keep & clear].all()
        sel &= clear
    r = {k: ref[k][sel] for k in ("loss_i", "grad", "proj", "rnorm")}
    r["loss"] = r["loss_i"]
    s = _sub(o, sel)
    s["loss"] = s["loss_i"]
    _check(s, r, rtol, mode)
    polar = keep & (regime == POLAR)
    c = np.linalg.norm(pred[polar].astype(np.float64), axis=1)
    assert (np.linalg.norm(o["proj"][polar], axis=1) <= 1e-2 * rtol * c + 1e-12).all()
    np.testing.assert_allclose(o["rnorm"][polar], c, rtol=rtol, atol=1e-12)


def _certificate(A, pred, o, keep, regime, At, precision):
    """Optimality of the device projection in float64, without scipy: q = c - p in the polar cone, <p, q> = 0, and p
    projects onto itself.  The bound is 1e-7 relative: the solver stops at a KKT residual of about 1e-8 relative (the
    kernel source reaches 1.3e-8 on mixed_batch), so 1e-9 would assert what it never promised."""
    from cave_b200 import cave_forward_backward
    c = -pred.astype(np.float64)
    for b in np.flatnonzero(keep):
        a = A[b].astype(np.float64)
        p = o["proj"][b]
        q = c[b] - p
        cn, an = np.linalg.norm(c[b]), np.linalg.norm(a, axis=1).max()
        assert (a @ q).max() <= 1e-7 * cn * an, (b, (a @ q).max() / (cn * an))
        assert abs(p @ q) <= 1e-7 * cn * cn, (b, abs(p @ q) / (cn * cn))
    # p projects onto itself: a second solve, from p, stops at its own relative residual, hence 1e-6
    again = keep
    pb = torch.tensor(o["proj"][again], device=At.device)
    o2 = cave_forward_backward(pb, At[torch.tensor(np.flatnonzero(again), device=At.device)], 1.0, 0, reduction="none",
                               precision=precision, want_proj=True, want_status=True)
    # the second solve starts at a point on a face of the cone; on the most degenerate cones (setup_cap) it may use all
    # its iterations: then it must still have returned p (checked below), never another point under status 0
    st2 = (o2["status"] & 0xff).cpu().numpy()
    assert np.isin(st2, (0, ST_ITER_CAP)).all(), st2
    p2 = o2["proj"]
    cn = torch.tensor(np.linalg.norm(c[again], axis=1), device=At.device)
    err = ((p2 - pb).norm(dim=1) / cn).cpu().numpy()
    assert (err <= 1e-6).all(), (np.flatnonzero(again)[err > 1e-6], err.max())


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("io64", [True, False])
@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("name", adv.FAMILIES)
def test_structured_setup_routes_match_the_oracle_and_each_other(name, precision, io64, mode, monkeypatch):
    A, pred, regime, info = _data(name)
    ref = _ref(name, mode)
    At, _, out = _routes(name, precision, io64, mode, monkeypatch)
    needs_dense = info["lh"] | info["overflow"]
    routes = [("one_shot", out["one_shot"][0]), ("pack", out["pack"]), ("pack_no_cache", out["pack_no_cache"]),
              ("sparse", out["sparse"])]
    for route, o in routes:
        st = o["status"]
        valid = ~needs_dense if route == "sparse" else np.ones(len(A), bool)
        if route == "sparse":       # no dense rows on the device: instances that need them must report, not guess
            assert ((st[needs_dense] & 0xff) == ST_NOSPACE).all(), route
        # which path ran: Newton for every instance with a singleton row, Lawson-Hanson for the others
        assert ((st[valid] & ST_LH) != 0).tolist() == info["lh"][valid].tolist(), route
        # the instances the float32 factor cannot finish (test_structured_setup_host.fp32_stall): flagged, checked
        stall = fp32_stall(name, A, regime) & (precision == "fp32")
        capped = (st & 0xff) == ST_ITER_CAP
        assert not (capped & ~stall).any(), (route, np.flatnonzero(capped))
        check_stalled(o, ref, stall & capped, mode)
        keep = valid & ~stall
        _check_against_reference(o, ref, regime, pred, info, precision, mode, keep)
        if io64 and route in ("one_shot", "pack"):      # float32 output rounds p beyond the certificate's bound
            _certificate(A, pred, o, keep & (regime != POLAR), regime, At, precision)
    # bit for bit where the code promises it: int8 rows, every route and repeated calls
    base = out["one_shot"][0]
    others = [o for _, o in routes[1:]] + out["one_shot"][1:]
    for o in others:
        for k in KEYS:
            assert np.array_equal(o[k][info["bits"]], base[k][info["bits"]]), (k, np.flatnonzero(
                (o[k][info["bits"]] != base[k][info["bits"]]).reshape(int(info["bits"].sum()), -1).any(axis=1)))
    # float rows: a tolerance (float atomics in the Hessian); 1e-10 relative with the float64 factor
    flt = info["newton"] & ~info["int8"] & ~info["overflow"]
    if precision == "fp64" and io64 and flt.any():
        for o in others:
            for k in KEYS:
                x, y = o[k][flt].reshape(int(flt.sum()), -1), base[k][flt].reshape(int(flt.sum()), -1)
                scale = np.maximum(np.abs(y).max(axis=1, keepdims=True), 1.0 if k == "loss_i" else 1e-30)
                assert (np.abs(x - y) <= 1e-10 * scale).all(), k


@pytest.mark.parametrize("cfg", range(5))
def test_every_solve_configuration_on_one_family(cfg, monkeypatch):
    """CAVE_SOLVE_CFG forces one launch configuration (threads x CTAs/SM, and the wide one): one family each."""
    name = adv.FAMILIES[cfg]
    A, pred, regime, info = _data(name)
    ref = _ref(name, 1)
    monkeypatch.setenv("CAVE_SOLVE_CFG", str(cfg))
    from cave_b200 import cave_forward_backward
    o = _np(cave_forward_backward(torch.tensor(pred, device=_dev(), dtype=torch.float64), torch.tensor(A, device=_dev()),
                                  -1.0, 1, 0.2, "none", want_proj=True, want_status=True))
    assert ((o["status"] & 0xff) == 0).all() and ((o["status"] & ST_LH) == 0).all()
    _check_against_reference(o, ref, regime, pred, info, "fp64", 1, np.ones(len(A), bool))


def test_csr_overflow_without_dense_rows_reports_nospace():
    """General rows beyond the packed CSR: with the dense rows dropped the solver cannot read them back from A and
    must report ST_NOSPACE (NaN results); the instance that fits is solved."""
    from cave_b200 import cave_forward_backward, pack_constraints
    A, pred, regime, info = _data("csr_overflow")
    dev = _dev()
    pk = pack_constraints(torch.tensor(A, device=dev), keep_dense=False)
    o = _np(cave_forward_backward(torch.tensor(pred, device=dev, dtype=torch.float64), None, -1.0, 0, 0.0, "none",
                                  want_proj=True, want_status=True, pack=pk,
                                  index=torch.arange(len(A), dtype=torch.int32, device=dev)))
    st = o["status"] & 0xff
    assert info["overflow"].any() and (st[info["overflow"]] == ST_NOSPACE).all()
    assert np.isnan(o["loss_i"][info["overflow"]]).all()
    assert (st[~info["overflow"]] == 0).all()
    _check_against_reference(o, _ref("csr_overflow", 0), regime, pred, info, "fp64", 0, ~info["overflow"])
