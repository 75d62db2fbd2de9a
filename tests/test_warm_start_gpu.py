"""Warm start of a resident pack on the B200 (pack_constraints(..., warm_start=True)): every structured solve starts from
the instance's last converged multipliers.  Results must equal cold results within the parity tolerances, iterations
must drop, and the state must be left alone wherever the rules say so."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ST_WARM = 0x400


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _packs(kind, n, seed, dev, sparse):
    from cave_b200 import SparseConstraints, pack_constraints, pack_constraints_sparse, synth
    insts = synth.make_batch(kind, n, seed=seed)
    pred = torch.tensor(synth.predictions(insts, seed, "near"), device=dev)
    if sparse:
        sc = SparseConstraints.from_instances(insts)
        return pred, pack_constraints_sparse(sc, device=dev), pack_constraints_sparse(sc, device=dev, warm_start=True)
    A = synth.densify(insts, device=dev)
    return pred, pack_constraints(A), pack_constraints(A, warm_start=True)


def _call(pred, pack, idx, **kw):
    from cave_b200 import cave_forward_backward
    return cave_forward_backward(pred, None, -1.0, kw.pop("mode", 1), 0.2, "none", want_proj=True, want_status=True,
                                 pack=pack, index=idx, **kw)


def _close(a, b, rtol):
    for k in ("loss", "grad", "proj", "rnorm"):
        x, y = a[k].double().cpu().numpy(), b[k].double().cpu().numpy()
        np.testing.assert_allclose(x, y, rtol=rtol, atol=rtol * max(np.abs(y).max(), 1e-6), err_msg=k)


@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("kind", ["tsp20", "tsp50", "sp5", "vrp20"])
def test_perturbed_epochs_match_cold_with_fewer_iterations(kind, sparse):
    dev = _cuda()
    n = 96
    pred0, cold_pack, warm_pack = _packs(kind, n, 41, dev, sparse)
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(1)).to(dev, torch.int32)
    g = torch.Generator(device=dev).manual_seed(2)
    for precision, io in (("fp64", torch.float64), ("fp32", torch.float64), ("fp64", torch.float32)):
        warm_pack.reset_warm_start()
        p = pred0.to(io)
        cold_it, warm_it = [], []
        for epoch in range(4):
            c = _call(p[idx.long()], cold_pack, idx, precision=precision)
            w = _call(p[idx.long()], warm_pack, idx, precision=precision)
            assert ((c["status"] & 0xff) == 0).all() and ((w["status"] & 0xff) == 0).all()
            _close(w, c, 1e-6 if io == torch.float64 else 1e-4)
            if epoch:
                assert (w["status"] & ST_WARM).all()
                cold_it.append(c["iters"].double().mean().item())
                warm_it.append(w["iters"].double().mean().item())
            else:
                assert not (w["status"] & ST_WARM).any() and torch.equal(w["iters"], c["iters"])
            p = p * (1 + 1e-2 * torch.randn(p.shape, device=dev, generator=g, dtype=p.dtype))
        assert np.mean(warm_it) < np.mean(cold_it), (precision, io, warm_it, cold_it)


def test_identical_predictions_reproduce_bit_for_bit_and_reset():
    dev = _cuda()
    pred, cold_pack, pk = _packs("tsp50", 64, 43, dev, False)
    idx = torch.arange(64, dtype=torch.int32, device=dev)
    first = _call(pred, pk, idx)
    again = _call(pred, pk, idx)
    zero = again["iters"] == 0
    assert zero.float().mean() > 0.5 and (again["status"] & ST_WARM).all()
    for k in ("loss", "grad", "proj", "rnorm"):
        assert torch.equal(again[k][zero], first[k][zero]), k
    pk.reset_warm_start()
    assert int(pk.warm.count_nonzero()) == 0
    reset = _call(pred, pk, idx)
    assert torch.equal(reset["iters"], first["iters"]) and not (reset["status"] & ST_WARM).any()
    cold = _call(pred, cold_pack, idx)
    for k in ("loss", "grad", "proj", "status", "iters"):
        assert torch.equal(cold[k], first[k]), k


def test_heuristic_mode_and_nan_predictions_leave_the_state_alone():
    dev = _cuda()
    pred, cold_pack, pk = _packs("vrp20", 48, 47, dev, False)
    idx = torch.arange(48, dtype=torch.int32, device=dev)
    _call(pred, pk, idx)
    before = pk.warm.clone()
    h = _call(pred, pk, idx, mode=2)
    assert ((h["status"] & 0xff) == 4).all() and torch.equal(pk.warm, before)
    bad = pred.clone()
    bad[5, 0] = float("nan")
    out = _call(bad * 1.01, pk, idx)
    assert (out["status"][5] & 0xff) == 5
    slot = pk.warm.numel() // 48
    assert torch.equal(pk.warm[5 * slot:6 * slot], before[5 * slot:6 * slot])
    later = _call(pred * 1.01, pk, idx)
    cold = _call(pred * 1.01, cold_pack, idx)
    assert ((later["status"] & 0xff) == 0).all()
    _close(later, cold, 1e-6)


def test_duplicate_indices_with_different_predictions():
    dev = _cuda()
    n = 64
    pred, cold_pack, pk = _packs("tsp20", n, 53, dev, False)
    idx = torch.cat([torch.arange(n), torch.arange(n)]).to(dev, torch.int32)
    g = torch.Generator(device=dev).manual_seed(4)
    for epoch in range(3):
        p = pred[idx.long()] * (1 + 0.05 * torch.randn(2 * n, pred.shape[1], device=dev, generator=g, dtype=pred.dtype))
        w = _call(p, pk, idx)
        c = _call(p, cold_pack, idx)
        assert ((w["status"] & 0xff) == 0).all()
        _close(w, c, 1e-6)


def test_mixed_batch_non_newton_instances_carry_no_flag():
    """Dense rows without singleton rows take the Lawson-Hanson path (and, at >= 128 rows, the dense Gram path); in one
    resident pack with structured instances they match the oracle and never report a warm start."""
    from cave_b200 import cave_forward_backward, pack_constraints, synth
    from oracle import cave_oracle as O
    dev = _cuda()
    insts = synth.make_batch("sp5", 8, seed=59)
    S = synth.densify(insts).numpy()                       # [8, m, 40]
    m, d = S.shape[1], S.shape[2]
    rng = np.random.default_rng(59)
    M = max(m, 160)
    A = np.zeros((16, M, d), np.float32)
    A[:8, :m] = S
    A[8:12, :20] = rng.standard_normal((4, 20, d))          # Lawson-Hanson
    A[12:, :160] = rng.standard_normal((4, 160, d))         # dense (Gram) path
    At = torch.tensor(A, device=dev)
    pk = pack_constraints(At, warm_start=True)
    pred = np.concatenate([synth.predictions(insts, 59, "near"), rng.standard_normal((8, d))])
    p = torch.tensor(pred, device=dev)
    ref = O.forward_backward(pred, A, mode=0, fp64=True, reduction="none")
    for _ in range(2):
        out = cave_forward_backward(p, At, -1.0, 0, 0.2, "none", want_proj=True, want_status=True, pack=pk, dense="on")
        st = out["status"].cpu().numpy()
        assert not (st[8:] & ST_WARM).any() and (st[8:] & 0x300).all()
        np.testing.assert_allclose(out["loss"].cpu().numpy(), ref["loss"], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(out["proj"].cpu().numpy(), ref["proj"], rtol=1e-6, atol=1e-6 * np.abs(ref["proj"]).max())
    assert (st[:8] & ST_WARM).all()


def test_module_hybrid_sequence_matches_a_plain_pack():
    from cave_b200 import EPO, innerConeAlignedCosine, pack_constraints, synth
    dev = _cuda()
    insts = synth.make_batch("tsp20", 64, seed=61)
    A = synth.densify(insts, device=dev)
    plain, warm = pack_constraints(A), pack_constraints(A, warm_start=True)
    pred = torch.tensor(synth.predictions(insts, 61, "near"), device=dev)

    class Model:
        modelSense = EPO.MINIMIZE

    la = innerConeAlignedCosine(Model(), solver="cuda", seed=7)
    lb = innerConeAlignedCosine(Model(), solver="cuda", seed=7)
    g = torch.Generator(device=dev).manual_seed(8)
    for step in range(10):
        idx = torch.randint(0, 64, (32,), device=dev, generator=g).to(torch.int32)
        x = (pred[idx.long()] * (1 + 0.01 * step)).clone()
        pa, pb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        a = la(pa, plain, index=idx)
        b = lb(pb, warm, index=idx)
        a.backward()
        b.backward()
        assert torch.allclose(a, b, rtol=1e-6, atol=1e-9)
        assert torch.allclose(pa.grad, pb.grad, rtol=1e-5, atol=1e-9 * float(pa.grad.abs().max()))
