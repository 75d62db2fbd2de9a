"""Warm start of the dense Gram-space Newton solve on the B200 (pack_constraints(..., warm_start=True, warm_dense=True)):
every dense-path solve starts from the instance's last converged multipliers.  Results must equal cold results within the
parity tolerances, iterations must drop, a slot that does not fit must not matter, and the dense buffer must be left alone
wherever the rules say so."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ST_WARM, ST_PATH_LH, ST_PATH_GRAM = 0x400, 0x100, 0x200


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _dataset(n, m, d, seed, dev):
    """A resident dense dataset: a plain pack and a pack with both warm-start buffers over the same tensor."""
    from cave_b200 import pack_constraints, synth
    A, c = synth.dense_batch(n, m, d, seed=seed, device=dev)
    return A, c, pack_constraints(A), pack_constraints(A, warm_start=True, warm_dense=True)


def _call(pred, pack, idx, mode=1, **kw):
    from cave_b200 import cave_forward_backward
    return cave_forward_backward(pred, None, -1.0, mode, 0.2, "none", want_proj=True, want_status=True, pack=pack, index=idx,
                                 **kw)


def _close(a, b, rtol, keys=("loss", "grad", "proj", "rnorm")):
    for k in keys:
        x, y = a[k].double().cpu().numpy(), b[k].double().cpu().numpy()
        np.testing.assert_allclose(x, y, rtol=rtol, atol=rtol * max(np.abs(y).max(), 1e-6), err_msg=k)


def _slots(pack):
    """(header int32 [N, 4], multipliers float64 [N, cap]) as views of the pack's dense warm-start buffer."""
    n = pack.shape[0]
    s = pack.warm_dense.view(n, -1)
    return s[:, :16].view(torch.int32), s[:, 16:].view(torch.float64)


def _perturb(p, g, delta=1e-2):
    return p * (1 + delta * torch.randn(p.shape, device=p.device, generator=g, dtype=p.dtype))


@pytest.mark.parametrize("io", [torch.float64, torch.float32])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("m,d,n", [(128, 190, 64), (512, 640, 96), (256, 1225, 148)])
def test_perturbed_epochs_match_cold_with_fewer_iterations(m, d, n, mode, io):
    from oracle import cave_oracle as O
    dev = _cuda()
    A, c0, cold_pack, warm_pack = _dataset(n, m, d, 100 + m, dev)
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(1)).to(dev, torch.int32)
    g = torch.Generator(device=dev).manual_seed(2)
    p = c0.to(io)
    cold_it, warm_it = [], []
    for epoch in range(4):
        x = p[idx.long()]
        c = _call(x, cold_pack, idx, mode)
        w = _call(x, warm_pack, idx, mode)
        assert ((c["status"] & 0xff) == 0).all() and ((w["status"] & 0xff) == 0).all()
        _close(w, c, 1e-6 if io == torch.float64 else 1e-4)
        dense = (c["status"] & ST_PATH_GRAM) != 0
        assert dense.float().mean() > 0.9
        if epoch:
            assert ((w["status"][dense] & (ST_WARM | ST_PATH_GRAM)) == (ST_WARM | ST_PATH_GRAM)).all()
            cold_it.append(c["iters"].double().mean().item())
            warm_it.append(w["iters"].double().mean().item())
        else:
            assert not (w["status"] & ST_WARM).any() and torch.equal(w["iters"], c["iters"])
        if epoch == 2:          # one sample against the float64 oracle
            s = slice(0, 3)
            ref = O.forward_backward(x[s].double().cpu().numpy(), A[idx[s].long()].cpu().numpy(), mode=mode, fp64=True,
                                     reduction="none")
            tol = 1e-6 if io == torch.float64 else 1e-4
            np.testing.assert_allclose(w["loss"][s].double().cpu().numpy(), ref["loss"], rtol=tol, atol=tol)
            np.testing.assert_allclose(w["proj"][s].double().cpu().numpy(), ref["proj"], rtol=tol,
                                       atol=tol * np.abs(ref["proj"]).max())
        p = _perturb(p, g)
    assert np.mean(warm_it) < np.mean(cold_it), (warm_it, cold_it)


def test_repeat_reset_and_an_empty_slot_run_the_cold_algorithm():
    dev = _cuda()
    n = 96
    _, c, cold_pack, pk = _dataset(n, 256, 640, 7, dev)
    idx = torch.arange(n, dtype=torch.int32, device=dev)
    first = _call(c, pk, idx)
    again = _call(c, pk, idx)
    assert ((again["status"] & (ST_WARM | ST_PATH_GRAM)) == (ST_WARM | ST_PATH_GRAM)).all()
    zero = again["iters"] == 0
    assert zero.float().mean() >= 0.5, again["iters"]
    for k in ("loss", "grad", "proj", "rnorm"):
        x, y = again[k][zero].double(), first[k][zero].double()
        assert torch.allclose(x, y, rtol=1e-12, atol=1e-12 * float(y.abs().max())), k
    pk.reset_warm_start()
    assert int(pk.warm.count_nonzero()) == 0 and int(pk.warm_dense.count_nonzero()) == 0
    reset = _call(c, pk, idx)
    cold = _call(c, cold_pack, idx)
    for k in ("loss", "grad", "proj", "status", "iters"):
        assert torch.equal(reset[k], cold[k]), k
    for k in ("loss", "grad", "proj", "status", "iters"):
        assert torch.equal(first[k], cold[k]), k


@pytest.mark.parametrize("fill", ["tag", "nan", "huge"])
def test_a_bad_slot_never_changes_the_result(fill):
    dev = _cuda()
    n = 64
    _, c, cold_pack, pk = _dataset(n, 128, 190, 11, dev)
    idx = torch.arange(n, dtype=torch.int32, device=dev)
    _call(c, pk, idx, mode=0)
    hdr, lam = _slots(pk)
    assert (hdr[:, 0] == 1).all() and (hdr[:, 1] == 128).all()
    if fill == "tag":
        hdr[:, 2] += 1
    elif fill == "nan":
        lam[:, :128] = torch.where(torch.arange(128, device=dev) % 2 == 0, float("nan"), float("inf")).double()
    else:
        lam[:, :128] = 1e30 * (1 + torch.rand(n, 128, device=dev, dtype=torch.float64))
    p = c * 1.001
    cold = _call(p, cold_pack, idx, mode=0)
    out = _call(p, pk, idx, mode=0)
    assert ((out["status"] & 0xff) == 0).all()
    _close(out, cold, 1e-6)
    flagged = (out["status"] & ST_WARM) != 0
    if fill == "tag":
        assert not flagged.any() and torch.equal(out["iters"], cold["iters"])
        for k in ("loss", "grad", "proj"):
            assert torch.equal(out[k], cold[k]), k
    assert (out["iters"][~flagged] >= cold["iters"][~flagged]).all()
    if fill == "huge":
        assert not flagged.any()
    assert (_slots(pk)[0][:, 0] == 1).all()         # every instance converged and stored its solution afresh


def test_mixed_pack_with_both_buffers():
    """Structured (Newton), Lawson-Hanson and dense instances in one resident pack with both warm-start buffers."""
    from cave_b200 import cave_forward_backward, pack_constraints, synth
    from oracle import cave_oracle as O
    dev = _cuda()
    insts = synth.make_batch("tsp20", 8, seed=59)
    S = synth.densify(insts).numpy()                       # [8, m, 190]
    m, d = S.shape[1], S.shape[2]
    rng = np.random.default_rng(59)
    M = max(m, 2 * d)
    A = np.zeros((16, M, d), np.float32)
    A[:8, :m] = S
    A[8:12, :20] = rng.standard_normal((4, 20, d))          # Lawson-Hanson
    A[12:14, :160] = rng.standard_normal((2, 160, d))       # dense path
    A[14:, :2 * d] = rng.standard_normal((2, 2 * d, d))     # m > d: dense path, or handed back to Lawson-Hanson
    At = torch.tensor(A, device=dev)
    pk = pack_constraints(At, warm_start=True, warm_dense=True)
    pred = np.concatenate([synth.predictions(insts, 59, "near"), rng.standard_normal((8, d))])
    p = torch.tensor(pred, device=dev)
    ref = O.forward_backward(pred, A, mode=0, fp64=True, reduction="none")
    sts = []
    for _ in range(2):
        out = cave_forward_backward(p, At, -1.0, 0, 0.2, "none", want_proj=True, want_status=True, pack=pk, dense="on")
        st = out["status"].cpu().numpy()
        sts.append(st)
        assert ((st & 0xff) == 0).all()
        np.testing.assert_allclose(out["loss"].cpu().numpy(), ref["loss"], rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(out["proj"].cpu().numpy(), ref["proj"], rtol=1e-6, atol=1e-6 * np.abs(ref["proj"]).max())
    first, second = sts
    assert (second[:8] & ST_WARM).all()                     # structured, as with warm_start=True alone
    gram = (first & ST_PATH_GRAM) != 0
    assert gram[12:14].all() and not gram[:12].any()
    assert (second[gram] & ST_WARM).all()
    lh = (second & ST_PATH_LH) != 0
    assert lh[8:12].all() and not (second[lh] & ST_WARM).any()
    hdr, _ = _slots(pk)
    written = (hdr[:, 0] == 1).cpu().numpy()
    assert np.array_equal(written, gram)                    # only converged dense-path instances store a solution
    rest = torch.tensor(~gram, device=dev)
    assert int(pk.warm_dense.view(16, -1)[rest].count_nonzero()) == 0


def test_the_dense_buffer_stays_untouched_without_a_dense_solve():
    dev = _cuda()
    n = 48
    _, c, cold_pack, pk = _dataset(n, 128, 190, 13, dev)
    idx = torch.arange(n, dtype=torch.int32, device=dev)
    out = _call(c, pk, idx, dense="off")
    assert not (out["status"] & (ST_PATH_GRAM | ST_WARM)).any()
    assert int(pk.warm_dense.count_nonzero()) == 0
    _call(c, pk, idx)
    before = pk.warm_dense.clone()
    h = _call(c * 1.01, pk, idx, mode=2)
    assert ((h["status"] & 0xff) == 4).all() and torch.equal(pk.warm_dense, before)
    bad = c * 1.01
    bad[5, 0] = float("nan")
    out = _call(bad, pk, idx)
    assert (out["status"][5] & 0xff) == 5
    slot = pk.warm_dense.numel() // n
    assert torch.equal(pk.warm_dense[5 * slot:6 * slot], before[5 * slot:6 * slot])
    assert not torch.equal(pk.warm_dense, before)
    later = _call(c * 1.02, pk, idx)
    cold = _call(c * 1.02, cold_pack, idx)
    assert ((later["status"] & 0xff) == 0).all()
    _close(later, cold, 1e-6)


def test_duplicate_indices_with_different_predictions():
    dev = _cuda()
    n = 64
    _, c, cold_pack, pk = _dataset(n, 256, 640, 17, dev)
    idx = torch.cat([torch.arange(n), torch.arange(n)]).to(dev, torch.int32)
    g = torch.Generator(device=dev).manual_seed(4)
    for _ in range(3):
        p = _perturb(c[idx.long()], g, 0.05)
        w = _call(p, pk, idx)
        k = _call(p, cold_pack, idx)
        assert ((w["status"] & 0xff) == 0).all()
        _close(w, k, 1e-6)


def test_module_sequence_matches_a_plain_pack():
    from cave_b200 import EPO, innerConeAlignedCosine
    dev = _cuda()
    _, c, plain, warm = _dataset(64, 128, 190, 19, dev)

    class Model:
        modelSense = EPO.MINIMIZE

    la = innerConeAlignedCosine(Model(), solver="cuda", seed=7)
    lb = innerConeAlignedCosine(Model(), solver="cuda", seed=7)
    g = torch.Generator(device=dev).manual_seed(8)
    for step in range(10):
        idx = torch.randint(0, 64, (32,), device=dev, generator=g).to(torch.int32)
        x = (c[idx.long()] * (1 + 0.01 * step)).double()
        pa, pb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        a = la(pa, plain, index=idx)
        b = lb(pb, warm, index=idx)
        a.backward()
        b.backward()
        assert torch.allclose(a, b, rtol=1e-6, atol=1e-9)
        assert torch.allclose(pa.grad, pb.grad, rtol=1e-5, atol=1e-9 * float(pa.grad.abs().max()))
    assert int(warm.warm_dense.count_nonzero()) > 0


def test_warm_dense_needs_warm_start():
    from cave_b200 import pack_constraints, synth
    dev = _cuda()
    A, _ = synth.dense_batch(4, 128, 190, device=dev)
    with pytest.raises(ValueError, match="warm_start"):
        pack_constraints(A, warm_dense=True)
