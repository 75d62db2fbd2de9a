"""Chunked calls on the B200 (cave_forward_backward(..., chunk=k)): every chunked result is compared with the same call
unchunked.  With a resident pack every instance is solved exactly as in the unchunked call and the finalize reduces the
whole batch in the same order, so all outputs are bit-identical.  A one-shot pack (dense host tensor or SparseConstraints)
selects the solve kernel's launch configuration from its own instances, so a chunk may run another configuration than the
whole batch; those inputs are bit-identical with the configuration fixed (CAVE_SOLVE_CFG=3) and agree to 1e-12 relative in
float64 without it."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

KEYS = ("loss", "loss_i", "grad", "proj", "rnorm", "status", "iters")
SIZES = {"tsp20": 13, "tsp50": 10, "vrp20": 13, "sp5": 13}


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _call(pred, ctrs, mode=1, reduction="mean", **kw):
    from cave_b200 import cave_forward_backward
    return cave_forward_backward(pred, ctrs, -1.0, mode, 0.2, reduction, want_proj=True, want_status=True, **kw)


def _equal(a, b, what="", mode=None):
    for k in KEYS:
        if k == "proj" and mode == 2:       # heuristic mode writes no projection (no solve), chunked or not
            continue
        x, y = a[k], b[k]
        assert torch.equal(x.cpu(), y.cpu()), f"{what} {k}"


def _close(a, b, rtol=1e-12):
    for k in ("loss", "loss_i", "grad", "proj", "rnorm"):
        x, y = a[k].double().cpu().numpy(), b[k].double().cpu().numpy()
        np.testing.assert_allclose(x, y, rtol=rtol, atol=rtol * max(np.abs(y).max(), 1e-30), err_msg=k)
    for k in ("status",):
        assert torch.equal(a[k].cpu() & 0xff, b[k].cpu() & 0xff), k


_DATA = {}


def _dataset(kind, dev):
    """A resident pack over N instances and a batch index (a permutation without duplicates) of B < N of them."""
    if kind not in _DATA:
        from cave_b200 import pack_constraints, synth
        B = SIZES[kind]
        N = B + 3
        insts = synth.make_batch(kind, N, seed=11)
        A = synth.densify(insts, device=dev)
        pred = torch.tensor(synth.predictions(insts, 11, "near"), device=dev)
        idx = torch.randperm(N, generator=torch.Generator().manual_seed(5))[:B].to(dev, torch.int32)
        _DATA[kind] = (pack_constraints(A), pred[idx.long()].contiguous(), idx, insts, A)
    return _DATA[kind]


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("io", [torch.float32, torch.float64])
@pytest.mark.parametrize("reduction", ["mean", "sum", "none"])
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("kind", ["tsp20", "tsp50", "vrp20", "sp5"])
def test_resident_chunks_are_bit_identical(kind, mode, reduction, io, precision):
    dev = _cuda()
    pack, pred, idx, _, _ = _dataset(kind, dev)
    B = pred.shape[0]
    p = pred.to(io)
    ref = _call(p, None, mode, reduction, pack=pack, index=idx, precision=precision)
    assert ((ref["status"] & 0xff) != 3).all()          # no instance beyond the scratch caps: the comparison is meaningful
    for chunk in (1, 4, 7, B - 1, B, B + 5):            # 4 and 7 do not divide B
        got = _call(p, None, mode, reduction, pack=pack, index=idx, precision=precision, chunk=chunk)
        _equal(got, ref, f"chunk={chunk}", mode)


@pytest.mark.parametrize("pinned", [False, True])
def test_resident_host_predictions(pinned):
    """Host predictions: pinned or pageable, the chunks' inputs go through the copy stream and the outputs come back as host
    tensors, bit-identical to the unchunked call."""
    dev = _cuda()
    pack, pred, idx, _, _ = _dataset("tsp20", dev)
    ref = _call(pred.double(), None, 1, "mean", pack=pack, index=idx)
    host = pred.double().cpu()
    if pinned:
        host = host.pin_memory()
    got = _call(host, None, 1, "mean", pack=pack, index=idx.cpu(), chunk=4)
    for k in KEYS:
        assert got[k].device.type == "cpu", k
    assert got["grad"].is_pinned()
    _equal(got, ref)


def test_warm_packs_over_two_calls():
    from cave_b200 import pack_constraints, synth
    dev = _cuda()
    N, B = 40, 33
    insts = synth.make_batch("tsp20", N, seed=23)
    A = synth.densify(insts, device=dev)
    pred = torch.tensor(synth.predictions(insts, 23, "near"), device=dev, dtype=torch.float64)
    idx = torch.randperm(N, generator=torch.Generator().manual_seed(3))[:B].to(dev, torch.int32)
    plain, chunked = pack_constraints(A, warm_start=True), pack_constraints(A, warm_start=True)
    g = torch.Generator(device=dev).manual_seed(4)
    p = pred[idx.long()]
    for call in range(2):
        ref = _call(p, None, pack=plain, index=idx)
        got = _call(p, None, pack=chunked, index=idx, chunk=8)
        _equal(got, ref, f"call {call}")
        assert torch.equal(plain.warm, chunked.warm)
        if call:
            assert (got["status"] & 0x400).any()         # the second call started from the first one's solutions
        p = p * (1 + 0.01 * torch.randn(p.shape, generator=g, device=dev, dtype=p.dtype))


def test_dense_batch_with_gram_cache_and_dense_warm_start():
    from cave_b200 import pack_constraints, synth
    dev = _cuda()
    A, c = synth.dense_batch(24, 256, 1225, seed=7, device=dev)
    plain = pack_constraints(A, warm_start=True, warm_dense=True, cache_gram=True)
    chunked = pack_constraints(A, warm_start=True, warm_dense=True, cache_gram=True)
    assert plain.gram is not None
    idx = torch.arange(24, dtype=torch.int32, device=dev)
    for call in range(2):
        p = c.double() * (1 + 0.01 * call)
        ref = _call(p, None, 0, "mean", pack=plain, index=idx)
        got = _call(p, None, 0, "mean", pack=chunked, index=idx, chunk=7)
        assert (ref["status"] & 0x200).all()
        _equal(got, ref, f"call {call}")
        assert torch.equal(plain.warm_dense, chunked.warm_dense)


def test_mixed_structured_and_lawson_hanson_batch():
    from cave_b200 import pack_constraints, synth
    dev = _cuda()
    insts = synth.make_batch("tsp20", 8, seed=59)
    S = synth.densify(insts).numpy()
    m, d = S.shape[1], S.shape[2]
    rng = np.random.default_rng(59)
    A = np.zeros((16, max(m, 2 * d), d), np.float32)
    A[:8, :m] = S
    A[8:12, :20] = rng.standard_normal((4, 20, d))          # Lawson-Hanson (fewer than 128 rows)
    A[12:14, :160] = rng.standard_normal((2, 160, d))       # dense path
    A[14:, :2 * d] = rng.standard_normal((2, 2 * d, d))     # the dense path may hand them back to Lawson-Hanson
    pred = np.concatenate([synth.predictions(insts, 59, "near"), rng.standard_normal((8, d))])
    A, pred = torch.tensor(A, device=dev), torch.tensor(pred, device=dev)
    pack = pack_constraints(A)
    idx = torch.randperm(16, generator=torch.Generator().manual_seed(9)).to(dev, torch.int32)
    for mode in (0, 1):
        ref = _call(pred[idx.long()], None, mode, "sum", pack=pack, index=idx, dense=True)
        assert (ref["status"] & 0x100).any() and not (ref["status"] & 0x100).all()
        for chunk in (1, 5, 15):
            got = _call(pred[idx.long()], None, mode, "sum", pack=pack, index=idx, dense=True, chunk=chunk)
            _equal(got, ref, f"mode {mode} chunk {chunk}")


def _one_shot_inputs(kind, dev, n=29):
    from cave_b200 import SparseConstraints, synth
    insts = synth.make_batch(kind, n, seed=31)
    A = synth.densify(insts)
    pred = torch.tensor(synth.predictions(insts, 31, "near"), dtype=torch.float64)
    return A, SparseConstraints.from_instances(insts, m_max=A.shape[1]), pred


def _sparse_to(sc, dev):
    return type(sc)(sc.inst_off.to(dev), sc.row_ptr.to(dev), sc.col.to(dev), sc.val.to(dev), sc.m_max, sc.d)


@pytest.mark.parametrize("where", ["device", "pinned", "pageable"])
@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("mode", [0, 1])
def test_one_shot_packs_with_the_launch_configuration_fixed(monkeypatch, mode, sparse, where):
    dev = _cuda()
    monkeypatch.setenv("CAVE_SOLVE_CFG", "3")
    A, sc, pred = _one_shot_inputs("tsp20", dev)
    on_dev = A.to(dev) if not sparse else _sparse_to(sc, dev)
    ctrs, p = sc if sparse else A, pred
    if where == "device":
        ctrs, p = on_dev, pred.to(dev)
    elif where == "pinned":
        ctrs, p = ctrs.pin_memory(), pred.pin_memory()
    ref = _call(pred.to(dev), on_dev, mode, "mean")
    for chunk in (1, 6, 28):
        got = _call(p, ctrs, mode, "mean", chunk=chunk)
        _equal(got, ref, f"chunk {chunk}")


@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("kind", ["tsp20", "tsp50"])
def test_one_shot_packs_agree_to_rounding(kind, sparse):
    """Without a fixed configuration a chunk's pack may launch the solve kernel with another thread count and shared-memory
    split than the whole batch's; the reductions inside the solve then sum in another order, so the results agree to
    rounding, not bit for bit."""
    dev = _cuda()
    A, sc, pred = _one_shot_inputs(kind, dev, n=40 if kind == "tsp20" else 24)
    ref = _call(pred.to(dev), _sparse_to(sc, dev) if sparse else A.to(dev), 1, "mean")
    for chunk in (3, 17):
        got = _call(pred, sc if sparse else A, 1, "mean", chunk=chunk)
        _close(got, ref)


def test_device_memory_is_bounded_by_the_chunk():
    from cave_b200 import _lib, synth
    from cave_b200.qpsolver import _opts
    dev = _cuda()
    lib = _lib.load()
    B, chunk = 1024, 128
    insts = synth.make_batch("tsp50", B, seed=2)
    A = synth.densify(insts)                         # host, pageable: ~6.5 GB
    _, m, d = A.shape
    pred = torch.tensor(synth.predictions(insts, 2, "near"))
    n = ctypes.c_size_t()

    def pack_scratch(b):
        lib.cave_pack_bytes(b, m, d, ctypes.byref(n))
        p = n.value
        lib.cave_scratch_bytes(b, m, d, _lib.F64, ctypes.byref(_opts()), ctypes.byref(n))
        return p + n.value

    staging = 2 * chunk * (m * d * 4 + d * 4 + 2 * d * 4)   # two sets of A and pred rows in, gradient rows out
    outputs = 16 * B + 4 * 32 * B                            # accumulator and per-instance outputs (generous)
    bound = staging + pack_scratch(chunk) + outputs + (64 << 20)
    unchunked = B * m * d * 4 + pack_scratch(B)
    assert bound < unchunked / 2
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    out = _call(pred, A, 1, "mean", chunk=chunk)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(dev) - base
    assert peak < bound, (peak, bound)
    assert np.isfinite(float(out["loss"])) and out["grad"].shape == (B, d)


@pytest.mark.parametrize("host", [False, True])
def test_module_with_chunk_matches_and_draws_the_same_branches(host):
    from cave_b200 import EPO, innerConeAlignedCosine, pack_constraints, synth
    dev = _cuda()
    N, B = 300, 150
    insts = synth.make_batch("tsp20", N, seed=71)
    pack = pack_constraints(synth.densify(insts, device=dev))
    pred_all = torch.tensor(synth.predictions(insts, 71, "near"), device=dev)

    class Model:
        modelSense = EPO.MINIMIZE

    for s in (0, 1):
        plain = innerConeAlignedCosine(Model(), solver="cuda", solve_ratio=0.3, seed=s)
        chunked = innerConeAlignedCosine(Model(), solver="cuda", solve_ratio=0.3, seed=s, solver_kwargs={"chunk": 64})
        g = torch.Generator().manual_seed(s)
        for step in range(10):
            idx = torch.randperm(N, generator=g)[:B]
            p = pred_all[idx.to(dev)]
            x = p.clone().requires_grad_(True)
            y = (p.cpu() if host else p.clone()).requires_grad_(True)
            lx = plain(x, pack, index=idx.to(dev, torch.int32))
            ly = chunked(y, pack, index=idx.to(dev, torch.int32))
            lx.backward()
            ly.backward()
            assert torch.equal(lx.detach().cpu(), ly.detach().cpu()), step
            assert torch.equal(x.grad.cpu(), y.grad.cpu()), step
        a, b = plain._branch_rng.get_state(), chunked._branch_rng.get_state()
        assert np.array_equal(a[1], b[1]) and a[2] == b[2]
