"""Gram cache of a resident dense dataset on the B200 (pack_constraints(..., cache_gram=True)): the cache holds exactly what
the tensor-core Gram kernel computes, and a call with it gives bit-identical results to the same call with a plain pack,
with one kernel launch per dense round fewer."""
import dataclasses

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ST_BADINPUT, ST_PATH_LH, ST_PATH_GRAM = 5, 0x100, 0x200
KEYS = ("loss", "loss_i", "grad", "proj", "rnorm", "status", "iters")


def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _call(pred, pack, idx, mode=1, reduction="mean", **kw):
    from cave_b200 import cave_forward_backward
    return cave_forward_backward(pred, None, -1.0, mode, 0.2, reduction, want_proj=True, want_status=True, pack=pack, index=idx,
                                 **kw)


def _equal(a, b):
    for k in KEYS:
        assert torch.equal(a[k], b[k]), k


def _cache(pack):
    """(header int32 [4], map int32 [N], slots float32 [n_cached, m_pad, m_pad]) as views of the pack's Gram cache."""
    N, m, _ = pack.shape
    mp = (m + 127) // 128 * 128
    base = (16 + 4 * N + 1023) // 1024 * 1024
    hdr = pack.gram[:16].view(torch.int32)
    mp_ = pack.gram[16:16 + 4 * N].view(torch.int32)
    return hdr, mp_, pack.gram[base:].view(torch.float32).view(-1, mp, mp)


def _mixed(dev, seed=59):
    """Structured (TSP-20), Lawson-Hanson, dense and handed-back instances in one dataset tensor."""
    from cave_b200 import synth
    insts = synth.make_batch("tsp20", 8, seed=seed)
    S = synth.densify(insts).numpy()
    m, d = S.shape[1], S.shape[2]
    rng = np.random.default_rng(seed)
    A = np.zeros((16, max(m, 2 * d), d), np.float32)
    A[:8, :m] = S
    A[8:12, :20] = rng.standard_normal((4, 20, d))          # Lawson-Hanson (fewer than 128 rows)
    A[12:14, :160] = rng.standard_normal((2, 160, d))       # dense path
    A[14:, :2 * d] = rng.standard_normal((2, 2 * d, d))     # m = 2d: the dense path may hand them back to Lawson-Hanson
    pred = np.concatenate([synth.predictions(insts, seed, "near"), rng.standard_normal((8, d))])
    return torch.tensor(A, device=dev), torch.tensor(pred, device=dev)


@pytest.mark.parametrize("m,d", [(128, 190), (512, 640), (1024, 1225)])
def test_cached_slots_equal_the_gram_kernel(m, d):
    from cave_b200 import pack_constraints, synth
    from cave_b200.qpsolver import dense_gram
    dev = _cuda()
    n = 5
    A, _ = synth.dense_batch(n, m, d, seed=m, device=dev)
    if m > 128:
        A[2, m - 200:] = 0.0                                # fewer valid rows: a smaller leading square than m_pad
    pk = pack_constraints(A, cache_gram=True)
    G, cnt = dense_gram(A)
    assert cnt == n
    hdr, qmap, slots = _cache(pk)
    mp = (m + 127) // 128 * 128
    assert hdr.tolist() == [1, n, mp, n]
    assert sorted(qmap.tolist()) == list(range(n))
    for q in range(n):
        lim = (int((A[q].abs().sum(1) > 0).sum()) + 127) // 128 * 128
        s = slots[int(qmap[q])]
        assert torch.equal(s[:lim, :lim], G[q, :lim, :lim]), q
        assert int(s[lim:].count_nonzero()) == 0 and int(s[:, lim:].count_nonzero()) == 0


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("io", [torch.float64, torch.float32])
@pytest.mark.parametrize("mode", [0, 1])
def test_cached_and_plain_packs_are_bit_identical(mode, io, precision):
    from cave_b200 import pack_constraints, synth
    dev = _cuda()
    n = 96
    A, c = synth.dense_batch(n, 256, 640, seed=3, device=dev)
    plain, cached = pack_constraints(A), pack_constraints(A, cache_gram=True)
    assert plain.gram is None and cached.gram is not None
    # a permuted index with duplicates, over several rounds of 16 dense slots
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(5))
    idx = torch.cat([perm, perm[:40]]).to(dev, torch.int32)
    pred = (c[idx.long()] * (1 + 0.1 * torch.arange(idx.numel(), device=dev)[:, None] / idx.numel())).to(io)
    a = _call(pred, plain, idx, mode, precision=precision, dense_slots=16)
    b = _call(pred, cached, idx, mode, precision=precision, dense_slots=16)
    assert ((a["status"] & ST_PATH_GRAM) != 0).float().mean() > 0.9
    _equal(a, b)


def test_ffma_cholesky_update_is_bit_identical(monkeypatch):
    from cave_b200 import pack_constraints, synth
    dev = _cuda()
    n = 48
    A, c = synth.dense_batch(n, 512, 640, seed=4, device=dev)
    plain, cached = pack_constraints(A), pack_constraints(A, cache_gram=True)
    idx = torch.arange(n, dtype=torch.int32, device=dev).flip(0)
    for tc in ("0", "1"):
        monkeypatch.setenv("CAVE_DENSE_TC", tc)
        _equal(_call(c, plain, idx, 0), _call(c, cached, idx, 0))


def test_mixed_dataset_with_handed_back_instances():
    from cave_b200 import pack_constraints
    dev = _cuda()
    A, pred = _mixed(dev)
    plain, cached = pack_constraints(A), pack_constraints(A, cache_gram=True)
    hdr, qmap, _ = _cache(cached)
    assert hdr.tolist()[:2] == [1, 4]
    assert qmap.tolist() == [-1] * 12 + [0, 1, 2, 3]          # structured and short instances have no slot
    idx = torch.arange(16, dtype=torch.int32, device=dev)
    handed_back = 0
    for mode in (0, 1):
        a = _call(pred, plain, idx, mode, reduction="none", dense="on")
        b = _call(pred, cached, idx, mode, reduction="none", dense="on")
        _equal(a, b)
        st = b["status"].cpu().numpy()
        assert ((st & 0xff) == 0).all()
        assert (st[12:14] & ST_PATH_GRAM).all() and not (st[:12] & ST_PATH_GRAM).any()
        lh, gram = (st[14:] & ST_PATH_LH) != 0, (st[14:] & ST_PATH_GRAM) != 0
        assert (lh ^ gram).all()                            # solved on the dense path, or handed back to Lawson-Hanson
        handed_back += int(lh.sum())
    assert handed_back > 0                                  # the cached call hands instances back exactly as the plain one


def test_warm_dense_with_and_without_the_cache_over_perturbed_epochs():
    from cave_b200 import pack_constraints, synth
    dev = _cuda()
    n = 96
    A, c = synth.dense_batch(n, 512, 640, seed=6, device=dev)
    warm = pack_constraints(A, warm_start=True, warm_dense=True)
    both = pack_constraints(A, warm_start=True, warm_dense=True, cache_gram=True)
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(7)).to(dev, torch.int32)
    g = torch.Generator(device=dev).manual_seed(8)
    p = c.clone()
    for _ in range(4):
        x = p[idx.long()]
        _equal(_call(x, warm, idx), _call(x, both, idx))
        assert torch.equal(warm.warm_dense, both.warm_dense)
        p = p * (1 + 1e-2 * torch.randn(p.shape, device=dev, generator=g))
    both.reset_warm_start()
    assert int(both.gram.count_nonzero()) > 0


def test_one_launch_fewer_per_round_and_the_cache_is_only_read():
    from cave_b200 import _lib, pack_constraints, synth
    lib = _lib.load()
    dev = _cuda()
    n = 100
    A, c = synth.dense_batch(n, 256, 640, seed=9, device=dev)
    plain, cached = pack_constraints(A), pack_constraints(A, cache_gram=True)
    before = cached.gram.clone()
    idx = torch.arange(n, dtype=torch.int32, device=dev)
    counts = []
    for pk in (plain, cached):
        n0 = lib.cave_launch_count()
        _call(c, pk, idx, dense_slots=16)
        counts.append(lib.cave_launch_count() - n0)
    assert counts[0] - counts[1] == (n + 15) // 16
    torch.cuda.synchronize()
    assert torch.equal(cached.gram, before)


def test_a_cache_that_was_never_built_reports_bad_input():
    from cave_b200 import pack_constraints
    dev = _cuda()
    A, pred = _mixed(dev, seed=61)
    plain, cached = pack_constraints(A), pack_constraints(A, cache_gram=True)
    zero = dataclasses.replace(cached, gram=torch.zeros_like(cached.gram))
    idx = torch.arange(16, dtype=torch.int32, device=dev)
    a = _call(pred, plain, idx, 0, reduction="none", dense="on")
    b = _call(pred, zero, idx, 0, reduction="none", dense="on")
    st = b["status"].cpu().numpy()
    dense = np.zeros(16, bool)
    dense[12:] = True
    assert (st[dense] == (ST_BADINPUT | ST_PATH_GRAM)).all(), st
    assert torch.isnan(b["loss_i"][12:]).all() and torch.isnan(b["grad"][12:]).all()
    for k in KEYS[1:]:
        assert torch.equal(a[k][:12], b[k][:12]), k
    # a cache of another pack (other N) is refused the same way
    other = pack_constraints(A[:14].contiguous(), cache_gram=True)
    pad = torch.zeros_like(cached.gram)
    pad[:other.gram.numel()] = other.gram
    c = _call(pred, dataclasses.replace(cached, gram=pad), idx, 0, reduction="none", dense="on")
    assert (c["status"][12:] == (ST_BADINPUT | ST_PATH_GRAM)).all()


def test_no_qualifying_instance_gives_no_cache():
    from cave_b200 import pack_constraints, synth
    dev = _cuda()
    insts = synth.make_batch("tsp20", 4, seed=3)
    A = synth.densify(insts).to(dev)
    assert pack_constraints(A, cache_gram=True).gram is None
    assert pack_constraints(torch.randn((4, 100, 64), device=dev), cache_gram=True).gram is None      # m < 128


def test_module_gradient_with_and_without_the_cache():
    from cave_b200 import EPO, innerConeAlignedCosine, pack_constraints, synth
    dev = _cuda()
    A, c = synth.dense_batch(64, 128, 190, seed=19, device=dev)
    plain, cached = pack_constraints(A), pack_constraints(A, cache_gram=True)

    class Model:
        modelSense = EPO.MINIMIZE

    la = innerConeAlignedCosine(Model(), solver="cuda", seed=7)
    lb = innerConeAlignedCosine(Model(), solver="cuda", seed=7)
    g = torch.Generator(device=dev).manual_seed(8)
    for step in range(4):
        idx = torch.randint(0, 64, (32,), device=dev, generator=g).to(torch.int32)
        x = (c[idx.long()] * (1 + 0.01 * step)).double()
        pa, pb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        a = la(pa, plain, index=idx)
        b = lb(pb, cached, index=idx)
        a.backward()
        b.backward()
        assert torch.equal(a, b) and torch.equal(pa.grad, pb.grad)
