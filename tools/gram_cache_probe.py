"""Gram cache of a resident dense dataset (pack_constraints(..., cache_gram=True)): what it saves, measured on the GPU.

At (d, m, B) = (1225, 256, 2368), (1225, 1024, 1184) and (4950, 1024, 296), exact and innerConeAlignedCosine modes, the
resident step (index = a fixed permutation of the dataset) is timed with device events for four packs of the same tensor,
alternated within every epoch:
    plain        pack_constraints(A)
    cached       pack_constraints(A, cache_gram=True)
    warm         pack_constraints(A, warm_start=True, warm_dense=True)
    warm+cached  the same with the Gram cache
Epochs perturb the prediction by p <- p * (1 + 1e-2 N(0, 1)) (as tools/dense_warm_probe.py).  Two epochs of warm-up, then
--epochs timed ones.  Every epoch checks that the cached arms return bit-identical outputs (loss, loss_i, grad, rnorm, status,
iters) to their uncached partners.  The one-time cost of the cache (pack_constraints with cache_gram=True minus without) and
its bytes are recorded.

    python tools/gram_cache_probe.py [--out profiles] [--epochs 6]
        prints a report and writes OUT/r3_gram_cache_probe.{json,txt}
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from dense_warm_probe import card, timed  # noqa: E402

POINTS = ((1225, 256, 2368), (1225, 1024, 1184), (4950, 1024, 296))
MODES = {"exact": 0, "inner": 1}
ARMS = ("plain", "cached", "warm", "warm+cached")
KEYS = ("loss", "loss_i", "grad", "rnorm", "status", "iters")


def call(pred, pack, idx, mode):
    from cave_b200 import cave_forward_backward
    return cave_forward_backward(pred, None, -1.0, mode, 0.2, "mean", pack=pack, index=idx, want_status=True)


def host_timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def point(d, m, B, dev, epochs, say):
    import numpy as np
    import torch
    from cave_b200 import _lib, pack_constraints, synth
    A, c0 = synth.dense_batch(B, m, d, seed=2000 + m, device=dev)
    pack_constraints(A)                                     # first use of the pack kernels at this shape
    t_plain, plain = host_timed(lambda: pack_constraints(A))
    t_cached, cached = host_timed(lambda: pack_constraints(A, cache_gram=True))
    warm = pack_constraints(A, warm_start=True, warm_dense=True)
    both = pack_constraints(A, warm_start=True, warm_dense=True)
    both.gram = cached.gram                                 # the cache is constant data of A: one copy serves both arms
    packs = dict(zip(ARMS, (plain, cached, warm, both)))
    n_cached = int(cached.gram[4:8].view(torch.int32).item())
    res = {"cache_bytes": int(cached.gram.numel()), "n_cached": n_cached, "A_bytes": int(A.numel() * 4),
           "pack_ms_plain": t_plain, "pack_ms_cached": t_cached, "build_ms": t_cached - t_plain, "modes": {}}
    say(f"{d} x {m} x {B}: cache {res['cache_bytes'] / 1e9:.3f} GB for {n_cached} instances (A {res['A_bytes'] / 1e9:.3f} GB); "
        f"pack {t_plain:.1f} ms, with the cache {t_cached:.1f} ms (build {res['build_ms']:.1f} ms, host clock around a "
        f"synchronised call)")
    idx = torch.randperm(B, generator=torch.Generator().manual_seed(3)).to(dev, torch.int32)
    for mname, mode in MODES.items():
        warm.reset_warm_start()
        both.reset_warm_start()
        g = torch.Generator(device=dev).manual_seed(7)
        p = c0.clone()
        ms = {a: [] for a in ARMS}
        identical, dense_frac, iters = True, [], {a: [] for a in ARMS}
        for e in range(2 + epochs):
            x = p[idx.long()]
            out = {}
            for a in ARMS:
                t, out[a] = timed(lambda: call(x, packs[a], idx, mode))  # noqa: B023
                if e >= 2:
                    ms[a].append(t)
                    iters[a].append(out[a]["iters"].double().mean().item())
            for a, b in (("plain", "cached"), ("warm", "warm+cached")):
                for k in KEYS:
                    identical &= bool(torch.equal(out[a][k], out[b][k]))
            dense_frac.append(((out["plain"]["status"] & _lib.ST_PATH_GRAM) != 0).double().mean().item())
            p = p * (1 + 1e-2 * torch.randn(p.shape, device=dev, generator=g, dtype=p.dtype))
        s = {a: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "ms": v,
                 "iters_mean": float(np.mean(iters[a]))} for a, v in ms.items()}
        res["modes"][mname] = {"arms": s, "bit_identical": identical, "dense_fraction": float(np.mean(dense_frac))}
        say(f"  {mname:5s}  dense {100 * np.mean(dense_frac):5.1f} %   outputs of cached arms bit-identical: {identical}")
        for a in ARMS:
            say(f"    {a:12s} median {s[a]['median_ms']:8.2f} ms  (min {s[a]['min_ms']:8.2f}, max {s[a]['max_ms']:8.2f})   "
                f"iters mean {s[a]['iters_mean']:5.2f}")
        for a, b in (("plain", "cached"), ("warm", "warm+cached")):
            say(f"    {b} / {a}: {s[b]['median_ms'] / s[a]['median_ms']:.3f} (median), saved "
                f"{s[a]['median_ms'] - s[b]['median_ms']:.2f} ms per step")
    del A, c0, packs, plain, cached, warm, both
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--epochs", type=int, default=6)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("gram_cache_probe needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    res = {"card": card(), "epochs": a.epochs, "points": {}}
    say(f"card: {res['card']}")
    say(f"resident step, device events, {a.epochs} timed epochs after 2 of warm-up, the four arms alternated in every epoch")
    for d, m, B in POINTS:
        res["points"][f"d{d}_m{m}_B{B}"] = point(d, m, B, dev, a.epochs, say)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "r3_gram_cache_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(a.out, "r3_gram_cache_probe.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
