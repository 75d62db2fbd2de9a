"""Warm start of the structured Newton solve (pack_constraints(..., warm_start=True)): what it saves, measured on the GPU.

(a) fixed and per-iteration cost of the solve: TSP-50 x 4096, resident pack, device time at max_iter in {1, 2, 4, 8, 200};
(b) perturbation sweep: TSP-50 and TSP-20 x 4096, resident pack, innerConeAlignedCosine mode, epochs of
    p <- p * (1 + delta * N(0, 1)); iterations, warm-flag fraction, fallbacks and the device-timed step, cold and warm
    alternated in one process;
(c) a real trajectory: TSP-20 CaVE+ (linear predictor, batch 32, Adam 1e-2) for 20 epochs, cold and warm, same seed.

    python tools/warm_start_probe.py [--out DIR]      (prints a report and writes DIR/warm_start_probe.json)
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cave_b200 import _lib, cave_forward_backward, pack_constraints, synth, tsp_exact  # noqa: E402

ST_WARM = _lib.ST_WARM


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def part_a(dev, say):
    insts = synth.make_batch("tsp50", 4096, seed=1000)
    A = synth.densify(insts, device=dev)
    pred = torch.tensor(synth.predictions(insts, 1000, "uniform"), device=dev)
    pack = pack_constraints(A)
    idx = torch.arange(4096, dtype=torch.int32, device=dev)
    rows = []
    for mi in (1, 2, 4, 8, 200):
        fn = lambda: cave_forward_backward(pred, None, -1.0, 1, 0.2, "mean", pack=pack, index=idx, max_iter=mi,  # noqa: E731
                                           want_status=True)
        for _ in range(3):
            fn()
        ms, out = timed(fn, 10)
        it = out["iters"].double().mean().item()
        rows.append({"max_iter": mi, "ms": ms, "mean_iters": it})
        say(f"  max_iter {mi:4d}: {ms:7.3f} ms   mean iterations {it:5.2f}")
    # least squares fit of time = fixed + per_iter * mean iterations over the capped points (the cap binds there)
    x = np.array([r["mean_iters"] for r in rows]); y = np.array([r["ms"] for r in rows])
    per_iter, fixed = np.polyfit(x, y, 1)
    say(f"  fit: {fixed:.3f} ms fixed + {per_iter:.3f} ms per mean Newton iteration")
    return {"points": rows, "fixed_ms": float(fixed), "per_iter_ms": float(per_iter)}


def part_b(dev, say, epochs=6):
    res = {}
    for kind in ("tsp50", "tsp20"):
        insts = synth.make_batch(kind, 4096, seed=2000)
        A = synth.densify(insts, device=dev)
        pred0 = torch.tensor(synth.predictions(insts, 2000, "uniform"), device=dev)
        cold = pack_constraints(A)
        warm = pack_constraints(A, warm_start=True)
        idx = torch.arange(4096, dtype=torch.int32, device=dev)
        for delta in (0.0, 1e-3, 1e-2, 1e-1):
            warm.reset_warm_start()
            g = torch.Generator(device=dev).manual_seed(7)
            p = pred0.clone()
            rec = {"cold_ms": [], "warm_ms": [], "cold_iters": [], "warm_iters_mean": [], "warm_iters_max": [],
                   "warm_flag_frac": [], "fallbacks": []}
            for e in range(epochs):
                fc = lambda: cave_forward_backward(p, None, -1.0, 1, 0.2, "mean", pack=cold, index=idx, want_status=True)  # noqa: E731
                fw = lambda: cave_forward_backward(p, None, -1.0, 1, 0.2, "mean", pack=warm, index=idx, want_status=True)  # noqa: E731
                if e == 0:
                    fc()
                    fw()        # fills the slots; the timed warm calls below repeat the same predictions
                    p = p * (1 + delta * torch.randn(p.shape, device=dev, generator=g, dtype=p.dtype))
                    continue
                # one warm call per epoch is the real use; time it once, alternating with the cold call
                snapshot = warm.warm.clone()
                tc, oc = timed(fc, 1)
                tw, ow = timed(fw, 1)
                for _ in range(2):          # more samples of the same epoch step: restore the state before each
                    warm.warm.copy_(snapshot)
                    tc2, _ = timed(fc, 1)
                    warm.warm.copy_(snapshot)
                    tw2, ow = timed(fw, 1)
                    tc, tw = min(tc, tc2), min(tw, tw2)
                st = ow["status"]
                it = ow["iters"].double()
                rec["cold_ms"].append(tc); rec["warm_ms"].append(tw)
                rec["cold_iters"].append(oc["iters"].double().mean().item())
                rec["warm_iters_mean"].append(it.mean().item()); rec["warm_iters_max"].append(int(it.max().item()))
                rec["warm_flag_frac"].append(((st & ST_WARM) != 0).double().mean().item())
                rec["fallbacks"].append(int((((st & ST_WARM) == 0) & ((st & 0xff) == 0)).sum().item()))
                p = p * (1 + delta * torch.randn(p.shape, device=dev, generator=g, dtype=p.dtype))
            s = {k: float(np.mean(v)) for k, v in rec.items()}
            s["warm_iters_max"] = int(max(rec["warm_iters_max"])); s["fallbacks"] = int(sum(rec["fallbacks"]))
            res[f"{kind}_delta{delta:g}"] = {"mean": s, "per_epoch": rec}
            say(f"  {kind} delta {delta:<6g}: iters cold {s['cold_iters']:5.2f}  warm mean {s['warm_iters_mean']:5.2f} "
                f"max {s['warm_iters_max']:3d}   warm flag {100 * s['warm_flag_frac']:5.1f} %   fallbacks {s['fallbacks']:3d}   "
                f"step cold {s['cold_ms']:6.3f} ms  warm {s['warm_ms']:6.3f} ms  ({s['warm_ms'] / s['cold_ms']:.3f}x)")
    return res


def part_c(dev, say, epochs=20, n_train=1000, batch=32, seed=0):
    x, c = tsp_exact.gen_data(n_train, 10, 20, 4, 0.5, seed=135)
    _, _, tours = tsp_exact.solve(c, 20)
    rng = np.random.default_rng(seed)
    insts = [tsp_exact.binding_constraints(t, rng, 8) for t in tours]
    A = synth.densify(insts, device=dev)
    X, C = torch.tensor(x, device=dev, dtype=torch.float32), torch.tensor(c, device=dev, dtype=torch.float32)
    out = {}
    for label, warm_start in (("cold", False), ("warm", True)):
        pack = pack_constraints(A, warm_start=warm_start)
        torch.manual_seed(seed)
        reg = torch.nn.Linear(X.shape[1], C.shape[1]).to(dev)
        opt = torch.optim.Adam(reg.parameters(), lr=1e-2)
        gen = torch.Generator().manual_seed(seed)
        rows = []
        for epoch in range(epochs):
            perm = torch.randperm(n_train, generator=gen).to(dev)
            it_sum, n_inst, loss_sum, steps = torch.zeros((), device=dev, dtype=torch.float64), 0, torch.zeros((), device=dev, dtype=torch.float64), 0
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for s in range(0, n_train, batch):
                idx = perm[s:s + batch]
                cp = reg(X[idx])
                # CaVE+ (innerConeAlignedCosine, solve_ratio 1): the module's forward / backward with the status words kept
                r = cave_forward_backward(cp, None, -1.0, 1, 0.2, "mean", pack=pack, index=idx.to(torch.int32), want_status=True)
                opt.zero_grad()
                cp.backward(r["grad"].to(cp.dtype))
                opt.step()
                it_sum += r["iters"].double().sum(); n_inst += idx.numel()
                loss_sum += r["loss"].double(); steps += 1
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            rows.append({"epoch": epoch, "mean_iters": it_sum.item() / n_inst, "step_ms": 1e3 * dt / steps,
                         "mean_loss": loss_sum.item() / steps})
        out[label] = rows
    for e in range(epochs):
        a, b = out["cold"][e], out["warm"][e]
        rel = abs(a["mean_loss"] - b["mean_loss"]) / abs(a["mean_loss"])
        say(f"  epoch {e:2d}: iters cold {a['mean_iters']:5.2f} warm {b['mean_iters']:5.2f}   step cold {a['step_ms']:6.3f} ms "
            f"warm {b['step_ms']:6.3f} ms   loss cold {a['mean_loss']:.9f} warm {b['mean_loss']:.9f}  rel diff {rel:.1e}")
    out["max_rel_loss_diff"] = max(abs(a["mean_loss"] - b["mean_loss"]) / abs(a["mean_loss"])
                                   for a, b in zip(out["cold"], out["warm"]))
    say(f"  largest relative difference of the per-epoch losses: {out['max_rel_loss_diff']:.2e}")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--parts", default="abc")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("warm_start_probe needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    res = {"card": card()}
    say(f"card: {res['card']}")
    if "a" in a.parts:
        say("(a) TSP-50 x 4096, resident pack, innerConeAlignedCosine mode, cold solve at capped iterations")
        res["a"] = part_a(dev, say)
    if "b" in a.parts:
        say("(b) perturbation sweep, 4096 instances, resident pack, 5 timed epochs after the first (best of 3 per epoch)")
        res["b"] = part_b(dev, say)
    if "c" in a.parts:
        say("(c) TSP-20 CaVE+ training, linear predictor, batch 32, Adam 1e-2, 1000 instances, 20 epochs")
        res["c"] = part_c(dev, say)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "warm_start_probe.json"), "w") as f:
            json.dump(res, f, indent=1)
        with open(os.path.join(a.out, "warm_start_probe.txt"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
