"""Warm start of the dense Gram-space Newton solve (pack_constraints(..., warm_start=True, warm_dense=True)): what it saves,
measured on the GPU.

(a) perturbation sweep: resident synth.dense_batch datasets at (d, m, B) = (1225, 256, 2368) and (1225, 1024, 1184), exact
    and innerConeAlignedCosine modes, epochs of p <- p * (1 + delta * N(0, 1)); mean / max iterations, share of
    CAVE_ST_WARM, fallbacks (instances with a valid slot that ended without the warm flag) and the device-timed step, cold
    and warm alternated in one process;
(b) cold A/B (--ab-root DIR): the cold step of the same resident datasets with another checkout of the package and its
    built library (DIR/cave_b200, loaded through CAVE_B200_LIB; e.g. the parent commit's) against this one, alternated in
    child processes; the outputs of both are hashed.

    python tools/dense_warm_probe.py --ab-root DIR [--out profiles]
        prints a report and writes OUT/r3_dense_warm_probe.{json,txt}; --skip-ab measures (a) alone and says so
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

POINTS = ((1225, 256, 2368), (1225, 1024, 1184))        # (d, m, B): DESIGN.md 4.3 sweep points
DELTAS = (0.0, 1e-3, 1e-2, 1e-1)
MODES = {"exact": 0, "inner": 1}


def card():
    """Name and power limit of the device the run uses, matched by PCI address (nvidia-smi lists every physical GPU,
    whatever CUDA_VISIBLE_DEVICES hides)."""
    import torch
    pr = torch.cuda.get_device_properties(torch.cuda.current_device())
    want = (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id,name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    for row in q:
        f = [x.strip() for x in row.split(",")]
        try:
            dom, b, dev_fn = f[0].split(":")
            if (int(dom, 16), int(b, 16), int(dev_fn.split(".")[0], 16)) == want:
                return f"{f[1]}, {f[2]}"
        except (ValueError, IndexError):
            continue
    return f"{pr.name}, power limit unknown"


def timed(fn):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def dataset(d, m, B, dev):
    from cave_b200 import synth
    return synth.dense_batch(B, m, d, seed=1000 + m, device=dev)


def call(pred, pack, idx, mode):
    from cave_b200 import cave_forward_backward
    return cave_forward_backward(pred, None, -1.0, mode, 0.2, "mean", pack=pack, index=idx, want_status=True)


def sweep(dev, say, epochs=6, samples=3):
    import numpy as np
    import torch
    from cave_b200 import _lib, pack_constraints
    res = {}
    for d, m, B in POINTS:
        A, c0 = dataset(d, m, B, dev)
        cold = pack_constraints(A)
        warm = pack_constraints(A, warm_start=True, warm_dense=True)
        idx = torch.arange(B, dtype=torch.int32, device=dev)
        slot = warm.warm_dense.numel() // B
        for mname, mode in MODES.items():
            for _ in range(2):              # warm-up of both kernels at this shape
                call(c0, cold, idx, mode)
                call(c0, warm, idx, mode)
            for delta in DELTAS:
                warm.reset_warm_start()
                g = torch.Generator(device=dev).manual_seed(7)
                p = c0.clone()
                rec = {k: [] for k in ("cold_ms", "warm_ms", "cold_iters", "cold_iters_max", "warm_iters_mean",
                                       "warm_iters_max", "warm_flag_frac", "fallbacks", "handed_back")}
                for e in range(epochs):
                    fc = lambda: call(p, cold, idx, mode)  # noqa: E731
                    fw = lambda: call(p, warm, idx, mode)  # noqa: E731
                    if e == 0:
                        fc()
                        fw()        # fills the slots
                        p = p * (1 + delta * torch.randn(p.shape, device=dev, generator=g, dtype=p.dtype))
                        continue
                    snapshot = warm.warm_dense.clone()
                    valid = snapshot.view(B, slot)[:, :4].view(torch.int32)[:, 0] == 1
                    tc, tw = float("inf"), float("inf")
                    for _ in range(samples):        # the same epoch step again: restore the state before each warm call
                        warm.warm_dense.copy_(snapshot)
                        t, oc = timed(fc)
                        tc = min(tc, t)
                        warm.warm_dense.copy_(snapshot)
                        t, ow = timed(fw)
                        tw = min(tw, t)
                    st, it = ow["status"], ow["iters"].double()
                    flag = (st & _lib.ST_WARM) != 0
                    rec["cold_ms"].append(tc); rec["warm_ms"].append(tw)
                    rec["cold_iters"].append(oc["iters"].double().mean().item())
                    rec["cold_iters_max"].append(int(oc["iters"].max().item()))
                    rec["warm_iters_mean"].append(it.mean().item()); rec["warm_iters_max"].append(int(it.max().item()))
                    rec["warm_flag_frac"].append(flag.double().mean().item())
                    rec["fallbacks"].append(int((valid & ~flag).sum().item()))
                    rec["handed_back"].append(int(((st & _lib.ST_PATH_LH) != 0).sum().item()))
                    p = p * (1 + delta * torch.randn(p.shape, device=dev, generator=g, dtype=p.dtype))
                s = {k: float(np.mean(v)) for k, v in rec.items()}
                for k in ("warm_iters_max", "cold_iters_max"):
                    s[k] = int(max(rec[k]))
                s["fallbacks"] = int(sum(rec["fallbacks"])); s["handed_back"] = int(sum(rec["handed_back"]))
                key = f"d{d}_m{m}_B{B}_{mname}_delta{delta:g}"
                res[key] = {"mean": s, "per_epoch": rec}
                say(f"  {d} x {m} x {B} {mname:5s} delta {delta:<6g}: iters cold {s['cold_iters']:5.2f} (max {s['cold_iters_max']:2d})"
                    f"  warm {s['warm_iters_mean']:5.2f} (max {s['warm_iters_max']:2d})   warm flag {100 * s['warm_flag_frac']:5.1f} %"
                    f"   fallbacks {s['fallbacks']:4d}   handed back {s['handed_back']:3d}   step cold {s['cold_ms']:7.2f} ms"
                    f"  warm {s['warm_ms']:7.2f} ms  ({s['warm_ms'] / s['cold_ms']:.3f}x)")
        del A, c0, cold, warm
        torch.cuda.empty_cache()
    return res


def child_cold(steps):
    """Cold-step measurements in this process (the library chosen by CAVE_B200_LIB) at every point and mode: one JSON line."""
    import torch
    import cave_b200
    from cave_b200 import _lib, pack_constraints
    dev = torch.device("cuda", torch.cuda.current_device())
    res = {}
    for d, m, B in POINTS:
        A, c = dataset(d, m, B, dev)
        pack = pack_constraints(A)
        idx = torch.arange(B, dtype=torch.int32, device=dev)
        for mname, mode in MODES.items():
            for _ in range(2):
                call(c, pack, idx, mode)
            ms, out = [], None
            for _ in range(steps):
                t, out = timed(lambda: call(c, pack, idx, mode))
                ms.append(t)
            h = hashlib.sha256()
            for k in ("loss", "grad", "status", "iters"):
                h.update(out[k].cpu().numpy().tobytes())
            res[f"d{d}_m{m}_B{B}_{mname}"] = {"ms": ms, "hash": h.hexdigest()[:16]}
        del A, c, pack
        torch.cuda.empty_cache()
    print(json.dumps({"package": os.path.dirname(cave_b200.__file__), "lib": _lib.LIB_PATH, "points": res}), flush=True)


def ab(root_a, say, reps=3, steps=5):
    """Cold step of the package in root_a ('parent') and of this one ('this'), alternated in child processes."""
    import numpy as np
    roots = {"parent": os.path.abspath(root_a), "this": ROOT}
    runs = {name: [] for name in roots}
    for _ in range(reps):
        for name, root in roots.items():
            env = dict(os.environ, CAVE_B200_LIB=os.path.join(root, "cave_b200", "_C", "libcave_b200.so"))
            pr = subprocess.run([sys.executable, os.path.abspath(__file__), "--child-cold", root, "--steps", str(steps)],
                                env=env, capture_output=True, text=True)
            if pr.returncode != 0:
                raise SystemExit(f"cold step with {root} failed:\n{pr.stderr[-4000:]}")
            r = json.loads(pr.stdout.strip().splitlines()[-1])
            if name == "parent" and not r["package"].startswith(roots["parent"]):
                raise SystemExit(f"the parent run imported {r['package']}")
            runs[name].append(r["points"])
    res = {}
    for key in runs["this"][0]:
        med = {name: [float(np.median(r[key]["ms"])) for r in rs] for name, rs in runs.items()}
        hashes = {name: sorted({r[key]["hash"] for r in rs}) for name, rs in runs.items()}
        same = hashes["parent"] == hashes["this"] and len(hashes["this"]) == 1
        res[key] = {"runs_ms": {name: [r[key]["ms"] for r in rs] for name, rs in runs.items()}, "median_per_run_ms": med,
                    "identical_outputs": same, "hashes": hashes}
        say(f"  {key:24s}: parent {' '.join(f'{x:7.2f}' for x in med['parent'])} ms   this "
            f"{' '.join(f'{x:7.2f}' for x in med['this'])} ms   (median of {steps} steps per run, runs alternated)   "
            f"outputs identical: {same}")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--ab-root", default="", help="directory holding another cave_b200 package, built (e.g. the parent "
                                                  "commit's), for the cold A/B")
    ap.add_argument("--skip-ab", action="store_true", help="measure the sweep alone (the report then says so)")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--child-cold", default="", help=argparse.SUPPRESS)
    ap.add_argument("--steps", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("dense_warm_probe needs a CUDA device")
    if a.child_cold:
        sys.path.insert(0, a.child_cold)        # the package under test
        child_cold(a.steps)
        return
    if not a.ab_root and not a.skip_ab:
        raise SystemExit("the cold A/B needs --ab-root DIR (a built checkout of the commit to compare against); "
                         "--skip-ab measures the sweep alone")
    dev = torch.device("cuda", torch.cuda.current_device())
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    res = {"card": card()}
    say(f"card: {res['card']}")
    if not a.no_sweep:
        say("(a) perturbation sweep, resident dense datasets, 5 timed epochs after the first (best of 3 device-timed steps "
            "per epoch, cold and warm alternated)")
        res["sweep"] = sweep(dev, say)
    if a.ab_root:
        say("(b) cold step, the package in --ab-root (parent) against this one, resident pack, alternated child processes")
        res["ab"] = ab(a.ab_root, say, steps=a.steps)
    else:
        say("(b) cold A/B SKIPPED (--skip-ab): this report does not show the cold step unchanged")
        res["ab"] = "skipped"
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "r3_dense_warm_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(a.out, "r3_dense_warm_probe.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
