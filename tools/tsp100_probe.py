"""TSP-100 (d = 4950) on the solve kernel's wide configuration (256 threads x 1 CTA/SM, the per-block maximum of shared
memory) against 256 x 2, where the Newton working set of a TSP-100 instance does not fit shared memory and is placed
generically (factor and part of the Hessian in the CTA's global slot).

(a) TSP-100 x {2048, 4096}, sparse resident pack (SparseConstraints -> pack_constraints_sparse, index=), innerConeAlignedCosine
    mode, uniform and near predictions: cold calls, and warm calls one perturbation of delta = 1e-2 away from the stored
    solution (the state is restored before every timed warm call).  The default launch plan (configuration 4) and
    CAVE_SOLVE_CFG=3 alternate call by call in one process (the ABI reads the variable on every call); device events;
    median / min / max per arm.  Outputs of the two arms are compared bit for bit.
(b) TSP-50 x 4096 A/B against another build of the library (--parent-lib, loaded through CAVE_B200_LIB in a child process;
    e.g. the parent commit's): cold one-shot call on the dense batch and cold call on the resident pack, the two builds
    alternated process by process.

    python tools/tsp100_probe.py [--out DIR] [--parent-lib PATH] [--reps N]
        (prints a report; with --out writes DIR/r3_tsp100_probe.{txt,json})
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

ST_WARM = 0x400


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed_once(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def stats(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "n": len(v)}


def set_cfg(cfg):
    if cfg is None:
        os.environ.pop("CAVE_SOLVE_CFG", None)
    else:
        os.environ["CAVE_SOLVE_CFG"] = str(cfg)


def part_a(dev, say, reps):
    from cave_b200 import SparseConstraints, cave_forward_backward, pack_constraints_sparse, synth
    arms = (("plan (cfg 4)", None), ("cfg 3", 3))
    res = {}
    insts_all = synth.make_batch("tsp100", 4096, seed=3000)
    for B in (2048, 4096):
        insts = insts_all[:B]
        sc = SparseConstraints.from_instances(insts)
        cold = pack_constraints_sparse(sc, device=dev)
        warm = pack_constraints_sparse(sc, device=dev, warm_start=True)
        plan = cold.launch_plan("fp64")
        idx = torch.arange(B, dtype=torch.int32, device=dev)
        say(f"  B = {B}: launch plan {plan['config']} ({plan['threads']} x {plan['ctas_per_sm']}, {plan['smem_bytes']} B), "
            f"largest hot set {plan['max_hot_bytes_f64'] / 1024:.1f} KiB (fp64 factor), "
            f"mean working set {plan['avg_work_bytes_f64'] / 1024:.1f} KiB")
        for regime in ("uniform", "near"):
            p0 = torch.tensor(synth.predictions(insts, 3000, regime), device=dev)
            g = torch.Generator(device=dev).manual_seed(11)
            p1 = p0 * (1 + 1e-2 * torch.randn(p0.shape, device=dev, generator=g, dtype=p0.dtype))

            def call(pack, p):
                return cave_forward_backward(p, None, -1.0, 1, 0.2, "mean", pack=pack, index=idx, want_proj=True,
                                             want_status=True)
            for label, cfg in arms:                 # warm-up of both arms (module load, attributes)
                set_cfg(cfg)
                call(cold, p0)
            set_cfg(None)
            warm.reset_warm_start()
            call(warm, p0)                          # the stored solutions the warm calls start from
            snapshot = warm.warm.clone()
            t = {f"{kind} {label}": [] for kind in ("cold", "warm") for label, _ in arms}
            outs, ok = {}, True
            for r in range(reps):
                for label, cfg in (arms if r % 2 == 0 else arms[::-1]):
                    set_cfg(cfg)
                    ms, oc = timed_once(lambda: call(cold, p0))
                    t[f"cold {label}"].append(ms)
                    warm.warm.copy_(snapshot)
                    ms, ow = timed_once(lambda: call(warm, p1))
                    t[f"warm {label}"].append(ms)
                    outs[label] = (oc, ow)
            set_cfg(None)
            a, b = outs[arms[0][0]], outs[arms[1][0]]
            for x, y in zip(a, b):
                for k in ("loss", "grad", "proj", "rnorm", "status", "iters"):
                    ok &= bool(torch.equal(x[k], y[k]))
            oc, ow = a
            conv = int(((oc["status"] & 0xff) == 0).sum().item()), int(((ow["status"] & 0xff) == 0).sum().item())
            wflag = int(((ow["status"] & ST_WARM) != 0).sum().item())
            row = {k: stats(v) for k, v in t.items()}
            row.update({"bit_identical": ok, "converged_cold": conv[0], "converged_warm": conv[1], "warm_flag": wflag,
                        "mean_iters_cold": oc["iters"].double().mean().item(),
                        "mean_iters_warm": ow["iters"].double().mean().item()})
            res[f"B{B}_{regime}"] = row
            say(f"    {regime:7s}: iterations cold {row['mean_iters_cold']:.2f} warm {row['mean_iters_warm']:.2f}; "
                f"converged {conv[0]}/{B} cold {conv[1]}/{B} warm, warm flag {wflag}/{B}; arms bit-identical: {ok}")
            for kind in ("cold", "warm"):
                s4, s3 = row[f"{kind} plan (cfg 4)"], row[f"{kind} cfg 3"]
                say(f"      {kind}: cfg 4 {s4['median_ms']:8.3f} ms [{s4['min_ms']:.3f}, {s4['max_ms']:.3f}]   "
                    f"cfg 3 {s3['median_ms']:8.3f} ms [{s3['min_ms']:.3f}, {s3['max_ms']:.3f}]   "
                    f"cfg 3 / cfg 4 = {s3['median_ms'] / s4['median_ms']:.2f}x   "
                    f"({B / s4['median_ms']:.0f} k inst/s vs {B / s3['median_ms']:.0f} k inst/s)")
        del cold, warm
        torch.cuda.empty_cache()
    return res


def tsp50_child(reps):
    """TSP-50 x 4096 (the bench workload's shape) in this process, with the library CAVE_B200_LIB names: one JSON line."""
    from cave_b200 import cave_forward_backward, pack_constraints, synth
    dev = torch.device("cuda", torch.cuda.current_device())
    insts = synth.make_batch("tsp50", 4096, seed=1000)
    A = synth.densify(insts, device=dev)
    pred = torch.tensor(synth.predictions(insts, 1000, "uniform"), device=dev)
    pack = pack_constraints(A)
    idx = torch.arange(4096, dtype=torch.int32, device=dev)
    one_shot = lambda: cave_forward_backward(pred, A, -1.0, 1, 0.2, "mean", want_status=True)            # noqa: E731
    resident = lambda: cave_forward_backward(pred, None, -1.0, 1, 0.2, "mean", pack=pack, index=idx, want_status=True)  # noqa: E731
    out = {}
    for name, fn in (("one_shot", one_shot), ("resident", resident)):
        for _ in range(3):
            fn()
        v = [timed_once(fn)[0] for _ in range(reps)]
        o = fn()
        out[name] = {**stats(v), "loss": float(o["loss"].item())}
    print("TSP50 " + json.dumps(out), flush=True)


def part_b(say, parent_lib, rounds=3, reps=10):
    libs = (("this build", os.path.join(ROOT, "cave_b200", "_C", "libcave_b200.so")), ("parent", os.path.abspath(parent_lib)))
    runs = {label: [] for label, _ in libs}
    for r in range(rounds):
        for label, path in (libs if r % 2 == 0 else libs[::-1]):
            env = dict(os.environ, CAVE_B200_LIB=path)
            env.pop("CAVE_SOLVE_CFG", None)
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--tsp50-child", "--reps", str(reps)], env=env,
                               capture_output=True, text=True, check=True)
            line = [s for s in p.stdout.splitlines() if s.startswith("TSP50 ")][-1]
            runs[label].append(json.loads(line[6:]))
    res = {}
    for name in ("one_shot", "resident"):
        res[name] = {}
        for label, _ in libs:
            med = [x[name]["median_ms"] for x in runs[label]]
            res[name][label] = {"median_of_medians_ms": float(np.median(med)), "medians_ms": med,
                                "min_ms": float(min(x[name]["min_ms"] for x in runs[label])),
                                "max_ms": float(max(x[name]["max_ms"] for x in runs[label])),
                                "loss": runs[label][0][name]["loss"]}
        a, b = res[name]["this build"], res[name]["parent"]
        say(f"  {name:8s}: this build {a['median_of_medians_ms']:.3f} ms [{a['min_ms']:.3f}, {a['max_ms']:.3f}]   parent "
            f"{b['median_of_medians_ms']:.3f} ms [{b['min_ms']:.3f}, {b['max_ms']:.3f}]   ratio "
            f"{a['median_of_medians_ms'] / b['median_of_medians_ms']:.3f}   loss equal: {a['loss'] == b['loss']}")
    return {"runs": runs, "summary": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--parent-lib", default="")
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--tsp50-child", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tsp100_probe needs a CUDA device")
    if a.tsp50_child:
        return tsp50_child(a.reps)
    dev = torch.device("cuda", torch.cuda.current_device())
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    res = {"card": card()}
    say(f"card: {res['card']}")
    say(f"(a) TSP-100, sparse resident pack, innerConeAlignedCosine mode, fp64 factor, float32 I/O; default plan vs "
        f"CAVE_SOLVE_CFG=3 alternated call by call, {a.reps} device-timed calls per arm: median [min, max]")
    res["a"] = part_a(dev, say, a.reps)
    if a.parent_lib:
        say("(b) TSP-50 x 4096 (bench shape, uniform predictions, innerConeAlignedCosine mode): this build vs the parent "
            "build, 3 processes each, alternated; median of the per-process medians [min, max over all calls]")
        res["b"] = part_b(say, a.parent_lib)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "r3_tsp100_probe.json"), "w") as f:
            json.dump(res, f, indent=1)
        with open(os.path.join(a.out, "r3_tsp100_probe.txt"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
