"""Chunked host-input calls against unchunked ones: the three end-to-end legs of DESIGN §7 (TSP-50, innerConeAlignedCosine, a
module step with host tensors in and host loss / gradient out), each unchunked and with solver_kwargs={"chunk": k}.

  dense_host     pinned dense [B, m, d] host tensor (the reference's own call): a one-shot pack per chunk
  host_csr       pinned SparseConstraints: a one-shot sparse pack per chunk
  resident       pack over the dataset on the device, pinned pred and index on the host: slices of both per chunk

The arms of a leg alternate step by step in one process (the order rotates every round).  Each step is timed with a host
clock around a synchronised step and with CUDA events on the current stream; peak device memory is recorded per arm; the
loss and gradient of every step are compared bit for bit with the first unchunked step of the leg.  The card's name and
power limit are read in the same run.  Writes <out>/r3_chunk_probe.{txt,json}.

    python tools/chunk_probe.py [--batch 4096] [--rounds 7] [--chunks 256 512 1024 2048] [--out profiles]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:      # the probe still runs; the record says why the card is not named
        q = f"nvidia-smi unavailable ({e})"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--chunks", type=int, nargs="+", default=[256, 512, 1024, 2048])
    ap.add_argument("--legs", nargs="+", default=["resident", "host_csr", "dense_host"])
    ap.add_argument("--out", default="profiles")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("chunk_probe needs a CUDA device")
    from cave_b200 import EPO, SparseConstraints, innerConeAlignedCosine, pack_constraints, synth

    dev = torch.device("cuda:0")
    B = args.batch
    insts = synth.make_batch("tsp50", B, seed=1000)
    pred = torch.tensor(synth.predictions(insts, 1000, "uniform"))
    pred_host = pred.pin_memory()
    A_dev = synth.densify(insts, device=dev)

    class Model:
        modelSense = EPO.MINIMIZE

    arms = [None] + list(args.chunks)
    mods = {c: innerConeAlignedCosine(Model(), solver="cuda", inner_ratio=0.2, seed=0,
                                      solver_kwargs={} if c is None else {"chunk": c}) for c in arms}
    result = {"card": card(), "batch": B, "shape": "tsp50", "rounds": args.rounds, "legs": {}}
    lines = [f"card: {result['card']}", f"TSP-50, innerConeAlignedCosine, B = {B}, {args.rounds} rounds per arm, arms alternate"]

    for leg in args.legs:
        if leg == "resident":
            pack = pack_constraints(A_dev)
            perm = torch.randperm(B, dtype=torch.int32, generator=torch.Generator().manual_seed(0)).pin_memory()
            p_in = torch.empty_like(pred_host).pin_memory()
            p_in.copy_(pred[perm.long()])
            Bl, h2d = B, p_in.numel() * 4 + B * 4
            inputs = lambda: (pack, dict(index=perm))       # noqa: E731
        elif leg == "host_csr":
            sc = SparseConstraints.from_instances(insts).pin_memory()
            p_in, Bl, h2d = pred_host, B, sc.nbytes() + pred_host.numel() * 4
            inputs = lambda: (sc, {})                       # noqa: E731
        else:
            # bounded, as bench.py bounds it, to 40 % of the available host memory for the pinned copy
            Bl = B
            try:
                import psutil
                Bl = int(max(64, min(B, 0.4 * psutil.virtual_memory().available // (A_dev.shape[1] * A_dev.shape[2] * 4))))
            except ImportError:
                pass
            A_host = torch.empty((Bl,) + tuple(A_dev.shape[1:]), dtype=A_dev.dtype, pin_memory=True)
            A_host.copy_(A_dev[:Bl])
            p_in = pred_host[:Bl]
            h2d = A_host.numel() * 4 + p_in.numel() * 4
            inputs = lambda: (A_host, {})                   # noqa: E731

        def step(c):
            ctrs, kw = inputs()
            p = p_in.detach().requires_grad_(True)
            loss = mods[c](p, ctrs, **kw)
            loss.backward()
            return loss.detach(), p.grad

        rec = {c: {"host_ms": [], "event_ms": [], "peak_bytes": 0, "bit_identical": True, "max_rel_diff": 0.0} for c in arms}
        ref = None
        for c in arms:      # warm-up of every arm (first launches, allocator)
            out = step(c)
            torch.cuda.synchronize()
            if ref is None:
                ref = (out[0].clone(), out[1].clone())
        for r in range(args.rounds):
            order = arms[r % len(arms):] + arms[:r % len(arms)]
            for c in order:
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats(dev)
                base = torch.cuda.memory_allocated(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                e0.record()
                loss, grad = step(c)
                e1.record()
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                a = rec[c]
                a["host_ms"].append((t1 - t0) * 1e3)
                a["event_ms"].append(e0.elapsed_time(e1))
                a["peak_bytes"] = max(a["peak_bytes"], torch.cuda.max_memory_allocated(dev) - base)
                same = torch.equal(loss.cpu(), ref[0].cpu()) and torch.equal(grad.cpu(), ref[1].cpu())
                a["bit_identical"] &= bool(same)
                g, gr = grad.double().cpu(), ref[1].double().cpu()
                rel = float(((g - gr).abs().max() / gr.abs().max().clamp(min=1e-300)).item())
                a["max_rel_diff"] = max(a["max_rel_diff"], rel, abs(float(loss) - float(ref[0])) / max(abs(float(ref[0])), 1e-300))
        lines.append(f"\n== {leg}: B = {Bl}, {h2d / 1e6:.1f} MB H2D per step")
        lines.append(f"{'chunk':>8} {'host ms (median, min-max)':>28} {'event ms (median)':>18} {'peak device MB':>15} "
                     f"{'bit-identical':>14} {'max rel diff':>13}")
        for c in arms:
            a = rec[c]
            hm, em = np.array(a["host_ms"]), np.array(a["event_ms"])
            a.update(host_ms_median=float(np.median(hm)), event_ms_median=float(np.median(em)), batch=Bl, h2d_bytes=int(h2d))
            lines.append(f"{str(c):>8} {np.median(hm):10.2f} ({hm.min():7.2f}-{hm.max():7.2f}) {np.median(em):18.2f} "
                         f"{a['peak_bytes'] / 1e6:15.1f} {str(a['bit_identical']):>14} {a['max_rel_diff']:13.2e}")
        result["legs"][leg] = {str(c): rec[c] for c in arms}
        print("\n".join(lines[-(len(arms) + 2):]), flush=True)
        pack = sc = A_host = None       # noqa: F841 (the leg's inputs)
        torch.cuda.empty_cache()

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r3_chunk_probe.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    with open(os.path.join(args.out, "r3_chunk_probe.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
