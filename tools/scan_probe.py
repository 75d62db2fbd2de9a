"""Times the scan (pack) pass alone and compares the pack content of two builds.

    python tools/scan_probe.py [--ab-root CHECKOUT] [--reps 20] [--out DIR]

Workloads: TSP-50, TSP-20, VRP-20 and SP 5x5 at B = 4096 (flags 0 pack pass through cave_pack_ex into one preallocated
buffer, as bench.py times kernels[0]), the dense 1225 x 1024 x 592 batch through the same pass (inner mode: the
instantiation with the average), and the same dense batch in a cold exact-mode call, whose one-shot pack runs the
instantiation without the average (scan kernel time from torch.profiler).  With --ab-root (a built checkout of another
revision) both libraries are loaded into this process and alternated rep by rep; the pack content of every instance is
compared between them: counts, the general rows with their CSR slices, hashes, average, cone types, csr_ok, maxl1, maxl2.
Raw CSR offsets are not compared: general rows take their offsets in the order the warps reach them.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _a256(v: int) -> int:
    return (v + 255) & ~255


def pack_layout(B: int, m: int, d: int) -> dict:
    """Byte offsets of the pack arrays the scan writes (mirror of make_pack_layout in cave_b200/csrc/layout.cuh)."""
    dpad = (d + 15) & ~15
    full, c = m * d, 16 * d + 4096
    cap = (c if c < full else full + 1) // 8 * 8 + 8
    L, o = {"dpad": dpad, "cap_nnz": cap}, 0
    for name, nb in (("nvalid", B * 4), ("navg", B * 4), ("ngen", B * 4), ("gennnz", B * 4), ("nsingc", B * 4),
                     ("gen", B * m * 16), ("ctype", B * dpad), ("avg", B * dpad * 4), ("csrok", B * 4), ("maxl1", B * 4),
                     ("maxl2", B * 4), ("ghash", B * m * 16), ("csr_col", B * cap * 2), ("csr_val", B * cap * 4)):
        L[name] = o
        o = _a256(o + nb)
    return L


def pack_content(buf, B: int, m: int, d: int) -> list:
    """Per-instance pack content as comparable tuples of bytes (independent of the order of the CSR slices)."""
    raw = buf.cpu().numpy() if hasattr(buf, "cpu") else np.asarray(buf)
    L = pack_layout(B, m, d)
    cap, dpad = L["cap_nnz"], L["dpad"]

    def arr(name, dtype, count):
        return np.frombuffer(raw, dtype=dtype, count=count, offset=L[name])

    cnt = {k: arr(k, np.int32, B) for k in ("nvalid", "navg", "ngen", "gennnz", "nsingc", "csrok")}
    maxl1, maxl2 = arr("maxl1", np.uint32, B), arr("maxl2", np.uint32, B)
    gen = arr("gen", np.int32, B * m * 4).reshape(B, m, 4)
    ghash = arr("ghash", np.uint64, B * m * 2).reshape(B, m, 2)
    ctype = arr("ctype", np.uint8, B * dpad).reshape(B, dpad)
    avg = arr("avg", np.uint32, B * dpad).reshape(B, dpad)
    col = arr("csr_col", np.uint16, B * cap).reshape(B, cap)
    val = arr("csr_val", np.uint32, B * cap).reshape(B, cap)
    out = []
    for b in range(B):
        ng, ok = int(cnt["ngen"][b]), int(cnt["csrok"][b])
        rows = []
        for r, n, off, _ in gen[b, :max(ng, 0)]:
            row = [int(r), int(n)]
            if ok != 0:     # (an instance that overflows the packed CSR keeps the hashes of the rows that happened to fit)
                row += [ghash[b, r].tobytes(), col[b, off:off + n].tobytes(), val[b, off:off + n].tobytes()]
            rows.append(tuple(row))
        out.append((tuple(int(cnt[k][b]) for k in cnt), int(maxl1[b]), int(maxl2[b]), tuple(rows),
                    ctype[b].tobytes(), avg[b].tobytes()))
    return out


def _load(lib_path: str):
    from cave_b200 import _lib
    saved, saved_path = _lib._lib, _lib.LIB_PATH
    _lib._lib, _lib.LIB_PATH = None, lib_path
    try:
        return _lib.load()
    finally:
        _lib._lib, _lib.LIB_PATH = saved, saved_path


def _gpu_info() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return {"nvidia_smi": q}


def _stats(ms: list) -> dict:
    s = sorted(ms)
    return {"median": statistics.median(s), "min": s[0], "max": s[-1], "p25": s[len(s) // 4], "p75": s[(3 * len(s)) // 4],
            "n": len(s)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--ab-root", default="", help="built checkout of another revision to alternate with")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=".", help="directory for scan_probe.txt and scan_probe.json")
    ap.add_argument("--only", default="", help="comma-separated subset of workload names")
    args = ap.parse_args()
    import torch
    from cave_b200 import _lib, cave_forward_backward, synth

    assert torch.cuda.is_available(), "scan_probe needs a CUDA device"
    dev = torch.device("cuda:0")
    arms = {"this": _lib.load()}
    if args.ab_root:
        arms["ab"] = _load(os.path.join(os.path.abspath(args.ab_root), "cave_b200", "_C", "libcave_b200.so"))
    names = list(arms)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    res = {"gpu": _gpu_info(), "reps": args.reps, "arms": {"this": ROOT, "ab": os.path.abspath(args.ab_root) if args.ab_root else None},
           "workloads": {}}
    lines = [f"# scan_probe  {res['gpu']['nvidia_smi']}", f"# reps per arm {args.reps}, arms alternated rep by rep"]

    def structured(kind):
        insts = synth.make_batch(kind, 4096, seed=1000)
        return synth.densify(insts, device=dev)

    def dense():
        g = torch.Generator(device=dev).manual_seed(1000)
        return torch.randn((592, 1024, 1225), generator=g, device=dev)

    wl = [("tsp50", lambda: structured("tsp50")), ("tsp20", lambda: structured("tsp20")), ("vrp20", lambda: structured("vrp20")),
          ("sp5", lambda: structured("sp5")), ("dense1225x1024_inner", dense), ("dense1225x1024_exact", dense)]
    if args.only:
        keep = set(args.only.split(","))
        wl = [w for w in wl if w[0] in keep]
    for name, make in wl:
        A = make()
        B, m, d = A.shape
        nbytes = B * m * d * 4
        entry = {"shape": [B, m, d], "bytes": nbytes}
        if name.endswith("_exact"):
            # cold exact-mode call: its one-shot pack skips the average (SKIPAVG instantiation); scan time from the profiler
            c = torch.randn((B, d), generator=torch.Generator(device=dev).manual_seed(7), device=dev, dtype=torch.float64)
            times = {a: [] for a in names}
            outs = {}
            for rep in range(args.reps + 1):
                for a in names:
                    _lib._lib = arms[a]
                    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                        o = cave_forward_backward(c, A, 1.0, 0, reduction="none")
                        torch.cuda.synchronize()
                    ks = [e for e in prof.events() if "scan_rows_kernel" in e.name]
                    assert len(ks) == 1, [e.name for e in prof.events()][:20]
                    if rep:
                        times[a].append(ks[0].device_time_total / 1e3)
                    outs[a] = o
            _lib._lib = arms["this"]
            if len(names) == 2:
                entry["outputs_equal"] = all(torch.equal(outs["this"][k], outs["ab"][k]) for k in ("loss_i", "grad"))
        else:
            nb = ctypes.c_size_t()
            _lib.check(arms["this"].cave_pack_bytes(B, m, d, ctypes.byref(nb)))
            bufs = {a: torch.empty(nb.value, dtype=torch.uint8, device=dev) for a in names}

            def run(a):
                _lib.check(arms[a].cave_pack_ex(ctypes.c_void_p(A.data_ptr()), None, B, m, d, 0,
                                                ctypes.c_void_p(bufs[a].data_ptr()), nb.value, stream))
            for a in names:
                run(a); run(a)
            torch.cuda.synchronize()
            times = {a: [] for a in names}
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            for rep in range(args.reps):
                for a in names:
                    ev[0].record(); run(a); ev[1].record(); ev[1].synchronize()
                    times[a].append(ev[0].elapsed_time(ev[1]))
            if len(names) == 2:
                ca, cb = pack_content(bufs["this"], B, m, d), pack_content(bufs["ab"], B, m, d)
                entry["instances_differing"] = sum(x != y for x, y in zip(ca, cb))
            del bufs
        for a in names:
            entry[a] = _stats(times[a])
            entry[a]["tb_s"] = nbytes / (entry[a]["median"] * 1e-3) / 1e12
        res["workloads"][name] = entry
        ln = f"{name:24s} {B}x{m}x{d}  " + "  ".join(
            f"{a}: {entry[a]['median']:.3f} ms [{entry[a]['min']:.3f}, {entry[a]['max']:.3f}] {entry[a]['tb_s']:.2f} TB/s" for a in names)
        for k in ("instances_differing", "outputs_equal"):
            if k in entry:
                ln += f"  {k}={entry[k]}"
        lines.append(ln)
        print(ln, flush=True)
        del A
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "scan_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(args.out, "scan_probe.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
