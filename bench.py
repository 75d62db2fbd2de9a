#!/usr/bin/env python
"""
bench.py — CaVE loss+grad throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload tsp50|tsp20|vrp20|sp5|sweep]

A "step" is one pass of the hot path (scan/pack of A + projection + push-inside + cosine loss +
reduction + analytic backward) over one synthetic batch.  Headline workload: TSP-50 DFJ binding constraints
(d = 1225, m = 1325 + k tight cuts, SURVEY.md App. B), CaVE+ inner_ratio 0.2, batch 4096 per GPU
(BASELINE.json configs[2], the configuration the metric is quoted on).  Instances shard across
GPUs by instance with no data-path collective (weak scaling: 4096 per GPU).

Prints ONE JSON line (rank 0).  `value` is device-resident throughput (inputs already in HBM, the
dense [B, m_max, d] float32 layout the reference API hands over, pack rebuilt every step = cold);
`e2e` is the same metric through the module call with HOST tensors (pinned), including the
host->device copy of pred_cost and tight_ctrs and the device->host read of loss and gradient.
Beside the headline the line carries
  `workloads`      every named shape of BASELINE.json configs (SP 5x5, TSP-20, VRP-20, dense sweep points) at this N:
                   inst/s, roofline fraction and the CPU baseline of the same instances,
  `strong`         strong scaling: a global batch of 4096 (and of 65 536 where it fits) split N ways,
  `parity_sample`  the timed batch's first instances re-computed by the CPU oracle (outside the timed region).
`--impl reference` times the reference's CPU path (scipy nnls per instance + the torch epilogue,
restated in oracle/cave_oracle.py; the Python reference itself cannot travel to the GPU box) on
all host cores on a bounded sample of the same workload.
`--dump-outputs DIR` writes what the last timed step returned (rank 0's `loss`, `loss_i`, `grad`) as
DIR/<name>.npy, so that two builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "cave_loss_grad_instances_per_sec"
UNIT = "instances/s"
WORKLOADS = {  # name -> (synth kind, per-GPU batch, mode, inner_ratio)
    "tsp50": ("tsp50", 4096, 1, 0.2),
    "tsp20": ("tsp20", 4096, 1, 0.2),
    "vrp20": ("vrp20", 4096, 1, 0.2),
    "sp5": ("sp5", 4096, 0, 0.0),
}
# dense sweep points (d, m, per-GPU batch) reported by default; --workload sweep runs the full grid
SWEEP_DEFAULT = [(1225, 256, 1184), (1225, 1024, 592), (4950, 256, 592)]
SWEEP_FULL = [(190, 64, 8192), (190, 256, 4096), (190, 1024, 1184), (1225, 64, 4096), (1225, 256, 2368), (1225, 1024, 1184),
              (1225, 2048, 148), (4950, 64, 2368), (4950, 256, 1184), (4950, 1024, 296), (4950, 2048, 148)]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="tsp50", choices=sorted(WORKLOADS) + ["sweep"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override (0 = workload default)")
    ap.add_argument("--precision", default="fp64", choices=["fp64", "fp32"])
    ap.add_argument("--regime", default="uniform", choices=["uniform", "near"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `workloads` and `strong` keys")
    ap.add_argument("--cpu-sample", type=int, default=0, help="instances in the CPU baseline sample (0 = 2 x cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "sweep"):
        ap.error("--dump-outputs applies to --impl ours on a structured workload")
    return args


DUMP_BYTES = 64_000_000


def dump_outputs(arrays, dirname, limit=DUMP_BYTES):
    """Write arrays as dirname/<name>.npy in float32 or float64 (other dtypes as float64).  If they exceed `limit` bytes in all,
    the per-instance arrays (leading dimension = the batch of `grad`) keep a fixed, seeded sample of instances, whose indices
    go to instance_index.npy."""
    arrays = {k: a if a.dtype in (np.float32, np.float64) else a.astype(np.float64) for k, a in arrays.items()}
    B = arrays["grad"].shape[0]
    per_inst = [k for k, a in arrays.items() if a.ndim and a.shape[0] == B]
    total = sum(a.nbytes for a in arrays.values())
    if total > limit - 4096:                  # 4 KB for the .npy headers
        row = sum(arrays[k].nbytes // B for k in per_inst) + 8
        keep = max(1, (limit - 4096 - (total - sum(arrays[k].nbytes for k in per_inst))) // row)
        idx = np.sort(np.random.default_rng(0).choice(B, size=keep, replace=False))
        arrays = {k: a[idx] if k in per_inst else a for k, a in arrays.items()}
        arrays["instance_index"] = idx.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), a)


# ----------------------------------------------------------------------------- CPU reference arm
def _cpu_one(args):
    """One instance through the reference's CPU path (oracle restatement): projection by
    scipy.optimize.nnls + target + loss + gradient.  Returns (loss_i, grad)."""
    from oracle import cave_oracle as O
    pred, ctr, mode, ratio = args
    out = O.forward_backward(pred[None], ctr[None], minimize=True, mode=mode, inner_ratio=ratio, reduction="none")
    return float(out["loss_i"][0]), out["grad"][0]


def _cpu_pool(cores):
    import multiprocessing as mp
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    return mp.get_context("fork").Pool(cores)


def _cpu_sample(kind, n, mode, ratio, regime, seed):
    """The first n instances of the batch that rank 0 times on the GPU (same generator, same seed)."""
    from cave_b200 import synth
    insts = synth.make_batch(kind, n, seed=seed)
    m_max = max(i.m for i in insts)
    pred = synth.predictions(insts, seed, regime)[:n]
    return [(pred[b], insts[b].dense(m_max), mode, ratio) for b in range(n)]


def _dense_sample(d, m, n, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    A = torch.randn((n, m, d), generator=g).numpy()
    c = torch.randn((n, d), generator=g).numpy()
    return [(-c[b], A[b], 0, 0.0) for b in range(n)]


def run_reference(args):
    """Reference arm: rank 0 alone; each step = `cores` instances of the workload on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = args.cpu_sample or cores
    if args.workload == "sweep":
        d, m, _ = SWEEP_DEFAULT[1]
        work = _dense_sample(d, m, per_step, seed=1000)
        desc = f"dense sweep point d={d}, m={m} (N(0,1) rows), exact projection, solver='nnls' CPU path"
    else:
        kind, batch, mode, ratio = WORKLOADS[args.workload]
        work = _cpu_sample(kind, per_step, mode, ratio, args.regime, seed=1000)
        desc = f"{args.workload} (SURVEY App. B synthetic), CaVE+ inner_ratio {ratio}, solver='nnls' CPU path"
    pool = _cpu_pool(cores)
    for _ in range(max(args.warmup, 0)):
        pool.map(_cpu_one, work[:cores])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pool.map(_cpu_one, work)
    dt = time.perf_counter() - t0
    pool.close()
    value = per_step * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "sample_instances_per_step": per_step, "regime": args.regime,
                   "instances": "the first instances of the batch the GPU arm times on rank 0 (same generator and seed)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{per_step} instances/step x {args.steps} steps, multiprocessing.Pool({cores}) over "
                                   "oracle.forward_backward (scipy.optimize.nnls + epilogue), BLAS threads = 1"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        self.thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {0x2: "applications_clocks", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
                 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake", 0x100: "display"}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.nv:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        self._stop.set()
        if self.thread:
            self.thread.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def _traffic_from_profile(workload, B):
    """DRAM bytes per step of the dominant kernels from the committed ncu --set full capture of this command
    (profiles/r2_traffic.json, written by tools/ncu_summary.py with the commit it was captured on); None if absent."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        if t.get("workload") == workload and int(t.get("batch", 0)) == int(B):
            return {"bytes_per_step": float(t["dram_bytes_per_step"]), "commit": t.get("commit"), "source": t.get("source")}
    except Exception:
        pass
    return None


# ----------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    from cave_b200 import (EPO, SparseConstraints, _lib, cave_forward_backward, innerConeAlignedCosine, exactConeAlignedCosine,
                           pack_constraints, synth)
    from cave_b200.qpsolver import dense_gram

    lib = _lib.load()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs CUDA devices (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = None
    if world > 1:           # one process per GPU: keep its pinned host buffers on the GPU's NUMA node (e2e legs)
        from cave_b200.parallel import bind_to_gpu_numa_node
        numa = bind_to_gpu_numa_node(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    cores = os.cpu_count() or 1
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
    # TF32 dense tensor peak: half of the measured bf16 GEMM figure (nominal 1.1 vs 2.25 PFLOP/s; the driver measures bf16 only)
    tf32_peak = (peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops") or 1590.0) / 2.0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        """n calls of fn bracketed by barrier + synchronize; CUDA events on the launching stream; max over ranks."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / n

    def cpu_rate(work):
        """inst/s of the oracle port on all host cores over `work` (rank 0, N = 1 only)."""
        pool = _cpu_pool(cores)
        pool.map(_cpu_one, work[:min(len(work), cores)])
        t0 = time.perf_counter()
        res = pool.map(_cpu_one, work)
        dt = time.perf_counter() - t0
        pool.close()
        return len(work) / dt, res

    def parity(work, res, loss_i, grad):
        """max relative error of the GPU loss / gradient against the oracle on the same instances (float32 I/O)."""
        n = len(work)
        l_ref = np.array([r[0] for r in res]); g_ref = np.stack([r[1] for r in res])
        l_gpu = loss_i[:n].double().cpu().numpy(); g_gpu = grad[:n].double().cpu().numpy()
        # relative to the largest reference entry, floored: a cone that is the whole space has loss = 0 and gradient = 0 exactly
        return {"n": n, "max_rel_err_loss": float(np.abs(l_gpu - l_ref).max() / max(np.abs(l_ref).max(), 1e-6)),
                "max_rel_err_grad": float(np.abs(g_gpu - g_ref).max() / max(np.abs(g_ref).max(), 1e-6)),
                "max_abs_err_grad": float(np.abs(g_gpu - g_ref).max()), "max_abs_grad_ref": float(np.abs(g_ref).max()),
                "note": "GPU (this run's precision mode, float32 I/O) vs oracle.forward_backward in the reference's dtypes on the first n "
                        "instances of the timed batch; computed outside the timed region"}

    def structured(kind, batch, mode, ratio, steps, seed, want_sparse=False):
        """Device-resident cold-pack measurement of one structured workload; returns (dict, tensors for later legs)."""
        insts = synth.make_batch(kind, batch, seed=seed)
        if want_sparse:
            sparse_host.append(SparseConstraints.from_instances(insts).pin_memory())
        A = synth.densify(insts, device=dev)
        B, m_max, d = A.shape
        pred = torch.tensor(synth.predictions(insts, seed, args.regime), device=dev)
        alg_bytes = float(sum(4 * i.m * d + 8 * d + 4 for i in insts))       # SURVEY 8d
        gen_rows = [int((np.bincount(i.rows, minlength=i.m) > 1).sum()) for i in insts]
        del insts
        step = lambda: cave_forward_backward(pred, A, -1.0, mode, ratio, "mean", precision=args.precision)  # noqa: E731
        for _ in range(3):
            step()
        ms = timed(step, steps)
        info = {"inst_per_s": B * world / (ms * 1e-3), "ms_per_step": ms, "batch_per_gpu": B, "m_max": m_max, "d": d,
                "roofline": {"bound": "hbm", "achieved": alg_bytes / ms / 1e6, "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg_bytes / ms / 1e6 / hbm_peak}}
        return info, A, pred, alg_bytes, gen_rows

    def sweep_point(d, m, batch, steps, want_cpu):
        g = torch.Generator(device=dev).manual_seed(1000 + rank)
        A = torch.randn((batch, m, d), generator=g, device=dev)
        c = -torch.randn((batch, d), generator=g, device=dev)       # pred_cost; the signed cost is -pred (MINIMIZE, src/cave.py:62-64)
        # the host gate of the dense path is `m_max <= d` (structured models have m > d); rows up to 1.7 d still have a
        # unique solution for Gaussian rows, so the sweep asks for the dense path there explicitly
        dense = True if (d < m <= 1.7 * d and m >= 128) else "auto"
        step = lambda: cave_forward_backward(c, A, -1.0, 0, 0.0, "mean", precision=args.precision, dense=dense)  # noqa: E731
        for _ in range(2):
            step()
        ms = timed(step, steps)
        st = cave_forward_backward(c, A, -1.0, 0, 0.0, "none", precision=args.precision, want_status=True, dense=dense)
        status = st["status"].cpu().numpy()
        flops = float(batch) * (float(m) * m * d + 4.0 * m * d)                # SURVEY 8d "Algorithmic flops"
        info = {"d": d, "m": m, "batch_per_gpu": batch, "dense_mode": str(dense), "inst_per_s": batch * world / (ms * 1e-3), "ms_per_step": ms,
                "iters_mean": float(st["iters"].float().mean()),
                "path_gram_frac": float(((status & _lib.ST_PATH_GRAM) != 0).mean()),
                "converged_frac": float(((status & 0xff) == 0).mean()),
                "roofline": {"bound": "tensor", "achieved": flops / ms / 1e9, "peak": tf32_peak, "unit": "TFLOP/s",
                             "frac": flops / ms / 1e9 / tf32_peak,
                             "note": "flops_alg = m^2 d + 4 m d per instance over the WHOLE step (Gram + Gram-space solve + polish); "
                                     "peak = TF32 dense = measured bf16 / 2; the tensor-core Gram kernel alone is in `gram_kernel`"}}
        if m >= 128 and m <= 2048:
            nb = min(batch, 296)
            dense_gram(A[:nb], dense_slots=nb)
            msg = timed(lambda: dense_gram(A[:nb], dense_slots=nb), 3)
            # cave_dense_gram = scan/pack + list + TF32 split + Gram + copy of G; the pack pass alone is timed and subtracted
            msp = timed(lambda: pack_constraints(A[:nb]), 3)
            gf = float(nb) * float(m) * m * d * 3.0          # executed: 3 TF32 MMAs per product on the symmetric half (FMA = 2)
            info["gram_kernel"] = {"ms_per_instance_chipwide": (msg - msp) / nb, "executed_tf32_tflops": gf / max(msg - msp, 1e-9) / 1e9,
                                   "frac_of_tf32_peak": gf / max(msg - msp, 1e-9) / 1e9 / tf32_peak,
                                   "note": "TF32 split + Gram + D2D copy of G, pack pass subtracted; executed flops = 3 x m^2 d"}
        if want_cpu:
            n = max(4, min(2 * cores, 16))
            work = [(c[b].cpu().numpy(), A[b].cpu().numpy(), 0, 0.0) for b in range(n)]
            rate, res = cpu_rate(work)
            info["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": f"{n} instances of this batch"}
            info["parity_sample"] = parity(work, res, st["loss_i"], st["grad"])
        del A, c
        torch.cuda.empty_cache()
        return info

    if args.workload == "sweep":
        pts = [sweep_point(d, m, args.batch or b, args.steps, rank == 0 and world == 1 and not args.no_cpu_baseline)
               for d, m, b in SWEEP_FULL]
        head = next(p for p in pts if (p["d"], p["m"]) == (1225, 1024))
        line = {"metric": METRIC, "value": head["inst_per_s"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": 3, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "tf32x3 Gram + f32 factor + f64 iterates", "data": "synthetic",
                "config": {"workload": "dense projection sweep (BASELINE.json configs[4]): A ~ N(0,1)^{m x d}, exact projection, cold pack; "
                                       "headline point d=1225, m=1024", "l2_policy": "inputs larger than L2"},
                "roofline": head["roofline"], "sweep": pts, "cpu_baseline": head.get("cpu_baseline"), "e2e": None, "gpu_launches": None}
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    kind, batch, mode, ratio = WORKLOADS[args.workload]
    batch = args.batch or batch
    # every rank owns its own shard of the global batch (no data-path collective)
    seed = 1000 + rank
    sparse_host = []
    head, A, pred, alg_bytes, gen_rows = structured(kind, batch, mode, ratio, 1, seed, want_sparse=not args.no_e2e)
    B, m_max, d = A.shape

    last = {}

    def step():
        last["out"] = cave_forward_backward(pred, A, -1.0, mode, ratio, "mean", precision=args.precision)

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local)
    sampler.start()
    n0 = lib.cave_launch_count()
    ms_step = timed(step, args.steps)
    launches = int(lib.cave_launch_count() - n0)
    clocks = sampler.stop()
    value = B * world / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs({k: v.cpu().numpy() for k, v in last["out"].items() if not k.startswith("_")}, args.dump_outputs)

    # ---- per-kernel timings for the roofline (same stream, CUDA events, same inputs)
    pack = pack_constraints(A)
    # the pack pass alone, through the C ABI into one preallocated buffer (no allocator traffic inside the timed region):
    # flags 0 = scan + plan + order (+ clearing the setup words): what a cold step runs; flags 1 = + the setup kernel
    import ctypes
    nb_pack = ctypes.c_size_t()
    _lib.check(lib.cave_pack_bytes(B, m_max, d, ctypes.byref(nb_pack)))
    pbuf = torch.empty(nb_pack.value, dtype=torch.uint8, device=dev)
    cur_stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def pack_pass(flags):
        _lib.check(lib.cave_pack_ex(ctypes.c_void_p(A.data_ptr()), None, B, m_max, d, flags, ctypes.c_void_p(pbuf.data_ptr()),
                                    nb_pack.value, cur_stream))

    pack_pass(0); pack_pass(1)
    ms_scan = timed(lambda: pack_pass(0), max(3, args.steps // 2))
    ms_pack = timed(lambda: pack_pass(1), max(3, args.steps // 2))
    del pbuf
    warm = lambda: cave_forward_backward(pred, A, -1.0, mode, ratio, "mean", precision=args.precision, pack=pack)  # noqa: E731
    warm()
    ms_solve = timed(warm, max(3, args.steps // 2))
    st = cave_forward_backward(pred, A, -1.0, mode, ratio, "none", precision=args.precision, want_status=True)
    status = st["status"].cpu().numpy()
    iters = st["iters"].cpu().numpy()
    loss_val = float(st["loss_i"].double().mean())
    scan_bytes = float(B) * m_max * d * 4
    solve_bytes = float(sum(gen_rows)) * d * 4 + 2.0 * B * d * 4
    kernels = [
        {"name": "scan_kernel", "ms": ms_scan, "bytes": scan_bytes, "gbs": scan_bytes / ms_scan / 1e6,
         "frac_of_hbm_peak": scan_bytes / ms_scan / 1e6 / hbm_peak},
        {"name": "solve_kernel+finalize", "ms": ms_solve, "bytes": solve_bytes, "gbs": solve_bytes / ms_solve / 1e6,
         "note": "shared-memory / latency bound; WARM pack (cached solver setup: copy-in); a cold step runs the in-solver setup "
                 "instead (step - scan)"},
        {"name": "setup_kernel (reusable packs only, not in the cold step)", "ms": ms_pack - ms_scan},
    ]
    dom = max(kernels[:2], key=lambda k: k["ms"])
    # step-level roofline: algorithmic bytes of the whole path over the whole step, against HBM
    achieved = alg_bytes / ms_step / 1e6
    tr = _traffic_from_profile(args.workload, B)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": tr["bytes_per_step"] if tr else None, "traffic_source": tr, "peak_source": peak_src,
                "dominant_kernel": dom["name"], "algorithmic_bytes_per_step": alg_bytes,
                "note": "achieved = sum_i (4 m_i d + 8 d + 4) bytes / step time; per-kernel split in `kernels`"}
    # the same roofline figure for the device-resident packed dataset (warm pack: no pass over A, cached solver setup);
    # SURVEY 8d: a packed resident layout may exceed 100 % of the dense-input figure; its own traffic is ~1 % of it
    roofline["resident_pack"] = {"ms_per_step": ms_solve, "inst_per_s": B * world / (ms_solve * 1e-3),
                                 "frac_of_dense_input_roofline": alg_bytes / ms_solve / 1e6 / hbm_peak,
                                 "note": "warm / dataset pack (what every epoch after the first runs): latency bound, not HBM bound"}

    # ---- end to end through the module call with host tensors
    e2e = None
    e2e_resident = None
    e2e_sparse = None
    if not args.no_e2e:
        class Model:
            modelSense = EPO.MINIMIZE
        mod = (innerConeAlignedCosine(Model(), solver="cuda", inner_ratio=ratio, seed=0,
                                      solver_kwargs={"precision": args.precision})
               if mode == 1 else exactConeAlignedCosine(Model(), solver="cuda", solver_kwargs={"precision": args.precision}))
        # pinned host copy of the dense constraints, bounded so that N ranks on one box never pin more than
        # ~40 % of the host's free memory between them (the leg is PCIe-bound, so the rate does not depend on Be)
        Be = B
        try:
            import psutil
            budget = 0.4 * psutil.virtual_memory().available / max(world, 1)
            Be = int(max(64, min(B, budget // (m_max * d * 4))))
        except ImportError:
            Be = B if world == 1 else min(B, 1024)
        A_host = torch.empty((Be,) + tuple(A.shape[1:]), dtype=A.dtype, pin_memory=True)
        A_host.copy_(A[:Be])
        pred_host_e = torch.empty((Be, d), dtype=pred.dtype, pin_memory=True)
        pred_host_e.copy_(pred[:Be])
        pred_host = torch.empty(pred.shape, dtype=pred.dtype, pin_memory=True)
        pred_host.copy_(pred)

        def e2e_step():
            p = pred_host_e.requires_grad_(True)
            p.grad = None
            loss = mod(p, A_host)        # H2D of pred_cost and tight_ctrs inside; loss and grad come back to host
            loss.backward()
            return loss.item()

        e2e_step()
        n_e2e = max(2, min(args.steps, 5))
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        barrier()
        dt = (time.perf_counter() - t0) / n_e2e
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": Be * world / dt, "unit": UNIT, "h2d_bytes_per_step": int(A_host.numel() * 4 + pred_host_e.numel() * 4),
               "d2h_bytes_per_step": int(pred_host_e.numel() * 4 + 4), "ms_per_step": dt * 1e3, "steps": n_e2e,
               "batch_per_gpu": Be,
               "note": "module call with pinned host pred_cost and tight_ctrs; PCIe copy of the dense constraints dominates"
                       + ("" if Be == B else f"; batch bounded to {Be}/GPU by host memory")}
        # the same module call with the constraints kept resident on the device (CavePack over the dataset +
        # per-step instance index): what a multi-epoch trainer does, since A_i never changes between epochs
        perm_host = torch.randperm(B, dtype=torch.int32).pin_memory()

        def e2e_resident_step():
            p = pred_host.requires_grad_(True)
            p.grad = None
            loss = mod(p, pack, index=perm_host)       # H2D: pred_cost + index; D2H: loss + gradient
            loss.backward()
            return loss.item()

        e2e_resident_step()
        n_res = max(3, args.steps)
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_res):
            e2e_resident_step()
        barrier()
        dtr = (time.perf_counter() - t0) / n_res
        if world > 1:
            t = torch.tensor([dtr], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtr = float(t.item())
        e2e_resident = {"value": B * world / dtr, "unit": UNIT, "h2d_bytes_per_step": int(pred_host.numel() * 4 + B * 4),
                        "d2h_bytes_per_step": int(pred_host.numel() * 4 + 4), "ms_per_step": dtr * 1e3, "steps": n_res,
                        "note": "device-resident packed dataset (pack built once, outside the timed region) + instance "
                                "index per step; host pred_cost in, host loss and gradient out"}
        del A_host
        # the same module call with the batch's constraints as per-instance CSR in pinned HOST memory (SparseConstraints):
        # what crosses PCIe every step is the non-zeros, not the zero padding of collate_fn
        sc_host = sparse_host[0]

        def e2e_sparse_step():
            p = pred_host.requires_grad_(True)
            p.grad = None
            loss = mod(p, sc_host)                     # H2D: CSR + pred_cost; pack from the non-zeros; D2H: loss + gradient
            loss.backward()
            return loss.item()

        e2e_sparse_step()
        n_sp = max(3, args.steps)
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_sp):
            e2e_sparse_step()
        barrier()
        dts = (time.perf_counter() - t0) / n_sp
        if world > 1:
            t = torch.tensor([dts], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dts = float(t.item())
        e2e_sparse = {"value": B * world / dts, "unit": UNIT, "h2d_bytes_per_step": int(sc_host.nbytes() + pred_host.numel() * 4),
                      "d2h_bytes_per_step": int(pred_host.numel() * 4 + 4), "ms_per_step": dts * 1e3, "steps": n_sp,
                      "note": "module call with pinned host pred_cost and the batch's binding constraints as per-instance CSR "
                              "(SparseConstraints) in pinned host memory: upload, cave_pack_sparse, solve, loss and gradient back to the host"}

    plan_info = pack.launch_plan(args.precision)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64" if args.precision == "fp64" else "f64 state + f32 factor", "data": "synthetic",
        "config": {"workload": f"{args.workload} DFJ synthetic (SURVEY App. B), CaVE+ inner_ratio {ratio}, batch {B}/GPU, "
                               f"pred regime {args.regime}, dense float32 [B,{m_max},{d}] resident in HBM, cold pack",
                   "batch_per_gpu": B, "m_max": m_max, "d": d, "l2_policy": "inputs larger than L2 (A = %.1f GB)" % (scan_bytes / 1e9)},
        "numa_binding": numa, "clocks": clocks, "e2e": e2e, "e2e_sparse_host": e2e_sparse, "e2e_resident_dataset": e2e_resident, "gpu_launches": launches,
        "gpu_launches_note": "kernels launched by libcave_b200.so inside the timed region (cave_launch_count): per step scan, plan, "
                             "order, clear-setup, four solve configurations of which the device selects one, finalize",
        "roofline": roofline, "kernels": kernels, "solve_launch_plan": plan_info,
        "solver": {"status_counts": {str(k): int(v) for k, v in zip(*np.unique(status, return_counts=True))},
                   "iters_mean": float(iters.mean()), "iters_max": int(iters.max()), "loss": loss_val},
    }

    # ---- CPU baseline and parity on the SAME instances as the timed batch (rank 0's first instances)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n = args.cpu_sample or 2 * cores
        work = _cpu_sample(kind, n, mode, ratio, args.regime, seed=seed)
        rate, res = cpu_rate(work)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"the first {n} instances of the timed batch, multiprocessing.Pool({cores}) over "
                                          "oracle.forward_backward (scipy.optimize.nnls + epilogue), BLAS threads = 1"}
        line["parity_sample"] = parity(work, res, st["loss_i"], st["grad"])

    # ---- strong scaling: a fixed global batch split N ways (first instances of every rank's shard)
    if not args.no_extras:
        strong = {}
        for gB in (4096, 65536):
            per = gB // world
            key = f"global_batch_{gB}"
            reps = -(-per // B)
            if per * m_max * d * 4 > 60e9:
                strong[key] = {"value": None, "reason": f"{per} instances/GPU of dense float32 A = {per * m_max * d * 4 / 1e9:.0f} GB do not fit beside the scratch"}
                continue
            if reps > 1:          # more instances than the generated shard: the shard is tiled (distinct memory, same work per instance)
                As, ps = torch.cat([A] * reps)[:per].contiguous(), torch.cat([pred] * reps)[:per].contiguous()
            else:
                As, ps = A[:per].contiguous(), pred[:per].contiguous()
            fn = lambda: cave_forward_backward(ps, As, -1.0, mode, ratio, "mean", precision=args.precision)  # noqa: E731
            fn(); fn()
            ms = timed(fn, max(3, args.steps // 2))
            strong[key] = {"value": per * world / (ms * 1e-3), "unit": UNIT, "batch_per_gpu": per, "ms_per_step": ms,
                           "tiled_from": B if reps > 1 else None}
            del As, ps
            torch.cuda.empty_cache()
        line["strong"] = strong

    # ---- every other named shape at this N (BASELINE.json configs[0], [1], [3], [4])
    if not args.no_extras:
        del A, pred, pack
        torch.cuda.empty_cache()
        wl = {args.workload: {"inst_per_s": value, "ms_per_step": ms_step, "roofline_frac": roofline["frac"],
                              "cpu_baseline": line.get("cpu_baseline", {}).get("value")}}
        for name in ("sp5", "tsp20", "vrp20"):
            if name == args.workload:
                continue
            k2, b2, m2, r2 = WORKLOADS[name]
            info, A2, p2, _, _ = structured(k2, b2, m2, r2, max(5, args.steps), seed)
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                n = 2 * cores
                work = _cpu_sample(k2, n, m2, r2, args.regime, seed=seed)
                rate, res = cpu_rate(work)
                st2 = cave_forward_backward(p2, A2, -1.0, m2, r2, "none", precision=args.precision)
                info["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": f"first {n} instances of this batch"}
                info["parity_sample"] = parity(work, res, st2["loss_i"], st2["grad"])
            wl[name] = info
            del A2, p2
            torch.cuda.empty_cache()
        wl["sweep"] = [sweep_point(d_, m_, b_, 3, rank == 0 and world == 1 and not args.no_cpu_baseline) for d_, m_, b_ in SWEEP_DEFAULT]
        line["workloads"] = wl

    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
