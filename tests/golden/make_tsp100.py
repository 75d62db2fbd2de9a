"""
Generates tests/golden/tsp100/tsp100_coo.npz: two TSP-100 instances (d = 4950, m ~ 5150) with the CPU oracle's results
(oracle.cave_oracle.forward_backward, fp64=True, i.e. scipy's nnls in float64: the arithmetic the reference calls).

    python tests/golden/make_tsp100.py

One nnls solve at this size takes one to two minutes of one CPU core; the eight solves (2 instances x 2 prediction
regimes x exact / inner mode) run in parallel processes.  The tests replay the stored results and never run scipy at
this size.  A dense TSP-100 instance is 102 MB, so the rows are stored as COO:

    d, m[2], off[3]                 instance b owns COO entries [off[b], off[b + 1])
    rows, cols (int32), vals (f32)  rows in the reference's order (cave_b200.synth)
    pred_<regime>      f32 [2, d]   regime in (uniform, near): cave_b200.synth.predictions(insts, 0, regime)
    proj_<regime>, rnorm_<regime>   f64 projection of -pred (minimisation) and ||proj + pred||_2
    loss_<mode>_<regime>, grad_<mode>_<regime>   f64 per-instance loss ([2]) and d loss_i / d pred ([2, d]), reduction
                                    'none', mode in (exact, inner); inner mode with inner_ratio = 0.2
"""
import os
import sys
from multiprocessing import Pool

for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ.setdefault(_v, "1")

import numpy as np  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from cave_b200 import synth  # noqa: E402
from oracle import cave_oracle as O  # noqa: E402

SEED, BATCH, INNER_RATIO = 0, 2, 0.2
MODES = {"exact": O.MODE_EXACT, "inner": O.MODE_INNER}
REGIMES = ("uniform", "near")


def _job(args):
    b, regime, mode = args
    insts = synth.make_batch("tsp100", BATCH, SEED)
    pred = synth.predictions(insts, SEED, regime)[b:b + 1]
    ctrs = insts[b].dense()[None]
    ref = O.forward_backward(pred, ctrs, minimize=True, mode=MODES[mode], inner_ratio=INNER_RATIO, reduction="none",
                             fp64=True)
    print(f"instance {b} {regime:7s} {mode}: loss {float(ref['loss_i'][0]):.6f} rnorm {float(ref['rnorm'][0]):.4e}",
          flush=True)
    return args, ref


def main():
    insts = synth.make_batch("tsp100", BATCH, SEED)
    jobs = [(b, r, m) for b in range(BATCH) for r in REGIMES for m in MODES]
    with Pool(len(jobs)) as pool:
        res = dict(pool.map(_job, jobs))
    out = dict(d=np.int32(insts[0].d), m=np.asarray([i.m for i in insts], np.int32),
               off=np.cumsum([0] + [len(i.vals) for i in insts]).astype(np.int64),
               rows=np.concatenate([i.rows for i in insts]).astype(np.int32),
               cols=np.concatenate([i.cols for i in insts]).astype(np.int32),
               vals=np.concatenate([i.vals for i in insts]).astype(np.float32),
               inner_ratio=np.float64(INNER_RATIO), seed=np.int32(SEED))
    for r in REGIMES:
        out[f"pred_{r}"] = synth.predictions(insts, SEED, r)
        # the projection does not depend on the mode: stored once, from the exact-mode run
        out[f"proj_{r}"] = np.concatenate([res[(b, r, "exact")]["proj"] for b in range(BATCH)]).astype(np.float64)
        out[f"rnorm_{r}"] = np.concatenate([res[(b, r, "exact")]["rnorm"] for b in range(BATCH)]).astype(np.float64)
        for m in MODES:
            out[f"loss_{m}_{r}"] = np.concatenate([res[(b, r, m)]["loss_i"] for b in range(BATCH)]).astype(np.float64)
            out[f"grad_{m}_{r}"] = np.concatenate([res[(b, r, m)]["grad"] for b in range(BATCH)]).astype(np.float64)
            assert np.array_equal(res[(0, r, m)]["proj"], res[(0, r, "exact")]["proj"])
    # in a subdirectory: the top-level *.npz of tests/golden are replayed through the dense oracle by other tests
    os.makedirs(os.path.join(HERE, "tsp100"), exist_ok=True)
    path = os.path.join(HERE, "tsp100", "tsp100_coo.npz")
    np.savez_compressed(path, **out)
    print(f"{path}: {os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
