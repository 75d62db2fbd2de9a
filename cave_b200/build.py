"""Compiles the CUDA sources into cave_b200/_C/libcave_b200.so for sm_100a (in-tree, so the
built library travels to the GPU box with the repo snapshot)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_C")
LIB = os.path.join(OUT_DIR, "libcave_b200.so")
SOURCES = ["scan_kernel.cu", "solve_kernel.cu", "solve_inst_f32_f32.cu", "solve_inst_f32_f64.cu",
           "solve_inst_f64_f32.cu", "solve_inst_f64_f64.cu", "gram_kernel.cu", "dense_solve.cu", "tsp_dp.cu", "chunk.cu", "abi.cu"]
HEADERS = ["ctx.cuh", "layout.cuh", "dense.cuh", "scan_kernel.cuh", "solve_kernel.cuh", "solve_kernel_impl.cuh", "solver_core.cuh",
           os.path.join("..", "..", "include", "cave_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


# dense_solve.cu is compiled as relocatable device code: its heavy phases are non-inlined functions, and only with the strict
# call ABI of -rdc does ptxas give every callee the full register budget (saving the caller's live registers at the call);
# without it the callees are cloned per kernel and squeezed into what the call site leaves free, which splits their load batches.
PER_FILE_FLAGS = {"dense_solve.cu": ["-rdc=true", "-maxrregcount=128"]}     # (512-thread kernel: 128 registers per thread, callees included)


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; cannot build the CUDA library")
    return nvcc


def is_fresh() -> bool:
    if not os.path.exists(LIB):
        return False
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return all(os.path.getmtime(p) <= t for p in deps)


def build(force: bool = False, verbose: bool = False, alt_name: str | None = None) -> str:
    """alt_name: write an alternative build (with CAVE_NVCC_EXTRA flags) next to the product library instead of replacing it."""
    if alt_name is None and not force and is_fresh():
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    objs, logs = [], []
    procs = []
    for s in SOURCES:
        obj = os.path.join(OUT_DIR, s.replace(".cu", ".o") if alt_name is None else s.replace(".cu", ".alt.o"))
        cmd = [_nvcc(), *NVCC_FLAGS, *PER_FILE_FLAGS.get(s, []), *os.environ.get("CAVE_NVCC_EXTRA", "").split(),
               "-c", os.path.join(CSRC, s), "-o", obj]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for s, pr in procs:
        out, _ = pr.communicate()
        logs.append(f"== {s}\n{out}")
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{out}")
    if alt_name is None:
        with open(os.path.join(OUT_DIR, "ptxas.log"), "w") as f:
            f.write("\n".join(logs))
    if verbose:
        print("\n".join(logs))
    target = LIB if alt_name is None else os.path.join(OUT_DIR, alt_name)
    subprocess.check_call([_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", target, *objs,
                           "-lcudart_static", "-lpthread", "-ldl", "-lrt"])
    return target


if __name__ == "__main__":
    import sys
    alt = [a for a in sys.argv[1:] if a.endswith(".so")]
    print(build(force=True, verbose="-v" in sys.argv, alt_name=alt[0] if alt else None))
