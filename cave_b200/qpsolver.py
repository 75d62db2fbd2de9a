"""
``solver='cuda'`` backend for the CaVE cone projection — the counterpart of the reference's
``src/qpsolver.py`` (which holds ``project_apgd``, src/qpsolver.py:11-63).

``project_cuda`` has the calling convention of ``project_apgd`` and plugs into the batched early
return of ``_batch_project`` (src/cave.py:242-244); unlike ``project_apgd`` its ``rnorm`` has the
**nnls meaning** ``||proj - c||_2`` (src/cave.py:307), which is what the inner push-inside test
``rnorm < 1e-7`` (src/cave.py:218) consumes.  ``cave_forward_backward`` is the fused variant
(projection + target + loss + analytic backward in one pass).

Host code here is plumbing only (argument checks, buffers, stream); all arithmetic runs in the
hand-written sm_100a kernels behind the C ABI of include/cave_b200.h.  No CPU fallback.
"""
from __future__ import annotations

import ctypes
import os
from dataclasses import dataclass

import torch

from . import _lib

_PRECISIONS = {"fp64": _lib.F64, "float64": _lib.F64, "double": _lib.F64,
               "fp32": _lib.F32, "float32": _lib.F32, "single": _lib.F32}


_DENSE = {"auto": 0, None: 0, True: 1, False: -1, "on": 1, "off": -1}


def _opts(max_iter=None, max_linesearch=None, tol=None, cap_rows=None, cap_nnz=None, warm=False,
          index=None, n_packed=0, dense="auto", dense_slots=None) -> _lib.SolverOpts:
    if dense not in _DENSE:
        raise ValueError("dense must be 'auto', True or False")
    return _lib.SolverOpts(int(max_iter or 0), int(max_linesearch or 0), float(tol or 0.0),
                           int(cap_rows or 0), int(cap_nnz or 0), int(bool(warm)), _DENSE[dense],
                           index.data_ptr() if index is not None else None, int(n_packed), int(dense_slots or 0))


def _device_of(t: torch.Tensor, device) -> torch.device:
    if device is not None:
        return torch.device(device)
    if t.is_cuda:
        return t.device
    if not torch.cuda.is_available():
        raise _lib.CaveLibraryError("solver='cuda' needs a CUDA device; there is no CPU fallback "
                                    "(use the reference's solver='nnls' on the CPU)")
    return torch.device("cuda", torch.cuda.current_device())


def _to_device(t: torch.Tensor, dev: torch.device, dtype=None) -> torch.Tensor:
    if t.device != dev:
        t = t.to(dev, non_blocking=True)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


@dataclass
class CavePack:
    """Device-resident packed description of a ``tight_ctrs`` tensor (row classes, singleton cone types,
    average normal, packed CSR of the general rows).  A_i is constant across epochs (SURVEY.md §7.2):

    * per batch: ``pack=pack_constraints(bctr)`` skips the streaming pass over A on later calls with the
      same batch tensor;
    * per dataset: pack ALL instances once (``pack_constraints(all_ctrs)``) and pass ``pack=..., index=idx``
      with ``idx[b]`` = dataset instance of batch row ``b`` — the device-resident replacement of
      DataLoader + ``collate_fn`` (src/dataset.py:133-144).  ``ctrs`` keeps the dense dataset tensor
      resident for instances whose general rows did not fit the packed CSR (``keep_dense=False`` drops it).

    ``warm`` (``warm_start=True`` at packing) is the solver state kept across calls: the multipliers of every instance's last
    converged structured solve, from which the next call on that instance starts (``cave_forward_backward_warm`` in
    include/cave_b200.h).  It changes where the Newton iteration starts, never what it converges to.  Calls that use one
    pack must run on one stream, in the order they are made; ``reset_warm_start()`` empties the state.

    ``warm_dense`` (``warm_dense=True`` as well) does the same for instances solved by the dense Gram-space Newton path
    (``cave_forward_backward_warm_ex``): 8 bytes per general row and instance, which a structured dataset never uses."""
    buf: torch.Tensor
    shape: tuple
    data_ptr: int
    ctrs: torch.Tensor | None = None
    version: int = 0            # tensor._version of tight_ctrs when it was packed (in-place edits invalidate the pack)
    warm: torch.Tensor | None = None    # uint8 warm-start slots, one per packed instance (None: every solve starts from zero)
    warm_dense: torch.Tensor | None = None  # uint8 slots of the dense path (None: dense-path solves start from zero)

    def reset_warm_start(self) -> None:
        """Forget the stored solutions (e.g. after re-initialising the predictor): the next calls start from zero."""
        for buf in (self.warm, self.warm_dense):
            if buf is not None:
                buf.zero_()

    def launch_plan(self, precision: str = "fp64", io_dtype: torch.dtype = torch.float32) -> dict:
        """Diagnostics (synchronises): the solve-kernel configuration the pack's statistics select on the device."""
        lib = _lib.load()
        B, m, d = self.shape
        off = ctypes.c_size_t()
        _lib.check(lib.cave_plan_offset(B, m, d, ctypes.byref(off)))
        words = self.buf[off.value:off.value + 64].cpu().view(torch.int64).tolist()
        arr = (ctypes.c_uint64 * 8)(*[w & 0xFFFFFFFFFFFFFFFF for w in words])
        t, c, sm = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        idx = lib.cave_plan_choice(arr, d, _lib.F64 if io_dtype == torch.float64 else _lib.F32,
                                   _lib.F32 if precision == "fp32" else _lib.F64, ctypes.byref(t), ctypes.byref(c), ctypes.byref(sm))
        n = max(words[0], 1)
        return {"config": idx, "threads": t.value, "ctas_per_sm": c.value, "smem_bytes": sm.value,
                "avg_work_bytes_f64": words[1] / n, "avg_work_bytes_f32": words[2] / n,
                "max_hot_bytes_f64": words[3], "max_hot_bytes_f32": words[4]}


def _warm_buffer(sizer, B: int, m: int, d: int, device) -> torch.Tensor:
    nbytes = ctypes.c_size_t()
    _lib.check(sizer(B, m, d, ctypes.byref(nbytes)))
    return torch.zeros(nbytes.value, dtype=torch.uint8, device=device)


def pack_constraints(tight_ctrs: torch.Tensor, m_rows: torch.Tensor | None = None, keep_dense: bool = True,
                     cache_setup: bool = True, warm_start: bool = False, warm_dense: bool = False) -> CavePack:
    """``warm_start=True``: also keep the solver state across calls (``CavePack.warm``): every structured solve of an
    instance starts from that instance's last converged solution.  ``warm_dense=True`` (with ``warm_start=True``): the
    same for the dense Gram-space path (``CavePack.warm_dense``)."""
    if warm_dense and not warm_start:
        raise ValueError("warm_dense=True needs warm_start=True")
    lib = _lib.load()
    if not tight_ctrs.is_cuda:
        raise ValueError("pack_constraints expects a CUDA tensor")
    A = tight_ctrs.detach()
    if A.dtype != torch.float32 or not A.is_contiguous():
        raise ValueError("tight_ctrs must be contiguous float32 [B, m, d] (the collate_fn layout)")
    B, m, d = A.shape
    nbytes = ctypes.c_size_t()
    _lib.check(lib.cave_pack_bytes(B, m, d, ctypes.byref(nbytes)))
    buf = torch.empty(nbytes.value, dtype=torch.uint8, device=A.device)
    with torch.cuda.device(A.device):
        stream = torch.cuda.current_stream(A.device).cuda_stream
        _lib.check(lib.cave_pack_ex(_ptr(A), _ptr(m_rows), B, m, d, 1 if cache_setup else 0, _ptr(buf), nbytes.value,
                                    ctypes.c_void_p(stream)))
    warm = _warm_buffer(lib.cave_warm_bytes, B, m, d, A.device) if warm_start else None
    wdense = _warm_buffer(lib.cave_dense_warm_bytes, B, m, d, A.device) if warm_dense else None
    return CavePack(buf, (B, m, d), A.data_ptr(), A if keep_dense else None, int(tight_ctrs._version), warm, wdense)


@dataclass
class SparseConstraints:
    """Binding-constraint rows of a batch / dataset as per-instance CSR (host or device tensors):
    rows ``[inst_off[b], inst_off[b+1])`` of ``row_ptr`` belong to instance ``b`` (the reference's row order,
    src/dataset.py:178-211), row ``r`` holds ``col/val[row_ptr[r]:row_ptr[r+1]]`` with ascending columns.
    The sparse counterpart of the padded ``[B, m_max, d]`` tensor of ``collate_fn`` (src/dataset.py:133-144): about
    90 KB instead of 6.5 MB per TSP-50 instance."""
    inst_off: torch.Tensor      # int64 [B + 1]
    row_ptr: torch.Tensor       # int64 [R + 1]
    col: torch.Tensor           # int32 [nnz]
    val: torch.Tensor           # float32 [nnz]
    m_max: int
    d: int

    @property
    def batch(self) -> int:
        return int(self.inst_off.numel() - 1)

    def nbytes(self) -> int:
        return int(sum(t.numel() * t.element_size() for t in (self.inst_off, self.row_ptr, self.col, self.val)))

    @staticmethod
    def from_dense(tight_ctrs: torch.Tensor) -> "SparseConstraints":
        """Host-side conversion of a padded dense ``[B, m, d]`` tensor (all-zero rows are padding and are dropped)."""
        import numpy as np
        A = tight_ctrs.detach().cpu().numpy()
        B, m, d = A.shape
        inst_off, row_ptr, cols, vals = [0], [0], [], []
        for b in range(B):
            keep = np.flatnonzero(np.abs(A[b]).sum(axis=1) > 0)
            for r in keep:
                k = np.flatnonzero(A[b, r])
                cols.append(k.astype(np.int32)); vals.append(A[b, r, k].astype(np.float32))
                row_ptr.append(row_ptr[-1] + len(k))
            inst_off.append(inst_off[-1] + len(keep))
        return SparseConstraints(torch.tensor(inst_off, dtype=torch.int64), torch.tensor(row_ptr, dtype=torch.int64),
                                 torch.from_numpy(np.concatenate(cols) if cols else np.zeros(0, np.int32)),
                                 torch.from_numpy(np.concatenate(vals) if vals else np.zeros(0, np.float32)), m, d)

    @staticmethod
    def from_instances(insts, m_max: int | None = None) -> "SparseConstraints":
        """From ``cave_b200.synth.SparseInstance`` objects (COO, rows in the reference's order)."""
        import numpy as np
        d = insts[0].d
        m_max = max(i.m for i in insts) if m_max is None else m_max
        inst_off = np.zeros(len(insts) + 1, np.int64)
        ptrs, cols, vals = [np.zeros(1, np.int64)], [], []
        base = 0
        for b, it in enumerate(insts):
            order = np.lexsort((it.cols, it.rows))
            cnt = np.bincount(it.rows, minlength=it.m).astype(np.int64)
            ptrs.append(base + np.cumsum(cnt)); base += int(cnt.sum())
            cols.append(it.cols[order].astype(np.int32)); vals.append(it.vals[order].astype(np.float32))
            inst_off[b + 1] = inst_off[b] + it.m
        return SparseConstraints(torch.from_numpy(inst_off), torch.from_numpy(np.concatenate(ptrs)),
                                 torch.from_numpy(np.concatenate(cols)), torch.from_numpy(np.concatenate(vals)), int(m_max), int(d))

    def pin_memory(self) -> "SparseConstraints":
        return SparseConstraints(self.inst_off.pin_memory(), self.row_ptr.pin_memory(), self.col.pin_memory(), self.val.pin_memory(),
                                 self.m_max, self.d)


def pack_constraints_sparse(sc: SparseConstraints, device=None, cache_setup: bool = True,
                            warm_start: bool = False) -> CavePack:
    """Builds the device-resident pack straight from per-instance CSR (``cave_pack_sparse``): no dense tensor exists on
    the device, so instances that would need it (no singleton row at all, or general rows beyond the packed-CSR
    capacity) report ``CAVE_ST_NOSPACE``.  Host tensors are uploaded on the current stream (pinned -> asynchronous).
    ``warm_start``: as for ``pack_constraints``."""
    lib = _lib.load()
    dev = _device_of(sc.val, device)
    B, m, d = sc.batch, int(sc.m_max), int(sc.d)
    io = _to_device(sc.inst_off, dev, torch.int64)
    rp = _to_device(sc.row_ptr, dev, torch.int64)
    col = _to_device(sc.col, dev, torch.int32)
    val = _to_device(sc.val, dev, torch.float32)
    nbytes = ctypes.c_size_t()
    _lib.check(lib.cave_pack_bytes(B, m, d, ctypes.byref(nbytes)))
    buf = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(lib.cave_pack_sparse(_ptr(io), _ptr(rp), _ptr(col), _ptr(val), B, m, d, 1 if cache_setup else 0,
                                        _ptr(buf), nbytes.value, ctypes.c_void_p(stream)))
    warm = _warm_buffer(lib.cave_warm_bytes, B, m, d, dev) if warm_start else None
    return CavePack(buf, (B, m, d), 0, None, 0, warm)


def _call_forward_backward(lib, pack: CavePack | None, *args) -> None:
    """cave_forward_backward, or cave_forward_backward_warm(_ex) with the pack's warm-start state when it has one."""
    if pack is not None and pack.warm_dense is not None:
        *head, stream = args
        nwarm = pack.warm.numel() if pack.warm is not None else 0
        _lib.check(lib.cave_forward_backward_warm_ex(*head, _ptr(pack.warm), nwarm, _ptr(pack.warm_dense),
                                                     pack.warm_dense.numel(), stream))
    elif pack is not None and pack.warm is not None:
        *head, stream = args
        _lib.check(lib.cave_forward_backward_warm(*head, _ptr(pack.warm), pack.warm.numel(), stream))
    else:
        _lib.check(lib.cave_forward_backward(*args))


def cave_forward_backward(pred_cost: torch.Tensor, tight_ctrs: torch.Tensor, sign: float, mode: int,
                          inner_ratio: float = 0.2, reduction: str = "mean", precision: str = "fp64",
                          want_proj: bool = False, want_status: bool = False, pack: CavePack | None = None,
                          index: torch.Tensor | None = None,
                          m_rows: torch.Tensor | None = None, device=None, max_iter=None, max_linesearch=None,
                          tol=None, cap_rows=None, cap_nnz=None, dense="auto", dense_slots=None) -> dict:
    """One call of the hot path through the C ABI.  Returns a dict with ``loss`` (scalar for
    mean/sum, [B] for none), ``loss_i`` [B], ``grad`` [B, d] (= d loss / d pred_cost for an upstream
    gradient of one), and optionally ``proj``, ``rnorm``, ``status``, ``iters`` — all on the
    compute device, in ``pred_cost``'s dtype."""
    lib = _lib.load()
    if isinstance(tight_ctrs, SparseConstraints):      # one-shot sparse batch: pack from the non-zeros, then the indexed path
        pack = pack_constraints_sparse(tight_ctrs, device=device, cache_setup=False)
        tight_ctrs = None
    if index is None and tight_ctrs is None and pack is not None and pack.shape[0] == pred_cost.shape[0]:
        index = torch.arange(pred_cost.shape[0], dtype=torch.int32, device=pack.buf.device)     # the pack IS the batch
    if index is not None:
        return _forward_backward_indexed(lib, pred_cost, tight_ctrs, sign, mode, inner_ratio, reduction, precision,
                                         want_proj, want_status, pack, index, device, max_iter, max_linesearch, tol,
                                         cap_rows, cap_nnz, dense, dense_slots)
    if pred_cost.dim() != 2 or tight_ctrs.dim() != 3 or tight_ctrs.shape[0] != pred_cost.shape[0] \
            or tight_ctrs.shape[2] != pred_cost.shape[1]:
        raise ValueError(f"shape mismatch: pred_cost {tuple(pred_cost.shape)}, tight_ctrs {tuple(tight_ctrs.shape)}")
    if reduction not in _lib.REDUCE:
        raise ValueError(f"No reduction '{reduction}'.")
    if precision not in _PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
    dev = _device_of(tight_ctrs if tight_ctrs.is_cuda else pred_cost, device)
    io_dtype = torch.float64 if pred_cost.dtype == torch.float64 else torch.float32
    pred = _to_device(pred_cost.detach(), dev, io_dtype)
    A = _to_device(tight_ctrs.detach(), dev, torch.float32)
    B, m, d = A.shape
    if B == 0:
        z = torch.zeros((), dtype=io_dtype, device=dev)
        return dict(loss=z if reduction != "none" else torch.zeros(0, dtype=io_dtype, device=dev),
                    loss_i=torch.zeros(0, dtype=io_dtype, device=dev), grad=torch.zeros_like(pred))
    if m == 0:      # no rows at all: behave like all-padding (src/cave.py:304-305)
        A = torch.zeros((B, 1, d), dtype=torch.float32, device=dev)
        m = 1
    compute = _PRECISIONS[precision]
    opts = _opts(max_iter, max_linesearch, tol, cap_rows, cap_nnz, warm=pack is not None, dense=dense, dense_slots=dense_slots)
    nb = ctypes.c_size_t()
    if pack is not None:
        # a pack describes ONE tensor: same storage, not modified since (a same-shape batch of other instances would be
        # projected onto the wrong cones without any error otherwise)
        if pack.shape != (B, m, d) or pack.buf.device != dev or pack.data_ptr != A.data_ptr() \
                or pack.version != int(tight_ctrs._version):
            raise ValueError("pack does not belong to this tight_ctrs tensor (other storage, shape or device, or the "
                             "tensor was modified in place after pack_constraints); for batches drawn from a dataset "
                             "pack the whole dataset once and pass index=")
        pack_buf = pack.buf
    else:
        _lib.check(lib.cave_pack_bytes(B, m, d, ctypes.byref(nb)))
        pack_buf = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    _lib.check(lib.cave_scratch_bytes(B, m, d, compute, ctypes.byref(opts), ctypes.byref(nb)))
    scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    loss = torch.empty((), dtype=io_dtype, device=dev)
    loss_i = torch.empty(B, dtype=io_dtype, device=dev)
    grad = torch.empty((B, d), dtype=io_dtype, device=dev)
    proj = torch.empty((B, d), dtype=io_dtype, device=dev) if want_proj else None
    rnorm = torch.empty(B, dtype=io_dtype, device=dev) if (want_proj or want_status) else None
    status = torch.empty(B, dtype=torch.int32, device=dev) if want_status else None
    iters = torch.empty(B, dtype=torch.int32, device=dev) if want_status else None
    if m_rows is not None:
        m_rows = _to_device(m_rows, dev, torch.int32)
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        _call_forward_backward(
            lib, pack, _ptr(A), _ptr(m_rows), _ptr(pred), B, m, d, float(sign), int(mode), float(inner_ratio),
            _lib.REDUCE[reduction], _lib.F64 if io_dtype == torch.float64 else _lib.F32, compute,
            ctypes.byref(opts), _ptr(loss), _ptr(loss_i), _ptr(grad), _ptr(proj), _ptr(rnorm), _ptr(status),
            _ptr(iters), _ptr(pack_buf), pack_buf.numel(), _ptr(scratch), scratch.numel(), ctypes.c_void_p(stream))
    out = dict(loss=loss_i if reduction == "none" else loss, loss_i=loss_i, grad=grad)
    if want_proj:
        out["proj"], out["rnorm"] = proj, rnorm
    if want_status:
        out["status"], out["iters"], out["rnorm"] = status, iters, rnorm
    if os.environ.get("CAVE_KEEP_SCRATCH"):       # diagnostics (tools/dense_profile.py reads the dense control block)
        out["_scratch"], out["_opts"] = scratch, opts
    return out


def _forward_backward_indexed(lib, pred_cost, ctrs, sign, mode, inner_ratio, reduction, precision, want_proj,
                              want_status, pack, index, device, max_iter, max_linesearch, tol, cap_rows, cap_nnz,
                              dense="auto", dense_slots=None) -> dict:
    """Batch = rows ``index`` of a dataset whose constraints were packed once (device-resident dataset)."""
    if pack is None:
        raise ValueError("index= needs pack= (pack_constraints over the whole dataset)")
    if reduction not in _lib.REDUCE:
        raise ValueError(f"No reduction '{reduction}'.")
    if precision not in _PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
    dev = pack.buf.device
    N, m, d = pack.shape
    if pred_cost.dim() != 2 or pred_cost.shape[1] != d or index.dim() != 1 or index.shape[0] != pred_cost.shape[0]:
        raise ValueError(f"shape mismatch: pred_cost {tuple(pred_cost.shape)}, index {tuple(index.shape)}, pack {pack.shape}")
    io_dtype = torch.float64 if pred_cost.dtype == torch.float64 else torch.float32
    pred = _to_device(pred_cost.detach(), dev, io_dtype)
    idx = _to_device(index.detach(), dev, torch.int32)
    A = ctrs if ctrs is not None else pack.ctrs
    if A is not None and (not A.is_cuda or A.device != dev or tuple(A.shape) != (N, m, d) or A.dtype != torch.float32):
        raise ValueError("the dense dataset tensor must be the float32 CUDA tensor the pack was built from")
    B = pred.shape[0]
    compute = _PRECISIONS[precision]
    opts = _opts(max_iter, max_linesearch, tol, cap_rows, cap_nnz, warm=True, index=idx, n_packed=N, dense=dense,
                 dense_slots=dense_slots)
    nb = ctypes.c_size_t()
    _lib.check(lib.cave_scratch_bytes(B, m, d, compute, ctypes.byref(opts), ctypes.byref(nb)))
    scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    loss = torch.empty((), dtype=io_dtype, device=dev)
    loss_i = torch.empty(B, dtype=io_dtype, device=dev)
    grad = torch.empty((B, d), dtype=io_dtype, device=dev)
    proj = torch.empty((B, d), dtype=io_dtype, device=dev) if want_proj else None
    rnorm = torch.empty(B, dtype=io_dtype, device=dev) if (want_proj or want_status) else None
    status = torch.empty(B, dtype=torch.int32, device=dev) if want_status else None
    iters = torch.empty(B, dtype=torch.int32, device=dev) if want_status else None
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        _call_forward_backward(
            lib, pack, _ptr(A), None, _ptr(pred), B, m, d, float(sign), int(mode), float(inner_ratio),
            _lib.REDUCE[reduction], _lib.F64 if io_dtype == torch.float64 else _lib.F32, compute,
            ctypes.byref(opts), _ptr(loss), _ptr(loss_i), _ptr(grad), _ptr(proj), _ptr(rnorm), _ptr(status),
            _ptr(iters), _ptr(pack.buf), pack.buf.numel(), _ptr(scratch), scratch.numel(), ctypes.c_void_p(stream))
    out = dict(loss=loss_i if reduction == "none" else loss, loss_i=loss_i, grad=grad)
    if want_proj:
        out["proj"], out["rnorm"] = proj, rnorm
    if want_status:
        out["status"], out["iters"], out["rnorm"] = status, iters, rnorm
    return out


def dense_gram(tight_ctrs: torch.Tensor, dense_slots=None) -> tuple[torch.Tensor, int]:
    """Diagnostic: G~ = A A^T of every (dense) instance from the tensor-core Gram kernel alone (``cave_dense_gram``):
    returns ``(G [B, m_pad, m_pad] float32, number of instances the device classified as dense)``."""
    lib = _lib.load()
    A = tight_ctrs.detach()
    if not A.is_cuda or A.dtype != torch.float32 or not A.is_contiguous() or A.dim() != 3:
        raise ValueError("tight_ctrs must be a contiguous float32 CUDA tensor [B, m, d]")
    B, m, d = A.shape
    opts = _opts(dense=True, dense_slots=dense_slots or B)
    nb = ctypes.c_size_t()
    _lib.check(lib.cave_pack_bytes(B, m, d, ctypes.byref(nb)))
    pack_buf = torch.empty(nb.value, dtype=torch.uint8, device=A.device)
    _lib.check(lib.cave_scratch_bytes(B, m, d, _lib.F64, ctypes.byref(opts), ctypes.byref(nb)))
    scratch = torch.empty(nb.value, dtype=torch.uint8, device=A.device)
    m_pad = (m + 127) // 128 * 128
    G = torch.zeros((B, m_pad, m_pad), dtype=torch.float32, device=A.device)
    cnt = torch.zeros(1, dtype=torch.int32, device=A.device)
    with torch.cuda.device(A.device):
        stream = torch.cuda.current_stream(A.device).cuda_stream
        _lib.check(lib.cave_dense_gram(_ptr(A), B, m, d, ctypes.byref(opts), _ptr(G), _ptr(cnt), _ptr(pack_buf), pack_buf.numel(),
                                       _ptr(scratch), scratch.numel(), ctypes.c_void_p(stream)))
    return G, int(cnt.item())


def project_cuda(tight_ctrs: torch.Tensor, signed_cost: torch.Tensor, precision: str = "fp64",
                 **solver_kwargs) -> tuple[torch.Tensor, torch.Tensor]:
    """Batched projection of ``signed_cost`` onto cone{lam @ tight_ctrs[i] : lam >= 0}.

    Drop-in for the batched branch of ``_batch_project`` (src/cave.py:242-244): returns
    ``(proj [B, d], rnorm [B])`` on ``signed_cost``'s device and dtype (src/cave.py:240, 262-263),
    ``rnorm = ||proj - c||_2`` as for ``_project_nnls`` (src/cave.py:307)."""
    out = cave_forward_backward(signed_cost, tight_ctrs, sign=1.0, mode=_lib.MODE_EXACT, reduction="none",
                                precision=precision, want_proj=True, **solver_kwargs)
    proj, rnorm = out["proj"], out["rnorm"]
    if proj.device != signed_cost.device:
        proj, rnorm = proj.to(signed_cost.device), rnorm.to(signed_cost.device)
    return proj.to(signed_cost.dtype), rnorm.to(signed_cost.dtype)
