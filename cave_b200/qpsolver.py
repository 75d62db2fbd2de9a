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
import numbers
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
    (``cave_forward_backward_warm_ex``): 8 bytes per general row and instance, which a structured dataset never uses.

    ``gram`` (``cache_gram=True`` at packing) holds G~ = A Aᵀ of every instance the dense path could take, computed once by
    the same tensor-core kernel a call runs (``cave_gram_cache_build``); calls with the pack then skip the TF32 split and the
    Gram kernel and give bit-identical results.  It is constant data, not solver state: ``reset_warm_start()`` keeps it."""
    buf: torch.Tensor
    shape: tuple
    data_ptr: int
    ctrs: torch.Tensor | None = None
    version: int = 0            # tensor._version of tight_ctrs when it was packed (in-place edits invalidate the pack)
    warm: torch.Tensor | None = None    # uint8 warm-start slots, one per packed instance (None: every solve starts from zero)
    warm_dense: torch.Tensor | None = None  # uint8 slots of the dense path (None: dense-path solves start from zero)
    gram: torch.Tensor | None = None    # uint8 Gram cache (None: every call computes G~ of its dense instances)

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
                     cache_setup: bool = True, warm_start: bool = False, warm_dense: bool = False,
                     cache_gram: bool = False) -> CavePack:
    """``warm_start=True``: also keep the solver state across calls (``CavePack.warm``): every structured solve of an
    instance starts from that instance's last converged solution.  ``warm_dense=True`` (with ``warm_start=True``): the
    same for the dense Gram-space path (``CavePack.warm_dense``).  ``cache_gram=True``: compute G~ = A Aᵀ of every
    instance the dense path could take once, here (``CavePack.gram``, m_pad² · 4 bytes per such instance, m_pad = m
    rounded up to 128; ``None`` if there is none); later calls with the pack reuse it."""
    if warm_dense and not warm_start:
        raise ValueError("warm_dense=True needs warm_start=True")
    if cache_gram and not keep_dense:
        raise ValueError("cache_gram=True needs keep_dense=True: the dense path reads the rows of the dataset tensor")
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
    gram = _gram_cache(lib, A, buf) if cache_gram else None
    return CavePack(buf, (B, m, d), A.data_ptr(), A if keep_dense else None, int(tight_ctrs._version), warm, wdense, gram)


def _gram_cache(lib, A: torch.Tensor, pack_buf: torch.Tensor) -> torch.Tensor | None:
    """The Gram cache of a packed dataset (None if no instance can take the dense path).  Reads the number of cached
    instances back once (a synchronisation) to size the buffer."""
    N, m, d = A.shape
    dev = A.device
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        cnt = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(lib.cave_gram_cache_count(_ptr(pack_buf), pack_buf.numel(), N, m, d, _ptr(cnt), stream))
        n_cached = int(cnt.item())
        if n_cached == 0:
            return None
        nb = ctypes.c_size_t()
        _lib.check(lib.cave_gram_cache_bytes(N, n_cached, m, d, ctypes.byref(nb)))
        gram = torch.zeros(nb.value, dtype=torch.uint8, device=dev)
        # one round per SM: the Gram kernel's grid is one CTA per SM, and the scratch stays small
        opts = _opts(dense=True, dense_slots=torch.cuda.get_device_properties(dev).multi_processor_count)
        _lib.check(lib.cave_scratch_bytes(N, m, d, _lib.F64, ctypes.byref(opts), ctypes.byref(nb)))
        scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
        _lib.check(lib.cave_gram_cache_build(_ptr(A), N, m, d, ctypes.byref(opts), _ptr(gram), gram.numel(), _ptr(pack_buf),
                                             pack_buf.numel(), _ptr(scratch), scratch.numel(), stream))
    return gram


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
    """cave_forward_backward, cave_forward_backward_warm(_ex) with the pack's warm-start state when it has one, or
    cave_forward_backward_resident when the pack also has a Gram cache."""
    if pack is not None and pack.gram is not None:
        *head, stream = args
        nwarm = pack.warm.numel() if pack.warm is not None else 0
        ndense = pack.warm_dense.numel() if pack.warm_dense is not None else 0
        _lib.check(lib.cave_forward_backward_resident(*head, _ptr(pack.warm), nwarm, _ptr(pack.warm_dense), ndense,
                                                      _ptr(pack.gram), pack.gram.numel(), stream))
    elif pack is not None and pack.warm_dense is not None:
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
                          tol=None, cap_rows=None, cap_nnz=None, dense="auto", dense_slots=None, chunk=None) -> dict:
    """One call of the hot path through the C ABI.  Returns a dict with ``loss`` (scalar for
    mean/sum, [B] for none), ``loss_i`` [B], ``grad`` [B, d] (= d loss / d pred_cost for an upstream
    gradient of one), and optionally ``proj``, ``rnorm``, ``status``, ``iters`` — all on the
    compute device, in ``pred_cost``'s dtype.

    ``chunk``: solve the batch ``chunk`` rows at a time, copying the next chunk's inputs to the device and the last chunk's
    gradient back while a chunk is solved (``_forward_backward_chunked``).  Device memory then scales with ``chunk``, not
    with the batch.  The results are those of the unchunked call (see there for the one-shot packs); ``None`` or
    ``chunk >= B`` is the unchunked call."""
    if chunk is not None and (isinstance(chunk, bool) or not isinstance(chunk, numbers.Integral) or chunk <= 0):
        raise ValueError(f"chunk must be a positive int or None (got {chunk!r})")
    lib = _lib.load()
    if chunk is not None and 0 < int(chunk) < pred_cost.shape[0]:
        return _forward_backward_chunked(lib, pred_cost, tight_ctrs, sign, mode, inner_ratio, reduction, precision, want_proj,
                                         want_status, pack, index, m_rows, device, int(chunk),
                                         dict(max_iter=max_iter, max_linesearch=max_linesearch, tol=tol, cap_rows=cap_rows,
                                              cap_nnz=cap_nnz, dense=dense, dense_slots=dense_slots))
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


def chunk_bounds(B: int, chunk: int) -> list[tuple[int, int]]:
    """Rows ``[lo, hi)`` of the consecutive chunks of a batch of ``B`` rows (the last one may be shorter)."""
    return [(lo, min(lo + chunk, B)) for lo in range(0, B, chunk)]


class _Ring:
    """Chunks of one host tensor on their way to the device: two device buffers that alternate between chunks, each sized for
    the largest chunk, and for pageable memory two pinned buffers in front of them (a pinned source is copied directly)."""

    def __init__(self, src: torch.Tensor, cap: int, dev: torch.device):
        self.src = src
        shape = (max(cap, 1),) + tuple(src.shape[1:])
        self.dev = [torch.empty(shape, dtype=src.dtype, device=dev) for _ in range(2)]
        self.pin = None if src.is_pinned() else [torch.empty(shape, dtype=src.dtype, pin_memory=True) for _ in range(2)]

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self.dev)

    def put(self, s: int, lo: int, hi: int, copied: torch.cuda.Event) -> torch.Tensor:
        """Enqueues the copy of rows [lo, hi) into set ``s`` on the current (copy) stream; ``copied`` is the event recorded
        after the previous copy out of set ``s`` (the host waits for it before it overwrites the pinned buffer)."""
        n = hi - lo
        src = self.src[lo:hi]
        if self.pin is not None:
            copied.synchronize()
            self.pin[s][:n].copy_(src)
            src = self.pin[s][:n]
        dst = self.dev[s][:n]
        dst.copy_(src, non_blocking=True)
        return dst


def _forward_backward_chunked(lib, pred_cost, ctrs, sign, mode, inner_ratio, reduction, precision, want_proj, want_status,
                              pack, index, m_rows, device, chunk, solver) -> dict:
    """``cave_forward_backward(..., chunk=chunk)`` for ``chunk < B``: the batch as consecutive chunks of ``chunk`` rows
    (``cave_forward_backward_chunk``), then one ``cave_chunk_finalize`` over the whole batch.

    Inputs: a dense ``[B, m, d]`` tensor (a one-shot pack per chunk), ``SparseConstraints`` (a one-shot sparse pack per
    chunk) or a resident pack with ``index`` (or a pack of exactly ``ctrs``: slices of the index and the predictions only).
    Host inputs are copied chunk by chunk on a side stream into two alternating device buffers (through two pinned buffers
    when the host memory is pageable), the kernels of each chunk run on the caller's current stream, and with a host
    ``pred_cost`` the gradient (and projection) of each chunk is copied on a second side stream into pinned host outputs; all
    outputs are then host tensors and the call synchronises.  Device inputs are sliced in place.  Pack and scratch are
    sized for one chunk.

    Every instance is solved on its own, so the per-instance results are the unchunked call's, and the finalize reduces the
    whole batch in the unchunked order.  A one-shot pack (dense or sparse input) selects the solve kernel's launch
    configuration from its own instances, so a chunk can run another configuration than the whole batch: its results then
    agree to rounding only (bit-identical with the configuration fixed, ``CAVE_SOLVE_CFG``).  A warm pack's slots are
    written by a chunk before the next chunk reads them (one stream); an index that holds an instance in two chunks can
    therefore start the second solve from the first one's solution."""
    if reduction not in _lib.REDUCE:
        raise ValueError(f"No reduction '{reduction}'.")
    if precision not in _PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
    sparse = isinstance(ctrs, SparseConstraints)
    resident = pack is not None and not sparse
    B = pred_cost.shape[0]
    if pred_cost.dim() != 2:
        raise ValueError(f"pred_cost must be [B, d], got {tuple(pred_cost.shape)}")
    if resident:
        dev = pack.buf.device
        N, m, d = pack.shape
        if index is None:
            if ctrs is None and N != B:
                raise ValueError("index= is needed unless the pack holds exactly the batch")
            if ctrs is not None and (pack.data_ptr != ctrs.data_ptr() or pack.version != int(ctrs._version)):
                raise ValueError("pack does not belong to this tight_ctrs tensor (other storage, or the tensor was modified "
                                 "in place after pack_constraints)")
            index = torch.arange(B, dtype=torch.int32, device=dev)
        A = ctrs if ctrs is not None else pack.ctrs
        if A is not None and (not A.is_cuda or A.device != dev or tuple(A.shape) != (N, m, d) or A.dtype != torch.float32):
            raise ValueError("the dense dataset tensor must be the float32 CUDA tensor the pack was built from")
        if index.dim() != 1 or index.shape[0] != B:
            raise ValueError(f"shape mismatch: pred_cost {tuple(pred_cost.shape)}, index {tuple(index.shape)}")
        idx = _to_device(index.detach(), dev, torch.int32)
    elif sparse:
        dev = _device_of(ctrs.val, device)
        m, d = int(ctrs.m_max), int(ctrs.d)
        if ctrs.batch != B:
            raise ValueError(f"shape mismatch: pred_cost {tuple(pred_cost.shape)}, SparseConstraints of {ctrs.batch} instances")
    else:
        if ctrs is None:
            raise ValueError("tight_ctrs is None and no pack= was given")
        if ctrs.dim() != 3 or ctrs.shape[0] != B:
            raise ValueError(f"shape mismatch: pred_cost {tuple(pred_cost.shape)}, tight_ctrs {tuple(ctrs.shape)}")
        dev = _device_of(ctrs if ctrs.is_cuda else pred_cost, device)
        _, m, d = ctrs.shape
        ctrs = ctrs.detach()
        if m == 0:      # no rows at all: behave like all-padding (src/cave.py:304-305)
            ctrs, m = torch.zeros((B, 1, d), dtype=torch.float32, device=dev), 1
        ctrs = _to_device(ctrs, dev, torch.float32) if ctrs.is_cuda else ctrs.to(torch.float32).contiguous()
    if pred_cost.shape[1] != d:
        raise ValueError(f"shape mismatch: pred_cost {tuple(pred_cost.shape)}, d = {d}")
    io_dtype = torch.float64 if pred_cost.dtype == torch.float64 else torch.float32
    io_code = _lib.F64 if io_dtype == torch.float64 else _lib.F32
    compute = _PRECISIONS[precision]
    host_out = not pred_cost.is_cuda
    pred = pred_cost.detach()
    pred = _to_device(pred, dev, io_dtype) if pred.is_cuda else pred.to(io_dtype).contiguous()
    mr = _to_device(m_rows, dev, torch.int32) if (m_rows is not None and not resident) else None
    bounds = chunk_bounds(B, chunk)
    cap = max(hi - lo for lo, hi in bounds)
    nb = ctypes.c_size_t()

    with torch.cuda.device(dev):
        cur = torch.cuda.current_stream(dev)
        h2d, d2h = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        rings = {}
        if not pred.is_cuda:
            rings["pred"] = _Ring(pred, cap, dev)
        if sparse:
            sc_dev = ctrs.val.is_cuda
            io_ = ctrs.inst_off.to(dev if sc_dev else "cpu", torch.int64).contiguous()
            rp_ = ctrs.row_ptr.to(dev if sc_dev else "cpu", torch.int64).contiguous()
            col_ = ctrs.col.to(dev if sc_dev else "cpu", torch.int32).contiguous()
            val_ = ctrs.val.to(dev if sc_dev else "cpu", torch.float32).contiguous()
            if not sc_dev:
                rows = [(int(io_[lo]), int(io_[hi])) for lo, hi in bounds]
                nnz = [(int(rp_[r0]), int(rp_[r1])) for r0, r1 in rows]
                rings["inst_off"] = _Ring(io_, cap + 1, dev)
                rings["row_ptr"] = _Ring(rp_, max(r1 - r0 for r0, r1 in rows) + 1, dev)
                rings["col"] = _Ring(col_, max(z1 - z0 for z0, z1 in nnz), dev)
                rings["val"] = _Ring(val_, max(z1 - z0 for z0, z1 in nnz), dev)
            local_idx = torch.arange(cap, dtype=torch.int32, device=dev)
        elif not resident and not ctrs.is_cuda:
            rings["A"] = _Ring(ctrs, cap, dev)

        # one pack and one scratch for the largest chunk, reused by every chunk (they run in order on the current stream)
        opts0 = _opts(**solver)
        _lib.check(lib.cave_scratch_bytes(cap, m, d, compute, ctypes.byref(opts0), ctypes.byref(nb)))
        scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
        if resident:
            pack_buf = pack.buf
        else:
            _lib.check(lib.cave_pack_bytes(cap, m, d, ctypes.byref(nb)))
            pack_buf = torch.empty(nb.value, dtype=torch.uint8, device=dev)
        _lib.check(lib.cave_chunk_acc_bytes(B, ctypes.byref(nb)))
        acc = torch.empty(nb.value, dtype=torch.uint8, device=dev)
        grad = torch.empty((B, d), dtype=io_dtype, device=dev) if not host_out else None
        proj = torch.empty((B, d), dtype=io_dtype, device=dev) if (want_proj and not host_out) else None
        if host_out:        # the chunks' outputs pass through two device buffers into pinned host memory
            grad_h = torch.empty((B, d), dtype=io_dtype, pin_memory=True)
            proj_h = torch.empty((B, d), dtype=io_dtype, pin_memory=True) if want_proj else None
            out_stage = [torch.empty((2, cap, d), dtype=io_dtype, device=dev) for _ in range(2 if want_proj else 1)]
        warm = ndense = gram = None
        if resident:
            warm, ndense, gram = pack.warm, pack.warm_dense, pack.gram
        stream = ctypes.c_void_p(cur.cuda_stream)
        copied = [torch.cuda.Event(), torch.cuda.Event()]       # on h2d: the inputs of the chunk in set s are on the device
        computed = [torch.cuda.Event(), torch.cuda.Event()]     # on cur: the chunk in set s is solved (its inputs are free)
        drained = [torch.cuda.Event(), torch.cuda.Event()]      # on d2h: the outputs of the chunk in set s reached the host
        staged = [None, None]

        def stage(k):
            lo, hi = bounds[k]
            s = k & 1
            got = {}
            with torch.cuda.stream(h2d):
                h2d.wait_event(computed[s])
                for name in ("pred", "A"):
                    if name in rings:
                        got[name] = rings[name].put(s, lo, hi, copied[s])
                if sparse and not sc_dev:
                    (r0, r1), (z0, z1) = rows[k], nnz[k]
                    got["inst_off"] = rings["inst_off"].put(s, lo, hi + 1, copied[s])
                    got["row_ptr"] = rings["row_ptr"].put(s, r0, r1 + 1, copied[s])
                    got["col"] = rings["col"].put(s, z0, z1, copied[s])
                    got["val"] = rings["val"].put(s, z0, z1, copied[s])
                    _lib.check(lib.cave_csr_rebase(_ptr(got["inst_off"]), hi - lo + 1, r0, _ptr(got["row_ptr"]), r1 - r0 + 1,
                                                   z0, ctypes.c_void_p(h2d.cuda_stream)))
                copied[s].record(h2d)
            staged[s] = got

        stage(0)
        for k, (lo, hi) in enumerate(bounds):
            s, n = k & 1, hi - lo
            got = staged[s]
            cur.wait_event(copied[s])
            p_pred = got["pred"] if "pred" in got else pred[lo:hi]
            if host_out:
                cur.wait_event(drained[s])
                g_k = out_stage[0][s][:n]
                p_k = out_stage[1][s][:n] if want_proj else None
            else:
                g_k, p_k = grad[lo:hi], (proj[lo:hi] if want_proj else None)
            if resident:
                A_k = A
                opts = _opts(**solver, warm=True, index=idx[lo:hi], n_packed=N)
            elif sparse:
                if sc_dev:      # absolute offsets into the whole CSR, which is on the device
                    io_k, rp_k, col_k, val_k = io_[lo:], rp_, col_, val_
                else:
                    io_k, rp_k, col_k, val_k = got["inst_off"], got["row_ptr"], got["col"], got["val"]
                _lib.check(lib.cave_pack_sparse(_ptr(io_k), _ptr(rp_k), _ptr(col_k), _ptr(val_k), n, m, d, 0, _ptr(pack_buf),
                                                pack_buf.numel(), stream))
                A_k = None
                opts = _opts(**solver, warm=True, index=local_idx[:n], n_packed=n)
            else:
                A_k = got["A"] if "A" in got else ctrs[lo:hi]
                opts = _opts(**solver)
            _lib.check(lib.cave_forward_backward_chunk(
                _ptr(A_k), _ptr(mr[lo:hi] if mr is not None else None), _ptr(p_pred), n, m, d, float(sign), int(mode),
                float(inner_ratio), _lib.REDUCE[reduction], io_code, compute, ctypes.byref(opts), None, None, _ptr(g_k),
                _ptr(p_k), None, None, None, _ptr(pack_buf), pack_buf.numel(), _ptr(scratch), scratch.numel(),
                _ptr(warm), warm.numel() if warm is not None else 0, _ptr(ndense), ndense.numel() if ndense is not None else 0,
                _ptr(gram), gram.numel() if gram is not None else 0, lo, B, _ptr(acc), acc.numel(), stream))
            computed[s].record(cur)
            if host_out:
                with torch.cuda.stream(d2h):
                    d2h.wait_event(computed[s])
                    grad_h[lo:hi].copy_(g_k, non_blocking=True)
                    if want_proj:
                        proj_h[lo:hi].copy_(p_k, non_blocking=True)
                    drained[s].record(d2h)
            if k + 1 < len(bounds):
                stage(k + 1)        # after the launches of chunk k: a pageable host copy overlaps its solve
        cur.wait_stream(h2d)
        cur.wait_stream(d2h)
        for t in [*(r.dev for r in rings.values())]:
            for b in t:
                b.record_stream(h2d)
        if host_out:
            for t in out_stage:
                t.record_stream(d2h)

        loss = torch.empty((), dtype=io_dtype, device=dev)
        loss_i = torch.empty(B, dtype=io_dtype, device=dev)
        rnorm = torch.empty(B, dtype=io_dtype, device=dev) if (want_proj or want_status) else None
        status = torch.empty(B, dtype=torch.int32, device=dev) if want_status else None
        iters = torch.empty(B, dtype=torch.int32, device=dev) if want_status else None
        _lib.check(lib.cave_chunk_finalize(_ptr(acc), acc.numel(), B, _lib.REDUCE[reduction], io_code, _ptr(loss), _ptr(loss_i),
                                           _ptr(rnorm), _ptr(status), _ptr(iters), stream))
        out = dict(loss=loss_i if reduction == "none" else loss, loss_i=loss_i, grad=grad)
        if want_proj:
            out["proj"], out["rnorm"] = proj, rnorm
        if want_status:
            out["status"], out["iters"], out["rnorm"] = status, iters, rnorm
        if host_out:
            for key, v in out.items():
                if v is not None and key not in ("grad", "proj"):
                    h = torch.empty(v.shape, dtype=v.dtype, pin_memory=True)
                    h.copy_(v, non_blocking=True)
                    out[key] = h
            out["loss"] = out["loss_i"] if reduction == "none" else out["loss"]
            out["grad"] = grad_h
            if want_proj:
                out["proj"] = proj_h
            cur.synchronize()
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
