"""
CaVE loss modules with the B200 ``solver='cuda'`` backend.

Host-side mirror of the reference's ``src/cave.py`` for the hot path only: same class names,
constructor arguments, ``forward`` / ``backward`` contract and error behaviour
(``abstractConeAlignedCosine`` src/cave.py:31-81, ``exactConeAlignedCosine`` :84-129,
``innerConeAlignedCosine`` :132-219).  The only solver shipped here is ``'cuda'``; the reference's
CPU backends (``'nnls'``, ``'clarabel'``) and ``'apgd'`` stay in the reference — asking for them
raises instead of silently computing on the CPU.

``forward`` runs the fused kernels (projection + push-inside + cosine + reduction + analytic
backward, one C-ABI call) through a ``torch.autograd.Function``; ``_get_projection`` keeps the
reference's two-step contract (projection, then the target arithmetic in torch) for callers that
use it directly (test/test_func.py:285-292).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._pyepo_compat import EPO, optModule
from .qpsolver import CavePack, SparseConstraints, cave_forward_backward, project_cuda

_REFERENCE_SOLVERS = ("apgd", "clarabel", "nnls")
# constructor-level solver_kwargs: properties of the solver, never of one particular batch (a pack, an index or a row-count
# hint belongs to a call; accepted here they would silently apply to every later batch)
_KERNEL_KWARGS = ("precision", "max_iter", "max_linesearch", "tol", "cap_rows", "cap_nnz", "device", "dense", "dense_slots", "strict",
                  "chunk")


class _CaveCudaFunction(torch.autograd.Function):
    """forward: one fused launch returning the reduced loss and stashing d loss / d pred;
    backward: upstream gradient times the stash (SURVEY.md §8b "fused variant")."""

    @staticmethod
    def forward(ctx, pred_cost, tight_ctrs, sign, mode, inner_ratio, reduction, kwargs):
        if isinstance(tight_ctrs, CavePack):      # device-resident dataset: kwargs carries index= (or the pack is the batch)
            kwargs = dict(kwargs, pack=tight_ctrs)
            tight_ctrs = None
        strict = bool(kwargs.get("strict", False))
        kwargs = {k: v for k, v in kwargs.items() if k != "strict"}
        out = cave_forward_backward(pred_cost, tight_ctrs, sign, mode, inner_ratio, reduction, want_status=strict, **kwargs)
        if strict:      # opt-in (synchronises): scipy's nnls raises at its iteration limit, so does this
            st = out["status"] & 0xff
            bad = (st != _lib.ST_CONVERGED) & (st != _lib.ST_SKIPPED)
            if bool(bad.any()):
                codes, counts = torch.unique(st[bad], return_counts=True)
                raise RuntimeError("solver='cuda': %d of %d instances did not converge (status: count) %s"
                                   % (int(bad.sum()), st.numel(), dict(zip(codes.tolist(), counts.tolist()))))
        grad, loss = out["grad"], out["loss"]
        if grad.device != pred_cost.device:       # host tensors in -> host tensors out
            if pred_cost.device.type == "cpu" and pred_cost.is_pinned():
                # pinned in -> pinned out: one asynchronous copy each on the kernels' stream, one synchronisation
                g_host = torch.empty(grad.shape, dtype=grad.dtype, pin_memory=True)
                l_host = torch.empty(loss.shape, dtype=loss.dtype, pin_memory=True)
                g_host.copy_(grad, non_blocking=True)
                l_host.copy_(loss, non_blocking=True)
                torch.cuda.current_stream(grad.device).synchronize()
                grad, loss = g_host, l_host
            else:
                grad, loss = grad.to(pred_cost.device), loss.to(pred_cost.device)
        ctx.save_for_backward(grad)
        ctx.per_instance = reduction == "none"
        return loss.to(pred_cost.dtype)

    @staticmethod
    def backward(ctx, grad_out):
        (grad,) = ctx.saved_tensors
        if not ctx.per_instance and grad.device.type == "cpu" and grad_out.device.type == "cpu" and float(grad_out) == 1.0:
            return grad, None, None, None, None, None, None       # loss.backward() on host tensors: no 4 B d host multiply
        g = grad_out.unsqueeze(1) * grad if ctx.per_instance else grad_out * grad
        return g.to(grad.dtype), None, None, None, None, None, None


class abstractConeAlignedCosine(optModule):
    """Base of the CaVE cone-aligned cosine losses (src/cave.py:31-81)."""

    def __init__(self, optmodel, processes: int = 1, reduction: str = "mean") -> None:
        super().__init__(optmodel, processes, solve_ratio=1.0, reduction=reduction)

    def _sign(self) -> float:
        # sense-aware sign (src/cave.py:62-68); read at every call
        if self.optmodel.modelSense == EPO.MINIMIZE:
            return -1.0
        if self.optmodel.modelSense == EPO.MAXIMIZE:
            return 1.0
        raise ValueError("Invalid modelSense. Must be EPO.MINIMIZE or EPO.MAXIMIZE.")

    def _kernel_kwargs(self) -> dict:
        return {k: v for k, v in self.solver_kwargs.items() if k in _KERNEL_KWARGS}

    def _mode(self) -> int:
        raise NotImplementedError

    def forward(self, pred_cost: torch.Tensor, tight_ctrs, index: torch.Tensor | None = None,
                pack: CavePack | None = None, m_rows: torch.Tensor | None = None) -> torch.Tensor:
        """``tight_ctrs``: the reference's padded [B, m, d] tensor (src/cave.py:55-57) — or, as an extension,
        a ``CavePack`` built once over the whole dataset together with ``index`` [B] (dataset instance of
        every batch row), which keeps the constraints resident on the device across epochs.  ``pack`` (a warm
        pack of exactly this ``tight_ctrs`` tensor) and ``m_rows`` are per-call arguments."""
        sign = self._sign()
        mode = self._mode()
        kw = self._kernel_kwargs()
        if index is not None:
            kw = dict(kw, index=index)
        if pack is not None:
            kw = dict(kw, pack=pack)
        if m_rows is not None:
            kw = dict(kw, m_rows=m_rows)
        return _CaveCudaFunction.apply(pred_cost, tight_ctrs, sign, mode, getattr(self, "inner_ratio", 0.0),
                                       self.reduction, kw)


class exactConeAlignedCosine(abstractConeAlignedCosine):
    """CaVE Exact (src/cave.py:84-129) with ``solver='cuda'``."""

    def __init__(self, optmodel, solver: str = "cuda", solver_kwargs: dict | None = None,
                 processes: int = 1, reduction: str = "mean") -> None:
        super().__init__(optmodel, processes, reduction)
        if solver not in _REFERENCE_SOLVERS + ("cuda",):
            raise ValueError(f"Invalid solver: {solver}. Must be 'apgd', 'clarabel', 'nnls' or 'cuda'.")
        if solver != "cuda":
            raise ValueError(f"solver='{solver}' is a reference backend (src/cave.py); this package ships only "
                             "solver='cuda' and never falls back to a CPU path.")
        unknown = set(solver_kwargs or {}) - set(_KERNEL_KWARGS)
        if unknown:
            raise ValueError(f"Unknown solver_kwargs for solver='cuda': {sorted(unknown)}")
        self.solver = solver
        self.solver_kwargs = solver_kwargs or {}

    def _mode(self) -> int:
        return _lib.MODE_EXACT

    def _get_projection(self, signed_cost: torch.Tensor, tight_ctrs: torch.Tensor) -> torch.Tensor:
        kw = {k: v for k, v in self._kernel_kwargs().items() if k != "strict"}
        proj, _ = project_cuda(tight_ctrs, signed_cost, **kw)
        return proj / proj.norm(dim=1, keepdim=True).clamp(min=1e-8)       # src/cave.py:129


class innerConeAlignedCosine(exactConeAlignedCosine):
    """CaVE+ / CaVE Hybrid (src/cave.py:132-219) with ``solver='cuda'``, which takes the **nnls**
    branch of the reference: exact projection pushed inside the cone by ``inner_ratio`` unless
    ``rnorm < 1e-7`` (src/cave.py:213-219).  ``max_iter`` is accepted for signature compatibility
    and ignored, exactly as the reference ignores it for ``'nnls'`` (src/cave.py:302)."""

    _INNER_DEFAULTS: dict[str, dict] = {"cuda": {}}   # counterpart of src/cave.py:146-150

    def __init__(self, optmodel, solver: str = "cuda", solver_kwargs: dict | None = None, max_iter: int = 3,
                 solve_ratio: float = 1.0, inner_ratio: float = 0.2, processes: int = 1,
                 reduction: str = "mean", seed: int | None = None) -> None:
        if solver_kwargs is None:
            solver_kwargs = dict(self._INNER_DEFAULTS.get(solver, {}))
        super().__init__(optmodel, solver, solver_kwargs, processes, reduction)
        if not 0 <= solve_ratio <= 1:
            raise ValueError(f"Invalid solve_ratio {solve_ratio}. It should be between 0 and 1.")
        if not 0 <= inner_ratio <= 1:
            raise ValueError(f"Invalid inner_ratio {inner_ratio}. It should be between 0 and 1.")
        self.max_iter = int(max_iter)
        self.solve_ratio = float(solve_ratio)
        self.inner_ratio = float(inner_ratio)
        if seed is not None:
            self._branch_rng = np.random.RandomState(seed)

    def _mode(self) -> int:
        # ONE host draw per forward call, consumed even when solve_ratio == 1 (src/cave.py:201)
        if self._branch_rng.uniform() > self.solve_ratio:
            return _lib.MODE_HEURISTIC
        return _lib.MODE_INNER

    def _get_projection(self, signed_cost: torch.Tensor, tight_ctrs: torch.Tensor) -> torch.Tensor:
        kw = {k: v for k, v in self._kernel_kwargs().items() if k != "strict"}
        mode = self._mode()
        # the target is what the fused kernel aligns against; recover it through the two-step contract
        avg = _average_ctrs(tight_ctrs)
        if mode == _lib.MODE_HEURISTIC:
            pred_norm = signed_cost / signed_cost.norm(dim=1, keepdim=True).clamp(min=1e-8)
            return (1 - self.inner_ratio) * pred_norm + self.inner_ratio * avg
        proj, rnorm = project_cuda(tight_ctrs, signed_cost, **kw)
        proj_norm = proj / proj.norm(dim=1, keepdim=True).clamp(min=1e-8)
        pushed = (1 - self.inner_ratio) * proj_norm + self.inner_ratio * avg.to(proj_norm.device)
        return torch.where((rnorm < 1e-7).unsqueeze(1), proj_norm, pushed)


def _average_ctrs(tight_ctrs: torch.Tensor) -> torch.Tensor:
    """torch restatement of src/cave.py:222-228, used only by ``_get_projection`` above (the fused
    forward takes the average from the scan kernel)."""
    norms = tight_ctrs.norm(dim=2, keepdim=True)
    valid = (norms > 1e-7).to(tight_ctrs.dtype)
    unit = tight_ctrs / norms.clamp(min=1e-8) * valid
    return unit.sum(dim=1) / valid.sum(dim=1).clamp(min=1.0)
