"""Splatfacto's bilateral grid (nerfstudio `lib_bilagrid`, `use_bilateral_grid=True`) as a trainer table.

One grid [12, L, Y, X] per training image: a 3x4 affine colour matrix per lattice cell, identity at init.  While training,
each view's clamped composite goes through its grid before the loss (model.py:300-302); the slice and its gradient run inside
the loss kernels (`qed_loss_fwd_bwd_bilagrid`, which writes one gradient row per view).

Per step: the rows of the local views -> their sum over the ranks -> `regularize()` (TV, overwrites `grad`) ->
`accumulate(ids, rows)` (all views' rows in view order) -> `step(t)`: Adam over every grid (dense, because TV touches all of
them), lr with nerfstudio's warm-up / exponential decay schedule (camera_opt.lr_at).

`backend="cuda"`: csrc/bilagrid.cu and `qed_adam_arena`.  `backend="torch"`: the same arithmetic in torch, for the CPU tests
of the trainer's host logic.
"""
from __future__ import annotations

import torch
from torch import Tensor

from .camera_opt import AdamTable

# (X, Y, L) bounds of the kernels (include/qed_splat.h, qed_loss_fwd_bwd_bilagrid)
MAX_XY, MAX_L = 1024, 16


def check_grid_shape(X: int, Y: int, L: int, num_grids: int = 1) -> None:
    if not (2 <= X <= MAX_XY and 2 <= Y <= MAX_XY and 2 <= L <= MAX_L):
        raise ValueError(f"bilateral grid shape (X, Y, L) = {(X, Y, L)} unsupported: 2 <= X, Y <= {MAX_XY} and 2 <= L <= {MAX_L}")
    if num_grids < 1 or num_grids * 12 * L * Y * X > 2**31 - 1:
        raise ValueError(f"{num_grids} bilateral grids of {(X, Y, L)}: need 1 <= num_grids and num_grids * 12 L Y X < 2^31")


def total_variation_torch(grids: Tensor, weight: float) -> Tensor:
    """weight / G * sum over the L, Y, X axes of sum (x[i+1] - x[i])^2 / (elements of one grid's difference)."""
    tv = 0.0
    for d in (2, 3, 4):
        n = grids.shape[d]
        diff = grids.narrow(d, 1, n - 1) - grids.narrow(d, 0, n - 1)
        tv = tv + (diff ** 2).sum() / diff[0].numel()
    return weight * tv / grids.shape[0]


class BilateralGridOptimizer(AdamTable):
    """The grids (identity at init), their gradient and Adam moments as flat [num_grids * 12 L Y X] buffers."""

    def __init__(self, num_grids: int, device, shape=(16, 16, 8), lr: float = 2e-3, lr_final: float = 1e-4, warmup_steps: int = 1000,
                 max_steps: int = 30000, tv_weight: float = 10.0, betas=(0.9, 0.999), eps: float = 1e-15, backend: str = "cuda"):
        X, Y, L = (int(v) for v in shape)
        check_grid_shape(X, Y, L, num_grids)
        self.num_grids, self.X, self.Y, self.L = int(num_grids), X, Y, L
        self.row = 12 * L * Y * X  # a multiple of 4: the table needs no padding
        super().__init__(self.num_grids * self.row, device, "bilateral grid", lr, lr_final, warmup_steps, max_steps, betas, eps, backend)
        self.grids.copy_(torch.eye(3, 4, device=self.device).reshape(1, 12, 1, 1, 1))
        self.tv_weight = tv_weight
        self.tv_loss = torch.zeros(1, device=self.device)
        self._partials = torch.empty(self.num_grids, dtype=torch.float64, device=self.device)

    @property
    def grids(self) -> Tensor:
        """[num_grids, 12, L, Y, X] view of the grids."""
        return self.param.view(self.num_grids, 12, self.L, self.Y, self.X)

    @property
    def grids_grad(self) -> Tensor:
        return self.grad.view(self.num_grids, 12, self.L, self.Y, self.X)

    def regularize(self) -> Tensor:
        """Overwrites `grad` with the TV gradient (call once per step, before `accumulate`); returns its value (device)."""
        if self.backend != "cuda":
            g = self.grids.detach().clone().requires_grad_(True)
            tv = total_variation_torch(g, self.tv_weight)
            (d,) = torch.autograd.grad(tv, g)
            self.grids_grad.copy_(d)
            self.tv_loss.copy_(tv.detach().reshape(1))
            return self.tv_loss
        from . import _lib

        _lib.check(self.lib.qed_bilagrid_tv(self.num_grids, self.X, self.Y, self.L, _lib.ptr(self.param), float(self.tv_weight), _lib.ptr(self.grad),
                                            _lib.ptr(self._partials), _lib.ptr(self.tv_loss), _lib.current_stream()), "qed_bilagrid_tv")
        return self.tv_loss

    def accumulate(self, ids: Tensor, rows: Tensor) -> None:
        """grad[ids[r]] += rows[r] in row order; ids int32 on the device (validated), rows [n, 12, L, Y, X] contiguous."""
        n = ids.numel()
        if self.backend != "cuda":
            g = self.grids_grad
            for r in range(n):
                g[int(ids[r])] += rows[r].view(12, self.L, self.Y, self.X)
            return
        from . import _lib

        _lib.check(self.lib.qed_bilagrid_accumulate(n, _lib.ptr(ids), _lib.ptr(rows), self.num_grids, self.X, self.Y, self.L, _lib.ptr(self.grad),
                                                    _lib.current_stream()), "qed_bilagrid_accumulate")
