"""Splatfacto's MCMC densification strategy (nerfstudio 1.1.5 `strategy="mcmc"` -> gsplat 1.4.0 `MCMCStrategy`) on a
trainer.GaussianArena.

gsplat's step_post_backward(step, lr), after Adam, restated ([UP] = from memory of the upstream code):
  * refine_start_iter < step < refine_stop_iter and step % refine_every == 0: relocate, then add;
      relocate: rows with o = sigmoid(logit) <= min_opacity are dead; as many rows are drawn (with replacement, p ~ o) from
        the alive ones, each drawn row s gets compute_relocation at ratio bincount(draws)[s] + 1 (clamped to 51) and its Adam
        moments zeroed, and every dead row becomes a copy of its draw (keeping its own moments, as gsplat's optimizer_fn
        only zeroes the drawn rows [UP]);
      add: n_new = max(0, min(cap_max, int(1.05 N)) - N) rows drawn from all (p ~ o), the same update on the drawn rows
        (moments kept), one copy per draw appended with zero moments;
  * every step (also after refine_stop_iter): means += R diag(s)^2 R^T (randn(3) * sigmoid(100 ((1 - o) - 0.995)) * lr * noise_lr).
Splatfacto adds mcmc_opacity_reg * mean(o) + mcmc_scale_reg * mean(exp(log-scales)) to the loss.

Deliberate deviations (INTEGRATION.md section 3): draws come from a counter-based Philox4x32-10 through an inverse CDF over the
exact int64 scan of floor(o * 2^24) (torch.multinomial's stream cannot be reproduced; this one is identical on every rank
and reproducible from numpy, tests/mcmc_oracle.py); the relocation denominator is evaluated in float64 by the hockey-stick
identity; with no alive Gaussian relocate and add do nothing (torch.multinomial would raise).

`impl="fused"`: the kernels of csrc/mcmc.cu plus qed_arena_gather for the append.  `impl="torch"`: the same updates in
torch on any device (the CPU gloo tests); it draws with torch.multinomial and a CPU generator seeded from (seed, step), so
its draws are not the Philox ones.  Drawing is separate from applying, so both can be fed the same draws.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

STRATEGIES = ("default", "mcmc")
N_MAX = 51  # gsplat's n_max: relocation ratios are clamped to [1, 51]
FLT_EPSILON = float(torch.finfo(torch.float32).eps)
MIN_OPACITY_FLOOR = 2.0 ** -23  # above this every alive row has a sampling weight floor(o * 2^24) >= 1
STREAM_NOISE, STREAM_RELOCATE, STREAM_ADD = 0, 1, 2  # Philox counter word 2


def is_refine_step(step: int, refine_start: int, refine_stop: int, refine_every: int) -> bool:
    """gsplat MCMCStrategy.step_post_backward: relocate + add at this 0-based step."""
    return refine_start < step < refine_stop and step % refine_every == 0


def growth(N: int, cap_max: int) -> int:
    """Rows the add step appends: max(0, min(cap_max, int(1.05 * N)) - N), as Python computes it."""
    return max(0, min(cap_max, int(1.05 * N)) - N)


def relocation_denominator(x: Tensor, n: Tensor) -> Tensor:
    """D(x, n) = sum_{j=1..n} C(n, j) (-1)^(j-1) x^j / sqrt(j) (float64): gsplat's double loop folded by the hockey-stick
    identity sum_{i=k+1..n} C(i-1, k) = C(n, k+1)."""
    x, n = x.double(), n.double()
    D = torch.zeros_like(x)
    binom = torch.ones_like(x)
    xp = torch.ones_like(x)
    for j in range(1, int(n.max()) + 1 if n.numel() else 1):
        binom = binom * (n - j + 1) / j
        xp = xp * x
        D = D + torch.where(n >= j, binom * xp / math.sqrt(j) * (1.0 if j % 2 else -1.0), torch.zeros_like(x))
    return D


def relocation_values(o: Tensor, scales: Tensor, ratio: Tensor, min_opacity: float) -> Tuple[Tensor, Tensor]:
    """gsplat compute_relocation + the clamp of relocate / sample_add, in float64 (as the kernel computes it):
    o [n] float32 opacities, scales [n,3] float32 (exp of the log-scales), ratio [n] -> (clamped o' float32, scale' float32)."""
    n = ratio.clamp(1, N_MAX).double()
    od = o.double()
    x = 1.0 - torch.pow(1.0 - od, 1.0 / n)
    coeff = od / relocation_denominator(x, n)
    scale_new = (coeff[:, None] * scales.double()).to(torch.float32)
    o_new = x.to(torch.float32).clamp(min=min_opacity, max=1.0 - FLT_EPSILON)
    return o_new, scale_new


class MCMCStrategy:
    """State-free apart from workspaces: every decision derives from (seed, step) and the arena, so replicas that call it
    with the same arguments stay bit-identical without any broadcast."""

    def __init__(self, device, cap_max: int = 1_000_000, noise_lr: float = 5e5, refine_start: int = 500, refine_stop: int = 15000,
                 refine_every: int = 100, min_opacity: float = 0.005, opacity_reg: float = 0.01, scale_reg: float = 0.01, seed: int = 42,
                 impl: Optional[str] = None):
        device = torch.device(device)
        self.device = device
        self.impl = impl or ("fused" if device.type == "cuda" else "torch")
        if self.impl not in ("fused", "torch"):
            raise ValueError(f"impl must be 'fused' or 'torch', got {self.impl!r}")
        self.cap_max, self.noise_lr = int(cap_max), float(noise_lr)
        self.refine_start, self.refine_stop, self.refine_every = int(refine_start), int(refine_stop), int(refine_every)
        self.min_opacity, self.opacity_reg, self.scale_reg = float(min_opacity), float(opacity_reg), float(scale_reg)
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.reg_loss = torch.zeros(2, device=device)  # [opacity term, scale term] of the last regularize()
        self.lib = None
        self._ws = None
        self._reg_ws = None
        if self.impl == "fused":
            from . import _lib

            self.lib = _lib.load()
            self._reg_ws = torch.zeros(self.lib.qed_mcmc_reg_workspace_bytes(), dtype=torch.uint8, device=device)

    # -- helpers -------------------------------------------------------------------------------
    @staticmethod
    def _starts(arena) -> Tensor:
        from .trainer import GROUPS

        # host array: the caller keeps it referenced until the C call has returned (a temporary's data_ptr() would dangle)
        return torch.tensor([arena.offsets[g][0] for g in GROUPS], dtype=torch.int64)

    def _workspace(self, N: int) -> Tensor:
        n = self.lib.qed_mcmc_workspace_bytes(N)
        if self._ws is None or self._ws.numel() < n:
            self._ws = torch.empty(n, dtype=torch.uint8, device=self.device)
        return self._ws

    def _generator(self, step: int, stream: int) -> torch.Generator:
        return torch.Generator().manual_seed((self.seed * 1_000_003 + step * 3 + stream) % (2 ** 63))

    # -- drawing -------------------------------------------------------------------------------
    def dead_rows(self, arena) -> Tuple[Tensor, int]:
        """-> (int32 dead rows [n_dead] ascending, n_dead).  The count is the one device-to-host read of a refine step."""
        op = arena.view(arena.param, "opacities")
        if self.impl == "torch":
            dead = torch.where(torch.sigmoid(op) <= self.min_opacity)[0].to(torch.int32)
            return dead, int(dead.numel())
        from . import _lib

        idx = torch.empty(max(arena.N, 1), dtype=torch.int32, device=self.device)
        n_dead = torch.empty(1, dtype=torch.int64, device=self.device)
        ws = self._workspace(arena.N)
        _lib.check(self.lib.qed_mcmc_census(arena.N, _lib.ptr(op), self.min_opacity, _lib.ptr(idx), _lib.ptr(n_dead), _lib.ptr(ws), ws.numel(),
                                            _lib.current_stream()), "qed_mcmc_census")
        n = int(n_dead.item())
        return idx[:n], n

    def draw(self, arena, n: int, step: int, stream: int, zero_dead: bool) -> Tuple[Tensor, Tensor]:
        """n rows drawn with replacement, p ~ o (dead rows excluded with zero_dead) -> (int32 draws [n], int32 counts [N] =
        bincount).  The caller makes sure some row has a positive weight."""
        op = arena.view(arena.param, "opacities")
        if self.impl == "torch":
            w = torch.sigmoid(op).double().cpu()
            if zero_dead:
                w = torch.where(torch.sigmoid(op).cpu() <= self.min_opacity, torch.zeros_like(w), w)
            draws = torch.multinomial(w, n, replacement=True, generator=self._generator(step, stream)) if n else torch.zeros(0, dtype=torch.int64)
            draws = draws.to(self.device)
            return draws.to(torch.int32), torch.bincount(draws, minlength=arena.N).to(torch.int32)
        from . import _lib

        draws = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
        counts = torch.empty(arena.N, dtype=torch.int32, device=self.device)
        total = torch.empty(1, dtype=torch.int64, device=self.device)
        ws = self._workspace(arena.N)
        _lib.check(self.lib.qed_mcmc_sample(arena.N, _lib.ptr(op), self.min_opacity, int(zero_dead), n, self.seed, step & 0xFFFFFFFF, stream,
                                            _lib.ptr(draws), _lib.ptr(counts), _lib.ptr(total), _lib.ptr(ws), ws.numel(), _lib.current_stream()),
                   "qed_mcmc_sample")
        return draws[:n], counts

    # -- applying ------------------------------------------------------------------------------
    def relocate(self, arena, draws: Tensor, dead: Tensor, counts: Optional[Tensor] = None) -> None:
        """gsplat relocate on given draws (one per dead row, same order).  `counts` = bincount(draws) over N (the sample
        kernel writes it; computed here when draws come from elsewhere)."""
        assert draws.numel() == dead.numel()
        if draws.numel() == 0:
            return
        counts = self._counts(arena, draws, counts)
        if self.impl == "torch":
            P, M, V = arena.views(arena.param), arena.views(arena.exp_avg), arena.views(arena.exp_avg_sq)
            rows = self._update_rows_torch(arena, counts)
            d, s = dead.long(), draws.long()
            for g in P:
                P[g][d] = P[g][s]
                M[g][rows] = 0.0  # only the drawn rows; the dead rows keep their moments (gsplat's optimizer_fn [UP])
                V[g][rows] = 0.0
            return
        from . import _lib

        starts = self._starts(arena)
        _lib.check(self.lib.qed_mcmc_relocate(arena.N, _lib.ptr(counts), self.min_opacity, 1, draws.numel(), _lib.ptr(draws.contiguous()),
                                              _lib.ptr(dead.contiguous()), _lib.ptr(arena.param), _lib.ptr(arena.exp_avg),
                                              _lib.ptr(arena.exp_avg_sq), starts.data_ptr(), _lib.current_stream()),
                   "qed_mcmc_relocate")

    def add(self, arena, draws: Tensor, counts: Optional[Tensor] = None) -> None:
        """gsplat sample_add on given draws: the drawn rows updated in place (moments kept), one copy per draw appended with
        zero moments.  Rebuilds the arena (N -> N + len(draws))."""
        n_new = draws.numel()
        if n_new == 0:
            return
        counts = self._counts(arena, draws, counts)
        N = arena.N
        if self.impl == "torch":
            self._update_rows_torch(arena, counts)
            s = draws.long()
            P, M, V = arena.views(arena.param), arena.views(arena.exp_avg), arena.views(arena.exp_avg_sq)
            arena._build({g: torch.cat([P[g], P[g][s]]) for g in P}, {g: torch.cat([M[g], torch.zeros_like(M[g][s])]) for g in M},
                         {g: torch.cat([V[g], torch.zeros_like(V[g][s])]) for g in V})
            return
        from . import _lib
        from .trainer import GaussianArena, GROUPS

        starts = self._starts(arena)
        _lib.check(self.lib.qed_mcmc_relocate(N, _lib.ptr(counts), self.min_opacity, 0, 0, None, None, _lib.ptr(arena.param), None, None,
                                              starts.data_ptr(), _lib.current_stream()), "qed_mcmc_relocate")
        new_off, n = GaussianArena.layout(N + n_new)
        new_param, new_m, new_v = (torch.zeros(n, device=self.device) for _ in range(3))
        src = torch.cat([torch.arange(N, dtype=torch.int32, device=self.device), draws.to(torch.int32)]).contiguous()
        fresh = torch.cat([torch.zeros(N, dtype=torch.uint8, device=self.device), torch.ones(n_new, dtype=torch.uint8, device=self.device)])
        new_starts = torch.tensor([new_off[g][0] for g in GROUPS], dtype=torch.int64)
        _lib.check(self.lib.qed_arena_gather(N + n_new, _lib.ptr(src), _lib.ptr(fresh), None, None, None, _lib.ptr(arena.param),
                                             _lib.ptr(arena.exp_avg), _lib.ptr(arena.exp_avg_sq), starts.data_ptr(),
                                             _lib.ptr(new_param), _lib.ptr(new_m), _lib.ptr(new_v), new_starts.data_ptr(),
                                             _lib.current_stream()), "qed_arena_gather")
        arena.adopt(N + n_new, new_param, new_m, new_v)

    def _counts(self, arena, draws: Tensor, counts: Optional[Tensor]) -> Tensor:
        if counts is None:
            counts = torch.bincount(draws.long(), minlength=arena.N)
        return counts.to(device=self.device, dtype=torch.int32).contiguous()

    def _update_rows_torch(self, arena, counts: Tensor) -> Tensor:
        """compute_relocation on the rows drawn at least once, each once, from its old values -> those rows (int64)."""
        rows = torch.where(counts > 0)[0]
        op = arena.view(arena.param, "opacities")
        ls = arena.view(arena.param, "scales")
        o_new, s_new = relocation_values(torch.sigmoid(op[rows]), torch.exp(ls[rows]), counts[rows].long() + 1, self.min_opacity)
        op[rows] = torch.logit(o_new)
        ls[rows] = torch.log(s_new)
        return rows

    # -- the strategy --------------------------------------------------------------------------
    def refine(self, arena, step: int) -> Dict[str, int]:
        """relocate + add of a refine step -> {"n_relocated", "n_added", "n"} (and "no_alive": 1 when every row is dead:
        then nothing happens, where torch.multinomial would raise)."""
        dead, n_dead = self.dead_rows(arena)
        info = {"n_relocated": 0, "n_added": 0}
        if n_dead == arena.N:
            info["no_alive"] = 1
        else:
            if n_dead:
                draws, counts = self.draw(arena, n_dead, step, STREAM_RELOCATE, zero_dead=True)
                self.relocate(arena, draws, dead, counts)
                info["n_relocated"] = n_dead
            n_new = growth(arena.N, self.cap_max)
            if n_new:
                draws, counts = self.draw(arena, n_new, step, STREAM_ADD, zero_dead=False)
                self.add(arena, draws, counts)
                info["n_added"] = n_new
        info["n"] = arena.N
        return info

    def inject_noise(self, arena, step: int, scaler: float) -> None:
        """means += R diag(s)^2 R^T (n * sigmoid(100 ((1 - o) - 0.995)) * scaler); n from Philox (fused) or the (seed, step)
        generator (torch)."""
        if self.impl == "torch":
            P = arena.views(arena.param)
            n = torch.randn(arena.N, 3, generator=self._generator(step, STREAM_NOISE)).to(self.device)
            apply_noise_torch(P["means"], P["quats"], P["scales"], P["opacities"], n, scaler)
            return
        from . import _lib

        starts = self._starts(arena)
        _lib.check(self.lib.qed_mcmc_noise(arena.N, _lib.ptr(arena.param), starts.data_ptr(), float(scaler), self.seed, step & 0xFFFFFFFF,
                                           _lib.current_stream()), "qed_mcmc_noise")

    def regularize(self, arena) -> Tensor:
        """Adds the gradients of splatfacto's two MCMC regularisers to arena.grad (once per step, after the cross-rank sum);
        -> reg_loss [opacity term, scale term] (device)."""
        if self.impl == "torch":
            op = arena.view(arena.param, "opacities").detach().clone().requires_grad_(True)
            ls = arena.view(arena.param, "scales").detach().clone().requires_grad_(True)
            lo, lsc = regularizers_torch(op, ls, self.opacity_reg, self.scale_reg)
            go, gs = torch.autograd.grad(lo + lsc, (op, ls))
            arena.view(arena.grad, "opacities").add_(go)
            arena.view(arena.grad, "scales").add_(gs)
            self.reg_loss.copy_(torch.stack([lo.detach(), lsc.detach()]))
            return self.reg_loss
        from . import _lib

        starts = self._starts(arena)
        _lib.check(self.lib.qed_mcmc_reg(arena.N, _lib.ptr(arena.param), starts.data_ptr(), self.opacity_reg, self.scale_reg,
                                         _lib.ptr(arena.grad), _lib.ptr(self.reg_loss), _lib.ptr(self._reg_ws), self._reg_ws.numel(),
                                         _lib.current_stream()), "qed_mcmc_reg")
        return self.reg_loss

    def step_post_backward(self, arena, step: int, lr: float) -> Optional[Dict[str, int]]:
        """After Adam of 0-based `step`, `lr` = the means learning rate after the scheduler step: relocate + add on gsplat's
        schedule (-> info), position noise every step (-> None on other steps)."""
        info = None
        if is_refine_step(step, self.refine_start, self.refine_stop, self.refine_every):
            info = self.refine(arena, step)
        self.inject_noise(arena, step, lr * self.noise_lr)
        return info


def apply_noise_torch(means: Tensor, quats: Tensor, log_scales: Tensor, logit_opacities: Tensor, normals: Tensor, scaler: float) -> None:
    """gsplat inject_noise_to_position given the normals [N,3], in place on `means`."""
    from .trainer import _quat_to_rotmat

    R = _quat_to_rotmat(quats)
    s2 = torch.exp(log_scales) ** 2
    o = torch.sigmoid(logit_opacities)
    v = normals * (1.0 / (1.0 + torch.exp(-100.0 * ((1.0 - o) - 0.995))))[:, None] * scaler
    u = s2 * torch.einsum("nji,nj->ni", R, v)
    means.add_(torch.einsum("nij,nj->ni", R, u))


def regularizers_torch(logit_opacities: Tensor, log_scales: Tensor, opacity_reg: float, scale_reg: float) -> Tuple[Tensor, Tensor]:
    """splatfacto get_loss_dict with strategy="mcmc": (opacity_reg * mean |sigmoid|, scale_reg * mean |exp|)."""
    return opacity_reg * torch.sigmoid(logit_opacities).abs().mean(), scale_reg * torch.exp(log_scales).abs().mean()
