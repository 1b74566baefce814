"""View-sharded multi-GPU training step for the qed-splatter hot path (SURVEY.md §8 rows a14-a16, §8e).

What the reference does per iteration through nerfstudio (`Trainer.train_iteration` -> `QEDSplatterModel
.get_outputs` model.py:199-321 -> `get_loss_dict` model.py:73-118 -> backward -> six Adam groups
config.py:44-68 -> gsplat `DefaultStrategy.step_post_backward` on `self.info` model.py:267,289-292),
restated as one process per GPU:

  * Gaussian parameters, Adam moments and densification state are replicated on every rank; rank r renders
    its slice of the view batch (one reference step per view: per-view depth fill / n_valid, loss = mean
    over ALL views of the batch, so gradients are pre-scaled by 1/total_views).
  * one all-reduce (SUM) over the flat gradient arena (59 floats per Gaussian); the densification
    statistics (grad2d, count: SUM; radii: MAX) are accumulated locally and all-reduced only when a refine
    step consumes them (SUM/MAX are associative, so this equals reducing every step).
  * fused Adam over the flat arena (one launch), then — every `refine_every` steps — duplicate / split /
    prune / opacity reset with an RNG seeded from (seed, step), so every replica takes identical decisions
    and no parameter broadcast is needed.

Semantics caveat (SURVEY §8e): the reference takes one optimizer step PER VIEW; one step on the mean
gradient of B views is a different schedule.  Parity is defined on the gradients/statistics of a single
step (tests/test_trainer_*.py), not on a 30k-iteration trajectory.

The parameter update and densification bookkeeping run as torch ops / the fused Adam kernel; `backend`
selects "cuda" (C-ABI kernels) or "torch" (pure torch, used by the CPU gloo tests of the host logic; it is
NOT a rendering fallback — rendering always needs the CUDA library).
"""
from __future__ import annotations

import dataclasses
import math
from dataclasses import dataclass, field
from typing import Any, Dict, Optional, Tuple

import torch
from torch import Tensor

GROUPS = ("means", "quats", "scales", "opacities", "sh")
GROUP_SHAPES = {"means": (3,), "quats": (4,), "scales": (3,), "opacities": (), "sh": (16, 3)}  # per Gaussian
GROUP_DIMS = {g: math.prod(GROUP_SHAPES[g]) for g in GROUPS}
FLOATS_PER_GAUSSIAN = sum(GROUP_DIMS.values())  # 59

# SplatTrainer.state_dict(): splatfacto's stored Gaussian parameters (and optimizer groups), per-Gaussian shapes
CHECKPOINT_FORMAT_VERSION = 1
SPLATFACTO_SHAPES = {"means": (3,), "scales": (3,), "quats": (4,), "features_dc": (3,), "features_rest": (15, 3), "opacities": (1,)}
STRATEGY_STATS = ("grad2d", "count", "radii")
# TrainConfig fields that decide which tables a state holds and their shapes: a resumed run cannot change them
LAYOUT_FIELDS = ("strategy", "camera_optimizer", "use_bilateral_grid", "bilateral_grid_shape")
# SplatTrainer.evaluate renders the local views at most this many at a time, so its buffers do not grow with the eval set
EVAL_CHUNK_VIEWS = 8


@dataclass
class TrainConfig:
    """Hyper-parameters: qed_splatter/config.py:39-68 + qed_splatter/model.py:41-47 + splatfacto defaults (SURVEY A.8)."""
    max_steps: int = 30000
    lr_means: float = 1.6e-4
    lr_means_final: float = 1.6e-6
    lr_features_dc: float = 0.0025
    lr_features_rest: float = 0.0025 / 20
    lr_opacities: float = 0.05
    lr_scales: float = 0.005
    lr_quats: float = 0.001
    adam_eps: float = 1e-15
    adam_betas: Tuple[float, float] = (0.9, 0.999)
    depth_lambda: float = 0.2
    depth_unit_scale: float = 0.001  # qed_splatter/dataparser.py:15 (x the dataparser's scene scale); used when gt_depth is raw uint16
    ssim_lambda: float = 0.2
    sh_degree: int = 3
    sh_degree_interval: int = 1000
    render_mode: str = "RGB+D"  # what qed_splatter/model.py:257 passes; "RGB+ED" is the north_star variant
    rasterize_mode: str = "classic"
    # densification (gsplat DefaultStrategy as configured by splatfacto + config.py:40-41)
    warmup_length: int = 500
    refine_every: int = 100
    reset_alpha_every: int = 30
    stop_split_at: int = 15000
    stop_screen_size_at: int = 4000
    densify_grad_thresh: float = 0.0005
    densify_size_thresh: float = 0.01
    split_screen_size: float = 0.05
    cull_alpha_thresh: float = 0.005
    cull_scale_thresh: float = 0.5
    cull_screen_size: float = 0.15
    n_split_samples: int = 2
    pause_refine_after_reset: int = 100  # nerfstudio: num_train_data + refine_every; no dataset here -> refine_every
    use_absgrad: bool = True
    scene_scale: float = 1.0
    seed: int = 42
    # world_size > 1, how the gradients are summed over the ranks:
    #   "exchange": this library's NVLink path (comm.ViewShardedGradients: per-view colour gradients stored into every rank's
    #               exchange buffer by the projection backward, one all-reduce kernel over the 11 non-SH floats per Gaussian,
    #               SH coefficient gradient rebuilt locally) -- no NCCL on the data path;  CUDA backend + NCCL group only
    #   "nccl"    : torch.distributed all-reduce of the arena, pipelined over `comm_chunks` Gaussian ranges (also gloo / CPU)
    #   "auto"    : "exchange" when available, else "nccl"
    comm: str = "auto"
    comm_chunks: int = 4  # "nccl": Gaussian ranges whose SH gradients are all-reduced / Adam-stepped in a pipeline
    chunk_project_bwd: bool = True  # "nccl": also split the projection backward so the first reductions start earlier
    # splatfacto's camera optimizer (camera_opt.py): "off" or "SO3xR3" (a [num_cameras, 6] pose table trained with the
    # Gaussians; SplatTrainer(num_cameras=...), step(None, ..., camera_to_worlds=, camera_ids=)).  [UP] = nerfstudio 1.1.5
    # defaults restated from memory of the upstream code (CameraOptimizerConfig, splatfacto's "camera_opt" param group).
    camera_optimizer: str = "off"
    camera_opt_lr: float = 1e-4  # [UP] Adam lr (eps = adam_eps 1e-15 [UP])
    camera_opt_lr_final: float = 5e-7  # [UP] ExponentialDecayScheduler lr_final, reached at max_steps
    camera_opt_warmup: int = 1000  # [UP] warm-up steps from lr 0 (cosine ramp)
    camera_opt_trans_l2_penalty: float = 1e-2  # [UP] weight of mean_rows |t| in the loss
    camera_opt_rot_l2_penalty: float = 1e-3  # [UP] weight of mean_rows |omega| in the loss
    # splatfacto's bilateral grid (bilateral_grid.py): one affine colour grid per training camera, applied to the training
    # views before the RGB loss; SplatTrainer(num_cameras=...), step(..., camera_ids=).  [UP] = nerfstudio >= 1.1.4 defaults
    # restated from memory of the upstream code (splatfacto's "bilateral_grid" param group and tv loss).
    use_bilateral_grid: bool = False
    bilateral_grid_shape: Tuple[int, int, int] = (16, 16, 8)  # [UP] (X, Y, L) = grid_X, grid_Y, grid_W
    bilateral_grid_lr: float = 2e-3  # [UP] Adam lr (eps = adam_eps 1e-15 [UP])
    bilateral_grid_lr_final: float = 1e-4  # [UP] ExponentialDecayScheduler lr_final, reached at max_steps
    bilateral_grid_warmup: int = 1000  # [UP] warm-up steps from lr 0
    bilateral_grid_tv_weight: float = 10.0  # [UP] weight of the total-variation loss
    # splatfacto's resolution schedule: steps [k * resolution_schedule, (k + 1) * resolution_schedule) render at 1 / 2^(n - k)
    # of the full resolution for k < n = num_downscales, with the ground truth box-downscaled to match.  Splatfacto's default
    # (and qed-splatter's) is num_downscales = 2; it stays 0 (always full resolution) here so existing runs are unchanged.
    num_downscales: int = 0
    resolution_schedule: int = 3000
    # densification strategy: "default" (gsplat DefaultStrategy: the fields above) or "mcmc" (gsplat MCMCStrategy, mcmc.py:
    # relocation of dead Gaussians and capped growth every refine_every steps in (warmup_length, stop_split_at), position
    # noise every step, no opacity reset; min_opacity = cull_alpha_thresh).  [UP] = nerfstudio 1.1.5 SplatfactoModelConfig
    # defaults restated from memory of the upstream code.
    strategy: str = "default"  # [UP]
    max_gs_num: int = 1_000_000  # [UP] MCMC cap_max: the add step never grows past it
    noise_lr: float = 5e5  # [UP] position noise scale = means lr * noise_lr
    mcmc_opacity_reg: float = 0.01  # [UP] weight of mean(sigmoid(logit-opacities)) in the loss (MCMC only)
    mcmc_scale_reg: float = 0.01  # [UP] weight of mean(exp(log-scales)) in the loss (MCMC only)

    def __post_init__(self):
        self.validate()

    def validate(self) -> None:
        """Raises ValueError for settings no code path accepts (checked at construction and by SplatTrainer)."""
        from .camera_opt import CAMERA_OPTIMIZER_MODES

        if self.camera_optimizer not in CAMERA_OPTIMIZER_MODES:
            raise ValueError(f"camera_optimizer must be one of {CAMERA_OPTIMIZER_MODES}, got {self.camera_optimizer!r}")
        from .mcmc import MIN_OPACITY_FLOOR, STRATEGIES

        if self.strategy not in STRATEGIES:
            raise ValueError(f"strategy must be one of {STRATEGIES}, got {self.strategy!r}")
        if self.max_gs_num < 1:
            raise ValueError(f"max_gs_num >= 1 expected, got {self.max_gs_num}")
        if self.noise_lr < 0 or self.mcmc_opacity_reg < 0 or self.mcmc_scale_reg < 0:
            raise ValueError("noise_lr, mcmc_opacity_reg and mcmc_scale_reg must be >= 0")
        if self.strategy == "mcmc" and not (MIN_OPACITY_FLOOR <= self.cull_alpha_thresh < 1.0):
            # every alive Gaussian then has a positive sampling weight floor(o * 2^24) (mcmc.py)
            raise ValueError(f"strategy='mcmc' needs 2^-23 <= cull_alpha_thresh < 1, got {self.cull_alpha_thresh}")
        if self.num_downscales < 0 or self.resolution_schedule < 1:
            raise ValueError(f"num_downscales >= 0 and resolution_schedule >= 1 expected, got {self.num_downscales} and {self.resolution_schedule}")
        if self.use_bilateral_grid:
            from .bilateral_grid import check_grid_shape

            shape = tuple(self.bilateral_grid_shape)
            if len(shape) != 3 or not all(isinstance(v, int) for v in shape):
                raise ValueError(f"bilateral_grid_shape must be three ints (X, Y, L), got {self.bilateral_grid_shape!r}")
            check_grid_shape(*shape)
            if self.bilateral_grid_lr < 0 or self.bilateral_grid_lr_final <= 0 or self.bilateral_grid_warmup < 0 or self.bilateral_grid_tv_weight < 0:
                raise ValueError("bilateral grid: lr >= 0, lr_final > 0, warmup >= 0 and tv_weight >= 0 expected")

    def lr_means_at(self, step: int) -> float:
        """nerfstudio ExponentialDecayScheduler (no warmup): log-linear from lr to lr_final over max_steps."""
        t = min(max(step / self.max_steps, 0.0), 1.0)
        return math.exp(math.log(self.lr_means) * (1 - t) + math.log(self.lr_means_final) * t)


class GaussianArena:
    """Flat arenas [param | grad | exp_avg | exp_avg_sq], each 59*N floats laid out group by group
    (means 3N | quats 4N | log-scales 3N | logit-opacities N | SH 48N), so Adam and the gradient
    all-reduce are single launches over contiguous memory.  Rebuilt whenever N changes."""

    def __init__(self, means: Tensor, quats: Tensor, log_scales: Tensor, logit_opacities: Tensor, sh: Tensor):
        N = means.shape[0]
        assert quats.shape == (N, 4) and log_scales.shape == (N, 3) and logit_opacities.shape == (N,) and sh.shape == (N, 16, 3)
        self.device = means.device
        self._build(dict(means=means, quats=quats, scales=log_scales, opacities=logit_opacities, sh=sh), None, None)

    def _build(self, params: Dict[str, Tensor], m: Optional[Dict[str, Tensor]], v: Optional[Dict[str, Tensor]]) -> None:
        """New arenas for the Gaussians of `params` (tensors shaped as `view` returns them); Adam moments from m / v, or zero."""
        n = self._set_layout(params["means"].shape[0])
        self.param, self.grad, self.exp_avg, self.exp_avg_sq = (torch.zeros(n, device=self.device) for _ in range(4))
        for g in GROUPS:
            a, b = self.offsets[g]
            self.param[a:b] = params[g].reshape(-1).to(torch.float32)
            if m is not None:
                self.exp_avg[a:b] = m[g].reshape(-1)
                self.exp_avg_sq[a:b] = v[g].reshape(-1)

    @staticmethod
    def layout(N: int):
        """-> (offsets {group: (start, end)}, total floats) of an arena for N Gaussians.  Every group starts on a 16-byte
        boundary (vectorised loads in the kernels); the <= 3 padding floats per group carry zero gradients, so Adam and the
        all-reduce leave them at zero."""
        offsets, o = {}, 0
        for g in GROUPS:
            d = GROUP_DIMS[g]
            offsets[g] = (o, o + d * N)
            o += (d * N + 3) // 4 * 4
        return offsets, o

    def _set_layout(self, N: int) -> int:
        """N, offsets and group_ends (each group's padded end: where the next one starts) for N Gaussians; -> total floats."""
        self.N = N
        self.offsets, n = self.layout(N)
        starts = [self.offsets[g][0] for g in GROUPS]
        self.group_ends = torch.tensor(starts[1:] + [n], dtype=torch.int64, device=self.device)
        return n

    def adopt(self, N: int, param: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor) -> None:
        """Take over freshly built arenas (qed_arena_gather) for N Gaussians; gradients start at zero."""
        n = self._set_layout(N)
        assert param.numel() == n and exp_avg.numel() == n and exp_avg_sq.numel() == n
        self.param, self.exp_avg, self.exp_avg_sq = param, exp_avg, exp_avg_sq
        self.grad = torch.zeros(n, device=self.device)

    def view(self, buf: Tensor, g: str) -> Tensor:
        a, b = self.offsets[g]
        return buf[a:b].view(self.N, *GROUP_SHAPES[g])

    def views(self, buf: Tensor) -> Dict[str, Tensor]:
        return {g: self.view(buf, g) for g in GROUPS}

    def splatfacto_views(self, buf: Tensor) -> Dict[str, Tensor]:
        """Views of `buf` in splatfacto's names and shapes (SPLATFACTO_SHAPES): the SH block as features_dc [N,3] and
        features_rest [N,15,3], the opacities as [N,1]."""
        v = self.views(buf)
        return {"means": v["means"], "scales": v["scales"], "quats": v["quats"], "features_dc": v["sh"][:, 0, :],
                "features_rest": v["sh"][:, 1:, :], "opacities": v["opacities"][:, None]}


@dataclass
class StrategyState:
    grad2d: Tensor
    count: Tensor
    radii: Tensor

    @staticmethod
    def zeros(N: int, device) -> "StrategyState":
        return StrategyState(torch.zeros(N, device=device), torch.zeros(N, device=device), torch.zeros(N, device=device))


def _quat_to_rotmat(q: Tensor) -> Tensor:
    q = q / q.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    w, x, y, z = q.unbind(-1)
    return torch.stack([
        1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
        2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
        2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], dim=-1).reshape(-1, 3, 3)


def refine_gaussians(arena: GaussianArena, state: StrategyState, cfg: TrainConfig, step: int, generator: torch.Generator,
                     impl: Optional[str] = None) -> Dict[str, int]:
    """gsplat DefaultStrategy._grow_gs + _prune_gs (+ optimizer-state surgery) on the arena, deterministic given
    `generator`, so all replicas stay identical.  Order of the Gaussians after the call follows gsplat
    ops.duplicate / ops.split / ops.remove.

    impl "fused" (CUDA arenas, the default there): the decisions are made on [N]-sized index / flag tensors and the
    59 floats x 3 arenas per Gaussian move ONCE, in `qed_arena_gather` (SURVEY.md section 8 a15 / f3).
    impl "torch": the same result with torch cat / index ops on every group (any device; the cross-check, and what
    the gloo tests run on CPU) -- 0.74 s instead of a few ms at 6 M Gaussians."""
    if impl is None:
        impl = "fused" if arena.param.is_cuda else "torch"
    if impl == "fused":
        return _refine_gaussians_fused(arena, state, cfg, step, generator)
    return _refine_gaussians_torch(arena, state, cfg, step, generator)


def _refine_gaussians_fused(arena: GaussianArena, state: StrategyState, cfg: TrainConfig, step: int, generator: torch.Generator) -> Dict[str, int]:
    from . import _lib

    lib = _lib.load()
    dev, N0 = arena.device, arena.N
    P = arena.views(arena.param)  # views, nothing is cloned
    info = {"n_dupli": 0, "n_split": 0, "n_prune": 0}
    idx = torch.arange(N0, device=dev)                        # old row each slot of the new set copies
    fresh = torch.zeros(N0, dtype=torch.bool, device=dev)     # Adam moments start at zero
    crow = torch.full((N0,), -1, dtype=torch.int32, device=dev)  # row in child_means / child_scales
    child_means = child_scales = None
    radii_cur = state.radii
    n_dupli = n_split = 0
    if step < cfg.stop_split_at:
        grads = state.grad2d / state.count.clamp_min(1)
        is_grad_high = grads > cfg.densify_grad_thresh
        is_small = torch.exp(P["scales"]).max(dim=-1).values <= cfg.densify_size_thresh * cfg.scene_scale
        is_dupli = is_grad_high & is_small
        is_split = is_grad_high & ~is_small
        if step < cfg.stop_screen_size_at:
            is_split |= state.radii > cfg.split_screen_size
        n_dupli, n_split = int(is_dupli.sum()), int(is_split.sum())
        info["n_dupli"], info["n_split"] = n_dupli, n_split
        if n_dupli:  # copies appended, optimizer state of the copies zero; freshly duplicated ones are not split
            sel = torch.where(is_dupli)[0]
            idx = torch.cat([idx, sel])
            fresh = torch.cat([fresh, torch.ones(n_dupli, dtype=torch.bool, device=dev)])
            crow = torch.cat([crow, torch.full((n_dupli,), -1, dtype=torch.int32, device=dev)])
            is_split = torch.cat([is_split, torch.zeros(n_dupli, dtype=torch.bool, device=dev)])
            radii_cur = torch.cat([radii_cur, radii_cur[sel]])
        if n_split:  # n_split_samples children replace the parent, appended at the end (sample-major)
            sel = torch.where(is_split)[0]
            rest = torch.where(~is_split)[0]
            par = idx[sel]
            scales = torch.exp(P["scales"][par])
            R = _quat_to_rotmat(P["quats"][par])
            ns = cfg.n_split_samples
            noise = torch.randn(ns, len(sel), 3, generator=generator, device="cpu").to(dev)
            samples = torch.einsum("nij,nj,bnj->bni", R, scales, noise)
            child_means = (P["means"][par][None] + samples).reshape(-1, 3).contiguous()
            child_scales = torch.log(scales / 1.6).repeat(ns, 1).contiguous()
            n_child = ns * len(sel)
            idx = torch.cat([idx[rest], par.repeat(ns)])
            fresh = torch.cat([fresh[rest], torch.ones(n_child, dtype=torch.bool, device=dev)])
            crow = torch.cat([crow[rest], torch.arange(n_child, dtype=torch.int32, device=dev)])
            radii_cur = torch.cat([radii_cur[rest], radii_cur[sel].repeat(ns)])
    # prune, decided on the new set
    is_prune = torch.sigmoid(P["opacities"][idx]) < cfg.cull_alpha_thresh
    if step > cfg.reset_alpha_every * cfg.refine_every:
        s_new = P["scales"][idx]
        if child_scales is not None:
            is_child = crow >= 0
            s_new[is_child] = child_scales[crow[is_child].long()]
        is_big = torch.exp(s_new).max(dim=-1).values > cfg.cull_scale_thresh * cfg.scene_scale
        if step < cfg.stop_screen_size_at:
            is_big |= radii_cur > cfg.cull_screen_size
        is_prune |= is_big
    n_prune = int(is_prune.sum())
    info["n_prune"] = n_prune
    if n_prune:
        keep = torch.where(~is_prune)[0]
        idx, fresh, crow = idx[keep], fresh[keep], crow[keep]
    N1 = idx.numel()
    if N1 != N0 or n_prune or n_split or n_dupli:
        new_off, n = GaussianArena.layout(N1)
        new_param, new_m, new_v = (torch.zeros(n, device=dev) for _ in range(3))
        old_starts = torch.tensor([arena.offsets[g][0] for g in GROUPS], dtype=torch.int64)  # host arrays
        new_starts = torch.tensor([new_off[g][0] for g in GROUPS], dtype=torch.int64)
        idx32 = idx.to(torch.int32).contiguous()
        fresh8 = fresh.to(torch.uint8).contiguous()
        _lib.check(lib.qed_arena_gather(N1, _lib.ptr(idx32), _lib.ptr(fresh8), _lib.ptr(crow.contiguous()) if child_means is not None else None,
                                        _lib.ptr(child_means), _lib.ptr(child_scales), _lib.ptr(arena.param), _lib.ptr(arena.exp_avg),
                                        _lib.ptr(arena.exp_avg_sq), old_starts.data_ptr(), _lib.ptr(new_param), _lib.ptr(new_m), _lib.ptr(new_v),
                                        new_starts.data_ptr(), _lib.current_stream()), "qed_arena_gather")
        arena.adopt(N1, new_param, new_m, new_v)
    state.grad2d = torch.zeros(arena.N, device=dev)
    state.count = torch.zeros(arena.N, device=dev)
    state.radii = torch.zeros(arena.N, device=dev)
    info["n"] = arena.N
    return info


def _refine_gaussians_torch(arena: GaussianArena, state: StrategyState, cfg: TrainConfig, step: int, generator: torch.Generator) -> Dict[str, int]:
    p = {g: arena.view(arena.param, g).clone() for g in GROUPS}
    m = {g: arena.view(arena.exp_avg, g).clone() for g in GROUPS}
    v = {g: arena.view(arena.exp_avg_sq, g).clone() for g in GROUPS}
    N0 = arena.N
    dev = arena.device
    info = {"n_dupli": 0, "n_split": 0, "n_prune": 0}

    if step < cfg.stop_split_at:
        count = state.count
        grads = state.grad2d / count.clamp_min(1)
        is_grad_high = grads > cfg.densify_grad_thresh
        is_small = torch.exp(p["scales"]).max(dim=-1).values <= cfg.densify_size_thresh * cfg.scene_scale
        is_dupli = is_grad_high & is_small
        is_split = is_grad_high & ~is_small
        if step < cfg.stop_screen_size_at:
            is_split |= state.radii > cfg.split_screen_size
        n_dupli, n_split = int(is_dupli.sum()), int(is_split.sum())
        info["n_dupli"], info["n_split"] = n_dupli, n_split
        # duplicate: copies appended, optimizer state of the copies zero
        if n_dupli:
            sel = torch.where(is_dupli)[0]
            for g in GROUPS:
                p[g] = torch.cat([p[g], p[g][sel]])
                m[g] = torch.cat([m[g], torch.zeros_like(m[g][sel])])
                v[g] = torch.cat([v[g], torch.zeros_like(v[g][sel])])
            extra = torch.zeros(n_dupli, dtype=torch.bool, device=dev)
            is_split = torch.cat([is_split, extra])  # freshly duplicated ones are not split
            state_vals = [torch.cat([t, t[sel]]) for t in (state.grad2d, state.count, state.radii)]
        else:
            state_vals = [state.grad2d, state.count, state.radii]
        # split: n_split_samples children replace the parent, appended at the end
        if n_split:
            sel = torch.where(is_split)[0]
            rest = torch.where(~is_split)[0]
            scales = torch.exp(p["scales"][sel])
            R = _quat_to_rotmat(p["quats"][sel])
            ns = cfg.n_split_samples
            noise = torch.randn(ns, len(sel), 3, generator=generator, device="cpu").to(dev)
            samples = torch.einsum("nij,nj,bnj->bni", R, scales, noise)
            newp = {
                "means": (p["means"][sel][None] + samples).reshape(-1, 3),
                "scales": torch.log(scales / 1.6).repeat(ns, 1),
                "quats": p["quats"][sel].repeat(ns, 1),
                "opacities": p["opacities"][sel].repeat(ns),
                "sh": p["sh"][sel].repeat(ns, 1, 1),
            }
            for g in GROUPS:
                p[g] = torch.cat([p[g][rest], newp[g]])
                m[g] = torch.cat([m[g][rest], torch.zeros_like(newp[g])])
                v[g] = torch.cat([v[g][rest], torch.zeros_like(newp[g])])
            state_vals = [torch.cat([t[rest], t[sel].repeat(ns)]) for t in state_vals]
    else:
        state_vals = [state.grad2d, state.count, state.radii]

    # prune
    is_prune = torch.sigmoid(p["opacities"]) < cfg.cull_alpha_thresh
    if step > cfg.reset_alpha_every * cfg.refine_every:
        is_big = torch.exp(p["scales"]).max(dim=-1).values > cfg.cull_scale_thresh * cfg.scene_scale
        if step < cfg.stop_screen_size_at:
            is_big |= state_vals[2] > cfg.cull_screen_size
        is_prune |= is_big
    n_prune = int(is_prune.sum())
    info["n_prune"] = n_prune
    if n_prune:
        keep = torch.where(~is_prune)[0]
        for g in GROUPS:
            p[g], m[g], v[g] = p[g][keep], m[g][keep], v[g][keep]
    if p["means"].shape[0] != N0 or n_prune or info["n_split"] or info["n_dupli"]:
        arena._build(p, m, v)
    # reset running stats (gsplat zeroes them after every refine)
    state.grad2d = torch.zeros(arena.N, device=dev)
    state.count = torch.zeros(arena.N, device=dev)
    state.radii = torch.zeros(arena.N, device=dev)
    info["n"] = arena.N
    return info


def reset_opacities(arena: GaussianArena, cfg: TrainConfig) -> None:
    """gsplat ops.reset_opa: clamp logit-opacities to logit(2*prune_opa), zero their Adam moments."""
    value = cfg.cull_alpha_thresh * 2.0
    cap = math.log(value / (1.0 - value))
    arena.view(arena.param, "opacities").clamp_(max=cap)
    arena.view(arena.exp_avg, "opacities").zero_()
    arena.view(arena.exp_avg_sq, "opacities").zero_()


def adam_step_torch(arena: GaussianArena, lrs: Dict[str, float], lr_sh_rest: float, cfg: TrainConfig, t: int) -> None:
    """torch.optim.Adam arithmetic on the arena (reference for qed_adam_arena; used by the CPU tests)."""
    b1, b2 = cfg.adam_betas
    bias1 = 1.0 - b1 ** t
    bias2_sqrt = math.sqrt(1.0 - b2 ** t)
    arena.exp_avg.mul_(b1).add_(arena.grad, alpha=1 - b1)
    arena.exp_avg_sq.mul_(b2).addcmul_(arena.grad, arena.grad, value=1 - b2)
    lr = torch.empty_like(arena.param)
    for g in GROUPS:
        a, b = arena.offsets[g]
        lr[a:b] = lrs[g]
    a, b = arena.offsets["sh"]
    lr[a:b].view(-1, 48)[:, 3:] = lr_sh_rest
    denom = arena.exp_avg_sq.sqrt() / bias2_sqrt + cfg.adam_eps
    arena.param.sub_(lr / bias1 * (arena.exp_avg / denom))


def rescaled_camera(Ks: Tensor, width: int, height: int, factor: int) -> Tuple[Tensor, int, int]:
    """The render camera of a step at 1/factor resolution, as nerfstudio's `Cameras.rescale_output_resolution(1 / factor)`
    builds it: rows 0-1 of the intrinsics [C,3,3] times 1/factor (float32), size floor(W / factor + 0.5) x
    floor(H / factor + 0.5).  ValueError when that size is not the size of the box-downscaled ground truth
    (data_side.downscaled_size: W // factor x H // factor), where splatfacto's L1 would fail to broadcast."""
    from .data_side import downscaled_size

    if factor == 1:
        return Ks, width, height
    w, h = math.floor(width / factor + 0.5), math.floor(height / factor + 0.5)
    gw, gh = downscaled_size(width, height, factor)
    if (w, h) != (gw, gh):
        raise ValueError(f"{width}x{height} at 1/{factor}: the rescaled camera is {w}x{h} but the downscaled ground truth is {gw}x{gh}")
    Ks = Ks.clone()
    Ks[..., :2, :] *= 1.0 / factor
    return Ks, w, h


def _owned_cpu(t: Tensor) -> Tensor:
    """A contiguous CPU copy of `t` whose storage holds exactly its elements (torch.save of a view writes the whole buffer
    behind it)."""
    out = torch.empty(t.shape, dtype=t.dtype, device="cpu")
    out.copy_(t.detach())
    return out


def _check_shape(what: str, t: Any, shape) -> None:
    if not isinstance(t, Tensor) or tuple(t.shape) != tuple(shape):
        got = tuple(t.shape) if isinstance(t, Tensor) else type(t).__name__
        raise ValueError(f"state {what}: expected a tensor of shape {tuple(shape)}, got {got}")


def _section(state: Dict, key: str) -> Dict:
    if not isinstance(state.get(key), dict):
        raise ValueError(f"state {key!r}: missing (the saved configuration needs it)")
    return state[key]


class SplatTrainer:
    """One process per GPU.  `step()` = render local views + loss + backward + gradient all-reduce + Adam
    (+ densify / opacity reset on schedule)."""

    def __init__(self, means: Tensor, quats: Tensor, log_scales: Tensor, logit_opacities: Tensor, sh: Tensor,
                 cfg: Optional[TrainConfig] = None, rank: int = 0, world_size: int = 1, process_group=None,
                 backend: str = "cuda", num_cameras: int = 0):
        """`num_cameras`: the training cameras: rows of the camera optimizer's pose table (cfg.camera_optimizer != "off") and
        the number of bilateral grids (cfg.use_bilateral_grid)."""
        self.cfg = cfg or TrainConfig()
        self.cfg.validate()  # fields may have been changed after construction
        self.rank, self.world = rank, world_size
        self.pg = process_group
        self.backend = backend
        self.device = means.device
        self.num_cameras = int(num_cameras)
        self.arena = GaussianArena(means, quats, log_scales, logit_opacities, sh)
        self.state = StrategyState.zeros(self.arena.N, self.device)
        self.step_count = 0
        self._fused = None
        if backend == "cuda":
            from .pipeline import FusedSplatStep

            self._fused = FusedSplatStep(self.device)
        self._lr_dev = None
        self._xg = None  # comm.ViewShardedGradients for the current (N, views per rank), built lazily
        self.comm = self._pick_comm()
        self.camera_opt = None
        if self.cfg.camera_optimizer != "off":
            from .camera_opt import CameraPoseOptimizer

            c = self.cfg
            self.camera_opt = CameraPoseOptimizer(num_cameras, self.device, lr=c.camera_opt_lr, lr_final=c.camera_opt_lr_final,
                                                  warmup_steps=c.camera_opt_warmup, max_steps=c.max_steps,
                                                  trans_weight=c.camera_opt_trans_l2_penalty, rot_weight=c.camera_opt_rot_l2_penalty,
                                                  betas=c.adam_betas, eps=c.adam_eps, backend=backend)
        self.bilagrid = None
        self._bg_buf = None  # rows + ids of the whole view batch ("nccl" / one rank; the exchange keeps its own, symmetric)
        if self.cfg.use_bilateral_grid:
            from .bilateral_grid import BilateralGridOptimizer

            c = self.cfg
            if num_cameras < 1:
                raise ValueError("the bilateral grid needs num_cameras >= 1")
            self.bilagrid = BilateralGridOptimizer(num_cameras, self.device, shape=c.bilateral_grid_shape, lr=c.bilateral_grid_lr,
                                                   lr_final=c.bilateral_grid_lr_final, warmup_steps=c.bilateral_grid_warmup, max_steps=c.max_steps,
                                                   tv_weight=c.bilateral_grid_tv_weight, betas=c.adam_betas, eps=c.adam_eps, backend=backend)
        self.mcmc = None
        if self.cfg.strategy == "mcmc":
            from .mcmc import MCMCStrategy

            c = self.cfg
            self.mcmc = MCMCStrategy(self.device, cap_max=c.max_gs_num, noise_lr=c.noise_lr, refine_start=c.warmup_length, refine_stop=c.stop_split_at,
                                     refine_every=c.refine_every, min_opacity=c.cull_alpha_thresh, opacity_reg=c.mcmc_opacity_reg,
                                     scale_reg=c.mcmc_scale_reg, seed=c.seed, impl="fused" if backend == "cuda" else "torch")

    @property
    def pose_adjustment(self) -> Optional[Tensor]:
        """The camera optimizer's [num_cameras, 6] table (translation, rotation log); None when it is off."""
        return None if self.camera_opt is None else self.camera_opt.pose_adjustment

    @property
    def camera_opt_loss(self) -> Optional[Tensor]:
        """The camera optimizer's regulariser of the last step (device scalar [1]); None when it is off."""
        return None if self.camera_opt is None else self.camera_opt.reg_loss

    @property
    def bilateral_grids(self) -> Optional[Tensor]:
        """The bilateral grids [num_cameras, 12, L, Y, X]; None when the grid is off."""
        return None if self.bilagrid is None else self.bilagrid.grids

    @property
    def bilagrid_tv_loss(self) -> Optional[Tensor]:
        """The grids' total-variation loss of the last step (device scalar [1]); None when the grid is off."""
        return None if self.bilagrid is None else self.bilagrid.tv_loss

    @property
    def mcmc_reg_loss(self) -> Optional[Tensor]:
        """The MCMC regularisers of the last step (device [2]: opacity term, scale term); None with strategy "default"."""
        return None if self.mcmc is None else self.mcmc.reg_loss

    def _pick_comm(self) -> str:
        c = self.cfg.comm
        if self.world <= 1:
            return "none"
        ok = self.backend == "cuda" and self.device.type == "cuda"
        if ok:
            import torch.distributed as dist

            ok = dist.is_initialized() and dist.get_backend(self.pg) == "nccl"
        if c == "exchange" and not ok:
            raise RuntimeError("comm='exchange' needs the CUDA backend and an NCCL process group (symmetric memory)")
        return "exchange" if (c in ("auto", "exchange") and ok) else "nccl"

    def _exchange_for(self, views_per_rank: int):
        """The symmetric gradient arena + exchange buffers for the current Gaussian count (rebuilt, collectively, when a
        refine step changed N: every rank refines at the same step).  With MCMC the set never grows past max_gs_num, so the
        buffers are sized for that once and never rebuilt."""
        from .comm import ViewShardedGradients

        x = self._xg
        if x is None or x.views_per_rank != views_per_rank or (x.N != self.arena.N and not x.resize(self.arena.N)):
            # headroom: densification grows the set gradually; most refine steps then reuse the symmetric buffers
            import torch.distributed as dist

            err = None
            try:
                if self.mcmc is not None:  # room for max_gs_num Gaussians: MCMC never grows past it
                    headroom = max(self.cfg.max_gs_num / self.arena.N - 1.0, 0.0)
                else:
                    headroom = 0.25 if self.step_count < self.cfg.stop_split_at else 0.0
                x = ViewShardedGradients(self.arena.N, views_per_rank, self.device, self.pg, headroom=headroom,
                                         num_cameras=0 if self.camera_opt is None else self.camera_opt.num_cameras,
                                         bilagrid_row=0 if self.bilagrid is None else self.bilagrid.row)
            except Exception as e:  # noqa: BLE001  (no peer mappings / symmetric memory on this box)
                x, err = None, e
            ok = torch.tensor([0.0 if x is None else 1.0], device=self.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.pg)  # every rank takes the same path
            if float(ok.item()) < 1.0:
                if self.cfg.comm == "exchange":
                    raise RuntimeError(f"comm='exchange': symmetric memory is not available on every rank ({err})")
                self.comm, self._xg = "nccl", None
                return None
            self._xg = x
        if self.arena.grad.data_ptr() != x.grad.data_ptr():
            assert x.grad.numel() == self.arena.grad.numel()
            self.arena.grad = x.grad  # Adam reads the summed gradients straight from the symmetric arena
        if self.camera_opt is not None and self.camera_opt.grad.data_ptr() != x.pose.buf.data_ptr():
            self.camera_opt.use_grad_buffer(x.pose.buf)
        return x

    # -- collectives --------------------------------------------------------------------------
    def _all_reduce(self, t: Tensor, sym=None, op: str = "sum") -> None:
        """`t` <- its sum (op "max": maximum) over the ranks, in place.  `sym`: the comm.SymmetricArena whose buffer holds
        `t`; then that whole buffer is summed by this library's all-reduce kernel.  Otherwise torch.distributed, and with one
        rank nothing."""
        if sym is not None:
            assert op == "sum"
            sym.all_reduce_()
        elif self.world > 1:
            import torch.distributed as dist

            dist.all_reduce(t, op=dist.ReduceOp.SUM if op == "sum" else dist.ReduceOp.MAX, group=self.pg)

    def _all_reduce_sh_async(self, works: list, n0: int, n1: int) -> None:
        """Starts the all-reduce of the SH gradient rows of Gaussians [n0, n1) on the NCCL stream; appends (work, lo, hi)."""
        import torch.distributed as dist

        sh0 = self.arena.offsets["sh"][0]
        lo, hi = sh0 + 48 * n0, sh0 + 48 * n1
        works.append((dist.all_reduce(self.arena.grad[lo:hi], group=self.pg, async_op=True), lo, hi))

    def _gaussian_update(self, pipelined: bool, chunked_bwd: bool, works: list) -> None:
        """The Gaussian gradients summed over the ranks, then Adam.  The exchange has summed them inside the fused step, and
        one rank has nothing to sum.  `pipelined` ("nccl", one view per rank): the SH rows are reduced in `comm_chunks`
        async ranges (started by the chunked projection backward, else here) and each range is Adam-stepped as soon as its
        sum has landed, while the head (means | quats | scales | opacities) is reduced."""
        c, a = self.cfg, self.arena
        if not pipelined:
            if self.comm == "nccl":
                self._all_reduce(a.grad)
            self._mcmc_regularize()
            self.optimizer_step()
            return
        import torch.distributed as dist

        if not chunked_bwd:  # one projection-backward launch, then chunked reductions
            step_n = ((a.N + c.comm_chunks - 1) // c.comm_chunks + 3) // 4 * 4
            for n0 in range(0, a.N, step_n):
                self._all_reduce_sh_async(works, n0, min(n0 + step_n, a.N))
        sh0 = a.offsets["sh"][0]
        head = dist.all_reduce(a.grad[:sh0], group=self.pg, async_op=True)
        for w, lo, hi in works:  # Adam on each SH range as soon as its reduction has landed
            w.wait()
            self.optimizer_step(lo, hi)
        head.wait()
        self._mcmc_regularize()  # opacities and scales lie in [0, sh0)
        self.optimizer_step(0, sh0)

    def _mcmc_regularize(self) -> None:
        """MCMC: the regularisers' gradients, added once to the gradients summed over the ranks (identical on every rank)."""
        if self.mcmc is not None:
            self.mcmc.regularize(self.arena)

    # -- pieces that the tests drive directly ---------------------------------------------------
    def sh_degree_to_use(self) -> int:
        c = self.cfg
        return min(self.step_count // c.sh_degree_interval, c.sh_degree)

    def downscale_factor(self) -> int:
        """splatfacto `_get_downscale_factor` while training: the resolution divisor of the current step."""
        c = self.cfg
        return 2 ** max(c.num_downscales - self.step_count // c.resolution_schedule, 0)

    def accumulate_stats(self, absgrad_or_packed: Tensor, radii: Tensor, width: int, height: int, packed: bool,
                         n_cameras: Optional[int] = None) -> None:
        """DefaultStrategy._update_state for the local views.  gsplat scales the image-plane gradient by
        (W/2, H/2) * n_cameras of the batch the loss was averaged over; here that batch is the whole
        view batch of the step (all ranks), because the local gradients already carry 1/total_views."""
        if self.step_count >= self.cfg.stop_split_at:
            return
        C, N = radii.shape
        n_cameras = n_cameras or C
        if packed and self.backend == "cuda":
            from . import _lib

            lib = _lib.load()
            _lib.check(lib.qed_strategy_update(C, N, _lib.ptr(absgrad_or_packed), int(self.cfg.use_absgrad), _lib.ptr(radii), width, height,
                                               n_cameras, _lib.ptr(self.state.grad2d), _lib.ptr(self.state.count),
                                               _lib.ptr(self.state.radii), _lib.current_stream()), "qed_strategy_update")
            return
        if packed:
            rec = absgrad_or_packed.view(C, N, 12)
            g = rec[..., 2:4] if self.cfg.use_absgrad else rec[..., 0:2]
        else:
            g = absgrad_or_packed
        g = g * torch.tensor([width / 2.0 * n_cameras, height / 2.0 * n_cameras], device=g.device)
        sel = radii > 0
        norm = g.norm(dim=-1) * sel
        self.state.grad2d += norm.sum(0)
        self.state.count += sel.sum(0).to(torch.float32)
        r = (radii.to(torch.float32) / float(max(width, height))) * sel
        self.state.radii = torch.maximum(self.state.radii, r.max(dim=0).values)

    def optimizer_step(self, lo: int = 0, hi: Optional[int] = None) -> None:
        """Adam on arena elements [lo, hi) (default: everything).  Ranges must not split a Gaussian's SH row."""
        c, a = self.cfg, self.arena
        t = self.step_count + 1
        hi = a.param.numel() if hi is None else hi
        lrs = {"means": c.lr_means_at(self.step_count), "quats": c.lr_quats, "scales": c.lr_scales, "opacities": c.lr_opacities,
               "sh": c.lr_features_dc}
        if self.backend == "cuda":
            from . import _lib

            lib = _lib.load()
            if self._lr_dev is None or self._lr_dev[0] != (self.step_count, a.N):
                lr = torch.tensor([lrs[g] for g in GROUPS], device=self.device)
                lr_alt = torch.tensor([lrs["means"], lrs["quats"], lrs["scales"], lrs["opacities"], c.lr_features_rest], device=self.device)
                period = torch.tensor([0, 0, 0, 0, 48], dtype=torch.int32, device=self.device)
                split = torch.tensor([0, 0, 0, 0, 3], dtype=torch.int32, device=self.device)
                self._lr_dev = ((self.step_count, a.N), lr, lr_alt, period, split)
            _, lr, lr_alt, period, split = self._lr_dev
            sh0 = a.offsets["sh"][0]
            if lo >= sh0:
                # a range inside the SH block: one group starting at `lo` (multiple of 48 floats past sh0)
                assert (lo - sh0) % 48 == 0
                ends = torch.tensor([hi - lo], dtype=torch.int64, device=self.device)
                _lib.check(lib.qed_adam_arena(hi - lo, _lib.ptr(a.param[lo:hi]), _lib.ptr(a.grad[lo:hi]), _lib.ptr(a.exp_avg[lo:hi]),
                                              _lib.ptr(a.exp_avg_sq[lo:hi]), 1, _lib.ptr(ends), _lib.ptr(lr[4:]), _lib.ptr(lr_alt[4:]),
                                              _lib.ptr(period[4:]), _lib.ptr(split[4:]), c.adam_betas[0], c.adam_betas[1], c.adam_eps, t,
                                              _lib.current_stream()), "qed_adam_arena")
            else:
                assert lo == 0
                ends = torch.clamp(a.group_ends, max=hi)
                _lib.check(lib.qed_adam_arena(hi, _lib.ptr(a.param), _lib.ptr(a.grad), _lib.ptr(a.exp_avg), _lib.ptr(a.exp_avg_sq),
                                              len(GROUPS), _lib.ptr(ends), _lib.ptr(lr), _lib.ptr(lr_alt), _lib.ptr(period),
                                              _lib.ptr(split), c.adam_betas[0], c.adam_betas[1], c.adam_eps, t, _lib.current_stream()),
                           "qed_adam_arena")
        else:
            assert lo == 0 and hi == a.param.numel()
            adam_step_torch(a, lrs, c.lr_features_rest, c, t)

    def camera_opt_update(self, v_viewmats: Tensor, camera_ids: Tensor, camera_to_worlds: Tensor, exchange=None) -> None:
        """The camera optimizer's part of a step, after the backward: table gradient of the local views, its sum over the
        ranks (this library's all-reduce kernel with `exchange`, else torch.distributed), the regulariser (once, identically
        on every rank) and Adam on the table.  Replicas keep bit-identical tables."""
        camera_to_worlds, camera_ids = self.camera_opt.prepare(camera_to_worlds, camera_ids)
        self._camera_opt_update(v_viewmats, camera_ids, camera_to_worlds, exchange)

    def _camera_opt_update(self, v_viewmats: Tensor, camera_ids: Tensor, camera_to_worlds: Tensor, exchange) -> None:
        """camera_opt_update on inputs already passed through CameraPoseOptimizer.prepare."""
        cam = self.camera_opt
        cam._backward(v_viewmats, camera_ids, camera_to_worlds)
        self._all_reduce(cam.grad, None if exchange is None else exchange.pose)
        cam.regularize()
        cam.step(self.step_count)

    def _bilagrid_slots(self, C: int, exchange=None):
        """-> (buffer, rows [world*C, 12, L, Y, X], ids as floats [world*C], this rank's rows [C, ...]): views of the buffer the
        ranks sum, the exchange's symmetric one or else an ordinary tensor.  Slots of other ranks are zero."""
        bg, slots = self.bilagrid, self.world * C
        n = slots * (bg.row + 1)
        if exchange is not None:
            buf = exchange.bilagrid.buf
        else:
            if self._bg_buf is None or self._bg_buf.numel() < n:
                self._bg_buf = torch.zeros(n, device=self.device)
            buf = self._bg_buf
        if exchange is not None or self.world > 1:
            buf.zero_()
        buf = buf[:n]
        rows = buf[:slots * bg.row].view(slots, 12, bg.L, bg.Y, bg.X)
        return buf, rows, buf[slots * bg.row:], rows[self.rank * C:(self.rank + 1) * C]

    def _bilagrid_finish(self, C: int, ids: Tensor, buf: Tensor, rows: Tensor, ids_f: Tensor, exchange) -> None:
        """After the local rows are written: the ids into their slots, the sum over the ranks, TV (overwrites the dense
        gradient), every view's row added in global view order, Adam.  Replicas keep bit-identical grids."""
        bg = self.bilagrid
        if exchange is not None or self.world > 1:
            ids_f[self.rank * C:(self.rank + 1) * C].copy_(ids)
            # with the exchange: its whole symmetric buffer; floats past this batch's slots are zero
            self._all_reduce(buf, None if exchange is None else exchange.bilagrid)
            ids = ids_f.to(torch.int32)
        bg.regularize()
        bg.accumulate(ids, rows)
        bg.step(self.step_count)

    def bilagrid_update(self, v_grid_rows: Tensor, camera_ids: Tensor) -> None:
        """The bilateral grid's part of a step from this rank's per-view grid gradients v_grid_rows [C,12,L,Y,X] (what the
        fused step writes; they already carry 1 / total_views): sum over the ranks, TV, accumulate, Adam."""
        from .camera_opt import check_camera_ids

        C = v_grid_rows.shape[0]
        ids = check_camera_ids(camera_ids, C, self.bilagrid.num_grids, self.device)
        buf, rows, ids_f, mine = self._bilagrid_slots(C)
        mine.copy_(v_grid_rows)
        self._bilagrid_finish(C, ids, buf, rows, ids_f, None)

    def maybe_refine(self, step: int) -> Optional[Dict[str, int]]:
        """DefaultStrategy.step_post_backward schedule, called after the optimizer step of 0-based iteration
        `step` (nerfstudio passes its 0-based step; note gsplat resets opacities at step 0 too).
        strategy "mcmc": MCMCStrategy.step_post_backward with the means lr after the scheduler step -> {"n_relocated",
        "n_added", "n"} on refine steps, position noise on every step."""
        c = self.cfg
        if self.mcmc is not None:
            return self.mcmc.step_post_backward(self.arena, step, c.lr_means_at(step + 1))
        info = None
        if step >= c.stop_split_at:
            return None
        reset_every = c.reset_alpha_every * c.refine_every
        if step > c.warmup_length and step % c.refine_every == 0 and step % reset_every >= c.pause_refine_after_reset:
            # the accumulators of every rank are combined only now (SUM / MAX are associative)
            self._all_reduce(self.state.grad2d)
            self._all_reduce(self.state.count)
            self._all_reduce(self.state.radii, op="max")
            gen = torch.Generator().manual_seed(c.seed * 1_000_003 + step)
            info = refine_gaussians(self.arena, self.state, c, step, gen)
        if step % reset_every == 0:
            reset_opacities(self.arena, c)
        return info

    # -- the full step --------------------------------------------------------------------------
    @torch.no_grad()
    def step(self, viewmats: Optional[Tensor], Ks: Tensor, width: int, height: int, gt_rgb: Tensor, gt_depth: Tensor,
             background: Tensor, total_views: Optional[int] = None, mask: Optional[Tensor] = None, *,
             camera_to_worlds: Optional[Tensor] = None, camera_ids: Optional[Tensor] = None):
        """Local views [C_local,...]; `mask` = the batch's optional loss mask (model.py:93-97).
        With the camera optimizer on, `viewmats` is None and the views come as `camera_to_worlds` [C,3|4,4] (nerfstudio
        camera-to-world) and `camera_ids` [C] (rows of the pose table); the viewmats are those of the adjusted poses.
        Returns (loss[3] device tensor of the local views -- a fresh copy, safe to keep for logging --, refine info|None);
        the camera optimizer's regulariser is `camera_opt_loss`.
        With the bilateral grid on, `camera_ids` [C] (the training camera of each view, the same ids the camera optimizer
        uses) selects each view's grid; the grids' TV loss is `bilagrid_tv_loss`.
        With cfg.num_downscales > 0 the camera (Ks, width, height) and gt_rgb / gt_depth / mask are at full resolution, as
        nerfstudio's datamanager supplies them; a step whose `downscale_factor()` d is above 1 renders at the camera
        `rescaled_camera` builds and trains against the ground truth box-downscaled by d."""
        if self._fused is None:
            raise RuntimeError("rendering needs the CUDA library (backend='cuda'); there is no CPU fallback")
        c, a, cam, bg = self.cfg, self.arena, self.camera_opt, self.bilagrid
        if cam is not None:
            if viewmats is not None or camera_to_worlds is None or camera_ids is None:
                raise ValueError("camera optimizer on: pass viewmats=None with camera_to_worlds= and camera_ids=")
            camera_to_worlds, camera_ids = cam.prepare(camera_to_worlds, camera_ids)  # validated once per step
            viewmats = cam._viewmats(camera_to_worlds, camera_ids)
        elif camera_to_worlds is not None:
            raise ValueError("camera_to_worlds= needs cfg.camera_optimizer != 'off'")
        elif camera_ids is not None and bg is None:
            raise ValueError("camera_ids= needs cfg.camera_optimizer != 'off' or cfg.use_bilateral_grid")
        elif bg is not None:
            from .camera_opt import check_camera_ids

            if camera_ids is None:
                raise ValueError("bilateral grid on: pass camera_ids= (the training camera of each view)")
            camera_ids = check_camera_ids(camera_ids, viewmats.shape[0], bg.num_grids, self.device)
        C = viewmats.shape[0]
        # the resolution schedule: every rank derives the same factor from step_count
        d = self.downscale_factor()
        Ks, width, height = rescaled_camera(Ks, width, height, d)
        total = total_views or C * self.world
        xg = self._exchange_for(C) if self.comm == "exchange" else None  # may fall back to "nccl" (comm="auto", no symmetric memory)
        # "nccl" with one view per rank: the SH gradients are all-reduced and Adam-stepped in `comm_chunks` Gaussian ranges
        pipelined = self.comm == "nccl" and C == 1 and c.comm_chunks > 1
        # pose gradients need the projection backward in one launch: the pipelined path then chunks only the reductions
        chunked_bwd = pipelined and c.chunk_project_bwd and cam is None
        works = []  # (async all-reduce, lo, hi) of the SH ranges in flight
        if xg is not None:  # the projection backward writes into the symmetric arena; the fused step ends with the sum
            comm_args = dict(exchange=xg)
        elif chunked_bwd:  # SH rows of a finished Gaussian range: all-reduce them now while the next range computes
            comm_args = dict(grad_out=a.views(a.grad), n_chunks=c.comm_chunks,
                             on_chunk=lambda k, n0, n1: self._all_reduce_sh_async(works, n0, n1))
        else:
            comm_args = dict(grad_out=a.views(a.grad))
        # this rank's grid rows are written by the loss kernels of the fused step
        bl = None if bg is None else self._bilagrid_slots(C, xg)
        # the stored parameters go straight in: exp / sigmoid (model.py:269-271) and their chain rule run inside the
        # projection kernels, the gradients land in the arena
        pv = a.views(a.param)
        out = self._fused.step(pv["means"], pv["quats"], pv["scales"], pv["opacities"], pv["sh"], viewmats, Ks, width, height, self.sh_degree_to_use(),
                               gt_rgb, gt_depth, background, render_mode=c.render_mode, rgb_weight=1.0 - c.ssim_lambda,
                               depth_lambda=c.depth_lambda, grad_scale=C / float(total), rasterize_mode=c.rasterize_mode,
                               activations=3,  # ACT_LOG_SCALES | ACT_LOGIT_OPACITIES (pipeline.py / include/qed_splat.h)
                               mask=mask, depth_unit_scale=c.depth_unit_scale, ssim_lambda=c.ssim_lambda, pose_gradients=cam is not None,
                               bilateral_grid=None if bl is None else (bg.grids, camera_ids, bl[3]), gt_downscale=d, **comm_args)
        if self.mcmc is None:  # MCMC uses no gradient statistics
            self.accumulate_stats(out.packed_grads, out.radii, width, height, packed=True, n_cameras=total)
        self._gaussian_update(pipelined, chunked_bwd, works)
        if cam is not None:
            self._camera_opt_update(out.v_viewmats, camera_ids, camera_to_worlds, xg)
        if bg is not None:
            self._bilagrid_finish(C, camera_ids, *bl[:3], xg)
        loss = out.loss.clone()  # out.loss is a buffer the next step overwrites in place
        info = self.maybe_refine(self.step_count)
        self.step_count += 1
        return loss, info

    # -- evaluation ------------------------------------------------------------------------------
    @torch.no_grad()
    def evaluate(self, viewmats: Tensor, Ks: Tensor, width: int, height: int, gt_rgb: Tensor, gt_depth: Tensor, background: Tensor, *,
                 depth_tolerance: float = 0.1) -> Dict[str, Tensor]:
        """Renders this rank's held-out views as splatfacto renders outside training and scores them (metrics.image_metrics)
        -> {name: [world_size * C] float64 device tensor} for every name of metrics.METRIC_NAMES: the rows of every rank's views,
        rank-major (rank r's C views in slots [r C, (r + 1) C)), identical on every rank.  With world_size > 1 it is collective,
        and every rank must pass the same number C of views.

        The views are rendered at full resolution (whatever num_downscales and the step), from the poses as given (viewmats
        [C,4,4], e.g. get_viewmat(camera_to_worlds): the camera optimizer's table is not applied), without the bilateral grid,
        with sh_degree_to_use(), cfg.rasterize_mode and cfg.render_mode, composited on `background` [3] (splatfacto's fixed
        colour when training uses a random one).  Ks [C,3,3]; gt_rgb / gt_depth at full resolution as for step(), depth in
        cfg.depth_unit_scale when raw uint16.  At most EVAL_CHUNK_VIEWS views are rendered at a time.
        No training state changes: the next step() computes exactly what it would have computed without this call, and costs
        what it would have cost.  The views are rendered by a FusedSplatStep of their own, dropped when the call returns: the
        step's buffers and intersection-list capacity stay sized for the training views."""
        if self._fused is None:
            raise RuntimeError("rendering needs the CUDA library (backend='cuda'); there is no CPU fallback")
        from .metrics import METRIC_NAMES, metric_rows
        from .pipeline import FusedSplatStep

        c, a = self.cfg, self.arena
        C = viewmats.shape[0]
        if Ks.shape[0] != C or gt_rgb.shape[0] != C or gt_depth.shape[0] != C:
            raise ValueError("viewmats, Ks, gt_rgb and gt_depth must hold the same views")
        rows = torch.zeros(self.world * C, len(METRIC_NAMES), dtype=torch.float64, device=self.device)
        pv = a.views(a.param)
        fused = FusedSplatStep(self.device)
        for c0 in range(0, C, EVAL_CHUNK_VIEWS):
            c1 = min(c0 + EVAL_CHUNK_VIEWS, C)
            render, alphas = fused.forward(pv["means"], pv["quats"], pv["scales"], pv["opacities"], pv["sh"], viewmats[c0:c1].contiguous(),
                                           Ks[c0:c1].contiguous(), width, height, self.sh_degree_to_use(), render_mode=c.render_mode,
                                           rasterize_mode=c.rasterize_mode, activations=3)  # ACT_LOG_SCALES | ACT_LOGIT_OPACITIES
            slot = self.rank * C
            metric_rows(render, alphas, gt_rgb[c0:c1], gt_depth[c0:c1], background, depth_unit_scale=c.depth_unit_scale,
                        depth_tolerance=depth_tolerance, out=rows[slot + c0:slot + c1])
        self._all_reduce(rows)  # every slot has one non-zero contributor: the sum is exact, the same bits on every rank
        return {name: rows[:, k] for k, name in enumerate(METRIC_NAMES)}

    # -- checkpoints -----------------------------------------------------------------------------
    def _gather_rows(self, t: Tensor) -> Tensor:
        """[world, N] on the CPU: row r = rank r's `t` (a collective with world_size > 1)."""
        if self.world <= 1:
            return _owned_cpu(t)[None]
        import torch.distributed as dist

        rows = [torch.empty_like(t) for _ in range(self.world)]
        dist.all_gather(rows, t.contiguous(), group=self.pg)
        return _owned_cpu(torch.stack(rows))

    @torch.no_grad()
    def state_dict(self) -> Dict[str, Any]:
        """Everything the run needs to continue (DESIGN.md section 0 lists it), as plain Python values and CPU tensors that own
        their storage, so `torch.save` writes exactly them and `torch.load(weights_only=True)` reads them back.  Call it
        between steps; with world_size > 1 it is collective (the strategy statistics of every rank are gathered) and every
        rank gets the same dict.  The live trainer is left as it was.

        Keys: format_version, config (dataclasses.asdict), step, num_cameras, world_size, gauss_params / exp_avg / exp_avg_sq
        (splatfacto's names and shapes: means, scales (log), quats (as stored), features_dc, features_rest, opacities (logit)
        [N,1]), strategy_state (strategy "default": grad2d, count, radii [world_size, N], row r from rank r),
        camera_optimizer (pose_adjustment, exp_avg, exp_avg_sq [num_cameras, 6]) and bil_grids (grids, exp_avg, exp_avg_sq
        [num_cameras, 12, L, Y, X]) when those are on."""
        a = self.arena
        out: Dict[str, Any] = dict(format_version=CHECKPOINT_FORMAT_VERSION, config=dataclasses.asdict(self.cfg), step=int(self.step_count),
                                   num_cameras=self.num_cameras, world_size=int(self.world))
        for key, buf in (("gauss_params", a.param), ("exp_avg", a.exp_avg), ("exp_avg_sq", a.exp_avg_sq)):
            out[key] = {k: _owned_cpu(v) for k, v in a.splatfacto_views(buf).items()}
        if self.mcmc is None:
            out["strategy_state"] = {k: self._gather_rows(getattr(self.state, k)) for k in STRATEGY_STATS}
        if self.camera_opt is not None:
            n = self.camera_opt.num_cameras * 6
            out["camera_optimizer"] = {k: _owned_cpu(getattr(self.camera_opt, b)[:n].view(-1, 6))
                                       for k, b in (("pose_adjustment", "param"), ("exp_avg", "exp_avg"), ("exp_avg_sq", "exp_avg_sq"))}
        if self.bilagrid is not None:
            shape = self.bilagrid.grids.shape
            out["bil_grids"] = {k: _owned_cpu(getattr(self.bilagrid, b).view(shape))
                                for k, b in (("grids", "param"), ("exp_avg", "exp_avg"), ("exp_avg_sq", "exp_avg_sq"))}
        return out

    @classmethod
    @torch.no_grad()
    def from_state_dict(cls, state: Dict[str, Any], cfg: Optional[TrainConfig] = None, *, rank: int = 0, world_size: int = 1,
                        process_group=None, backend: str = "cuda", device=None) -> "SplatTrainer":
        """A trainer that continues the run `state` (from `state_dict()`, possibly through torch.save / torch.load) at step
        state["step"]: the next `step()` is the one the saved run would have taken.

        `cfg=None` uses the saved configuration; a `cfg` passed in may change hyper-parameters (max_steps, learning rates,
        comm, ...) but not the layout fields (LAYOUT_FIELDS: ValueError naming the field).  ValueError also for an unknown
        format_version, a tensor whose shape disagrees with N, num_cameras or the grid shape, and an MCMC state with more
        than cfg.max_gs_num Gaussians.

        Strategy statistics ("default"): at the saved world size rank r takes row r, so the run continues exactly.  At another
        world size rank 0 takes the rows' sum (radii: their maximum) and the other ranks zeros; the next refine step reduces
        them over the ranks to the same totals (grad2d up to the float summation order).

        Nothing else needs loading: the multi-GPU exchange buffers are built by the first `step()` as for a new trainer.
        `device`: default the current CUDA device with backend "cuda", the CPU with backend "torch" (which opens a
        checkpoint of a CUDA run on a machine without a GPU)."""
        version = state.get("format_version") if isinstance(state, dict) else None
        if version != CHECKPOINT_FORMAT_VERSION:
            raise ValueError(f"state format_version {version!r} unknown: this trainer reads version {CHECKPOINT_FORMAT_VERSION}")
        saved = TrainConfig(**state["config"])
        if cfg is None:
            cfg = saved
        for f in LAYOUT_FIELDS:
            old, new = getattr(saved, f), getattr(cfg, f)
            if f == "bilateral_grid_shape":
                if not saved.use_bilateral_grid:
                    continue
                old, new = tuple(old), tuple(new)
            if old != new:
                raise ValueError(f"cfg.{f} = {new!r} would change the state's layout (saved with {old!r})")
        cfg.validate()
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if backend == "cuda" else torch.device("cpu")
        device = torch.device(device)
        # shapes, before anything is allocated
        num_cameras = int(state["num_cameras"])
        saved_world = int(state["world_size"])
        gp = _section(state, "gauss_params")
        if not isinstance(gp.get("means"), Tensor) or gp["means"].dim() != 2:
            raise ValueError("state gauss_params['means']: expected a tensor of shape (N, 3)")
        N = gp["means"].shape[0]
        for key in ("gauss_params", "exp_avg", "exp_avg_sq"):
            sec = _section(state, key)
            for k, shape in SPLATFACTO_SHAPES.items():
                _check_shape(f"{key}[{k!r}]", sec.get(k), (N, *shape))
        if cfg.strategy == "mcmc" and N > cfg.max_gs_num:
            raise ValueError(f"state holds {N} Gaussians, more than cfg.max_gs_num = {cfg.max_gs_num} (strategy 'mcmc')")
        if cfg.strategy == "default":
            sec = _section(state, "strategy_state")
            for k in STRATEGY_STATS:
                _check_shape(f"strategy_state[{k!r}]", sec.get(k), (saved_world, N))
        tables = []
        if cfg.camera_optimizer != "off":
            tables.append(("camera_optimizer", ("pose_adjustment", "exp_avg", "exp_avg_sq"), (num_cameras, 6)))
        if cfg.use_bilateral_grid:
            X, Y, L = cfg.bilateral_grid_shape
            tables.append(("bil_grids", ("grids", "exp_avg", "exp_avg_sq"), (num_cameras, 12, L, Y, X)))
        for key, names, shape in tables:
            sec = _section(state, key)
            for k in names:
                _check_shape(f"{key}[{k!r}]", sec.get(k), shape)

        sh = torch.cat([gp["features_dc"][:, None, :], gp["features_rest"]], dim=1)
        tr = cls(gp["means"].to(device), gp["quats"].to(device), gp["scales"].to(device), gp["opacities"].reshape(N).to(device), sh.to(device),
                 cfg=cfg, rank=rank, world_size=world_size, process_group=process_group, backend=backend, num_cameras=num_cameras)
        a = tr.arena
        for key, buf in (("exp_avg", a.exp_avg), ("exp_avg_sq", a.exp_avg_sq)):
            for k, v in a.splatfacto_views(buf).items():
                v.copy_(state[key][k])
        tr.step_count = int(state["step"])
        if tr.mcmc is None:
            for k in STRATEGY_STATS:
                rows = state["strategy_state"][k]
                if saved_world == world_size:
                    v = rows[rank]
                elif rank == 0:
                    v = rows.amax(0) if k == "radii" else rows.sum(0)
                else:
                    continue  # zeros, as built
                getattr(tr.state, k).copy_(v)
        if tr.camera_opt is not None:
            sec, n = state["camera_optimizer"], num_cameras * 6
            for k, b in (("pose_adjustment", "param"), ("exp_avg", "exp_avg"), ("exp_avg_sq", "exp_avg_sq")):
                getattr(tr.camera_opt, b)[:n].copy_(sec[k].reshape(-1))
        if tr.bilagrid is not None:
            sec = state["bil_grids"]
            for k, b in (("grids", "param"), ("exp_avg", "exp_avg"), ("exp_avg_sq", "exp_avg_sq")):
                getattr(tr.bilagrid, b).copy_(sec[k].reshape(-1))
        return tr
