"""`depth_supervised_loss` — the tail of `QEDSplatterModel.get_outputs` and its `get_loss_dict` as ONE call.

Replaces, for a render produced by `rasterization(..., render_mode="RGB+D" | "RGB+ED")`:
  * /root/reference/qed_splatter/model.py:295-306 — background composite, clamp to [0,1], depth fill of
    never-hit pixels with the maximum rendered depth;
  * /root/reference/qed_splatter/model.py:73-118 (+ splatfacto's RGB loss it inherits) —
    rgb_weight * L1 + ssim_lambda * (1 - SSIM) + depth_lambda * masked depth-L1 (22-38: `depth_loss`),
with a torch.autograd.Function over the C-ABI `qed_loss_fwd_bwd`: the forward launch computes the loss AND its
gradient with respect to (render, alphas); backward only scales it.  The dozen element-wise torch kernels of the
reference formulation (each a full pass over the image) become four launches.

Semantics are per camera (one camera = one reference step: its own depth fill and valid-pixel count) and the
mean over cameras; for the reference's single-camera steps that is the reference's number.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import check, current_stream, ptr


class _DepthSupervisedLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, render: Tensor, alphas: Tensor, gt_rgb: Tensor, gt_depth: Tensor, background: Tensor, rgb_weight: float,
                depth_lambda: float, ssim_lambda: float, mask: Optional[Tensor], depth_unit_scale: float) -> Tuple[Tensor, Tensor, Tensor]:
        # raw pointers cross the C-ABI: a CPU tensor (e.g. nerfstudio's image cache under cache_images="cpu") or one
        # on another device would hand the kernel a pointer it cannot read -> raise here instead
        _lib.require_cuda(render, alphas, gt_rgb, gt_depth, background, mask)
        _lib.require_dtype(gt_rgb, (torch.float32, torch.uint8), "gt_rgb")
        _lib.require_dtype(gt_depth, (torch.float32, torch.uint16, torch.int16), "gt_depth")
        _lib.require_dtype(background, (torch.float32,), "background")
        _lib.require_dtype(render, (torch.float32,), "render")
        _lib.require_dtype(alphas, (torch.float32,), "alphas")
        _lib.require_dtype(mask, (torch.float32, torch.uint8, torch.bool), "mask")
        C, H, W, D = render.shape
        if D != 4:
            raise ValueError("depth_supervised_loss needs a 4-channel render (render_mode 'RGB+D' or 'RGB+ED')")
        if gt_rgb.shape != (C, H, W, 3) or gt_depth.numel() != C * H * W or alphas.numel() != C * H * W or background.numel() != 3:
            raise ValueError("shapes: render [C,H,W,4], alphas [C,H,W,1], gt_rgb [C,H,W,3], gt_depth [C,H,W(,1)], background [3]")
        if mask is not None and mask.numel() != C * H * W:
            raise ValueError("mask must be [C,H,W] or [C,H,W,1]")
        lib = _lib.load()
        dev = render.device
        r = render.detach().contiguous()
        a = alphas.detach().contiguous()
        rgb = gt_rgb.detach().contiguous()  # float32 in [0,1], or the uint8 image cache (converted in-kernel, u8 / 255)
        dep = gt_depth.detach().contiguous()
        bg = background.detach().contiguous()
        mk = None
        if mask is not None:
            mk = mask.detach().contiguous()
            if mk.dtype == torch.bool:
                mk = mk.view(torch.uint8)
        stats = torch.zeros(C * 8, dtype=torch.float64, device=dev)
        loss = torch.empty(3, device=dev)
        v_render = torch.empty_like(r)
        v_alphas = torch.empty_like(a)
        ws_bytes = lib.qed_loss_workspace_bytes(C, W, H, float(ssim_lambda))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev) if ws_bytes else None
        check(lib.qed_loss_fwd_bwd(C, W, H, ptr(r), ptr(a), ptr(rgb), int(rgb.dtype == torch.uint8), ptr(dep), int(dep.dtype != torch.float32), float(depth_unit_scale),
                                   ptr(mk), int(mk is not None and mk.dtype == torch.uint8), ptr(bg), float(rgb_weight), float(depth_lambda),
                                   float(ssim_lambda), 1.0, ptr(stats), ptr(loss), ptr(v_render), ptr(v_alphas), ptr(ws), ws_bytes,
                                   current_stream()), "qed_loss_fwd_bwd")
        ctx.save_for_backward(v_render, v_alphas)
        total, l_rgb, l_depth = loss.unbind(0)
        ctx.mark_non_differentiable(l_rgb, l_depth)
        return total, l_rgb, l_depth

    @staticmethod
    def backward(ctx, g_total, g_rgb, g_depth):
        v_render, v_alphas = ctx.saved_tensors
        # d(total)/d(render, alphas) was computed by the forward launch; the components are reported for logging only
        return v_render * g_total, v_alphas * g_total, None, None, None, None, None, None, None, None


def _check_grids(grids: Tensor) -> None:
    from .bilateral_grid import check_grid_shape

    _lib.require_dtype(grids, (torch.float32,), "bilateral_grids")
    if grids.dim() != 5 or grids.shape[1] != 12:
        raise ValueError("bilateral_grids must be [G,12,L,Y,X]")
    G, _, L, Y, X = grids.shape
    check_grid_shape(X, Y, L, G)


class _DepthSupervisedLossBilagrid(torch.autograd.Function):
    """The loss with the bilateral grid of each view applied to its clamped composite: one `qed_loss_fwd_bwd_bilagrid` launch
    chain computes the loss, d loss / d (render, alphas) and the per-view grid rows; `qed_bilagrid_accumulate` sums the rows
    into the [G,12,L,Y,X] gradient in view order."""

    @staticmethod
    def forward(ctx, render, alphas, grids, grid_ids, gt_rgb, gt_depth, background, rgb_weight, depth_lambda, ssim_lambda, mask, depth_unit_scale):
        _lib.require_cuda(render, alphas, gt_rgb, gt_depth, background, mask, grids)
        _lib.require_dtype(gt_rgb, (torch.float32, torch.uint8), "gt_rgb")
        _lib.require_dtype(gt_depth, (torch.float32, torch.uint16, torch.int16), "gt_depth")
        _lib.require_dtype(background, (torch.float32,), "background")
        _lib.require_dtype(render, (torch.float32,), "render")
        _lib.require_dtype(alphas, (torch.float32,), "alphas")
        _lib.require_dtype(mask, (torch.float32, torch.uint8, torch.bool), "mask")
        _check_grids(grids)
        C, H, W, D = render.shape
        if D != 4:
            raise ValueError("depth_supervised_loss needs a 4-channel render (render_mode 'RGB+D' or 'RGB+ED')")
        if gt_rgb.shape != (C, H, W, 3) or gt_depth.numel() != C * H * W or alphas.numel() != C * H * W or background.numel() != 3:
            raise ValueError("shapes: render [C,H,W,4], alphas [C,H,W,1], gt_rgb [C,H,W,3], gt_depth [C,H,W(,1)], background [3]")
        if mask is not None and mask.numel() != C * H * W:
            raise ValueError("mask must be [C,H,W] or [C,H,W,1]")
        from .camera_opt import check_camera_ids

        G, _, L, Y, X = grids.shape
        ids = check_camera_ids(grid_ids, C, G, render.device)
        lib = _lib.load()
        dev = render.device
        r = render.detach().contiguous()
        a = alphas.detach().contiguous()
        g = grids.detach().contiguous()
        rgb = gt_rgb.detach().contiguous()
        dep = gt_depth.detach().contiguous()
        bg = background.detach().contiguous()
        mk = None
        if mask is not None:
            mk = mask.detach().contiguous()
            if mk.dtype == torch.bool:
                mk = mk.view(torch.uint8)
        stats = torch.zeros(C * 8, dtype=torch.float64, device=dev)
        loss = torch.empty(3, device=dev)
        v_render = torch.empty_like(r)
        v_alphas = torch.empty_like(a)
        v_rows = torch.empty(C, 12, L, Y, X, device=dev)
        ws_bytes = lib.qed_loss_bilagrid_workspace_bytes(C, W, H, float(ssim_lambda))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(lib.qed_loss_fwd_bwd_bilagrid(C, W, H, ptr(r), ptr(a), ptr(rgb), int(rgb.dtype == torch.uint8), ptr(dep), int(dep.dtype != torch.float32),
                                            float(depth_unit_scale), ptr(mk), int(mk is not None and mk.dtype == torch.uint8), ptr(bg), float(rgb_weight),
                                            float(depth_lambda), float(ssim_lambda), 1.0, ptr(stats), ptr(loss), ptr(v_render), ptr(v_alphas), ptr(g),
                                            ptr(ids), G, X, Y, L, ptr(v_rows), ptr(ws), ws_bytes, current_stream()), "qed_loss_fwd_bwd_bilagrid")
        v_grids = torch.zeros_like(g)
        check(lib.qed_bilagrid_accumulate(C, ptr(ids), ptr(v_rows), G, X, Y, L, ptr(v_grids), current_stream()), "qed_bilagrid_accumulate")
        ctx.save_for_backward(v_render, v_alphas, v_grids)
        total, l_rgb, l_depth = loss.unbind(0)
        ctx.mark_non_differentiable(l_rgb, l_depth)
        return total, l_rgb, l_depth

    @staticmethod
    def backward(ctx, g_total, g_rgb, g_depth):
        v_render, v_alphas, v_grids = ctx.saved_tensors
        return v_render * g_total, v_alphas * g_total, v_grids * g_total, None, None, None, None, None, None, None, None, None


class _BilateralGridTV(torch.autograd.Function):
    @staticmethod
    def forward(ctx, grids: Tensor, weight: float) -> Tensor:
        _lib.require_cuda(grids)
        _check_grids(grids)
        G, _, L, Y, X = grids.shape
        lib = _lib.load()
        g = grids.detach().contiguous()
        v = torch.empty_like(g)
        partials = torch.empty(G, dtype=torch.float64, device=g.device)
        loss = torch.empty(1, device=g.device)
        check(lib.qed_bilagrid_tv(G, X, Y, L, ptr(g), float(weight), ptr(v), ptr(partials), ptr(loss), current_stream()), "qed_bilagrid_tv")
        ctx.save_for_backward(v)
        return loss[0]

    @staticmethod
    def backward(ctx, g_out):
        (v,) = ctx.saved_tensors
        return v * g_out, None


def bilateral_grid_tv_loss(grids: Tensor, weight: float = 10.0) -> Tensor:
    """Splatfacto's total-variation regulariser of the bilateral grids [G,12,L,Y,X] (added once per training step):
    weight / G * sum over the L, Y and X axes of the mean squared difference of neighbouring cells of one grid.
    A 0-dim tensor carrying its gradient to `grids` (one launch computes both)."""
    return _BilateralGridTV.apply(grids, weight)


def depth_supervised_loss(render: Tensor, alphas: Tensor, gt_rgb: Tensor, gt_depth: Tensor, background: Tensor, rgb_weight: float = 0.8,
                          depth_lambda: float = 0.2, ssim_lambda: float = 0.0, mask: Optional[Tensor] = None,
                          depth_unit_scale: float = 0.001, bilateral_grids: Optional[Tensor] = None,
                          grid_ids: Optional[Tensor] = None, gt_downscale: int = 1) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (total, rgb_term, depth_term), 0-dim tensors; `total` carries the gradient to `render` and `alphas`.

    render [C,H,W,4] (RGB + depth; expected depth for 'RGB+ED'), alphas [C,H,W,1], gt_rgb [C,H,W,3] float in [0,1] or uint8
    (nerfstudio's image cache, config.py:37; converted as splatfacto's `image.float() / 255.0` inside the kernels),
    gt_depth [C,H,W] or [C,H,W,1] (<= 0 or non-finite = no supervision): float32 metres, or the raw uint16 sensor image
    (torch.uint16, or its bits as torch.int16), converted in-kernel with `depth_unit_scale` (qed_splatter/dataparser.py:15:
    0.001, times the dataparser's scene scale) as nerfstudio's depth loader does; background [3]; mask [C,H,W(,1)] float32 / uint8 /
    bool or None = `batch["mask"]`: rendered and ground-truth depth are multiplied by it before the validity test
    (model.py:93-97), predicted and ground-truth RGB before L1 / SSIM (splatfacto's parent loss).  All tensors must be
    on the render's CUDA device (CPU tensors raise; copy nerfstudio's CPU image cache explicitly).
    total = rgb_weight * mean|clamp(rgb + (1 - alpha) bg, 0, 1) - gt| + ssim_lambda * (1 - SSIM) + depth_lambda *
    mean_valid|depth_filled - gt_depth|  (qed-splatter: depth_lambda = 0.2; splatfacto: rgb_weight = 0.8, ssim_lambda = 0.2).

    bilateral_grids [G,12,L,Y,X] float32 (splatfacto's `bil_grids.grids`, may require grad) with grid_ids [C] (int32/int64,
    the training image of each view): the clamped composite of every view goes through its grid's affine colour transform
    (nerfstudio lib_bilagrid `slice`) before the mask, L1 and SSIM, as splatfacto does for training views; the depth term is
    unchanged.  `total` then carries the gradient to the grids too.  Supported grid shapes: 2 <= X, Y <= 1024, 2 <= L <= 16.

    gt_downscale d > 1 (splatfacto's resolution schedule, `_get_downscale_factor()`): render / alphas are [C,h,w,...] at the
    rescaled camera and gt_rgb / gt_depth / mask are at full resolution [C,H,W,...] with H // d == h and W // d == w; they
    are box-downscaled first as splatfacto's `_downscale_if_required` does (data_side.downscale_ground_truth, one launch).
    """
    if (bilateral_grids is None) != (grid_ids is None):
        raise ValueError("bilateral_grids and grid_ids go together")
    if gt_downscale != 1:
        from .data_side import downscale_ground_truth, downscaled_size

        if render.dim() != 4 or gt_rgb.dim() != 4:
            raise ValueError("gt_downscale: render [C,h,w,4] and full-resolution gt_rgb [C,H,W,3] expected")
        size = downscaled_size(gt_rgb.shape[2], gt_rgb.shape[1], gt_downscale)
        if size != (render.shape[2], render.shape[1]) or gt_rgb.shape[0] != render.shape[0]:
            raise ValueError(f"gt_downscale={gt_downscale}: {gt_rgb.shape[2]}x{gt_rgb.shape[1]} ground truth downscales to {size[0]}x{size[1]}, "
                             f"the render is {render.shape[2]}x{render.shape[1]}")
        gt_rgb, gt_depth, mask = downscale_ground_truth(gt_rgb, gt_depth, mask, gt_downscale, depth_unit_scale)
    if bilateral_grids is not None:
        return _DepthSupervisedLossBilagrid.apply(render, alphas, bilateral_grids, grid_ids, gt_rgb, gt_depth, background, rgb_weight, depth_lambda,
                                                  ssim_lambda, mask, depth_unit_scale)
    total, l_rgb, l_depth = _DepthSupervisedLoss.apply(render, alphas, gt_rgb, gt_depth, background, rgb_weight, depth_lambda, ssim_lambda, mask, depth_unit_scale)
    return total, l_rgb, l_depth
