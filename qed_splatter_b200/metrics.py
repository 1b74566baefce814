"""Held-out evaluation metrics: what nerfstudio's eval reports for qed-splatter (`QEDSplatterModel.get_metrics_dict`,
metrics.py:83-156), computed by one C-ABI call (`qed_eval_metrics`, csrc/metrics.cu) per batch of views.

  * psnr, ssim, rgb_mse: torchmetrics' PeakSignalNoiseRatio(data_range=1.0) and StructuralSimilarityIndexMeasure(data_range=1.0)
    on one image (the SSIM is the loss's: 11x11 Gaussian window, sigma 1.5, valid windows);
  * abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3 over the pixels whose ground-truth depth is finite and > depth_tolerance,
    and n_depth, their number (qed-splatter's DepthMetrics, restated from the dn-splatter code it follows).

LPIPS is not computed: it needs AlexNet / VGG weights, which this package neither ships nor downloads.
"""
from __future__ import annotations

import math
from typing import Dict

import torch
from torch import Tensor

from . import _lib
from ._lib import check, current_stream, ptr

METRIC_NAMES = ("psnr", "ssim", "rgb_mse", "abs_rel", "sq_rel", "rmse", "rmse_log", "a1", "a2", "a3", "n_depth")  # QED_EVAL_METRICS columns
DEPTH_METRICS = METRIC_NAMES[3:10]


def _require(t: Tensor, dtypes, what: str) -> None:
    if t.dtype not in dtypes:
        raise ValueError(f"{what}: expected {' or '.join(str(d) for d in dtypes)}, got {t.dtype}")


def metric_rows(render: Tensor, alphas: Tensor, gt_rgb: Tensor, gt_depth: Tensor, background: Tensor, *, depth_unit_scale: float = 0.001,
                depth_tolerance: float = 0.1, out: Tensor = None) -> Tensor:
    """-> [C, len(METRIC_NAMES)] float64 device tensor, one row per view (`out`, a contiguous tensor of that shape, when given).
    Arguments as for `image_metrics`."""
    _require(render, (torch.float32,), "render")
    _require(alphas, (torch.float32,), "alphas")
    _require(gt_rgb, (torch.float32, torch.uint8), "gt_rgb")
    _require(gt_depth, (torch.float32, torch.uint16, torch.int16), "gt_depth")
    _require(background, (torch.float32,), "background")
    if render.dim() != 4 or render.shape[-1] != 4:
        raise ValueError("image_metrics needs a 4-channel render [C,H,W,4] (render_mode 'RGB+D' or 'RGB+ED')")
    C, H, W, _ = render.shape
    if (gt_rgb.shape != (C, H, W, 3) or alphas.shape not in ((C, H, W), (C, H, W, 1)) or gt_depth.shape not in ((C, H, W), (C, H, W, 1))
            or background.numel() != 3):
        raise ValueError("shapes: render [C,H,W,4], alphas [C,H,W(,1)], gt_rgb [C,H,W,3], gt_depth [C,H,W(,1)], background [3]")
    if W <= 10 or H <= 10:
        raise ValueError(f"SSIM's 11x11 window needs width and height > 10, got {W}x{H}")
    _lib.require_cuda(render, alphas, gt_rgb, gt_depth, background, out)
    if out is None:
        out = torch.empty(C, len(METRIC_NAMES), dtype=torch.float64, device=render.device)
    elif out.shape != (C, len(METRIC_NAMES)) or out.dtype != torch.float64 or not out.is_contiguous():
        raise ValueError(f"out: a contiguous float64 [{C}, {len(METRIC_NAMES)}] tensor expected")
    lib = _lib.load()
    r, a, rgb, dep, bg = (t.detach().contiguous() for t in (render, alphas, gt_rgb, gt_depth, background))
    ws_bytes = lib.qed_eval_metrics_workspace_bytes(C, W, H)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=r.device)
    check(lib.qed_eval_metrics(C, W, H, ptr(r), ptr(a), ptr(rgb), int(rgb.dtype == torch.uint8), ptr(dep), int(dep.dtype != torch.float32),
                               float(depth_unit_scale), ptr(bg), float(depth_tolerance), ptr(out), ptr(ws), ws_bytes, current_stream()),
          "qed_eval_metrics")
    return out


def image_metrics(render: Tensor, alphas: Tensor, gt_rgb: Tensor, gt_depth: Tensor, background: Tensor, *, depth_unit_scale: float = 0.001,
                  depth_tolerance: float = 0.1) -> Dict[str, Tensor]:
    """Per-view metrics of C rendered views -> {name: [C] float64 device tensor} for every name of METRIC_NAMES; nothing is
    read back to the host.

    render [C,H,W,4] (RGB + depth, as `rasterization(..., render_mode="RGB+D" | "RGB+ED")` returns it), alphas [C,H,W(,1)],
    gt_rgb [C,H,W,3] float32 in [0,1] or uint8 (u8 / 255), gt_depth [C,H,W(,1)] float32 metres or raw uint16 (its bits as
    int16 too) times depth_unit_scale, background [3].  The prediction is the one the loss sees: clamp(rgb + (1 - alpha) bg,
    0, 1), and the depth channel where alpha > 0, else the view's maximum rendered depth (model.py:295-306).
    psnr = 10 log10(1 / rgb_mse) (+inf for a perfect image); the depth metrics are NaN for a view with n_depth = 0.
    A CPU tensor raises RuntimeError; a dtype or shape mismatch, a render without the depth channel or an image of width or
    height <= 10 raises ValueError."""
    rows = metric_rows(render, alphas, gt_rgb, gt_depth, background, depth_unit_scale=depth_unit_scale, depth_tolerance=depth_tolerance)
    return {name: rows[:, k] for k, name in enumerate(METRIC_NAMES)}


def summarize(per_view: Dict[str, Tensor]) -> Dict[str, float]:
    """The eval set's averages (one host read), as nerfstudio's `get_average_eval_image_metrics` averages per-image values:
    psnr, ssim and rgb_mse over all views; the depth metrics over the views with n_depth > 0 only (NaN when there is none),
    whose number is n_views_depth -- where nerfstudio's plain mean would be NaN as soon as one view has no valid depth.
    Also n_views."""
    t = torch.stack([per_view[name].to(torch.float64) for name in METRIC_NAMES]).cpu()
    has_depth = t[METRIC_NAMES.index("n_depth")] > 0
    n_depth_views = int(has_depth.sum())
    out: Dict[str, float] = {}
    for k, name in enumerate(METRIC_NAMES[:3]):
        out[name] = float(t[k].mean())
    for name in DEPTH_METRICS:
        out[name] = float(t[METRIC_NAMES.index(name)][has_depth].mean()) if n_depth_views else math.nan
    out["n_views"] = int(t.shape[1])
    out["n_views_depth"] = n_depth_views
    return out
