"""Float64 restatement of the held-out metrics (qed_eval_metrics, qed_splatter_b200.metrics) for the tests.

Inputs are converted as the kernels convert them (u8 * float32(1/255), float32(float64(u16) * depth_unit_scale)); the
prediction is oracle.composite_and_fill's, except that the fill value starts at 0 as the loss's does (the depth channel is
>= 0, so this is the same value).  Everything after that is float64: torchmetrics' PSNR on one image, the loss's SSIM
(oracle.ssim, valid windows), and qed-splatter's DepthMetrics over the pixels with finite ground truth > tolerance."""
from __future__ import annotations

import numpy as np
import torch

import oracle

NAMES = ("psnr", "ssim", "rgb_mse", "abs_rel", "sq_rel", "rmse", "rmse_log", "a1", "a2", "a3", "n_depth")


def gt_rgb_f32(gt_rgb: torch.Tensor) -> torch.Tensor:
    gt_rgb = gt_rgb.cpu()
    if gt_rgb.dtype == torch.uint8:
        return gt_rgb.to(torch.float32) * np.float32(1.0 / 255.0)
    return gt_rgb.to(torch.float32)


def gt_depth_f32(gt_depth: torch.Tensor, depth_unit_scale: float) -> np.ndarray:
    gt_depth = gt_depth.cpu()
    if gt_depth.dtype in (torch.int16, torch.uint16):
        raw = gt_depth.view(torch.int16).numpy().view(np.uint16)
        return (raw.astype(np.float64) * depth_unit_scale).astype(np.float32)
    return gt_depth.to(torch.float32).numpy()


def depth_metrics(d: np.ndarray, g: np.ndarray, tolerance: float = 0.1) -> np.ndarray:
    """[abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3, n] over the pixels whose g is finite and > tolerance (float32 compare),
    in float64; NaN for the seven means when there is none, non-finite values propagate."""
    g32 = np.asarray(g, np.float32).ravel()
    valid = np.isfinite(g32) & (g32 > np.float32(tolerance))
    g64 = g32[valid].astype(np.float64)
    d64 = np.asarray(d, np.float32).ravel()[valid].astype(np.float64)
    n = float(valid.sum())
    with np.errstate(all="ignore"):
        diff = g64 - d64
        t = np.maximum(g64 / d64, d64 / g64)
        lg = np.log(g64) - np.log(d64)
        sums = [np.abs(diff) / g64, diff * diff / g64, diff * diff, lg * lg, t < 1.25, t < 1.25 ** 2, t < 1.25 ** 3]
        m = [float(np.sum(s)) / n if n else float("nan") for s in sums]
        m[2], m[3] = np.sqrt(m[2]), np.sqrt(m[3])
    return np.array(m + [n])


def image_metrics(render, alphas, gt_rgb, gt_depth, background, depth_unit_scale=0.001, depth_tolerance=0.1) -> np.ndarray:
    """-> [C, 11] float64, columns NAMES."""
    render = render.detach().cpu().to(torch.float32)
    C, H, W, _ = render.shape
    alphas = alphas.detach().cpu().to(torch.float32).reshape(C, H, W, 1)
    bg = background.detach().cpu().to(torch.float32)
    rgb_gt = gt_rgb_f32(gt_rgb)
    dep_gt = gt_depth_f32(gt_depth, depth_unit_scale).reshape(C, H, W)
    out = np.zeros((C, len(NAMES)))
    for c in range(C):
        rgb, _ = oracle.composite_and_fill(render[c:c + 1], alphas[c:c + 1], bg)
        fill = max(float(render[c, ..., 3].max()), 0.0)
        depth = torch.where(alphas[c:c + 1] > 0, render[c:c + 1, ..., 3:4], torch.tensor(fill, dtype=torch.float32))
        p64, g64 = rgb.double(), rgb_gt[c:c + 1].double()
        mse = float(((p64 - g64) ** 2).mean())
        with np.errstate(divide="ignore"):
            psnr = float(10.0 * np.log10(np.float64(1.0) / mse))
        ssim = float(oracle.ssim(p64, g64))
        out[c, :3] = [psnr, ssim, mse]
        out[c, 3:] = depth_metrics(depth.numpy(), dep_gt[c], depth_tolerance)
    return out
