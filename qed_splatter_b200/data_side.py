"""Camera / data side of the hot path (SURVEY.md §8 rows a1 and f4), CUDA only, same names as the reference's functions.

* `get_viewmat(optimized_camera_to_world)` — /root/reference/qed_splatter/model.py:22-38 (called at model.py:246):
  nerfstudio camera-to-world -> gsplat world-to-camera.  One launch of `qed_viewmat_from_c2w` instead of six tiny torch
  kernels; rebind it with `qed_splatter.model.get_viewmat = qed_splatter_b200.get_viewmat` (INTEGRATION.md).
* `backproject_frame(...)`, `voxel_down_sample(...)`, `merge_pointclouds(...)`, `create_pointcloud_from_frames(...)` —
  the arithmetic of `qed-init-pc` (/root/reference/qed_splatter/create_init_pointcloud.py:148-196, :85-91, :100-145,
  :199-261), which the reference runs on the host through Open3D with every intermediate cloud written to disk as PLY.
  Here the frames' depth images go through `qed_backproject_depth` / `qed_voxel_downsample` and the pairwise tree merge
  stays on the device.  File handling (transforms.json, PLY, the on-disk cache, colourising from RGB) stays the
  reference's: these functions take arrays, not dataset paths.
* `downscale_ground_truth(...)` — splatfacto's `_downscale_if_required` (resolution schedule): the full-resolution image,
  depth and mask of a step box-downscaled in one launch of `qed_downscale_ground_truth`, read in their cached types.

No CPU fallback: CPU tensors raise.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch import Tensor

from . import _lib
from ._lib import check, current_stream, ptr


def _viewmat_from_c2w(c2w: Tensor) -> Tensor:
    C = c2w.shape[0]
    out = torch.empty(C, 4, 4, dtype=torch.float32, device=c2w.device)
    check(_lib.load().qed_viewmat_from_c2w(C, int(c2w.shape[1]), ptr(c2w), ptr(out), current_stream()), "qed_viewmat_from_c2w")
    return out


class _GetViewmat(torch.autograd.Function):
    @staticmethod
    def forward(ctx, c2w):
        c2w = c2w.detach().contiguous()
        ctx.save_for_backward(c2w)
        return _viewmat_from_c2w(c2w)

    @staticmethod
    def backward(ctx, v_viewmats):
        (c2w,) = ctx.saved_tensors
        v_viewmats = v_viewmats.to(torch.float32).contiguous()
        v_c2w = torch.empty_like(c2w)
        check(_lib.load().qed_viewmat_from_c2w_bwd(c2w.shape[0], int(c2w.shape[1]), ptr(c2w), ptr(v_viewmats), ptr(v_c2w), current_stream()),
              "qed_viewmat_from_c2w_bwd")
        return v_c2w


def get_viewmat(optimized_camera_to_world: Tensor, pose_gradients: bool = False) -> Tensor:
    """model.py:22-38: c2w [C,3|4,4] (OpenGL camera axes) -> gsplat world-to-camera [C,4,4].

    `pose_gradients=True`: when c2w requires grad, the result carries the gradient back to it (the camera optimizer's
    pose; bind `functools.partial(get_viewmat, pose_gradients=True)`, INTEGRATION.md section 2b).  The forward values are
    the same bits either way."""
    c2w = optimized_camera_to_world
    _lib.require_cuda(c2w)
    _lib.require_dtype(c2w, (torch.float32,), "optimized_camera_to_world")
    if c2w.dim() != 3 or c2w.shape[1] not in (3, 4) or c2w.shape[2] != 4:
        raise ValueError("optimized_camera_to_world must be [C,3,4] or [C,4,4]")
    if c2w.requires_grad and torch.is_grad_enabled():
        if pose_gradients:
            return _GetViewmat.apply(c2w)
        # camera_optimizer.mode != "off" without asking for pose gradients: refuse rather than train with zero gradients
        raise NotImplementedError("get_viewmat: c2w requires grad (camera optimisation): pass pose_gradients=True, or c2w.detach()")
    return _viewmat_from_c2w(c2w.detach().contiguous())


def downscaled_size(width: int, height: int, factor: int) -> Tuple[int, int]:
    """(w, h) of ground truth of size width x height box-downscaled by `factor`: rounded down, as conv2d(stride=factor)
    drops trailing rows and columns that fill no block.  ValueError when the factor is below 1 or nothing is left."""
    if int(factor) != factor or factor < 1:
        raise ValueError(f"downscale factor must be an integer >= 1, got {factor!r}")
    w, h = int(width) // int(factor), int(height) // int(factor)
    if w < 1 or h < 1:
        raise ValueError(f"{width}x{height} ground truth has no full {factor}x{factor} block")
    return w, h


def downscale_ground_truth(gt_rgb: Tensor, gt_depth: Tensor, mask: Optional[Tensor], factor: int, depth_unit_scale: float = 0.001,
                           out: Optional[Tuple[Tensor, Tensor, Optional[Tensor]]] = None) -> Tuple[Tensor, Tensor, Optional[Tensor]]:
    """Splatfacto's `_downscale_if_required` (nerfstudio `resize_image`: a factor x factor box filter) on the ground truth of
    a step, one launch of `qed_downscale_ground_truth`.

    gt_rgb [C,H,W,3] float32 or the uint8 image cache (u8 / 255 before the filter, as `get_gt_img` does), gt_depth
    [C,H,W(,1)] float32 metres or the raw uint16 sensor image (torch.uint16, or its bits as torch.int16; converted with
    `depth_unit_scale` before the filter), mask [C,H,W(,1)] float32 / uint8 / bool or None (bool -> 0 / 1 floats, so the
    result is fractional).  -> float32 (rgb [C,h,w,3], depth [C,h,w,1] metres, mask [C,h,w,1] or None) with
    (w, h) = downscaled_size(W, H, factor); each value is the row-major sum of (1/factor^2) * x over its block.
    `out`: tensors of those shapes to write into (the mask slot may be None when mask is None)."""
    _lib.require_cuda(gt_rgb, gt_depth, mask)
    _lib.require_dtype(gt_rgb, (torch.float32, torch.uint8), "gt_rgb")
    _lib.require_dtype(gt_depth, (torch.float32, torch.uint16, torch.int16), "gt_depth")
    _lib.require_dtype(mask, (torch.float32, torch.uint8, torch.bool), "mask")
    if gt_rgb.dim() != 4 or gt_rgb.shape[3] != 3:
        raise ValueError("gt_rgb must be [C,H,W,3]")
    C, H, W, _ = gt_rgb.shape
    w, h = downscaled_size(W, H, factor)
    if gt_depth.numel() != C * H * W or (mask is not None and mask.numel() != C * H * W):
        raise ValueError("shapes: gt_rgb [C,H,W,3], gt_depth [C,H,W(,1)], mask [C,H,W(,1)]")
    shapes = ((C, h, w, 3), (C, h, w, 1), (C, h, w, 1))
    if out is None:
        out = tuple(torch.empty(s, dtype=torch.float32, device=gt_rgb.device) for s in shapes)
    out_rgb, out_depth, out_mask = out
    out_mask = out_mask if mask is not None else None
    for t, s in zip((out_rgb, out_depth, out_mask), shapes):
        if t is not None and (tuple(t.shape) != s or t.dtype != torch.float32 or not t.is_contiguous() or t.device != gt_rgb.device):
            raise ValueError(f"out: contiguous float32 tensors of shapes {shapes} on {gt_rgb.device} expected")
    if mask is not None and out_mask is None:
        raise ValueError("out: a mask tensor is needed when mask is given")
    rgb, dep = gt_rgb.contiguous(), gt_depth.contiguous()
    mk = None if mask is None else mask.contiguous()
    if mk is not None and mk.dtype == torch.bool:
        mk = mk.view(torch.uint8)
    check(_lib.load().qed_downscale_ground_truth(C, W, H, int(factor), ptr(rgb), int(rgb.dtype == torch.uint8), ptr(dep),
                                                 int(dep.dtype != torch.float32), float(depth_unit_scale), ptr(mk),
                                                 int(mk is not None and mk.dtype == torch.uint8), ptr(out_rgb), ptr(out_depth),
                                                 ptr(out_mask), current_stream()), "qed_downscale_ground_truth")
    return out_rgb, out_depth, out_mask


def _host_f32(x, shape, what: str) -> np.ndarray:
    a = np.ascontiguousarray(x.detach().cpu().numpy() if isinstance(x, Tensor) else np.asarray(x), dtype=np.float32)
    if a.shape != shape:
        raise ValueError(f"{what} must be {shape}, got {a.shape}")
    return a


def opengl_c2w_to_opencv_w2c(c2w_opengl) -> np.ndarray:
    """create_init_pointcloud.py:59-70 `_opengl_c2w_to_opencv_w2c` (host, float64 inverse, float32 result)."""
    c2w = np.array(c2w_opengl, dtype=np.float64).copy()
    c2w[:3, 1:3] *= -1
    return np.linalg.inv(c2w).astype(np.float32)


def backproject_frame(depth: Tensor, intrinsic, w2c, depth_unit_scale_factor: float = 0.001, depth_max: float = 100.0, stride: int = 1,
                      frame_voxel_size: Optional[float] = 0.05) -> Optional[Tensor]:
    """create_init_pointcloud.py:148-196: one depth frame -> world points [n,3] (float32, CUDA), or None when no pixel
    survives.  depth [H,W] float32 or the raw uint16 image; intrinsic [3,3]; w2c [4,4] OpenCV world-to-camera
    (`opengl_c2w_to_opencv_w2c` of the frame's transform_matrix)."""
    _lib.require_cuda(depth)
    if depth.dim() == 3:
        depth = depth[..., 0]
    if depth.dtype == torch.int16:
        depth = depth.view(torch.uint16)
    _lib.require_dtype(depth, (torch.float32, torch.uint16), "depth")
    depth = depth.contiguous()
    H, W = depth.shape
    K = _host_f32(intrinsic, (3, 3), "intrinsic")
    E = _host_f32(w2c, (4, 4), "w2c")
    lib = _lib.load()
    dev = depth.device
    cap = ((W + stride - 1) // stride) * ((H + stride - 1) // stride)
    points = torch.empty(cap, 3, dtype=torch.float32, device=dev)
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    ws = torch.empty(max(int(lib.qed_backproject_workspace_bytes(W, H, stride)), 8), dtype=torch.uint8, device=dev)
    check(lib.qed_backproject_depth(W, H, ptr(depth), 1 if depth.dtype == torch.uint16 else 0, float(depth_unit_scale_factor), float(depth_max),
                                    int(stride), K.ctypes.data, E.ctypes.data, ptr(points), ptr(count), ptr(ws), ws.numel(), current_stream()),
          "qed_backproject_depth")
    if frame_voxel_size is not None and frame_voxel_size > 0:
        # the count stays on the device between the two passes; the only host read is the final size
        return _voxel_down_sample(points, float(frame_voxel_size), n_dev=count, empty_is_none=True)
    n = int(count.item())
    return points[:n] if n > 0 else None


def _voxel_down_sample(points: Tensor, voxel_size: float, n_dev: Optional[Tensor] = None, empty_is_none: bool = False):
    lib = _lib.load()
    n = points.shape[0]
    dev = points.device
    out = torch.empty(max(n, 1), 3, dtype=torch.float32, device=dev)
    n_out = torch.zeros(1, dtype=torch.int64, device=dev)
    ws = torch.empty(max(int(lib.qed_voxel_downsample_workspace_bytes(n)), 8), dtype=torch.uint8, device=dev)
    check(lib.qed_voxel_downsample(n, ptr(n_dev), ptr(points), float(voxel_size), ptr(out), ptr(n_out), ptr(ws), ws.numel(), current_stream()),
          "qed_voxel_downsample")
    m = int(n_out.item())
    if m == 0 and empty_is_none:
        return None
    return out[:m]


def voxel_down_sample(points: Tensor, voxel_size: float) -> Tensor:
    """Open3D `PointCloud.voxel_down_sample(voxel_size)` (create_init_pointcloud.py:89, :194, :260): mean of the points
    of every occupied voxel floor(p / voxel_size); rows sorted by voxel index."""
    _lib.require_cuda(points)
    _lib.require_dtype(points, (torch.float32,), "points")
    if points.dim() != 2 or points.shape[1] != 3:
        raise ValueError("points must be [n,3]")
    if not voxel_size > 0:
        raise ValueError("voxel_size must be positive")
    return _voxel_down_sample(points.contiguous(), float(voxel_size))


def merge_pointclouds(clouds: Sequence[Tensor], voxel_size: float = 0.03, max_points: int = 2_000_000) -> Tensor:
    """create_init_pointcloud.py:100-145 `tree_merge_pointclouds_on_disk` without the disk: pairwise merge level by level,
    a merged pair is voxel-downsampled only when it exceeds max_points (:85-91), an odd cloud is carried forward."""
    current: List[Tensor] = list(clouds)
    if not current:
        raise RuntimeError("No valid point clouds could be generated from the dataset.")  # :246
    while len(current) > 1:
        nxt: List[Tensor] = []
        for i in range(0, len(current), 2):
            if i + 1 < len(current):
                merged = torch.cat([current[i], current[i + 1]], dim=0)
                if merged.shape[0] > max_points:
                    merged = voxel_down_sample(merged, voxel_size)
                nxt.append(merged)
            else:
                nxt.append(current[i])
        current = nxt
    return current[0]


def create_pointcloud_from_frames(depths: Sequence[Tensor], intrinsics: Sequence, c2w_opengl: Sequence, depth_unit_scale_factor: float = 0.001,
                                  voxel_size: float = 0.05, merge_voxel_size: float = 0.03, frame_voxel_size: Optional[float] = 0.05,
                                  max_points: int = 2_000_000, depth_max: float = 100.0, stride: int = 1) -> Tensor:
    """create_init_pointcloud.py:199-261 `create_pointcloud_from_transforms` on arrays: back-project every frame (frames
    without a valid pixel are skipped, :169-171 / :238), tree-merge, final voxel_down_sample(voxel_size)."""
    clouds = []
    for depth, K, c2w in zip(depths, intrinsics, c2w_opengl):
        pcd = backproject_frame(depth, K, opengl_c2w_to_opencv_w2c(c2w), depth_unit_scale_factor, depth_max, stride, frame_voxel_size)
        if pcd is not None:
            clouds.append(pcd)
    merged = merge_pointclouds(clouds, voxel_size=merge_voxel_size, max_points=max_points)
    return voxel_down_sample(merged, voxel_size)
