"""Test oracle of the resolution schedule's ground-truth pass (qed_downscale_ground_truth): float32 conversion as the loss
kernels convert (u8 * (1/255), float(double(u16) * unit scale), bool -> 0/1), then per output the sum over its d x d block,
in row-major order starting from 0, of (1/d^2) * x -- one torch op per product and per sum, so nothing is fused.
Also loads the nerfstudio stand-ins (tests/stubs) whose `_downscale_if_required` and `rescale_output_resolution` this
restates, without putting the `nerfstudio` stand-in package on sys.path."""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

STUBS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "stubs", "nerfstudio")


def _load_stub(rel: str, name: str):
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(STUBS, rel))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod  # dataclasses look their module up there
    spec.loader.exec_module(mod)
    return mod


def stub_downscale(image: torch.Tensor, d: int) -> torch.Tensor:
    """splatfacto `_downscale_if_required` (tests/stubs/nerfstudio/models/splatfacto.py) at factor d on one [H,W,K] image."""
    sf = _load_stub(os.path.join("models", "splatfacto.py"), "_qed_stub_splatfacto")
    fake = types.SimpleNamespace(_get_downscale_factor=lambda: d)
    return sf.SplatfactoModel._downscale_if_required(fake, image)


def stub_cameras():
    return _load_stub(os.path.join("cameras", "cameras.py"), "_qed_stub_cameras").Cameras


def to_float(x: torch.Tensor, kind: str, depth_unit_scale: float = 0.001) -> torch.Tensor:
    """kind "rgb" / "depth" / "mask": the float32 value the loss kernels read (GtImage / GtDepth / PixelMask)."""
    if kind == "rgb" and x.dtype == torch.uint8:
        return x.float() * torch.tensor(1.0 / 255.0, dtype=torch.float32)
    if kind == "depth" and x.dtype in (torch.uint16, torch.int16):
        return (x.view(torch.uint16).to(torch.float64) * depth_unit_scale).to(torch.float32)
    return x.to(torch.float32)


def downscale(x: torch.Tensor, d: int) -> torch.Tensor:
    """[C,H,W,K] float32 -> [C,H//d,W//d,K] float32, row-major block sums of (1/d^2) * x."""
    C, H, W, K = x.shape
    h, w = H // d, W // d
    blocks = x[:, :h * d, :w * d].reshape(C, h, d, w, d, K)
    inv = torch.tensor(1.0 / (d * d), dtype=torch.float32)
    acc = torch.zeros(C, h, w, K, dtype=torch.float32, device=x.device)
    for dy in range(d):
        for dx in range(d):
            acc = acc + inv.to(x.device) * blocks[:, :, dy, :, dx]
    return acc


def downscale_ground_truth(gt_rgb, gt_depth, mask, d: int, depth_unit_scale: float = 0.001):
    """The oracle of data_side.downscale_ground_truth: (rgb [C,h,w,3], depth [C,h,w,1], mask [C,h,w,1] | None)."""
    C, H, W, _ = gt_rgb.shape
    rgb = downscale(to_float(gt_rgb, "rgb"), d)
    dep = downscale(to_float(gt_depth, "depth", depth_unit_scale).reshape(C, H, W, 1), d)
    mk = None if mask is None else downscale(to_float(mask, "mask").reshape(C, H, W, 1), d)
    return rgb, dep, mk


def make_inputs(C: int, H: int, W: int, rgb: str, depth: str, mask: str, seed: int = 0):
    """Ground truth in the cached types: rgb "u8" / "f32", depth "u16" / "f32" (zeros = invalid, and NaN for f32),
    mask None / "bool" / "u8" / "f32"."""
    g = np.random.default_rng(seed)
    if rgb == "u8":
        gt_rgb = torch.from_numpy(g.integers(0, 256, (C, H, W, 3), dtype=np.uint8))
    else:
        gt_rgb = torch.from_numpy(g.random((C, H, W, 3), dtype=np.float32))
    if depth == "u16":
        raw = g.integers(300, 20000, (C, H, W), dtype=np.uint16)
        raw[g.random((C, H, W)) < 0.1] = 0
        gt_depth = torch.from_numpy(raw)
    else:
        dep = (0.3 + 19.7 * g.random((C, H, W), dtype=np.float32)).astype(np.float32)
        dep[g.random((C, H, W)) < 0.1] = 0.0
        dep[g.random((C, H, W)) < 0.005] = np.nan
        gt_depth = torch.from_numpy(dep)
    m = None
    if mask is not None:
        bits = g.random((C, H, W)) > 0.3
        m = {"bool": torch.from_numpy(bits), "u8": torch.from_numpy(bits.astype(np.uint8)),
             "f32": torch.from_numpy(g.random((C, H, W), dtype=np.float32))}[mask]
    return gt_rgb, gt_depth, m


def ulp_distance(a: torch.Tensor, b: torch.Tensor) -> int:
    """Largest distance in units in the last place between float32 tensors of non-negative values; NaN must sit at the
    same places in both (returns a huge number otherwise)."""
    a, b = a.detach().cpu().float().contiguous(), b.detach().cpu().float().contiguous()
    na, nb = torch.isnan(a), torch.isnan(b)
    if not torch.equal(na, nb):
        return 1 << 40
    ia, ib = a[~na].view(torch.int32).long(), b[~nb].view(torch.int32).long()
    return int((ia - ib).abs().max()) if ia.numel() else 0
