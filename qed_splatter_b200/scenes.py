"""Seeded synthetic scenes for parity tests and benchmarks (SURVEY.md §8d: S0..S4).

Everything is generated on the CPU with a fixed `torch.Generator` so the same
bytes are produced here, on the GPU box and in the golden-fixture script.
Parameters are returned in the *activated* form the reference passes to
`rasterization` (`qed_splatter/model.py:267-273`): normalised quats, exp'd
scales, sigmoid'd opacities, SH coefficients `[N,K,3]`.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import torch
from torch import Tensor


@dataclass
class Scene:
    means: Tensor  # [N,3]
    quats: Tensor  # [N,4] wxyz, normalised
    scales: Tensor  # [N,3] (post-exp)
    opacities: Tensor  # [N] (post-sigmoid)
    sh: Tensor  # [N,K,3]
    viewmats: Tensor  # [C,4,4]
    Ks: Tensor  # [C,3,3]
    width: int
    height: int
    sh_degree: int
    gt_rgb: Optional[Tensor] = None  # [C,H,W,3]
    gt_depth: Optional[Tensor] = None  # [C,H,W,1]
    name: str = ""

    def to(self, device) -> "Scene":
        kw = {}
        for k, v in self.__dict__.items():
            kw[k] = v.to(device) if isinstance(v, Tensor) else v
        return Scene(**kw)

    @property
    def N(self) -> int:
        return self.means.shape[0]

    @property
    def C(self) -> int:
        return self.viewmats.shape[0]


def camera_to_worlds(viewmats: Tensor) -> Tensor:
    """Inverse of `get_viewmat` (model.py:22-38) for rigid world->camera viewmats [C,4,4] -> nerfstudio camera-to-world
    [C,3,4] (OpenGL camera axes): R = W^T with the y / z columns flipped back, T = -W^T t."""
    W, t = viewmats[:, :3, :3], viewmats[:, :3, 3:]
    R = W.transpose(1, 2)
    flip = torch.tensor([[[1.0, -1.0, -1.0]]], dtype=R.dtype, device=R.device)
    return torch.cat([R * flip, -(R @ t)], dim=-1).contiguous()


def look_at(eye: Tensor, target: Tensor, up=(0.0, -1.0, 0.0)) -> Tensor:
    """World->camera [4,4] in gsplat/OpenCV convention (+z forward, +y down)."""
    eye = eye.to(torch.float64)
    target = target.to(torch.float64)
    f = target - eye
    f = f / f.norm()
    upv = torch.tensor(up, dtype=torch.float64)
    r = torch.linalg.cross(f, -upv)
    if r.norm() < 1e-8:
        r = torch.tensor([1.0, 0.0, 0.0], dtype=torch.float64)
    r = r / r.norm()
    d = torch.linalg.cross(f, r)
    R = torch.stack([r, d, f], dim=0)  # rows: camera x,y,z axes in world coords
    t = -R @ eye
    V = torch.eye(4, dtype=torch.float64)
    V[:3, :3] = R
    V[:3, 3] = t
    return V.to(torch.float32)


def _intrinsics(C: int, f: float, width: int, height: int) -> Tensor:
    K = torch.zeros(C, 3, 3)
    K[:, 0, 0] = f
    K[:, 1, 1] = f
    K[:, 0, 2] = width / 2.0
    K[:, 1, 2] = height / 2.0
    K[:, 2, 2] = 1.0
    return K


def _gaussians(g: torch.Generator, N: int, lo, hi, smin: float, smax: float, K: int = 16, aniso: float = 0.0):
    lo_t = torch.tensor(lo, dtype=torch.float32)
    hi_t = torch.tensor(hi, dtype=torch.float32)
    means = lo_t + (hi_t - lo_t) * torch.rand(N, 3, generator=g)
    ls = math.log(smin) + (math.log(smax) - math.log(smin)) * torch.rand(N, 3, generator=g)
    if aniso > 0:
        ls[:, 1] += aniso  # stretched along local y
    scales = torch.exp(ls)
    quats = torch.randn(N, 4, generator=g)
    quats = quats / quats.norm(dim=-1, keepdim=True)
    opac = 0.05 + 0.9 * torch.rand(N, generator=g)
    sh = torch.empty(N, K, 3)
    sh[:, 0, :] = (torch.rand(N, 3, generator=g) * 2 - 1) / 0.2820947917738781 * 0.5
    if K > 1:
        sh[:, 1:, :] = torch.randn(N, K - 1, 3, generator=g) * 0.05
    return means, quats, scales, opac, sh


def _targets(g: torch.Generator, C: int, H: int, W: int, dmin: float, dmax: float):
    gt_rgb = torch.rand(C, H, W, 3, generator=g)
    gt_depth = dmin + (dmax - dmin) * torch.rand(C, H, W, 1, generator=g)
    invalid = torch.rand(C, H, W, 1, generator=g) < 0.1
    gt_depth = torch.where(invalid, torch.zeros(()), gt_depth)
    return gt_rgb, gt_depth


def scene_s0(N: int = 10_000, C: int = 8, size: int = 256, seed: int = 42, sh_degree: int = 3) -> Scene:
    """BASELINE.json config[0]: 10k Gaussians, 8 cameras 256x256 on a radius-3 circle."""
    g = torch.Generator().manual_seed(seed)
    K = (sh_degree + 1) ** 2
    means, quats, scales, opac, sh = _gaussians(g, N, (-1, -1, -1), (1, 1, 1), 0.01, 0.1, K)
    vms = []
    for i in range(C):
        a = 2 * math.pi * i / C
        eye = torch.tensor([3.0 * math.cos(a), 0.3 * math.sin(2 * a), 3.0 * math.sin(a)])
        vms.append(look_at(eye, torch.zeros(3)))
    gt_rgb, gt_depth = _targets(g, C, size, size, 1.0, 5.0)
    return Scene(means, quats, scales, opac, sh, torch.stack(vms), _intrinsics(C, float(size), size, size),
                 size, size, sh_degree, gt_rgb, gt_depth, name=f"S0-{N}x{C}@{size}")


def scene_s1(N: int = 1_000_000, width: int = 1920, height: int = 1080, seed: int = 42, C: int = 1,
             f: float = 1200.0, sh_degree: int = 3, targets: bool = True) -> Scene:
    """BASELINE.json config[1]: 1M Gaussians in [-10,10]x[-2,4]x[-10,10], camera at the box edge looking in."""
    g = torch.Generator().manual_seed(seed)
    K = (sh_degree + 1) ** 2
    means, quats, scales, opac, sh = _gaussians(g, N, (-10, -2, -10), (10, 4, 10), 0.005, 0.08, K)
    vms = []
    for i in range(C):
        a = 2 * math.pi * i / max(C, 1) * 0.25
        eye = torch.tensor([10.0 * math.sin(a), 1.0, -10.0 * math.cos(a)])
        vms.append(look_at(eye, torch.tensor([0.0, 1.0, 0.0])))
    gt_rgb = gt_depth = None
    if targets:
        gt_rgb, gt_depth = _targets(g, C, height, width, 1.0, 20.0)
    return Scene(means, quats, scales, opac, sh, torch.stack(vms), _intrinsics(C, f, width, height),
                 width, height, sh_degree, gt_rgb, gt_depth, name=f"S1-{N}x{C}@{width}x{height}")


def scene_s2(N: int = 3_000_000, C: int = 8, width: int = 1440, height: int = 1080, seed: int = 42,
             sh_degree: int = 3, view_offset: int = 0, total_views: Optional[int] = None) -> Scene:
    """BASELINE.json config[2]: 3M Gaussians, views on a walk-through path, 1440x1080, f=1000.

    `view_offset`/`total_views` select a rank's slice of the global view batch while keeping the
    Gaussian set (which is drawn first from the generator) identical on every rank.
    """
    g = torch.Generator().manual_seed(seed)
    K = (sh_degree + 1) ** 2
    means, quats, scales, opac, sh = _gaussians(g, N, (-10, -2, -10), (10, 4, 10), 0.005, 0.08, K)
    total = total_views if total_views is not None else C
    vms = []
    for i in range(view_offset, view_offset + C):
        s = i / max(total - 1, 1)
        eye = torch.tensor([-6.0 + 12.0 * s, 1.0, -9.5 + 2.0 * math.sin(3.0 * s)])
        tgt = torch.tensor([-3.0 + 6.0 * s, 1.0, 2.0])
        vms.append(look_at(eye, tgt))
    g2 = torch.Generator().manual_seed(seed * 1000 + 17 + view_offset)
    gt_rgb, gt_depth = _targets(g2, C, height, width, 1.0, 20.0)
    return Scene(means, quats, scales, opac, sh, torch.stack(vms), _intrinsics(C, 1000.0, width, height),
                 width, height, sh_degree, gt_rgb, gt_depth, name=f"S2-{N}x{C}@{width}x{height}")


def scene_s3(N: int = 6_000_000, C: int = 1, width: int = 1440, height: int = 1080, seed: int = 42,
             sh_degree: int = 3, view_offset: int = 0, total_views: Optional[int] = None) -> Scene:
    """BASELINE.json config[3]: 'forest' — 70% of the mass in vertical cylinders (trunks) + a ground plane."""
    g = torch.Generator().manual_seed(seed)
    K = (sh_degree + 1) ** 2
    n_trunk = int(0.7 * N)
    n_ground = N - n_trunk
    n_trees = 400
    centres = (torch.rand(n_trees, 2, generator=g) * 2 - 1) * 10.0
    tree = torch.randint(0, n_trees, (n_trunk,), generator=g)
    ang = torch.rand(n_trunk, generator=g) * 2 * math.pi
    rad = 0.15 + 0.1 * torch.rand(n_trunk, generator=g)
    hgt = torch.rand(n_trunk, generator=g) * 6.0 - 2.0
    trunk = torch.stack([centres[tree, 0] + rad * torch.cos(ang), hgt, centres[tree, 1] + rad * torch.sin(ang)], -1)
    ground = torch.stack([(torch.rand(n_ground, generator=g) * 2 - 1) * 10.0,
                          3.9 + 0.1 * torch.rand(n_ground, generator=g),
                          (torch.rand(n_ground, generator=g) * 2 - 1) * 10.0], -1)
    _, quats, scales, opac, sh = _gaussians(g, N, (0, 0, 0), (1, 1, 1), 0.004, 0.04, K, aniso=1.0)
    means = torch.cat([trunk, ground], 0)
    total = total_views if total_views is not None else C
    vms = []
    for i in range(view_offset, view_offset + C):
        a = 2 * math.pi * i / max(total, 1)
        eye = torch.tensor([9.0 * math.cos(a), 1.0, 9.0 * math.sin(a)])
        vms.append(look_at(eye, torch.tensor([0.0, 1.0, 0.0])))
    g2 = torch.Generator().manual_seed(seed * 1000 + 29 + view_offset)
    gt_rgb, gt_depth = _targets(g2, C, height, width, 1.0, 20.0)
    return Scene(means, quats, scales, opac, sh, torch.stack(vms), _intrinsics(C, 1000.0, width, height),
                 width, height, sh_degree, gt_rgb, gt_depth, name=f"S3-{N}x{C}@{width}x{height}")
