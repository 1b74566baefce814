"""Float64 restatement of splatfacto's bilateral grid (nerfstudio lib_bilagrid), test infrastructure only.

`slice_grid_sample` is the op nerfstudio runs: torch's own F.grid_sample on the 5-D grid [12, L, Y, X] with
(x, y, z) = (column / (W-1), row / (H-1), BT.601 gray) mapped to [-1, 1], bilinear, align_corners=True, border padding.
`slice_trilinear` restates the same lookup by hand, the way the CUDA kernel computes it; the CPU tests pin the two
together.  `total_variation` is the grids' TV regulariser and `loss` the full chain the fused kernels compute.
"""
import torch
import torch.nn.functional as F

import oracle

LUMA = (0.299, 0.587, 0.114)


def identity_grids(G, X=16, Y=16, L=8, dtype=torch.float32):
    """[G,12,L,Y,X]: every cell the 3x4 identity, row-major in the 12 channels."""
    eye = torch.eye(3, 4, dtype=dtype).reshape(12)
    return eye.view(1, 12, 1, 1, 1).repeat(G, 1, L, Y, X)


def _gray(rgb):
    return rgb[..., 0] * LUMA[0] + rgb[..., 1] * LUMA[1] + rgb[..., 2] * LUMA[2]


def _apply(A, rgb):  # A [C,H,W,12], rgb [C,H,W,3] -> out_i = sum_j A[i][j] c_j + A[i][3]
    A = A.reshape(*A.shape[:-1], 3, 4)
    return (A[..., :3] @ rgb[..., None]).squeeze(-1) + A[..., 3]


def slice_grid_sample(grids, ids, rgb):
    """grids [G,12,L,Y,X], ids [C] (long), rgb [C,H,W,3] -> corrected rgb [C,H,W,3] (nerfstudio's slice)."""
    C, H, W, _ = rgb.shape
    gy, gx = torch.meshgrid(torch.linspace(0, 1, H, dtype=rgb.dtype), torch.linspace(0, 1, W, dtype=rgb.dtype), indexing="ij")
    coords = torch.stack([gx.expand(C, H, W), gy.expand(C, H, W), _gray(rgb)], -1) * 2 - 1
    A = F.grid_sample(grids[ids], coords[:, None], mode="bilinear", align_corners=True, padding_mode="border")  # [C,12,1,H,W]
    return _apply(A[:, :, 0].permute(0, 2, 3, 1), rgb)


def slice_trilinear(grids, ids, rgb):
    """The same lookup written out: lattice coordinate g = coord (n-1) clamped to [0, n-1], cell i0 = min(floor g, n-2),
    weight g - i0 of cell i0 + 1, trilinear over the 8 cells."""
    C, H, W, _ = rgb.shape
    _, _, L, Y, X = grids.shape

    def axis(coord, n):
        g = (coord * (n - 1)).clamp(0, n - 1)
        i0 = torch.clamp(torch.floor(g), max=n - 2).long()
        return i0, g - i0

    xs = torch.arange(W, dtype=rgb.dtype) / max(W - 1, 1)
    ys = torch.arange(H, dtype=rgb.dtype) / max(H - 1, 1)
    x0, fx = axis(xs.view(1, 1, W).expand(C, H, W), X)
    y0, fy = axis(ys.view(1, H, 1).expand(C, H, W), Y)
    z0, fz = axis(_gray(rgb), L)
    g = grids[ids]  # [C,12,L,Y,X]
    cidx = torch.arange(C).view(C, 1, 1).expand(C, H, W)
    A = 0.0
    for dz, wz in ((0, 1 - fz), (1, fz)):
        for dy, wy in ((0, 1 - fy), (1, fy)):
            for dx, wx in ((0, 1 - fx), (1, fx)):
                cell = g[cidx, :, z0 + dz, y0 + dy, x0 + dx]  # [C,H,W,12]
                A = A + (wz * wy * wx)[..., None] * cell
    return _apply(A, rgb)


def total_variation(grids, weight=10.0):
    """weight / G * sum over the L, Y, X axes of sum (x[i+1] - x[i])^2 / (elements of one grid's difference)."""
    tv = 0.0
    for d in (2, 3, 4):
        n = grids.shape[d]
        diff = grids.narrow(d, 1, n - 1) - grids.narrow(d, 0, n - 1)
        tv = tv + (diff ** 2).sum() / diff[0].numel()
    return weight * tv / grids.shape[0]


def loss(render, alphas, grids, ids, gt_rgb, gt_depth, bg, rgb_weight=0.8, depth_lambda=0.2, ssim_lambda=0.2, mask=None):
    """composite -> clamp -> slice -> mask -> rgb_weight L1 + ssim_lambda (1 - SSIM), + the unchanged depth term; mean over views."""
    C = render.shape[0]
    total = 0.0
    for c in range(C):
        rgb, depth = oracle.composite_and_fill(render[c:c + 1], alphas[c:c + 1], bg)
        out = slice_grid_sample(grids, ids[c:c + 1], rgb)
        gt = gt_rgb[c:c + 1]
        m = None
        if mask is not None:
            m = mask[c:c + 1].reshape(1, *render.shape[1:3], 1).to(render.dtype)
            out, gt = out * m, gt * m
        t = rgb_weight * (out - gt).abs().mean()
        if ssim_lambda > 0:
            t = t + ssim_lambda * (1 - oracle.ssim(out, gt))
        total = total + t + oracle.depth_l1_loss(depth, gt_depth[c:c + 1].reshape(depth.shape), depth_lambda, mask=m)
    return total / C
