"""CPU: the oracle as a reference for camera pose gradients (v_viewmats).

In float64, torch autograd of `oracle.rasterization` with respect to `viewmats` -- and through `oracle.get_viewmat` with
respect to the camera-to-world pose -- matches central finite differences of the whole render.  That makes the oracle a
checked reference for the pose gradient of `qed_project_bwd_pose` (tests/test_gpu_pose_grad.py)."""
import pytest
import torch

import oracle
from test_oracle import _tiny


def _c2w_of(viewmats: torch.Tensor) -> torch.Tensor:
    """Inverse of oracle.get_viewmat for a rigid viewmat: R = W^T, T = -W^T t, y / z columns flipped back."""
    W, t = viewmats[:, :3, :3], viewmats[:, :3, 3:]
    R = W.transpose(1, 2)
    c2w = torch.cat([R * torch.tensor([[[1.0, -1.0, -1.0]]], dtype=R.dtype), -(R @ t)], dim=-1)
    return c2w.contiguous()


def _fd_check(f, x, g, eps=1e-6, trials=3):
    """Directional central differences of the scalar f at x against autograd."""
    leaf = x.clone().requires_grad_(True)
    f(leaf).backward()
    for _ in range(trials):
        d = torch.randn(x.shape, generator=g, dtype=torch.float64)
        d = d / d.norm()
        fd = (f(x + eps * d) - f(x - eps * d)) / (2 * eps)
        an = (leaf.grad * d).sum()
        assert abs(float(fd - an)) <= 1e-5 * max(1.0, abs(float(an))), (float(fd), float(an))
    return leaf.grad


@pytest.mark.parametrize("render_mode,rasterize_mode", [("RGB+ED", "classic"), ("RGB+ED", "antialiased")])
def test_viewmats_autograd_vs_finite_differences(render_mode, rasterize_mode):
    s, a = _tiny(N=8, C=2, size=24, seed=5)
    g = torch.Generator().manual_seed(3)
    r0, al0, _ = oracle.rasterization(**a, width=s.width, height=s.height, sh_degree=3, render_mode=render_mode, rasterize_mode=rasterize_mode)
    wr = torch.randn(r0.shape, generator=g, dtype=torch.float64)
    wa = torch.randn(al0.shape, generator=g, dtype=torch.float64)

    def f(vm):
        r, al, _ = oracle.rasterization(**{**a, "viewmats": vm}, width=s.width, height=s.height, sh_degree=3, render_mode=render_mode,
                                        rasterize_mode=rasterize_mode)
        return (r * wr).sum() + (al * wa).sum()

    grad = _fd_check(f, a["viewmats"], g)
    assert float(grad[:, :3].abs().max()) > 0
    assert torch.equal(grad[:, 3], torch.zeros_like(grad[:, 3]))  # row 3 is constant for every caller


@pytest.mark.parametrize("rows", [3, 4])
def test_c2w_chain_autograd_vs_finite_differences(rows):
    s, a = _tiny(N=8, C=2, size=24, seed=7)
    c2w = _c2w_of(a["viewmats"])
    if rows == 4:
        c2w = torch.cat([c2w, torch.tensor([[[0.0, 0.0, 0.0, 1.0]]], dtype=c2w.dtype).expand(c2w.shape[0], 1, 4)], dim=1)
    assert torch.allclose(oracle.get_viewmat(c2w), a["viewmats"], atol=1e-12)
    g = torch.Generator().manual_seed(4)
    r0, al0, _ = oracle.rasterization(**a, width=s.width, height=s.height, sh_degree=3, render_mode="RGB+ED")
    wr = torch.randn(r0.shape, generator=g, dtype=torch.float64)
    wa = torch.randn(al0.shape, generator=g, dtype=torch.float64)

    def f(pose):
        r, al, _ = oracle.rasterization(**{**a, "viewmats": oracle.get_viewmat(pose)}, width=s.width, height=s.height, sh_degree=3,
                                        render_mode="RGB+ED")
        return (r * wr).sum() + (al * wa).sum()

    grad = _fd_check(f, c2w, g)
    assert float(grad[:, :3].abs().max()) > 0
