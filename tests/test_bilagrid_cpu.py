"""CPU: the bilateral-grid oracle pins grid_sample's axis order and align_corners mapping, its gradient matches finite
differences through the whole loss chain, and the host-side validation of the new keywords."""
import pytest
import torch

import bilagrid_oracle as bo


def test_identity_grid_is_the_identity():
    rgb = torch.rand(2, 5, 7, 3, dtype=torch.float64)
    g = bo.identity_grids(3, X=4, Y=3, L=5, dtype=torch.float64)
    ids = torch.tensor([2, 0])
    assert torch.allclose(bo.slice_grid_sample(g, ids, rgb), rgb, atol=1e-12)
    assert torch.allclose(bo.slice_trilinear(g, ids, rgb), rgb, atol=1e-12)
    assert float(bo.total_variation(g)) == 0.0


@pytest.mark.parametrize("shape", [(16, 16, 8), (4, 3, 5), (32, 32, 16), (2, 2, 2)])
@pytest.mark.parametrize("HW", [(9, 13), (1, 6), (17, 1)])
def test_hand_written_trilinear_is_grid_sample(shape, HW):
    """Random grids; colours whose gray lands on cell borders, inside cells, and outside [0, 1] (clamped)."""
    X, Y, L = shape
    H, W = HW
    gen = torch.Generator().manual_seed(X * 100 + H)
    grids = torch.randn(3, 12, L, Y, X, generator=gen, dtype=torch.float64)
    rgb = torch.rand(2, H, W, 3, generator=gen, dtype=torch.float64) * 1.4 - 0.2
    # grey pixels on every lattice level (gray = level / (L-1)), and beyond both ends
    flat = rgb.view(-1, 3)
    levels = torch.cat([torch.arange(L, dtype=torch.float64) / (L - 1), torch.tensor([-0.3, 1.3], dtype=torch.float64)])
    k = min(len(levels), flat.shape[0])
    flat[:k] = levels[:k, None]
    ids = torch.tensor([1, 2])
    a = bo.slice_grid_sample(grids, ids, rgb)
    b = bo.slice_trilinear(grids, ids, rgb)
    assert torch.allclose(a, b, rtol=1e-10, atol=1e-10)


def test_axis_order_and_corners():
    """A grid that varies along one axis only changes the output along the matching image / colour axis."""
    X, Y, L = 5, 4, 3
    g = bo.identity_grids(1, X, Y, L, dtype=torch.float64)
    g[0, 3] += torch.arange(X, dtype=torch.float64).view(1, 1, X)  # red offset grows with the column
    g[0, 7] += torch.arange(Y, dtype=torch.float64).view(1, Y, 1)  # green offset grows with the row
    g[0, 11] += torch.arange(L, dtype=torch.float64).view(L, 1, 1)  # blue offset grows with the gray level
    H, W = 4, 5
    rgb = torch.zeros(1, H, W, 3, dtype=torch.float64)
    out = bo.slice_grid_sample(g, torch.tensor([0]), rgb)
    assert torch.allclose(out[0, :, :, 0], torch.arange(W, dtype=torch.float64).expand(H, W) * (X - 1) / (W - 1))
    assert torch.allclose(out[0, :, :, 1], torch.arange(H, dtype=torch.float64).view(H, 1).expand(H, W) * (Y - 1) / (H - 1))
    assert torch.allclose(out[0, :, :, 2], torch.zeros(H, W, dtype=torch.float64))
    out1 = bo.slice_grid_sample(g, torch.tensor([0]), torch.ones(1, H, W, 3, dtype=torch.float64))
    assert torch.allclose(out1[0, :, :, 2], torch.full((H, W), 1.0 + (L - 1), dtype=torch.float64))


def test_total_variation_by_hand():
    g = torch.zeros(2, 12, 2, 2, 3, dtype=torch.float64)
    g[0, 0, 0, 0, 0] = 1.0  # one cell: neighbours along X (1), Y (1), L (1)
    tv = bo.total_variation(g, weight=10.0)
    # counts of one grid's differences: X 12*2*2*2 = 96, Y 12*2*1*3 = 72, L 12*1*2*3 = 72
    assert float(tv) == pytest.approx(10.0 / 2 * (1 / 96 + 1 / 72 + 1 / 72))


@pytest.mark.parametrize("ssim,masked", [(0.0, False), (0.2, True)])
def test_loss_chain_gradient_matches_finite_differences(ssim, masked):
    """render, alphas, grids -> composite -> clamp -> slice -> mask -> L1 + SSIM (+ depth), plus TV, in float64 with
    random non-identity grids (at the identity the guidance term through the gray level is exactly zero)."""
    gen = torch.Generator().manual_seed(3)
    C, H, W = 2, 12, 13
    X, Y, L = 3, 4, 4
    render = torch.rand(C, H, W, 4, generator=gen, dtype=torch.float64) * 0.9
    render[..., 3] += 1.0
    alphas = torch.rand(C, H, W, 1, generator=gen, dtype=torch.float64)
    grids = bo.identity_grids(2, X, Y, L, dtype=torch.float64) + 0.2 * torch.randn(2, 12, L, Y, X, generator=gen, dtype=torch.float64)
    gt_rgb = torch.rand(C, H, W, 3, generator=gen, dtype=torch.float64)
    gt_depth = 1 + torch.rand(C, H, W, 1, generator=gen, dtype=torch.float64)
    bg = torch.tensor([0.3, 0.1, 0.6], dtype=torch.float64)
    mask = (torch.rand(C, H, W, generator=gen) > 0.2).double() if masked else None
    ids = torch.tensor([1, 0])

    def f(r, a, g):
        return bo.loss(r, a, g, ids, gt_rgb, gt_depth, bg, rgb_weight=1 - ssim, ssim_lambda=ssim, mask=mask) + bo.total_variation(g)

    inputs = (render.requires_grad_(True), alphas.requires_grad_(True), grids.requires_grad_(True))
    assert torch.autograd.gradcheck(f, inputs, eps=1e-6, atol=1e-6, rtol=1e-4)


def test_keywords_go_together_and_ids_are_checked():
    from qed_splatter_b200 import depth_supervised_loss
    from qed_splatter_b200.camera_opt import check_camera_ids

    r = torch.zeros(1, 4, 4, 4)
    with pytest.raises(ValueError, match="go together"):
        depth_supervised_loss(r, r[..., :1], r[..., :3], r[..., :1], torch.zeros(3), bilateral_grids=bo.identity_grids(1))
    with pytest.raises(ValueError, match="go together"):
        depth_supervised_loss(r, r[..., :1], r[..., :3], r[..., :1], torch.zeros(3), grid_ids=torch.zeros(1, dtype=torch.int32))
    with pytest.raises(ValueError):
        check_camera_ids(torch.tensor([3]), 1, 3, torch.device("cpu"))
    with pytest.raises(RuntimeError, match="CUDA"):  # no CPU fallback
        depth_supervised_loss(r, r[..., :1], r[..., :3], r[..., :1], torch.zeros(3), bilateral_grids=bo.identity_grids(1),
                              grid_ids=torch.zeros(1, dtype=torch.int32))
