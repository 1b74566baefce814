"""-m gpu: the bilateral grid fused into the loss (qed_loss_fwd_bwd_bilagrid), its TV regulariser and the row
accumulation, against the float64 oracle of tests/bilagrid_oracle.py."""
import pytest
import torch

import bilagrid_oracle as bo
from qed_splatter_b200 import _lib, bilateral_grid_tv_loss, depth_supervised_loss, rasterization
from qed_splatter_b200.scenes import scene_s0
from helpers import assert_close_frac, scene_args

pytestmark = pytest.mark.gpu


def _inputs(C, H, W, G, shape, seed=0, masked=False, u8=False, noise=0.2):
    gen = torch.Generator().manual_seed(seed)
    X, Y, L = shape
    render = torch.rand(C, H, W, 4, generator=gen) * 1.2 - 0.1  # some composites clamp at both ends
    render[..., 3] = 1 + 4 * torch.rand(C, H, W, generator=gen)
    alphas = torch.rand(C, H, W, 1, generator=gen)
    alphas[torch.rand(C, H, W, 1, generator=gen) < 0.05] = 0.0
    grids = bo.identity_grids(G, X, Y, L) + noise * torch.randn(G, 12, L, Y, X, generator=gen)
    gt_rgb = torch.rand(C, H, W, 3, generator=gen)
    if u8:
        gt_rgb = (gt_rgb * 255).round().to(torch.uint8)
    gt_depth = 1 + 4 * torch.rand(C, H, W, 1, generator=gen)
    gt_depth[torch.rand(C, H, W, 1, generator=gen) < 0.1] = 0.0
    mask = (torch.rand(C, H, W, generator=gen) > 0.2) if masked else None
    return render, alphas, grids, gt_rgb, gt_depth, mask


def _oracle(render, alphas, grids, ids, gt_rgb, gt_depth, bg, ssim, mask):
    d = lambda t: None if t is None else t.double().requires_grad_(t.is_floating_point())  # noqa: E731
    r, a, g = d(render), d(alphas), d(grids)
    gt = gt_rgb.double() / 255.0 if gt_rgb.dtype == torch.uint8 else gt_rgb.double()
    loss = bo.loss(r, a, g, ids.long(), gt, gt_depth.double(), bg.double(), rgb_weight=1 - ssim, ssim_lambda=ssim,
                   mask=None if mask is None else mask.double())
    loss.backward()
    return loss.detach(), r.grad, a.grad, g.grad


def _check(cuda, C, H, W, G, ids, shape, ssim, masked=False, u8=False, seed=0):
    render, alphas, grids, gt_rgb, gt_depth, mask = _inputs(C, H, W, G, shape, seed, masked, u8)
    bg = torch.tensor([0.3, 0.1, 0.6])
    lo, vr_o, va_o, vg_o = _oracle(render, alphas, grids, ids, gt_rgb, gt_depth, bg, ssim, mask)
    r, a, g = (t.to(cuda).requires_grad_(True) for t in (render, alphas, grids))
    tot, l_rgb, l_d = depth_supervised_loss(r, a, gt_rgb.to(cuda), gt_depth.to(cuda), bg.to(cuda), rgb_weight=1 - ssim, depth_lambda=0.2,
                                            ssim_lambda=ssim, mask=None if mask is None else mask.to(cuda), bilateral_grids=g,
                                            grid_ids=ids.to(cuda))
    tot.backward()
    assert float(tot) == pytest.approx(float(lo), rel=2e-5)
    assert float(l_rgb + l_d) == pytest.approx(float(tot), rel=1e-5)
    for name, got, ref in (("v_render", r.grad, vr_o), ("v_alphas", a.grad, va_o), ("v_grids", g.grad, vg_o)):
        scale = float(ref.abs().max()) + 1e-30
        assert_close_frac(got, ref, 1e-3, 1e-4 * scale, 2e-3, name, max_outlier=2e-2)


@pytest.mark.parametrize("C,ids", [(1, [0]), (8, [3, 1, 3, 0, 1, 1, 2, 3])])
@pytest.mark.parametrize("ssim,masked,u8", [(0.0, False, False), (0.2, True, False), (0.2, False, True)])
def test_loss_matches_oracle(cuda, C, ids, ssim, masked, u8):
    _check(cuda, C, 40, 53, 4, torch.tensor(ids, dtype=torch.int32), (16, 16, 8), ssim, masked, u8)


@pytest.mark.parametrize("shape", [(32, 32, 16), (5, 7, 3)])
def test_loss_matches_oracle_other_grid_shapes(cuda, shape):
    _check(cuda, 2, 64, 96, 2, torch.tensor([1, 0], dtype=torch.int32), shape, 0.2, masked=True)


def test_loss_matches_oracle_at_1080p(cuda):
    _check(cuda, 1, 1080, 1920, 3, torch.tensor([2], dtype=torch.int32), (16, 16, 8), 0.2)


@pytest.mark.parametrize("mode", ["RGB+D", "RGB+ED"])
def test_rendered_views_match_oracle(cuda, mode):
    """S0 scene at its 256 px size, rendered by the library: the grid loss on a real render."""
    s = scene_s0(N=3000, C=2, size=256)
    render, alpha, _ = rasterization(**scene_args(s, cuda), width=s.width, height=s.height, sh_degree=3, render_mode=mode)
    gen = torch.Generator().manual_seed(5)
    grids = bo.identity_grids(3) + 0.1 * torch.randn(3, 12, 8, 16, 16, generator=gen)
    ids = torch.tensor([2, 0], dtype=torch.int32)
    bg = torch.tensor([0.3, 0.1, 0.6])
    lo, vr_o, va_o, vg_o = _oracle(render.cpu(), alpha.cpu(), grids, ids, s.gt_rgb, s.gt_depth, bg, 0.2, None)
    r, a, g = render.detach().requires_grad_(True), alpha.detach().requires_grad_(True), grids.to(cuda).requires_grad_(True)
    tot, _, _ = depth_supervised_loss(r, a, s.gt_rgb.to(cuda), s.gt_depth.to(cuda), bg.to(cuda), rgb_weight=0.8, ssim_lambda=0.2,
                                      bilateral_grids=g, grid_ids=ids.to(cuda))
    tot.backward()
    assert float(tot) == pytest.approx(float(lo), rel=2e-5)
    for name, got, ref in (("v_render", r.grad, vr_o), ("v_alphas", a.grad, va_o), ("v_grids", g.grad, vg_o)):
        assert_close_frac(got, ref, 1e-3, 1e-4 * float(ref.abs().max()), 2e-3, name, max_outlier=2e-2)


def _raw_call(cuda, C, H, W, grids, ids, ssim):
    lib = _lib.load()
    render, alphas, _, gt_rgb, gt_depth, _ = _inputs(C, H, W, 1, grids.shape[2:][::-1], seed=1)
    G, _, L, Y, X = grids.shape
    t = [x.to(cuda).contiguous() for x in (render, alphas, gt_rgb, gt_depth, grids, ids)]
    bg = torch.tensor([0.3, 0.1, 0.6], device=cuda)
    stats = torch.zeros(C * 8, dtype=torch.float64, device=cuda)
    loss = torch.empty(3, device=cuda)
    v_render, v_alphas = torch.empty_like(t[0]), torch.empty_like(t[1])
    rows = torch.full((C, 12, L, Y, X), float("nan"), device=cuda)
    nb = lib.qed_loss_bilagrid_workspace_bytes(C, W, H, ssim)
    ws = torch.empty(nb, dtype=torch.uint8, device=cuda)
    rc = lib.qed_loss_fwd_bwd_bilagrid(C, W, H, _lib.ptr(t[0]), _lib.ptr(t[1]), _lib.ptr(t[2]), 0, _lib.ptr(t[3]), 0, 1.0, None, 0, _lib.ptr(bg),
                                       1 - ssim, 0.2, ssim, 1.0, _lib.ptr(stats), _lib.ptr(loss), _lib.ptr(v_render), _lib.ptr(v_alphas),
                                       _lib.ptr(t[4]), _lib.ptr(t[5]), G, X, Y, L, _lib.ptr(rows), _lib.ptr(ws), nb, _lib.current_stream())
    return rc, loss, v_render, v_alphas, rows


def test_deterministic_and_rows_overwritten(cuda):
    gen = torch.Generator().manual_seed(2)
    grids = bo.identity_grids(3) + 0.2 * torch.randn(3, 12, 8, 16, 16, generator=gen)
    ids = torch.tensor([1, 1, 0], dtype=torch.int32)
    a = _raw_call(cuda, 3, 300, 411, grids, ids, 0.2)
    b = _raw_call(cuda, 3, 300, 411, grids, ids, 0.2)
    assert a[0] == 0 and b[0] == 0
    for x, y in zip(a[1:], b[1:]):
        assert torch.equal(x, y)
    assert torch.isfinite(a[4]).all()  # every row element written
    # the rows of the two views sharing grid 1 are summed by qed_bilagrid_accumulate in view order
    lib = _lib.load()
    v = torch.zeros(3, 12, 8, 16, 16, device=cuda)
    idc = ids.to(cuda)
    assert lib.qed_bilagrid_accumulate(3, _lib.ptr(idc), _lib.ptr(a[4]), 3, 16, 16, 8, _lib.ptr(v), _lib.current_stream()) == 0
    assert torch.equal(v[1], a[4][0] + a[4][1]) and torch.equal(v[0], a[4][2]) and torch.equal(v[2], torch.zeros_like(v[2]))


def test_unsupported_shapes(cuda):
    for shape in ((1, 16, 8), (16, 16, 17)):
        X, Y, L = shape
        rc = _raw_call(cuda, 1, 32, 32, torch.zeros(1, 12, L, Y, X), torch.zeros(1, dtype=torch.int32), 0.0)[0]
        assert rc == -2  # QED_ERR_UNSUPPORTED
        with pytest.raises(ValueError, match="unsupported"):
            bilateral_grid_tv_loss(torch.zeros(1, 12, L, Y, X, device=cuda))
    with pytest.raises(ValueError):
        r = torch.zeros(1, 8, 8, 4, device=cuda)
        depth_supervised_loss(r, r[..., :1], r[..., :3], r[..., 3:], torch.zeros(3, device=cuda), bilateral_grids=bo.identity_grids(2).to(cuda),
                              grid_ids=torch.tensor([2], dtype=torch.int32))


def test_identity_grids_match_the_plain_loss(cuda):
    render, alphas, _, gt_rgb, gt_depth, mask = _inputs(2, 96, 128, 1, (16, 16, 8), seed=4, masked=True)
    args = [t.to(cuda) for t in (gt_rgb, gt_depth)] + [torch.tensor([0.3, 0.1, 0.6], device=cuda)]
    out = {}
    for name, kw in (("plain", {}), ("grid", dict(bilateral_grids=bo.identity_grids(2).to(cuda), grid_ids=torch.tensor([1, 0], dtype=torch.int32)))):
        r, a = render.to(cuda).requires_grad_(True), alphas.to(cuda).requires_grad_(True)
        tot, _, _ = depth_supervised_loss(r, a, *args, ssim_lambda=0.2, rgb_weight=0.8, mask=mask.to(cuda), **kw)
        tot.backward()
        out[name] = (tot.detach(), r.grad, a.grad)
    assert float(out["grid"][0]) == pytest.approx(float(out["plain"][0]), abs=1e-6)
    for i in (1, 2):
        assert (out["grid"][i] - out["plain"][i]).abs().max() <= 1e-6 * max(float(out["plain"][i].abs().max()), 1e-3)


def test_tv_matches_oracle(cuda):
    gen = torch.Generator().manual_seed(7)
    for shape in ((16, 16, 8), (32, 32, 16), (3, 5, 2)):
        X, Y, L = shape
        grids = bo.identity_grids(5, X, Y, L) + 0.1 * torch.randn(5, 12, L, Y, X, generator=gen)
        go = grids.double().requires_grad_(True)
        ref = bo.total_variation(go, 10.0)
        ref.backward()
        g = grids.to(cuda).requires_grad_(True)
        tv = bilateral_grid_tv_loss(g, 10.0)
        tv.backward()
        assert float(tv) == pytest.approx(float(ref), rel=1e-5)
        assert torch.allclose(g.grad.double().cpu(), go.grad, rtol=1e-4, atol=1e-6 * float(go.grad.abs().max()))
        tv2 = bilateral_grid_tv_loss(g.detach(), 10.0)
        assert torch.equal(tv2, tv.detach())


def test_recovers_a_per_camera_colour_change(cuda):
    """Ground truth rendered by the library, then a known affine colour change per camera (gains 0.8-1.2, offsets
    +-0.05); only the grids train (the Gaussians stay fixed).  The L1 error has to fall by a large factor: on a B200 it went
    from 0.0506 to 0.0022 (22.7x) in 300 steps; the threshold leaves room for a different summation order."""
    s = scene_s0(N=4000, C=4, size=128)
    a = scene_args(s, cuda)
    bg = torch.tensor([0.0, 0.0, 0.0], device=cuda)
    with torch.no_grad():
        render, alpha, _ = rasterization(**a, width=128, height=128, sh_degree=3, render_mode="RGB+D")
        clean = torch.clamp(render[..., :3] + (1 - alpha) * bg, 0, 1)
        gen = torch.Generator().manual_seed(11)
        gain = (0.8 + 0.4 * torch.rand(4, 1, 1, 3, generator=gen)).to(cuda)
        off = (0.1 * torch.rand(4, 1, 1, 3, generator=gen) - 0.05).to(cuda)
        gt_rgb = clean * gain + off
    ids = torch.arange(4, dtype=torch.int32, device=cuda)
    grids = bo.identity_grids(4).to(cuda).requires_grad_(True)
    opt = torch.optim.Adam([grids], lr=2e-2, eps=1e-15)
    l1 = []
    for it in range(300):
        opt.zero_grad()
        tot, l_rgb, _ = depth_supervised_loss(render, alpha, gt_rgb, render[..., 3:], bg, rgb_weight=1.0, depth_lambda=0.0, bilateral_grids=grids,
                                              grid_ids=ids)
        (tot + bilateral_grid_tv_loss(grids, 10.0)).backward()
        opt.step()
        l1.append(float(l_rgb))
    assert l1[-1] < l1[0] / 8, (l1[0], l1[-1])
