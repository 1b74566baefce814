"""GPU: qed_eval_metrics / image_metrics against the float64 restatement, its determinism, and SplatTrainer.evaluate."""
import os
import sys

import numpy as np
import pytest
import torch

import metrics_oracle as mo
from qed_splatter_b200 import get_viewmat, image_metrics, rasterization
from qed_splatter_b200.metrics import METRIC_NAMES, metric_rows
from qed_splatter_b200.scenes import camera_to_worlds, scene_s0
from qed_splatter_b200.trainer import EVAL_CHUNK_VIEWS, SplatTrainer, TrainConfig
from reference_model import ROOT, reference_root

pytestmark = pytest.mark.gpu


def _views(C, W, H, rgb_u8, depth_u16, seed=0):
    """Renders with clamped colours, zero-alpha pixels, NaN / zero / below-tolerance ground-truth depth; with C >= 3 view 1
    has no hit at all (the fill path everywhere) and view 2 no valid ground-truth depth."""
    g = torch.Generator().manual_seed(seed)
    render = torch.rand(C, H, W, 4, generator=g) * 1.2 - 0.1
    render[..., 3] = 0.3 + 4.0 * torch.rand(C, H, W, generator=g)
    alphas = torch.rand(C, H, W, 1, generator=g)
    alphas[torch.rand(C, H, W, 1, generator=g) < 0.2] = 0.0
    if rgb_u8:
        gt_rgb = torch.randint(0, 256, (C, H, W, 3), generator=g, dtype=torch.uint8)
    else:
        gt_rgb = torch.rand(C, H, W, 3, generator=g)
    depth_m = 0.05 + 4.0 * torch.rand(C, H, W, generator=g)
    drop = torch.rand(C, H, W, generator=g) < 0.1
    depth_m[drop] = 0.0
    if C >= 3:
        alphas[1] = 0.0
        depth_m[2] = 0.0
    if depth_u16:
        gt_depth = (depth_m * 1000.0).round().to(torch.int32).to(torch.uint16)
    else:
        gt_depth = depth_m.clone()
        gt_depth[torch.rand(C, H, W, generator=g) < 0.02] = float("nan")
    return render, alphas, gt_rgb, gt_depth, torch.tensor([0.1, 0.4, 0.7])


def _compare(got: np.ndarray, want: np.ndarray, what: str, depth_rtol=1e-9):
    psnr_g, psnr_w = got[:, 0], want[:, 0]
    assert np.array_equal(np.isinf(psnr_g), np.isinf(psnr_w)), what
    fin = np.isfinite(psnr_w)
    np.testing.assert_allclose(psnr_g[fin], psnr_w[fin], rtol=0, atol=1e-4, err_msg=f"{what} psnr")
    np.testing.assert_allclose(got[:, 1], want[:, 1], rtol=0, atol=1e-4, err_msg=f"{what} ssim")
    np.testing.assert_allclose(got[:, 2], want[:, 2], rtol=1e-4, atol=0, err_msg=f"{what} rgb_mse")
    np.testing.assert_allclose(got[:, 3:], want[:, 3:], rtol=depth_rtol, atol=0, equal_nan=True, err_msg=f"{what} depth")


SIZES = [(37, 23, 1), (37, 23, 3), (1920, 1080, 1)]


@pytest.mark.parametrize("W,H,C", SIZES)
@pytest.mark.parametrize("rgb_u8", [False, True])
@pytest.mark.parametrize("depth_u16", [False, True])
def test_image_metrics_against_the_oracle(cuda, W, H, C, rgb_u8, depth_u16):
    render, alphas, gt_rgb, gt_depth, bg = _views(C, W, H, rgb_u8, depth_u16)
    for tol in (0.1, 1.5):
        got = image_metrics(render.to(cuda), alphas.to(cuda), gt_rgb.to(cuda), gt_depth.to(cuda), bg.to(cuda), depth_tolerance=tol)
        assert all(got[n].shape == (C,) and got[n].dtype == torch.float64 and got[n].is_cuda for n in METRIC_NAMES)
        got = torch.stack([got[n] for n in METRIC_NAMES], 1).cpu().numpy()
        want = mo.image_metrics(render, alphas, gt_rgb, gt_depth, bg, depth_tolerance=tol)
        _compare(got, want, f"{W}x{H} C={C} tol={tol}")
        if C >= 3:
            assert got[2, 10] == 0 and np.all(np.isnan(got[2, 3:10]))  # no valid depth
            assert got[1, 10] > 0  # the fill path only


def test_perfect_prediction(cuda):
    render, _, _, gt_depth, bg = _views(2, 40, 30, False, False)
    render[..., :3] = render[..., :3].clamp(0, 1)
    alphas = torch.ones(2, 30, 40, 1)
    gt_depth = render[..., 3].clone()
    got = image_metrics(render.to(cuda), alphas.to(cuda), render[..., :3].contiguous().to(cuda), gt_depth.to(cuda), bg.to(cuda))
    assert torch.all(torch.isposinf(got["psnr"])) and torch.all(got["rgb_mse"] == 0)
    assert torch.allclose(got["ssim"].cpu(), torch.ones(2, dtype=torch.float64), atol=1e-5)
    assert torch.all(got["abs_rel"] == 0) and torch.all(got["a1"] == 1)


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.int64).cpu()


def test_deterministic_and_independent_of_the_batch(cuda):
    render, alphas, gt_rgb, gt_depth, bg = (t.to(cuda) for t in _views(3, 1920, 1080, True, True))
    a = metric_rows(render, alphas, gt_rgb, gt_depth, bg)
    b = metric_rows(render, alphas, gt_rgb, gt_depth, bg)
    assert torch.equal(_bits(a), _bits(b))
    for c in range(3):
        one = metric_rows(render[c:c + 1], alphas[c:c + 1], gt_rgb[c:c + 1], gt_depth[c:c + 1], bg)
        assert torch.equal(_bits(one[0]), _bits(a[c])), c


# -- SplatTrainer.evaluate ---------------------------------------------------------------------------------------------


def _scene(C, size=96):
    return scene_s0(N=4000, C=C, size=size)


def _trainer(s, cuda, cfg, num_cameras=0):
    return SplatTrainer(s.means.to(cuda), s.quats.to(cuda), torch.log(s.scales).to(cuda), torch.logit(s.opacities).to(cuda), s.sh.to(cuda),
                        cfg=cfg, num_cameras=num_cameras)


def _expected(tr, s, cuda, bg):
    """rasterization() of the trainer's Gaussians (activated on the host) at full resolution, then the oracle's metrics."""
    p = tr.arena.views(tr.arena.param)
    render, alphas, _ = rasterization(p["means"], p["quats"], torch.exp(p["scales"]), torch.sigmoid(p["opacities"]), p["sh"], s.viewmats.to(cuda),
                                      s.Ks.to(cuda), s.width, s.height, sh_degree=tr.sh_degree_to_use(), render_mode=tr.cfg.render_mode,
                                      rasterize_mode=tr.cfg.rasterize_mode)
    return mo.image_metrics(render, alphas, s.gt_rgb, s.gt_depth, bg)


def _check_against_rasterization(tr, s, cuda, bg, what):
    got = tr.evaluate(s.viewmats.to(cuda), s.Ks.to(cuda), s.width, s.height, s.gt_rgb.to(cuda), s.gt_depth.to(cuda), bg.to(cuda))
    got = torch.stack([got[n] for n in METRIC_NAMES], 1).cpu().numpy()
    want = _expected(tr, s, cuda, bg)
    # two renders of the same Gaussians (exp / sigmoid in the kernel or on the host): forward tolerances, not bits
    np.testing.assert_allclose(got[:, 0], want[:, 0], rtol=0, atol=2e-3, err_msg=f"{what} psnr")
    np.testing.assert_allclose(got[:, 1], want[:, 1], rtol=0, atol=2e-4, err_msg=f"{what} ssim")
    np.testing.assert_allclose(got[:, 2:10], want[:, 2:10], rtol=2e-3, atol=2e-3, err_msg=f"{what} metrics")
    np.testing.assert_array_equal(got[:, 10], want[:, 10])
    return got


@pytest.mark.parametrize("case", ["downscales", "camera_opt", "bilagrid", "chunks"])
def test_evaluate_equals_rasterization_and_oracle(cuda, case):
    C = EVAL_CHUNK_VIEWS + 3 if case == "chunks" else 3
    s = _scene(C)
    bg = torch.tensor([0.2, 0.3, 0.4])
    cfg = dict(downscales=TrainConfig(num_downscales=2), camera_opt=TrainConfig(camera_optimizer="SO3xR3"),
               bilagrid=TrainConfig(use_bilateral_grid=True, bilateral_grid_shape=(4, 4, 4)), chunks=TrainConfig())[case]
    tr = _trainer(s, cuda, cfg, num_cameras=C)
    if case == "camera_opt":
        tr.pose_adjustment.copy_(0.05 * torch.randn(C, 6, generator=torch.Generator().manual_seed(1)).to(cuda))
    if case == "bilagrid":
        g = tr.bilateral_grids
        g.add_(0.2 * torch.randn(g.shape, generator=torch.Generator().manual_seed(2)).to(cuda))
    assert tr.downscale_factor() == (4 if case == "downscales" else 1)
    got = _check_against_rasterization(tr, s, cuda, bg, case)
    if case == "chunks":  # a view's row does not depend on the chunk it is rendered in (what the multi-GPU rows rely on)
        for c in (0, C - 1):
            one = tr.evaluate(s.viewmats[c:c + 1].to(cuda), s.Ks[c:c + 1].to(cuda), s.width, s.height, s.gt_rgb[c:c + 1].to(cuda),
                              s.gt_depth[c:c + 1].to(cuda), bg.to(cuda))
            one = torch.stack([one[n] for n in METRIC_NAMES], 1).cpu().numpy()
            assert np.array_equal(one[0].view(np.int64), got[c].view(np.int64)), c


def test_evaluate_changes_no_training_state(cuda):
    s = _scene(3)
    bg = torch.tensor([0.2, 0.3, 0.4]).to(cuda)
    cfg = TrainConfig(camera_optimizer="SO3xR3", use_bilateral_grid=True, bilateral_grid_shape=(4, 4, 4), warmup_length=0, refine_every=2)
    trs = [_trainer(s, cuda, cfg, num_cameras=3) for _ in range(2)]
    c2w = camera_to_worlds(s.viewmats).to(cuda)
    ids = torch.arange(3, device=cuda)
    args = (s.Ks.to(cuda), s.width, s.height, s.gt_rgb.to(cuda), s.gt_depth.to(cuda), bg)
    for tr in trs:
        tr.step(None, *args, camera_to_worlds=c2w, camera_ids=ids)
    before = trs[0].state_dict()
    f = trs[0]._fused
    sizing = (f._cap_isects, {k: (v.dtype, v.numel(), v.data_ptr()) for k, v in f._buf.items()})
    for _ in range(2):  # a batch larger than the step's, whose lists and buffers would be larger than the step's
        trs[0].evaluate(get_viewmat(c2w).repeat(4, 1, 1), s.Ks.to(cuda).repeat(4, 1, 1), s.width, s.height, s.gt_rgb.to(cuda).repeat(4, 1, 1, 1),
                        s.gt_depth.to(cuda).repeat(4, 1, 1, 1), bg)
    after = trs[0].state_dict()
    # the step's buffers and intersection capacity stay those of its own views: what the next step launches is unchanged
    assert (f._cap_isects, {k: (v.dtype, v.numel(), v.data_ptr()) for k, v in f._buf.items()}) == sizing

    def same(x, y):
        if isinstance(x, dict):
            return x.keys() == y.keys() and all(same(x[k], y[k]) for k in x)
        if isinstance(x, torch.Tensor):
            return x.dtype == y.dtype and x.shape == y.shape and torch.equal(x.view(torch.uint8), y.view(torch.uint8))
        return x == y

    assert same(before, after)
    # training continues, and the next step is the one the twin without evaluate() takes (up to the atomics of the backward)
    losses = [tr.step(None, *args, camera_to_worlds=c2w, camera_ids=ids)[0].cpu() for tr in trs]
    assert torch.isfinite(losses[0]).all() and torch.allclose(losses[0], losses[1], rtol=1e-5, atol=0)
    for k, v in trs[0].state_dict()["gauss_params"].items():
        w = trs[1].state_dict()["gauss_params"][k]
        assert torch.allclose(v, w, rtol=1e-4, atol=1e-6), k


@pytest.mark.skipif(reference_root() is None, reason="reference package not found")
def test_depth_columns_match_the_reference_depth_metrics(cuda):
    ref = reference_root()
    paths = [os.path.join(ROOT, "tests", "stubs"), ref]
    sys.path[:0] = paths
    try:
        from qed_splatter.metrics import DepthMetrics
    finally:
        for p in paths:
            sys.path.remove(p)
    render, alphas, gt_rgb, gt_depth, bg = _views(3, 64, 48, False, False, seed=3)
    gt_depth = torch.nan_to_num(gt_depth, nan=0.0)  # DepthMetrics takes gt > tolerance, without the finiteness test
    got = image_metrics(render.to(cuda), alphas.to(cuda), gt_rgb.to(cuda), gt_depth.to(cuda), bg.to(cuda), depth_tolerance=0.1)
    for c in (0, 1):
        depth = torch.where(alphas[c] > 0, render[c, ..., 3:4], render[c, ..., 3].max().clamp_min(0))
        want = DepthMetrics(tolerance=0.1)(depth[None].permute(0, 3, 1, 2).double(), gt_depth[c][None, None].double())
        for name, w in zip(("abs_rel", "sq_rel", "rmse", "rmse_log", "a1", "a2", "a3"), want):
            assert float(got[name][c]) == pytest.approx(float(w), rel=1e-6), name
