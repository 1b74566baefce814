"""-m gpu: compositing at the opacity clamp (alpha = min(0.999, opacity * exp(-sigma))) and at the transmittance cutoff.

Trained splatfacto scenes have many opacities above sigmoid(6.9) = 0.999.  There the compositors clamp alpha, the
backward passes no gradient through a clamped alpha and reconstructs the transmittance through 1 / (1 - 0.999), and
a pixel stops after a few opaque layers (T <= 1e-4).  The scenes here are built so that a real share of the composited
pairs is clamped and of the pixels terminates, checked against the float64 oracle with the suite's standard tolerances.
"""
import functools
import math

import pytest
import torch

import oracle
from oracle import torch_impl
from qed_splatter_b200 import ops
from qed_splatter_b200.pipeline import FusedSplatStep
from qed_splatter_b200.scenes import scene_s0
from helpers import assert_close_frac

pytestmark = pytest.mark.gpu

OPACITY_LEVELS = (1.0, 0.99999, 0.9992, 0.999, 0.9989, 0.995)
W, H, C, LAYERS = 72, 56, 2, 4  # 4.5 x 3.5 tiles: clipped tiles on the right and bottom edges
SEEDS = {False: 1, True: 12}


def _cov_to_conic(cov):
    a, b, c = cov[..., 0, 0], cov[..., 0, 1], cov[..., 1, 1]
    det = a * c - b * b
    return torch.stack([c / det, -b / det, a / det], -1)


def _stacks(g, n_cols, lo, hi):
    """n_cols pixel positions per view, each with a stack of 1..LAYERS Gaussians (layer k at depth ~1 + k), centred
    0.004..0.010 px from the pixel centre: at a 0.3..1.2 px Gaussian's pixel alpha_raw = opacity * (0.9989 .. 0.99999), so
    opacities >= 0.99999 are mostly clamped there and 0.9992 sometimes, and a stack of near-opaque layers ends the pixel's loop after two to four layers.
    -> means2d [C,n,2], covariance [C,n,2,2], depth [C,n] (float64); n = n_cols * LAYERS, unused slots have radius 0."""
    px = torch.randint(0, W, (C, n_cols), generator=g).double() + 0.5
    py = torch.randint(0, H, (C, n_cols), generator=g).double() + 0.5
    height = torch.randint(1, LAYERS + 1, (C, n_cols), generator=g)
    n = n_cols * LAYERS
    off = 0.004 + 0.006 * torch.rand(C, n, 2, generator=g, dtype=torch.float64)
    off = off * torch.where(torch.rand(C, n, 2, generator=g) < 0.5, -1.0, 1.0).double()
    means2d = torch.stack([px, py], -1).repeat(1, LAYERS, 1) + off  # slot k * n_cols + j: layer k of column j
    sx = lo + (hi - lo) * torch.rand(C, n, generator=g, dtype=torch.float64)
    sy = lo + (hi - lo) * torch.rand(C, n, generator=g, dtype=torch.float64)
    rho = 0.6 * torch.rand(C, n, generator=g, dtype=torch.float64) - 0.3
    cov = torch.stack([torch.stack([sx * sx, rho * sx * sy], -1), torch.stack([rho * sx * sy, sy * sy], -1)], -2)
    layer = torch.arange(n) // n_cols
    present = layer[None] < height.repeat(1, LAYERS)
    depths = 1.0 + layer.double()[None] + 0.5 * torch.rand(C, n, generator=g, dtype=torch.float64)  # distinct, layer by layer
    return means2d, cov, depths, present


@functools.lru_cache(maxsize=None)
def layered_scene(antialiased: bool):
    """Stacks of 2D Gaussians (`_stacks`) with opacities from OPACITY_LEVELS, sizes 0.3..1.2 px.  Antialiased: the
    opacities times the compensation sqrt(det S / det (S + 0.3 I)) and the conics of S + 0.3 I, plus stacks of large
    Gaussians (20..40 px) whose compensation is close enough to 1 that opacity x compensation lies on both sides of
    0.999.  The seeds are ones whose pairs all keep a margin from the clamp and the cutoff (asserted below).
    -> float32 CPU tensors."""
    g = torch.Generator().manual_seed(SEEDS[antialiased])
    means2d, cov, depths, present = _stacks(g, 200, 0.3, 1.2)
    if antialiased:  # the large ones in front: their clamped centres are not hidden behind opaque small ones
        m_big, c_big, d_big, p_big = _stacks(g, 15, 20.0, 40.0)
        means2d, cov, depths, present = (torch.cat(t, 1) for t in ((means2d, m_big), (cov, c_big), (depths, d_big - 0.6), (present, p_big)))
    n = means2d.shape[1]
    op = torch.tensor(OPACITY_LEVELS, dtype=torch.float64)[torch.randint(0, len(OPACITY_LEVELS), (C, n), generator=g)]
    if antialiased:
        blurred = cov + 0.3 * torch.eye(2, dtype=torch.float64)
        comp = torch.sqrt(torch.linalg.det(cov) / torch.linalg.det(blurred))
        op, cov = op * comp, blurred
    conics = _cov_to_conic(cov)
    eig = torch.linalg.eigvalsh(cov)[..., 1]
    radii = torch.ceil(3.0 * torch.sqrt(eig)).to(torch.int32) * present
    colors = torch.rand(C, n, 4, generator=g)
    f32 = lambda t: t.float().contiguous()
    m2, cn, opac, dep = f32(means2d), f32(conics), f32(op), f32(depths)
    tw, th = ops.tile_grid(W, H, 16)
    _, ids, flat = oracle.isect_tiles(m2, radii, dep, 16, tw, th)
    offsets = oracle.isect_offset_encode(ids, C, tw, th)
    return dict(means2d=m2, conics=cn, opacities=opac, colors=colors, offsets=offsets, flat=flat)


def pair_stats(means2d, conics, opacities, width, height, offsets, flat, max_alpha=torch_impl.MAX_ALPHA):
    """From the oracle's per-tile arithmetic (float64): composited pairs, how many of them are clamped, pixels whose
    transmittance reaches the cutoff, and the smallest relative distances of a pair to the clamp and (pairs that weigh
    in a pixel) to the cutoff."""
    Cn, Nn = opacities.shape
    th, tw = offsets.shape[1:]
    m2, cn, op = (t.double().reshape(Cn * Nn, -1) for t in (means2d, conics, opacities))
    op = op[:, 0]
    fid = flat.to(torch.int64)
    st = dict(pairs=0, clamped=0, pixels=0, terminated=0, clamp_margin=math.inf, cutoff_margin=math.inf)
    for c, ty, tx, s, e in torch_impl._tile_iter(Cn, th, tw, offsets, flat.numel()):
        _, _, px, py = torch_impl._tile_pixels(ty, tx, 16, width, height, torch.float64)
        st["pixels"] += px.numel()
        if e <= s:
            continue
        gi = fid[s:e]
        _, _, _, _, alpha_raw, alpha, T_before, included = torch_impl._tile_forward(px, py, m2[gi], cn[gi], op[gi])
        valid = alpha > 0
        T_after = T_before * (1.0 - alpha)
        st["pairs"] += int(included.sum())
        st["clamped"] += int((included & (alpha_raw > max_alpha)).sum())
        st["terminated"] += int((valid & (T_after <= torch_impl.TRANSMITTANCE_THRESHOLD)).any(1).sum())
        live = valid & (T_before > torch_impl.TRANSMITTANCE_THRESHOLD)  # pairs the loop reaches (or stops at)
        if bool(live.any()):
            st["clamp_margin"] = min(st["clamp_margin"], float((alpha_raw[live] / max_alpha - 1.0).abs().min()))
        # (the cutoff flips a pair in or out of a pixel; only pairs of weight alpha * T >= 1e-5 could move a pixel visibly)
        heavy = live & (alpha * T_before >= 1e-5)
        if bool(heavy.any()):
            st["cutoff_margin"] = min(st["cutoff_margin"], float((T_after[heavy] / torch_impl.TRANSMITTANCE_THRESHOLD - 1.0).abs().min()))
    return st


@functools.lru_cache(maxsize=None)
def reference(antialiased: bool, D: int, bg: bool):
    sc = layered_scene(antialiased)
    gen = torch.Generator().manual_seed(100 * D + int(bg))
    cols = sc["colors"][..., :D].contiguous()
    bgs = torch.rand(C, D, generator=gen) if bg else None
    vr = torch.randn(C, H, W, D, generator=gen)
    va = torch.randn(C, H, W, 1, generator=gen)
    d = lambda t: None if t is None else t.double()
    args = (d(sc["means2d"]), d(sc["conics"]), d(cols), d(sc["opacities"]))
    render, alpha, last = oracle.rasterize_to_pixels(*args, W, H, 16, sc["offsets"], sc["flat"], backgrounds=d(bgs))
    grads = oracle.rasterize_to_pixels_bwd(*args, W, H, 16, sc["offsets"], sc["flat"], vr.double(), va[..., 0].double(), backgrounds=d(bgs))
    return dict(cols=cols, bgs=bgs, vr=vr, va=va, render=render, alpha=alpha, last=last, grads=grads)


@pytest.mark.timeout(120)
@pytest.mark.parametrize("antialiased", [False, True], ids=["classic", "antialiased"])
def test_scenes_reach_the_clamp_and_the_cutoff(cuda, antialiased):
    """The scenes are what the comparisons below rely on: many clamped pairs, pixels that terminate after a few layers
    and pixels that never do, and no pair so close to the clamp or the cutoff that float32 rounding could flip it."""
    sc = layered_scene(antialiased)
    st = pair_stats(sc["means2d"], sc["conics"], sc["opacities"], W, H, sc["offsets"], sc["flat"])
    # (a Gaussian is clamped within ~0.04 sigma of its centre and composited out to ~3.3 sigma: only the small ones give
    # a large share; the large ones of the antialiased scene add few clamped pairs and many composited ones)
    assert st["clamped"] >= (10 if antialiased else max(100, 0.005 * st["pairs"])), st
    assert st["terminated"] >= 0.02 * st["pixels"], st
    if not antialiased:  # (the large Gaussians of the antialiased scene end nearly every pixel)
        assert st["terminated"] <= 0.5 * st["pixels"], st
    assert st["clamp_margin"] > 2e-6 and st["cutoff_margin"] > 5e-5, st
    if antialiased:
        op = sc["opacities"].double()
        assert int(((op > 0.999) & (op < 0.99999)).sum()) > 10 and int(((op < 0.999) & (op > 0.998)).sum()) > 10, "compensated opacities straddle 0.999"


VARIANTS = {"packed": dict(packed=True, cull=True), "scalar": dict(packed=False, cull=True), "no_cull": dict(packed=True, cull=False)}


@pytest.mark.timeout(180)
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("D,bg", [(1, False), (1, True), (3, False), (3, True), (4, False), (4, True)])
@pytest.mark.parametrize("antialiased", [False, True], ids=["classic", "antialiased"])
def test_compositing_at_the_clamp_matches_oracle(cuda, antialiased, D, bg, variant):
    """Forward (render, alpha, last ids), backward (means2d, conics, colours, opacities) and absgrad of the compositors
    against the float64 oracle, for the packed kernels, the scalar kernels and with the warp-level culling off."""
    sc = layered_scene(antialiased)
    ref = reference(antialiased, D, bg)
    v = VARIANTS[variant]
    gl = [t.to(cuda).requires_grad_(True) for t in (sc["means2d"], sc["conics"], ref["cols"], sc["opacities"])]
    old_packed = ops.set_raster_packed(v["packed"])
    old_cull = ops.set_raster_cull(v["cull"])
    try:
        render, alpha, last = ops.rasterize_to_pixels(*gl, W, H, 16, sc["offsets"].to(cuda), sc["flat"].to(cuda),
                                                      backgrounds=ref["bgs"].to(cuda) if bg else None, absgrad=True, return_last_ids=True)
        ((render * ref["vr"].to(cuda)).sum() + (alpha * ref["va"].to(cuda)).sum()).backward()
        torch.cuda.synchronize()
    finally:
        ops.set_raster_packed(old_packed)
        ops.set_raster_cull(old_cull)
    assert_close_frac(render, ref["render"], 1e-4, 1e-4, 2e-3, "render")
    assert_close_frac(alpha, ref["alpha"], 1e-4, 1e-4, 2e-3, "alpha")
    assert float((last.cpu() != ref["last"]).float().mean()) < 2e-3, "last_ids"
    v_m, v_mabs, v_cn, v_co, v_op = ref["grads"]
    for name, got, want in (("means2d", gl[0].grad, v_m), ("conics", gl[1].grad, v_cn), ("colors", gl[2].grad, v_co),
                            ("opacities", gl[3].grad, v_op), ("absgrad", gl[0].absgrad, v_mabs)):
        scale = float(want.abs().mean()) + 1e-12
        assert_close_frac(got, want, 1e-3, 1e-3 * scale, 5e-3, f"v_{name}")


NAMES = ("means", "quats", "scales", "opacities", "sh")


def _ref_loss(render, alpha, gt_rgb, gt_depth, bg):
    total = 0.0
    for c in range(render.shape[0]):
        rgb, depth = oracle.composite_and_fill(render[c:c + 1], alpha[c:c + 1], bg)
        total = total + oracle.rgb_l1_loss(rgb, gt_rgb[c:c + 1]) + oracle.depth_l1_loss(depth, gt_depth[c:c + 1], 0.2)
    return total / render.shape[0]


@pytest.mark.timeout(300)
@pytest.mark.parametrize("mode", ["classic", "antialiased"])
def test_fused_step_with_saturated_logit_opacities(cuda, mode):
    """FusedSplatStep with the trainer's parametrisation (log scales, logit opacities in [6.5, 12], i.e. opacities
    0.9985 .. 0.999994) against the oracle's autograd through exp and sigmoid."""
    s = scene_s0(N=3000, C=2, size=80)
    g = torch.Generator().manual_seed(5)
    log_s = torch.log(s.scales * 2.0)
    logit = 6.5 + 5.5 * torch.rand(s.N, generator=g)
    leaves = {"means": s.means, "quats": s.quats, "scales": log_s, "opacities": logit, "sh": s.sh}
    lo = {k: v.clone().requires_grad_(True) for k, v in leaves.items()}
    bg = torch.tensor([0.3, 0.1, 0.6])
    ro, ao, io = oracle.rasterization(lo["means"], lo["quats"], torch.exp(lo["scales"]), torch.sigmoid(lo["opacities"]), lo["sh"], s.viewmats,
                                      s.Ks, s.width, s.height, sh_degree=3, render_mode="RGB+ED", rasterize_mode=mode)
    loss_o = _ref_loss(ro, ao, s.gt_rgb, s.gt_depth, bg)
    loss_o.backward()
    st = pair_stats(io["means2d"].detach(), io["conics"].detach(), io["opacities"].detach(), s.width, s.height, io["isect_offsets"], io["flatten_ids"])
    assert st["terminated"] >= 0.1 * st["pixels"], st
    if mode == "classic":  # (antialiased: the compensation keeps these small Gaussians' opacities well below the clamp)
        assert st["clamped"] >= 10, st

    fs = FusedSplatStep(cuda)
    d = {k: v.to(cuda) for k, v in leaves.items()}
    out = fs.step(d["means"], d["quats"], d["scales"], d["opacities"], d["sh"], s.viewmats.to(cuda), s.Ks.to(cuda), s.width, s.height, 3,
                  s.gt_rgb.to(cuda), s.gt_depth.to(cuda), bg.to(cuda), rasterize_mode=mode, activations=3)
    assert float(out.loss[0]) == pytest.approx(float(loss_o.detach()), rel=1e-4)
    assert_close_frac(out.render[..., :3], ro[..., :3], 1e-4, 1e-4, 2e-3, "render")
    assert_close_frac(out.alphas, ao, 1e-4, 1e-4, 2e-3, "alpha")
    for k in NAMES:
        scale = float(lo[k].grad.abs().mean()) + 1e-12
        assert_close_frac(out.grads[k], lo[k].grad, 1e-3, 1e-3 * scale, 5e-3, f"v_{k}")
