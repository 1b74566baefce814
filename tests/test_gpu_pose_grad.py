"""-m gpu: camera pose gradients (v_viewmats) of the projection backward, get_viewmat and the fused step, against the
oracle's autograd (itself checked against finite differences in tests/test_pose_grad_cpu.py)."""
import functools
import json
import math
import os

import pytest
import torch

import oracle
from oracle import torch_impl as ti
from qed_splatter_b200 import _lib, depth_supervised_loss, get_viewmat, ops, rasterization
from qed_splatter_b200.pipeline import FusedSplatStep
from qed_splatter_b200.scenes import scene_s0
import reference_model as rm
from helpers import scene_args

pytestmark = pytest.mark.gpu

_LOG = os.environ.get("QED_PARITY_LOG")
# Largest per-camera error / block norm measured on a B200 (1000 W power limit) over this file: stage parity 3.0e-6
# (against 1e-4), end to end 7.4e-5 (RGB; compositor threshold flips and float atomics), fused step vs autograd 6.5e-9.
E2E_TOL = 1e-3


def _block_close(got, ref, tol, what):
    """v_viewmats [C,4,4]: v_W and v_t of every camera within tol x that block's norm of the reference; row 3 zero."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert torch.equal(got[:, 3], torch.zeros_like(got[:, 3])), f"{what}: row 3 not zero"
    worst = 0.0
    for c in range(ref.shape[0]):
        for name, sl in (("v_W", (slice(0, 3), slice(0, 3))), ("v_t", (slice(0, 3), 3))):
            r, g = ref[c][sl], got[c][sl]
            err = float((g - r).abs().max())
            norm = float(r.norm())
            rel = err / max(norm, 1e-30)
            worst = max(worst, rel if norm > 0 else 0.0)
            if _LOG:
                with open(_LOG, "a") as f:
                    f.write(json.dumps({"what": f"{what} cam{c} {name}", "max_abs_err": err, "norm": norm, "rel": rel, "tol": tol}) + "\n")
            assert err <= tol * norm + 1e-30, f"{what} camera {c} {name}: max error {err:.3e} > {tol:g} x norm {norm:.3e}"
    return worst


def _oracle_projection(a, width, height, sh_degree, antialiased, viewmats):
    """The projection stage of oracle.rasterization (RGB+D): -> means2d, depths, conics, colors[C,N,4], opacities."""
    radii, means2d, depths, conics, comps = oracle.fully_fused_projection(a["means"], a["quats"], a["scales"], viewmats, a["Ks"], width,
                                                                        height, calc_compensations=antialiased)
    C, N = radii.shape
    opac = a["opacities"][None].expand(C, N)
    if comps is not None:
        opac = opac * comps
    if sh_degree is None:
        cols = a["colors"][None].expand(C, N, 3)
    else:
        dirs = a["means"][None] - ti.camera_positions(viewmats)[:, None]
        cols = torch.clamp_min(oracle.spherical_harmonics(sh_degree, dirs, a["colors"][None].expand(C, *a["colors"].shape), masks=radii > 0) + 0.5, 0.0)
    cols = torch.cat([cols, depths[..., None]], dim=-1)
    return radii, means2d, depths, conics, cols, opac


TERMS = {"mean": ("means2d", "depths"), "conic": ("conics",), "color": ("colors",), "opacity": ("opacities",),
         "all": ("means2d", "depths", "conics", "colors", "opacities")}


def _scene(C, sh_degree):
    s = scene_s0(C=8)
    if C == 1:
        s.viewmats, s.Ks = s.viewmats[:1].contiguous(), s.Ks[:1].contiguous()
    a = scene_args(s)
    if sh_degree is None:
        a["colors"] = torch.rand(a["means"].shape[0], 3, generator=torch.Generator().manual_seed(7))
    return s, a


def _gpu_projection(a, cuda, s, sh_degree, antialiased, pose):
    leaves = {k: a[k].to(cuda).requires_grad_(True) for k in ("means", "quats", "scales", "opacities", "colors")}
    vm = a["viewmats"].to(cuda).requires_grad_(pose)
    out = ops.project_gaussians(leaves["means"], leaves["quats"], leaves["scales"], leaves["opacities"], leaves["colors"], vm,
                                a["Ks"].to(cuda), s.width, s.height, calc_compensations=antialiased, sh_degree=sh_degree)
    radii, means2d, depths, conics, _, cols, opac = out[:7]
    return leaves, vm, dict(radii=radii, means2d=means2d, depths=depths, conics=conics, colors=cols, opacities=opac)


@pytest.mark.parametrize("C", [1, 8])
@pytest.mark.parametrize("antialiased", [False, True])
@pytest.mark.parametrize("sh_degree", [None, 0, 3])
def test_stage_parity_per_term(cuda, C, antialiased, sh_degree):
    """ops.project_gaussians backward with fixed upstream gradients, one term at a time: no compositing, so no threshold
    flip can hide a missing term (the SH direction term in particular)."""
    s, a = _scene(C, sh_degree)
    vm_o = a["viewmats"].clone().requires_grad_(True)
    leaves_o = {k: a[k].clone().requires_grad_(True) for k in ("means", "quats", "scales", "opacities", "colors")}
    radii_o, *outs_o = _oracle_projection({**a, **leaves_o}, s.width, s.height, sh_degree, antialiased, vm_o)
    outs_o = dict(zip(("means2d", "depths", "conics", "colors", "opacities"), outs_o))
    leaves_g, vm_g, outs_g = _gpu_projection(a, cuda, s, sh_degree, antialiased, pose=True)
    assert torch.equal(outs_g["radii"].cpu(), radii_o)
    gen = torch.Generator().manual_seed(11)
    ups = {k: torch.randn(v.shape, generator=gen) * (radii_o > 0)[(...,) + (None,) * (v.dim() - 2)] for k, v in outs_o.items()}
    for term, keys in TERMS.items():
        got = torch.autograd.grad([outs_g[k] for k in keys], vm_g, [ups[k].to(cuda) for k in keys], retain_graph=True)[0]
        assert got.dtype == vm_g.dtype and got.shape == (C, 4, 4)
        if term == "opacity" and not antialiased:
            assert float(got.abs().max()) == 0.0  # opacity * compensation: no pose dependence without compensation
            continue
        ref = torch.autograd.grad([outs_o[k] for k in keys], vm_o, [ups[k] for k in keys], retain_graph=True)[0]
        _block_close(got, ref, 1e-4, f"stage {term} C={C} aa={antialiased} sh={sh_degree}")

    # the other parameter gradients do not change when the pose gradient is computed too
    keys = TERMS["all"]
    g_pose = torch.autograd.grad([outs_g[k] for k in keys], list(leaves_g.values()), [ups[k].to(cuda) for k in keys])
    leaves_d, _, outs_d = _gpu_projection(a, cuda, s, sh_degree, antialiased, pose=False)
    g_def = torch.autograd.grad([outs_d[k] for k in keys], list(leaves_d.values()), [ups[k].to(cuda) for k in keys])
    # (the pose variants are separate compilations: in the degree-3 kernels ptxas contracts a few products of v_means
    # differently -- measured 5.4e-8 of max |v_means| on a B200; every other gradient was bit-identical)
    for name, x, y in zip(leaves_g, g_pose, g_def):
        err, scale = float((x - y).abs().max()), float(y.abs().max())
        if _LOG:
            with open(_LOG, "a") as f:
                f.write(json.dumps({"what": f"other grads v_{name} C={C} aa={antialiased} sh={sh_degree}", "bit_identical": bool(torch.equal(x, y)),
                                    "rel": err / max(scale, 1e-30)}) + "\n")
        assert err <= 1e-6 * scale, f"v_{name} changed with pose gradients on: {err:.3e} vs max |v| {scale:.3e}"


def _call_pose_bwd(lib, s, a, dev, packed, radii, conics, C, N):
    """qed_project_bwd_pose on a fixed packed gradient record (fused path, RGB+D, SH degree 3)."""
    t = {k: v.to(dev).contiguous() for k, v in a.items()}
    outs = dict(v_means=torch.empty(N, 3, device=dev), v_quats=torch.empty(N, 4, device=dev), v_scales=torch.empty(N, 3, device=dev),
                v_opac=torch.empty(N, device=dev), v_sh=torch.empty(N, 16, 3, device=dev), v_vm=torch.full((C, 4, 4), float("nan"), device=dev))
    ws_bytes = lib.qed_project_bwd_pose_workspace_bytes(C, N)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
    p = _lib.ptr
    _lib.check(lib.qed_project_bwd_pose(C, N, p(t["means"]), p(t["quats"]), p(t["scales"]), p(t["opacities"]), 0, p(t["colors"]), 16, 3, 0,
                                        p(t["viewmats"]), p(t["Ks"]), s.width, s.height, 0.3, 0, 3, 1, p(radii), p(conics), None, None, None,
                                        None, None, None, p(packed), p(outs["v_means"]), p(outs["v_quats"]), p(outs["v_scales"]),
                                        p(outs["v_opac"]), p(outs["v_sh"]), p(outs["v_vm"]), p(ws), ws_bytes, _lib.current_stream()),
               "qed_project_bwd_pose")
    torch.cuda.synchronize()
    return outs


def test_deterministic_culled_and_empty(cuda):
    lib = _lib.load()
    s = scene_s0()
    a = scene_args(s)
    N, C = s.N, s.C
    radii, _, _, conics = ops.project_gaussians(*(a[k].to(cuda) for k in ("means", "quats", "scales", "opacities", "colors", "viewmats", "Ks")),
                                                s.width, s.height, sh_degree=3)[:4]
    packed = torch.randn(C * N, 12, generator=torch.Generator().manual_seed(5)).to(cuda)
    o1 = _call_pose_bwd(lib, s, a, cuda, packed, radii, conics, C, N)
    o2 = _call_pose_bwd(lib, s, a, cuda, packed, radii, conics, C, N)
    assert float(o1["v_vm"].abs().max()) > 0
    for k in o1:
        assert torch.equal(o1[k], o2[k]), k  # bit-identical: no atomics, fixed-order sums
    # every Gaussian culled: exactly zero
    o3 = _call_pose_bwd(lib, s, a, cuda, packed, torch.zeros_like(radii), conics, C, N)
    assert torch.equal(o3["v_vm"], torch.zeros_like(o3["v_vm"]))
    # C = 0 and N = 0 return cleanly; N = 0 writes zeros
    e = _call_pose_bwd(lib, s, {k: (v[:0] if k in ("means", "quats", "scales", "opacities", "colors") else v) for k, v in a.items()}, cuda,
                       packed[:0], radii[:, :0].contiguous(), conics[:, :0].contiguous(), C, 0)
    assert torch.equal(e["v_vm"], torch.zeros_like(e["v_vm"]))
    _call_pose_bwd(lib, s, {**a, "viewmats": a["viewmats"][:0], "Ks": a["Ks"][:0]}, cuda, packed[:0], radii[:0], conics[:0], 0, N)


def _loss_oracle(render, alpha, mode, gt_rgb, gt_depth, bg):
    """depth-L1 + RGB-L1 of test_config0_full_parity, per camera (depth_supervised_loss averages per camera), for any mode."""
    total = 0.0
    for c in range(render.shape[0]):
        r, al = render[c:c + 1], alpha[c:c + 1]
        if mode in ("RGB", "RGB+D", "RGB+ED"):
            rgb = torch.clamp(r[..., :3] + (1 - al) * bg, 0.0, 1.0)
            total = total + oracle.rgb_l1_loss(rgb, gt_rgb[c:c + 1])
        if mode != "RGB":
            d = r[..., -1:]
            d = torch.where(al > 0, d, d.detach().max())
            total = total + oracle.depth_l1_loss(d, gt_depth[c:c + 1], 0.2)
    return total / render.shape[0]


@pytest.mark.parametrize("mode", ["RGB", "D", "ED", "RGB+D", "RGB+ED"])
def test_end_to_end_parity(cuda, mode):
    """rasterization(pose_gradients=True) through the compositor against oracle.rasterization's viewmats.grad."""
    s = scene_s0()
    a = scene_args(s)
    bg = torch.tensor([0.2, 0.5, 0.8])
    vm_o = a["viewmats"].clone().requires_grad_(True)
    ro, ao, _ = oracle.rasterization(**{**a, "viewmats": vm_o}, width=s.width, height=s.height, render_mode=mode, sh_degree=3)
    _loss_oracle(ro, ao, mode, s.gt_rgb, s.gt_depth[..., None] if s.gt_depth.dim() == 3 else s.gt_depth, bg).backward()
    ag = scene_args(s, cuda)
    vm_g = ag["viewmats"].requires_grad_(True)
    rg, alg, _ = rasterization(**ag, width=s.width, height=s.height, render_mode=mode, sh_degree=3, pose_gradients=True)
    gd = s.gt_depth.to(cuda)
    _loss_oracle(rg, alg, mode, s.gt_rgb.to(cuda), gd[..., None] if gd.dim() == 3 else gd, bg.to(cuda)).backward()
    _block_close(vm_g.grad, vm_o.grad, E2E_TOL, f"e2e {mode}")


def test_get_viewmat_backward(cuda):
    from test_data_side_cpu import _rand_c2w

    for rows in (3, 4):
        c2w = torch.from_numpy(_rand_c2w(9, seed=13, rows=rows))
        w = torch.randn(9, 4, 4, generator=torch.Generator().manual_seed(rows))
        x_o = c2w.clone().requires_grad_(True)
        (oracle.get_viewmat(x_o) * w).sum().backward()
        x_g = c2w.to(cuda).requires_grad_(True)
        out = get_viewmat(x_g, pose_gradients=True)
        assert torch.equal(out.detach(), get_viewmat(c2w.to(cuda)))  # same forward bits
        (out * w.to(cuda)).sum().backward()
        assert x_g.grad.shape == c2w.shape
        torch.testing.assert_close(x_g.grad.cpu(), x_o.grad, rtol=1e-6, atol=1e-6)
        if rows == 4:
            assert float(x_g.grad[:, 3].abs().max()) == 0.0


def _c2w_of(viewmats):
    W, t = viewmats[:, :3, :3], viewmats[:, :3, 3:]
    R = W.transpose(1, 2)
    return torch.cat([R * torch.tensor([[[1.0, -1.0, -1.0]]], dtype=R.dtype, device=R.device), -(R @ t)], dim=-1).contiguous()


def test_c2w_chain_matches_oracle(cuda):
    """c2w -> get_viewmat -> rasterization -> depth_supervised_loss against the oracle chain's c2w.grad."""
    s = scene_s0(C=2, size=128)
    a = scene_args(s)
    bg = torch.tensor([0.2, 0.5, 0.8])
    c2w = _c2w_of(a["viewmats"])
    x_o = c2w.clone().requires_grad_(True)
    ro, ao, _ = oracle.rasterization(**{**a, "viewmats": oracle.get_viewmat(x_o)}, width=s.width, height=s.height, render_mode="RGB+ED", sh_degree=3)
    gd = s.gt_depth[..., None] if s.gt_depth.dim() == 3 else s.gt_depth
    _loss_oracle(ro, ao, "RGB+ED", s.gt_rgb, gd, bg).backward()
    ag = scene_args(s, cuda)
    x_g = c2w.to(cuda).requires_grad_(True)
    rg, alg, _ = rasterization(**{**ag, "viewmats": get_viewmat(x_g, pose_gradients=True)}, width=s.width, height=s.height,
                               render_mode="RGB+ED", sh_degree=3, pose_gradients=True)
    total, _, _ = depth_supervised_loss(rg, alg, s.gt_rgb.to(cuda), s.gt_depth.to(cuda), bg.to(cuda))
    total.backward()
    g, r = x_g.grad.double().cpu(), x_o.grad.double()
    for c in range(s.C):
        for sl in ((slice(0, 3), slice(0, 3)), (slice(0, 3), 3)):
            err, norm = float((g[c][sl] - r[c][sl]).abs().max()), float(r[c][sl].norm())
            assert err <= E2E_TOL * norm, (c, err, norm)


def test_fused_step_pose_gradients(cuda):
    s = scene_s0(C=2, size=128)
    a = scene_args(s, cuda)
    bg = torch.tensor([0.2, 0.5, 0.8], device=cuda)
    gt_rgb, gt_depth = s.gt_rgb.to(cuda), s.gt_depth.to(cuda)
    fs = FusedSplatStep(cuda)
    args = (a["means"], a["quats"], a["scales"], a["opacities"], a["colors"], a["viewmats"], a["Ks"], s.width, s.height, 3, gt_rgb, gt_depth, bg)
    assert fs.step(*args).v_viewmats is None
    calls = []
    out = fs.step(*args, pose_gradients=True, on_chunk=lambda k, n0, n1: calls.append((k, n0, n1)))
    assert calls == [(0, 0, s.N)]  # the per-range callback fires on the pose path too
    v_step = out.v_viewmats.clone()
    vm = a["viewmats"].clone().requires_grad_(True)
    rg, alg, _ = rasterization(**{**a, "viewmats": vm}, width=s.width, height=s.height, render_mode="RGB+ED", sh_degree=3, pose_gradients=True)
    depth_supervised_loss(rg, alg, gt_rgb, gt_depth, bg)[0].backward()
    _block_close(v_step, vm.grad, E2E_TOL, "fused step vs autograd")
    with pytest.raises(ValueError):
        fs.step(*args, pose_gradients=True, exchange=object())
    with pytest.raises(ValueError):
        fs.step(*args, pose_gradients=True, n_chunks=2)


def _rodrigues(w):
    th = torch.sqrt((w * w).sum() + 1e-24)
    k = w / th
    Kx = torch.stack([torch.stack([0 * th, -k[2], k[1]]), torch.stack([k[2], 0 * th, -k[0]]), torch.stack([-k[1], k[0], 0 * th])])
    return torch.eye(3, device=w.device) + torch.sin(th) * Kx + (1 - torch.cos(th)) * (Kx @ Kx)


def test_pose_recovery(cuda):
    """Adam on a 6-vector pose adjustment through get_viewmat and rasterization recovers a perturbed camera.
    Measured on a B200: 1.5 deg -> below the float32 resolution of the angle, 0.06 -> 1.1e-4 in translation."""
    s = scene_s0(C=1, size=128)
    a = scene_args(s, cuda)
    bg = torch.tensor([0.2, 0.5, 0.8], device=cuda)
    c2w_true = _c2w_of(a["viewmats"])[0]
    with torch.no_grad():
        gt, gt_a, _ = rasterization(**a, width=128, height=128, render_mode="RGB+ED", sh_degree=3)
    gt_rgb = torch.clamp(gt[..., :3] + (1 - gt_a) * bg, 0, 1)
    gt_depth = torch.where(gt_a[..., 0] > 0.5, gt[..., 3], torch.zeros_like(gt[..., 3]))
    dist = float(c2w_true[:, 3].norm())
    gen = torch.Generator().manual_seed(3)
    axis = torch.randn(3, generator=gen)
    axis = axis / axis.norm()
    dirn = torch.randn(3, generator=gen)
    dirn = dirn / dirn.norm()
    R0 = c2w_true[:, :3] @ _rodrigues((axis * math.radians(1.5)).to(cuda))
    T0 = c2w_true[:, 3] + (dirn * 0.02 * dist).to(cuda)
    delta = torch.zeros(6, device=cuda, requires_grad=True)
    opt = torch.optim.Adam([delta], lr=5e-3)
    sched = torch.optim.lr_scheduler.ExponentialLR(opt, gamma=0.99)

    def pose():
        return torch.cat([R0 @ _rodrigues(delta[:3]), (T0 + delta[3:])[:, None]], dim=1)[None]

    def errors():
        with torch.no_grad():
            p = pose()[0]
            cosang = ((torch.trace(c2w_true[:, :3].T @ p[:, :3]) - 1) / 2).clamp(-1, 1)
            return math.degrees(float(torch.acos(cosang))), float((p[:, 3] - c2w_true[:, 3]).norm())

    e_rot0, e_t0 = errors()
    trace = []
    for it in range(200):
        if it % 20 == 0:
            trace.append(errors())
        opt.zero_grad()
        vm = get_viewmat(pose(), pose_gradients=True)
        r, al, _ = rasterization(**{**a, "viewmats": vm}, width=128, height=128, render_mode="RGB+ED", sh_degree=3, pose_gradients=True)
        depth_supervised_loss(r, al, gt_rgb, gt_depth, bg)[0].backward()
        opt.step()
        sched.step()
    e_rot, e_t = errors()
    if _LOG:
        with open(_LOG, "a") as f:
            f.write(json.dumps({"what": "pose recovery", "rot_deg": [e_rot0, e_rot], "trans": [e_t0, e_t], "trace": trace}) + "\n")
    assert e_rot <= e_rot0 / 5 and e_t <= e_t0 / 5, (e_rot0, e_rot, e_t0, e_t)


def _adjust(c2w, adj):
    """Pose adjustment applied to nerfstudio camera-to-world [C,3,4]: rotation exp(adj[:3]) on the right, translation + adj[3:]."""
    R = c2w[:, :3, :3] @ _rodrigues(adj[:3]).to(c2w.dtype)
    return torch.cat([R, c2w[:, :3, 3:] + adj[3:].to(c2w.dtype)[None, :, None]], dim=-1)


class _PoseAdjustment(torch.nn.Module):
    """Stands in for splatfacto's CameraOptimizer in a mode other than "off": a learnable 6-vector per model, applied where
    model.py:212 asks `self.camera_optimizer.apply_to_camera(camera)`."""

    def __init__(self, init):
        super().__init__()
        self.adj = torch.nn.Parameter(init.clone())

    def apply_to_camera(self, camera):
        return _adjust(camera.camera_to_worlds, self.adj)


@pytest.mark.skipif(rm.reference_root() is None, reason="reference package not available (see tests/reference_model.py)")
def test_reference_model_with_pose_gradients(cuda):
    """The unmodified QEDSplatterModel with `rasterization` and `get_viewmat` bound with pose_gradients=True (INTEGRATION.md
    2b) and a pose adjustment as its camera optimizer: the adjustment's gradient equals the same chain written with the
    oracle (`oracle_reference_step` on the adjusted pose)."""
    s = scene_s0(N=3000, C=2, size=96)
    cam = 1
    init = torch.tensor([0.004, -0.006, 0.003, 0.02, -0.01, 0.015])
    with rm.reference_modules("cuda") as mod:
        mod.rasterization = functools.partial(rasterization, pose_gradients=True)
        mod.get_viewmat = functools.partial(get_viewmat, pose_gradients=True)
        model = rm.build_model(mod, s, cuda, step=3000)
        model.camera_optimizer = _PoseAdjustment(init.to(cuda))
        model.train()
        camera = rm.make_camera(s, cam, cuda)
        out = model.get_outputs(camera)
        loss = model.get_loss_dict(out, {"image": s.gt_rgb[cam].to(cuda), "depth_image": s.gt_depth[cam].to(cuda)})
        sum(loss.values()).backward()
        got = model.camera_optimizer.adj.grad.detach().double().cpu()
        bg = model._get_background_color().detach().cpu()
        c2w = camera.camera_to_worlds.detach().cpu()
    adj = init.clone().requires_grad_(True)
    _, ref_loss, _ = rm.oracle_reference_step(s, cam, _adjust(c2w, adj), bg, step=3000)
    sum(ref_loss.values()).backward()
    ref = adj.grad.double()
    for name, sl in (("rotation", slice(0, 3)), ("translation", slice(3, 6))):
        err, norm = float((got[sl] - ref[sl]).abs().max()), float(ref[sl].norm())
        assert norm > 0 and err <= E2E_TOL * norm, f"{name}: max error {err:.3e} > {E2E_TOL:g} x norm {norm:.3e}"
