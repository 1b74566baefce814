"""-m gpu: splatfacto's SO3xR3 camera optimizer on the device -- the apply / backward / regulariser kernels against the float64
restatement (tests/camera_opt_oracle.py), the pose gradient of the multi-GPU exchange's projection backward, and the trainer
with the optimizer on (pose recovery; a frozen table renders exactly what the optimizer-off trainer renders)."""
import ctypes
import math
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import camera_opt_oracle as co
from helpers import scene_args
from qed_splatter_b200 import _lib, get_viewmat, rasterization
from qed_splatter_b200.camera_opt import CameraPoseOptimizer
from qed_splatter_b200.pipeline import FusedSplatStep
from qed_splatter_b200.scenes import camera_to_worlds, scene_s0
from qed_splatter_b200.trainer import GROUPS, SplatTrainer, TrainConfig

pytestmark = pytest.mark.gpu


def _cameras(C, rows=3):
    c2w = camera_to_worlds(scene_s0(N=10, C=C).viewmats)
    if rows == 4:
        c2w = torch.cat([c2w, torch.tensor([[[0.0, 0.0, 0.0, 1.0]]]).expand(C, 1, 4)], dim=1)
    return c2w.contiguous()


def _table(n, seed, small_row=None):
    g = torch.Generator().manual_seed(seed)
    adj = torch.randn(n, 6, generator=g) * torch.tensor([0.05] * 3 + [0.03] * 3)
    if small_row is not None:
        adj[small_row, 3:] = torch.tensor([2e-3, -3e-3, 1e-3])  # |omega| below the clamp of theta
    return adj


@pytest.mark.parametrize("rows", [3, 4])
def test_apply_matches_oracle_and_zero_rows_are_bit_identical(cuda, rows):
    C, n = 6, 4
    c2w = _cameras(C, rows)
    ids = torch.tensor([3, 0, 1, 3, 2, 1])
    adj = _table(n, 1, small_row=2)
    adj[1] = 0.0  # views 2 and 5 use a zero row
    cam = CameraPoseOptimizer(n, cuda)
    cam.pose_adjustment.copy_(adj.to(cuda))
    got = cam.viewmats(c2w.to(cuda), ids)
    ref = co.viewmats(c2w[:, :3].double(), ids, adj.double())
    assert torch.allclose(got.double().cpu(), ref, rtol=0, atol=2e-6)
    plain = get_viewmat(c2w.to(cuda))
    for c in (2, 5):
        assert torch.equal(got[c].view(torch.int32), plain[c].view(torch.int32))
    cam.pose_adjustment.zero_()
    assert torch.equal(cam.viewmats(c2w.to(cuda), ids).view(torch.int32), plain.view(torch.int32))
    with pytest.raises(ValueError):
        cam.viewmats(c2w.to(cuda), torch.tensor([0, 1, 2, 3, 4, 0]))


def test_bwd_and_regularizer_match_oracle_autograd(cuda):
    C, n = 7, 5
    c2w = _cameras(C)
    ids = torch.tensor([0, 2, 0, 1, 2, 2, 3])  # duplicates; row 4 has no view
    adj = _table(n, 2, small_row=3)
    g = torch.Generator().manual_seed(5)
    v = torch.randn(C, 4, 4, generator=g)
    v[:, 3] = 0.0
    cam = CameraPoseOptimizer(n, cuda)
    cam.pose_adjustment.copy_(adj.to(cuda))
    cam.backward(v.to(cuda), ids.to(cuda), c2w.to(cuda))
    first = cam.grad.clone()
    cam.backward(v.to(cuda), ids.to(cuda), c2w.to(cuda))
    assert torch.equal(first.view(torch.int32), cam.grad.view(torch.int32))  # no atomics: the same bits every call
    x = adj.double().requires_grad_(True)
    (co.viewmats(c2w.double(), ids, x) * v.double()).sum().backward()
    got = cam.pose_grad.double().cpu()
    assert torch.equal(got[4], torch.zeros(6, dtype=torch.float64))
    assert float((got - x.grad).abs().max()) <= 1e-6 * float(x.grad.abs().max()), (got, x.grad)
    cam.grad.zero_()  # the regulariser's gradient alone (it accumulates)
    val = cam.regularize()
    y = adj.double().requires_grad_(True)
    r = co.regularizer(y)
    r.backward()
    assert float(val) == pytest.approx(float(r.detach()), rel=1e-6)
    assert torch.allclose(cam.pose_grad.double().cpu(), y.grad, rtol=1e-5, atol=1e-10)


@pytest.mark.parametrize("deg,C", [(3, 3), (1, 2)])
def test_exchange_pose_equals_batched_pose_gradient(cuda, deg, C):
    """Emulated ranks on one device (as tests/test_gpu_exchange.py): each rank's qed_project_bwd_exchange_pose returns the
    v_viewmats row that one qed_project_bwd_pose over the whole batch returns for its view."""
    lib = _lib.load()
    s = scene_s0(N=5000, C=C, size=96).to(cuda)
    bg = torch.tensor([0.3, 0.2, 0.1], device=cuda)
    fs = FusedSplatStep(cuda)
    whole = fs.step(s.means, s.quats, s.scales, s.opacities, s.sh, s.viewmats, s.Ks, s.width, s.height, deg, s.gt_rgb, s.gt_depth, bg,
                    pose_gradients=True)
    ref = whole.v_viewmats.clone()
    N, K = s.N, s.sh.shape[1]
    xch = torch.zeros((C * N + C) * 4, device=cuda)
    peers = (ctypes.c_void_p * 1)(xch.data_ptr())
    ws_bytes = lib.qed_project_bwd_pose_workspace_bytes(1, N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=cuda)
    for r in range(C):
        sl = slice(r, r + 1)
        vm, Ks = s.viewmats[sl].contiguous(), s.Ks[sl].contiguous()
        fs.step(s.means, s.quats, s.scales, s.opacities, s.sh, vm, Ks, s.width, s.height, deg, s.gt_rgb[sl].contiguous(), s.gt_depth[sl].contiguous(), bg,
                grad_scale=1.0 / C)
        f = fs._fwd
        packed = fs._get("packed", (N, 12))
        out = {k: torch.empty_like(whole.grads[k]) for k in ("means", "quats", "scales", "opacities")}
        v_vm = torch.full((1, 4, 4), float("nan"), device=cuda)
        args = (1, N, _lib.ptr(s.means), _lib.ptr(s.quats), _lib.ptr(s.scales), _lib.ptr(s.opacities), 0, _lib.ptr(s.sh), K, deg, _lib.ptr(vm),
                _lib.ptr(Ks), s.width, s.height, 0.3, 0, 1, _lib.ptr(f["radii"]), _lib.ptr(f["conics"]), None, _lib.ptr(packed),
                _lib.ptr(out["means"]), _lib.ptr(out["quats"]), _lib.ptr(out["scales"]), _lib.ptr(out["opacities"]), None, peers, 1, r, C, 7.0)
        _lib.check(lib.qed_project_bwd_exchange_pose(*args, _lib.ptr(v_vm), _lib.ptr(ws), ws_bytes, _lib.current_stream()),
                   "qed_project_bwd_exchange_pose")
        plain = {k: torch.empty_like(t) for k, t in out.items()}
        _lib.check(lib.qed_project_bwd_exchange(*args[:21], _lib.ptr(plain["means"]), _lib.ptr(plain["quats"]), _lib.ptr(plain["scales"]),
                                                _lib.ptr(plain["opacities"]), None, peers, 1, r, C, 7.0, _lib.current_stream()), "qed_project_bwd_exchange")
        for k in out:  # the pose variant leaves the Gaussian gradients of the exchange kernel as they were (up to contraction)
            assert float((out[k] - plain[k]).abs().max()) <= 1e-7 * float(plain[k].abs().max()) + 1e-30, k
        g, e = v_vm[0].double().cpu(), ref[r].double().cpu()
        assert torch.equal(g[3], torch.zeros(4, dtype=torch.float64))
        for sl2 in ((slice(0, 3), slice(0, 3)), (slice(0, 3), 3)):
            err, norm = float((g[sl2] - e[sl2]).abs().max()), float(e[sl2].norm())
            assert norm > 0 and err <= 1e-4 * norm, (r, err, norm)


def _trainer_scene(C, size=96, N=6000):
    s = scene_s0(N=N, C=C, size=size)
    a = scene_args(s)
    return s, a


def _gaussian_args(s, cuda):
    return (s.means.to(cuda), s.quats.to(cuda), torch.log(s.scales).to(cuda), torch.logit(s.opacities).to(cuda), s.sh.to(cuda))


def test_trainer_pose_recovery(cuda):
    """Gaussians frozen, 4 training cameras whose poses are off by 1.5 degrees and 2 % of their distance: the SO3xR3 table
    trained by SplatTrainer cuts both errors at least 5x (the bar of tests/test_gpu_pose_grad.py::test_pose_recovery)."""
    C, size = 4, 128
    s, a = _trainer_scene(C, size)
    bg = torch.tensor([0.2, 0.5, 0.8], device=cuda)
    with torch.no_grad():
        r, al, _ = rasterization(**{k: v.to(cuda) for k, v in a.items()}, width=size, height=size, render_mode="RGB+ED", sh_degree=3)
    gt_rgb = torch.clamp(r[..., :3] + (1 - al) * bg, 0, 1).contiguous()
    gt_depth = torch.where(al[..., 0] > 0.5, r[..., 3], torch.zeros_like(r[..., 3])).contiguous()
    c2w_true = camera_to_worlds(s.viewmats).double()
    gen = torch.Generator().manual_seed(3)
    pert = torch.zeros(C, 6, dtype=torch.float64)
    for c in range(C):
        axis = torch.randn(3, generator=gen, dtype=torch.float64)
        dirn = torch.randn(3, generator=gen, dtype=torch.float64)
        pert[c, 3:] = axis / axis.norm() * math.radians(1.5)
        pert[c, :3] = dirn / dirn.norm() * 0.02 * float(c2w_true[c, :, 3].norm())
    ids = torch.arange(C)
    c2w_bad = co.adjusted_c2w(c2w_true, ids, pert)  # what the training data claims

    def errors(table):
        p = co.adjusted_c2w(c2w_bad, ids, table.double().cpu())
        rot = [math.degrees(math.acos(max(-1.0, min(1.0, (float(torch.trace(c2w_true[c, :, :3].T @ p[c, :, :3])) - 1) / 2)))) for c in range(C)]
        return max(rot), float((p[:, :, 3] - c2w_true[:, :, 3]).norm(dim=-1).max())

    cfg = TrainConfig(camera_optimizer="SO3xR3", camera_opt_lr=5e-3, camera_opt_lr_final=5e-3 * 0.99 ** 200, camera_opt_warmup=0, max_steps=200,
                      camera_opt_trans_l2_penalty=0.0, camera_opt_rot_l2_penalty=0.0, lr_means=1e-30, lr_means_final=1e-30, lr_quats=0.0,
                      lr_scales=0.0, lr_opacities=0.0, lr_features_dc=0.0, lr_features_rest=0.0, stop_split_at=0, render_mode="RGB+ED",
                      sh_degree_interval=1)
    tr = SplatTrainer(*_gaussian_args(s, cuda), cfg=cfg, num_cameras=C)
    e_rot0, e_t0 = errors(tr.pose_adjustment)
    c2w_dev = c2w_bad.float().to(cuda)
    for _ in range(200):
        tr.step(None, s.Ks.to(cuda), size, size, gt_rgb, gt_depth, bg, camera_to_worlds=c2w_dev, camera_ids=ids)
    e_rot, e_t = errors(tr.pose_adjustment)
    print("pose recovery", dict(rot_deg=[e_rot0, e_rot], trans=[e_t0, e_t]))
    assert e_rot <= e_rot0 / 5 and e_t <= e_t0 / 5, (e_rot0, e_rot, e_t0, e_t)


def test_frozen_table_trains_like_optimizer_off(cuda):
    """Optimizer on with lr 0: the same viewmats, hence the same renders bit for bit (the forward has no atomics), as the
    trainer without it.  The loss and the Gaussian gradients are compared within float tolerance: the compositor's backward
    and the loss statistics accumulate with atomics, so two runs differ in the last bits whatever the pose kernel does
    (1e-6 of the largest value, the bound of tests/test_gpu_pose_grad.py; the pose kernels' own contraction differences
    are below 1e-7)."""
    C, size = 2, 96
    s, _ = _trainer_scene(C, size)
    bg = torch.tensor([0.3, 0.3, 0.3], device=cuda)
    gt_rgb, gt_depth = s.gt_rgb.to(cuda), s.gt_depth.to(cuda)
    c2w = camera_to_worlds(s.viewmats).to(cuda)
    base = dict(stop_split_at=0, sh_degree_interval=1)
    off = SplatTrainer(*_gaussian_args(s, cuda), cfg=TrainConfig(**base))
    on = SplatTrainer(*_gaussian_args(s, cuda), cfg=TrainConfig(camera_optimizer="SO3xR3", camera_opt_lr=0.0, **base), num_cameras=3)
    ids = torch.tensor([2, 0])
    for it in range(3):
        l_off, _ = off.step(get_viewmat(c2w), s.Ks.to(cuda), size, size, gt_rgb, gt_depth, bg)
        r_off = off._fused._fwd["render"].clone()
        l_on, _ = on.step(None, s.Ks.to(cuda), size, size, gt_rgb, gt_depth, bg, camera_to_worlds=c2w, camera_ids=ids)
        r_on = on._fused._fwd["render"]
        if it == 0:  # identical parameters: identical renders, equal losses and gradients
            assert torch.equal(r_on.view(torch.int32), r_off.view(torch.int32))
            assert torch.allclose(l_on, l_off, rtol=1e-6, atol=0)
            for g in GROUPS:
                a, b = off.arena.view(off.arena.grad, g), on.arena.view(on.arena.grad, g)
                assert float((a - b).abs().max()) <= 1e-6 * float(a.abs().max()), g
    assert float(on.pose_adjustment.abs().max()) == 0.0 and float(on.camera_opt.pose_grad.abs().max()) > 0
    assert float(on.camera_opt_loss) == 0.0
    with pytest.raises(ValueError):
        on.step(get_viewmat(c2w), s.Ks.to(cuda), size, size, gt_rgb, gt_depth, bg)
    with pytest.raises(ValueError):
        off.step(get_viewmat(c2w), s.Ks.to(cuda), size, size, gt_rgb, gt_depth, bg, camera_to_worlds=c2w, camera_ids=ids)


def _exchange_worker(rank, port, out):
    """One process, an NCCL group of one: a trainer forced onto the exchange path (symmetric gradient arena, symmetric pose
    buffer, this library's all-reduce kernels) next to the plain single-GPU trainer, both with frozen Gaussians."""
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    res = {}
    try:
        s = scene_s0(N=6000, C=2, size=96)
        frozen = dict(lr_means=1e-30, lr_means_final=1e-30, lr_quats=0.0, lr_scales=0.0, lr_opacities=0.0, lr_features_dc=0.0,
                      lr_features_rest=0.0, stop_split_at=0, camera_optimizer="SO3xR3", camera_opt_lr=1e-3, camera_opt_warmup=0)
        xt = SplatTrainer(*_gaussian_args(s, dev), cfg=TrainConfig(comm="exchange", **frozen), num_cameras=4)
        xt.comm = "exchange"  # world 1 picks no collective; one rank runs the multi-GPU code path unchanged
        ref = SplatTrainer(*_gaussian_args(s, dev), cfg=TrainConfig(**frozen), num_cameras=4)
        bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
        c2w, ids = camera_to_worlds(s.viewmats).to(dev), torch.tensor([3, 1])
        res.update(grad_err=[], grad_scale=[], grad_in_symmetric=[], exchanges=[])
        for v in (slice(0, 1), slice(0, 1), slice(0, 2), slice(0, 2)):  # 1 -> 2 views per rank: new symmetric buffers
            for tr in (xt, ref):
                tr.step(None, s.Ks[v].to(dev), s.width, s.height, s.gt_rgb[v].to(dev), s.gt_depth[v].to(dev), bg, camera_to_worlds=c2w[v],
                        camera_ids=ids[v])
            res["grad_err"].append(float((xt.camera_opt.pose_grad - ref.camera_opt.pose_grad).abs().max()))
            res["grad_scale"].append(float(ref.camera_opt.pose_grad.abs().max()))
            res["grad_in_symmetric"].append(xt.camera_opt.grad.data_ptr() == xt._xg.pose.buf.data_ptr())
            res["exchanges"].append(id(xt._xg))
        res["comm"] = xt.comm
        res["table_err"] = float((xt.pose_adjustment - ref.pose_adjustment).abs().max())
        res["table_scale"] = float(ref.pose_adjustment.abs().max())
        res["reg"] = [float(xt.camera_opt_loss), float(ref.camera_opt_loss)]
    except RuntimeError as e:  # no symmetric memory on this machine
        res["error"] = str(e)
    torch.save(res, out)
    dist.destroy_process_group()


def test_trainer_exchange_path_on_one_gpu(cuda, tmp_path):
    """The trainer's exchange integration -- pose gradient from qed_project_bwd_exchange_pose, the table gradient living in
    the symmetric pose buffer and summed by its all-reduce kernel, the buffers rebuilt when the views per rank change -- gives
    the table gradients and tables of the plain single-GPU trainer."""
    out = str(tmp_path / "xchg.pt")
    mp.spawn(_exchange_worker, args=(29500 + (os.getpid() + 11) % 2000, out), nprocs=1, join=True)
    r = torch.load(out)
    if "error" in r and "symmetric memory" in r["error"]:
        pytest.skip(r["error"])
    assert "error" not in r, r
    assert r["comm"] == "exchange" and all(r["grad_in_symmetric"]), r
    assert r["exchanges"][0] == r["exchanges"][1] != r["exchanges"][2] == r["exchanges"][3], r  # rebuilt once, re-pointed
    for err, scale in zip(r["grad_err"], r["grad_scale"]):
        assert scale > 0 and err <= 1e-4 * scale, r
    assert r["table_scale"] > 0 and r["table_err"] <= 1e-3 * r["table_scale"], r
    assert r["reg"][0] == pytest.approx(r["reg"][1], rel=1e-4) and r["reg"][0] > 0
