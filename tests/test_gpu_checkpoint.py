"""-m gpu: SplatTrainer.state_dict() / SplatTrainer.from_state_dict() on real steps of the CUDA trainer.

The raster backward sums with float atomics, so two uninterrupted runs of the same steps can differ in the last bits (see
tests/test_gpu_edge_cases.py).  The state is therefore checked bit for bit across a save and a load, and a resumed run is
checked against the spread of uninterrupted control runs: the same N and refine decisions after every step, and losses and
states no further from the first run than a small multiple of the controls' distance from it (equal when the controls are
equal).  A state with one piece lost (the Adam moments) is shown to fail that check."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from qed_splatter_b200.scenes import camera_to_worlds, scene_s0
from qed_splatter_b200.trainer import SplatTrainer, TrainConfig
from test_checkpoint_cpu import _bits, _tensors, _through_file, assert_states_equal

pytestmark = pytest.mark.gpu
NUM_CAMERAS = 3
# refine at steps 3 and 9 (opacity reset at 6), full resolution from step 6, both tables on
DEFAULT = dict(warmup_length=1, refine_every=3, reset_alpha_every=2, pause_refine_after_reset=3, sh_degree_interval=3, num_downscales=1,
               resolution_schedule=6, camera_optimizer="SO3xR3", camera_opt_warmup=0, use_bilateral_grid=True, bilateral_grid_warmup=0)
# relocate + add at steps 3, 6, 9
MCMC = dict(DEFAULT, strategy="mcmc", max_gs_num=3400)
SPREAD_MULTIPLE = 10.0  # B may differ from A by this many times the controls' largest distance from A ...
SPREAD_FLOOR = 1e-6     # ... plus this fraction of the tensor's largest magnitude


def _scene():
    s = scene_s0(N=3000, C=2, size=96)
    o = s.opacities.clone()
    o[::17] = 0.002  # pruned by the first DefaultStrategy refine, dead for MCMC's first relocation
    return s, o


def _new(cfg, dev):
    s, o = _scene()
    p = (s.means.to(dev), s.quats.to(dev), torch.log(s.scales).to(dev), torch.logit(o).to(dev), s.sh.to(dev))
    return SplatTrainer(*p, cfg=TrainConfig(**cfg), num_cameras=NUM_CAMERAS)


class _Inputs:
    def __init__(self, dev):
        s, _ = _scene()
        t = s.to(dev)
        self.args = (t.Ks, s.width, s.height, t.gt_rgb, t.gt_depth, torch.tensor([0.3, 0.4, 0.5], device=dev))
        self.c2w, self.ids = camera_to_worlds(s.viewmats).to(dev), torch.tensor([2, 0])

    def step(self, tr):
        loss, info = tr.step(None, *self.args, camera_to_worlds=self.c2w, camera_ids=self.ids)
        return loss, info


def _run(cfg, dev, steps, save_at=None, corrupt=None):
    """-> (final state, losses [steps, 3], N after every step, refine infos); saved, written, read and resumed at `save_at`."""
    x = _Inputs(dev)
    tr = _new(cfg, dev)
    losses, ns, infos = [], [], []
    for i in range(steps):
        if i == save_at:
            state = _through_file(tr.state_dict())
            if corrupt is not None:
                corrupt(state)
            tr = SplatTrainer.from_state_dict(state)
        loss, info = x.step(tr)
        losses.append(loss)
        ns.append(tr.arena.N)
        infos.append(info)
    return tr.state_dict(), torch.stack(losses).cpu(), ns, infos


def spread_violations(a, controls, b):
    """Tensors (and the losses) where b is further from a than SPREAD_MULTIPLE x the controls' largest distance from a plus
    SPREAD_FLOOR x max|a|; when every control equals a bit for bit, b must equal a bit for bit."""
    ta, tb = _tensors(a), _tensors(b)
    tcs = [_tensors(c) for c in controls]
    exact = all(torch.equal(_bits(ta[k]), _bits(tc[k])) for tc in tcs for k in ta)
    bad = []
    for k in ta:
        if exact:
            if not torch.equal(_bits(ta[k]), _bits(tb[k])):
                bad.append((k, "controls equal a bit for bit, b does not"))
            continue
        x = ta[k].double()
        spread = max(float((tc[k].double() - x).abs().max()) for tc in tcs) if x.numel() else 0.0
        err = float((tb[k].double() - x).abs().max()) if x.numel() else 0.0
        bound = SPREAD_MULTIPLE * spread + SPREAD_FLOOR * (float(x.abs().max()) if x.numel() else 0.0)
        if err > bound:
            bad.append((k, err, spread, bound))
    return bad


@pytest.mark.parametrize("cfg", [DEFAULT, MCMC], ids=["default", "mcmc"])
def test_round_trip_is_bitwise(cuda, cfg):
    x = _Inputs(cuda)
    tr = _new(cfg, cuda)
    n0 = tr.arena.N
    infos = [x.step(tr)[1] for _ in range(5)]
    assert any(i is not None and i["n"] != n0 for i in infos), infos
    s1 = tr.state_dict()
    s2 = SplatTrainer.from_state_dict(_through_file(s1)).state_dict()
    assert_states_equal(s1, s2)
    assert s1["step"] == 5 and s1["gauss_params"]["means"].shape[0] == tr.arena.N
    assert tr.downscale_factor() == 2  # the state was saved at half resolution


@pytest.mark.parametrize("cfg", [DEFAULT, MCMC], ids=["default", "mcmc"])
def test_continuation_within_the_spread_of_uninterrupted_runs(cuda, cfg):
    steps, K = 10, 5  # saved mid refine interval (statistics of step 4 in flight), resolution change and refine after it
    A, A1, A2, B = (_run(cfg, cuda, steps, save_at=K if r == "B" else None) for r in ("A", "A1", "A2", "B"))
    for r in (A1, A2, B):
        assert r[2] == A[2] and r[3] == A[3], (A[2], r[2], A[3], r[3])
    assert any(i is not None for i in A[3][K:]) and len(set(A[2])) > 1, A[3]

    def with_loss(r):
        return dict(r[0], loss=r[1])

    bad = spread_violations(with_loss(A), [with_loss(A1), with_loss(A2)], with_loss(B))
    assert not bad, bad
    # a lost piece of state: the continuation no longer passes

    def drop_moments(state):
        for k in state["exp_avg"]:
            state["exp_avg"][k].zero_()
            state["exp_avg_sq"][k].zero_()

    broken = _run(cfg, cuda, steps, save_at=K, corrupt=drop_moments)
    bad = spread_violations(with_loss(A), [with_loss(A1), with_loss(A2)], with_loss(broken))
    assert any(k[0].startswith("gauss_params.") for k in bad), bad
    print("checkpoint continuation", dict(cfg=cfg.get("strategy", "default"), broken=bad[:4]))


FROZEN = dict(lr_means=1e-30, lr_means_final=1e-30, lr_quats=0.0, lr_scales=0.0, lr_opacities=0.0, lr_features_dc=0.0, lr_features_rest=0.0)


def _exchange_worker(rank, port, out):
    """One process, an NCCL group of one: a state saved by the plain trainer, resumed on the exchange path next to the plain
    trainer resumed from the same state."""
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    res = {}
    try:
        cfg = dict(strategy="mcmc", max_gs_num=3400, warmup_length=1, refine_every=2, camera_optimizer="SO3xR3", camera_opt_lr=1e-3,
                   camera_opt_warmup=0, **FROZEN)
        x = _Inputs(dev)
        tr = _new(cfg, dev)
        for _ in range(3):
            x.step(tr)
        state = _through_file(tr.state_dict())
        xt = SplatTrainer.from_state_dict(state, TrainConfig(**dict(state["config"], comm="exchange")))
        xt.comm = "exchange"  # world 1 picks no collective; one rank runs the multi-GPU code path unchanged
        ref = SplatTrainer.from_state_dict(state)
        res.update(grad_err=[], grad_scale=[], pose_err=[], pose_scale=[], in_symmetric=[], exchanges=[], N=[])
        for _ in range(6):
            infos = [x.step(t)[1] for t in (xt, ref)]
            if infos[1] is None:  # a step that grew the set leaves fresh (zero) gradient arenas behind, re-pointed by the next step
                res["grad_err"].append(float((xt.arena.grad - ref.arena.grad).abs().max()))
                res["grad_scale"].append(float(ref.arena.grad.abs().max()))
                res["in_symmetric"].append(xt.arena.grad.data_ptr() == xt._xg.grad.data_ptr())
            res["in_symmetric"].append(xt.camera_opt.grad.data_ptr() == xt._xg.pose.buf.data_ptr())
            res["pose_err"].append(float((xt.camera_opt.pose_grad - ref.camera_opt.pose_grad).abs().max()))
            res["pose_scale"].append(float(ref.camera_opt.pose_grad.abs().max()))
            res["exchanges"].append(id(xt._xg))
            res["N"].append((xt.arena.N, ref.arena.N))
        res["comm"] = xt.comm
        res["capacity"] = xt._xg.capacity
        res["N_saved"] = state["gauss_params"]["means"].shape[0]
        res["param_err"] = float((xt.arena.param - ref.arena.param).abs().max())
        res["table_err"] = float((xt.pose_adjustment - ref.pose_adjustment).abs().max())
        res["table_scale"] = float(ref.pose_adjustment.abs().max())
    except RuntimeError as e:  # no symmetric memory available
        res["error"] = str(e)
    torch.save(res, out)
    dist.destroy_process_group()


def test_resumed_trainer_on_the_exchange_path(cuda, tmp_path):
    out = str(tmp_path / "xchg.pt")
    mp.spawn(_exchange_worker, args=(29500 + (os.getpid() + 47) % 2000, out), nprocs=1, join=True)
    r = torch.load(out)
    if "error" in r and "symmetric memory" in r["error"]:
        pytest.skip(r["error"])
    assert "error" not in r, r
    assert r["comm"] == "exchange" and r["capacity"] >= 3400, r
    assert len(r["in_symmetric"]) >= 9 and all(r["in_symmetric"]), r  # arena gradient and pose gradient in the symmetric buffers
    assert len(set(r["exchanges"])) == 1, r  # sized for max_gs_num by the first step: never rebuilt while N grows
    assert r["N_saved"] < r["N"][-1][0] and all(a == b for a, b in r["N"]), r
    assert len(r["grad_err"]) >= 3, r
    for err, scale in zip(r["grad_err"], r["grad_scale"]):
        assert scale > 0 and err <= 1e-4 * scale, r
    for err, scale in zip(r["pose_err"], r["pose_scale"]):
        assert scale > 0 and err <= 1e-4 * scale, r
    assert r["param_err"] <= 1e-6, r
    assert r["table_scale"] > 0 and r["table_err"] <= 1e-3 * r["table_scale"], r
