"""-m gpu: splatfacto's MCMC strategy on the device (csrc/mcmc.cu through qed_splatter_b200/mcmc.py) against
tests/mcmc_oracle.py -- the Philox draws, their distribution, relocation values, relocate / add, noise, the regularisers,
the fused path against impl="torch" on the same draws -- and SplatTrainer(strategy="mcmc") on one GPU and on the exchange
path.  Constructed opacities keep a margin from min_opacity, so a 1-ulp sigmoid difference cannot change the dead set."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import mcmc_oracle as mo
from qed_splatter_b200 import _lib, mcmc
from qed_splatter_b200.scenes import camera_to_worlds, scene_s0
from qed_splatter_b200.trainer import GROUPS, GaussianArena, SplatTrainer, TrainConfig

pytestmark = pytest.mark.gpu
FROZEN = dict(lr_means=1e-30, lr_means_final=1e-30, lr_quats=0.0, lr_scales=0.0, lr_opacities=0.0, lr_features_dc=0.0, lr_features_rest=0.0)


def _arena(N, dev, seed=0, dead_every=0):
    g = torch.Generator().manual_seed(seed)
    o = torch.rand(N, generator=g) * 0.96 + 0.02  # alive: >= 0.02, four times min_opacity
    if dead_every:
        o[::dead_every] = torch.rand(o[::dead_every].shape, generator=g) * 0.003 + 1e-4  # dead: <= 0.0031
    p = (torch.randn(N, 3, generator=g), torch.randn(N, 4, generator=g), torch.log(torch.rand(N, 3, generator=g) * 0.05 + 0.001), torch.logit(o),
         torch.randn(N, 16, 3, generator=g))
    a = GaussianArena(*(t.to(dev) for t in p))
    a.exp_avg.copy_(torch.rand(a.exp_avg.shape, generator=g).to(dev))
    a.exp_avg_sq.copy_(torch.rand(a.exp_avg_sq.shape, generator=g).to(dev))
    return a


def _np(a, buf):
    return {g: a.view(buf, g).double().cpu().numpy().copy() for g in GROUPS}


def _check_against(a, P, M, V, what):
    """copied floats and moments bit-exact, recomputed opacity / scale within 1e-5 (compared as o and exp(log-scale))."""
    for g in ("means", "quats", "sh"):
        assert np.array_equal(a.view(a.param, g).double().cpu().numpy(), P[g]), (what, g)
    for g in GROUPS:
        assert np.array_equal(a.view(a.exp_avg, g).double().cpu().numpy(), M[g]), (what, g)
        assert np.array_equal(a.view(a.exp_avg_sq, g).double().cpu().numpy(), V[g]), (what, g)
    o = torch.sigmoid(a.view(a.param, "opacities").double()).cpu().numpy()
    assert np.allclose(o, 1 / (1 + np.exp(-P["opacities"])), rtol=1e-5, atol=1e-9), what
    s = torch.exp(a.view(a.param, "scales").double()).cpu().numpy()
    assert np.allclose(s, np.exp(P["scales"]), rtol=1e-5, atol=1e-12), what


@pytest.mark.parametrize("zero_dead", [False, True])
def test_draws_equal_the_numpy_restatement(cuda, zero_dead):
    a = _arena(5000, cuda, seed=1, dead_every=7)
    st = mcmc.MCMCStrategy(cuda)
    op = a.view(a.param, "opacities").cpu().numpy()
    for step, stream, n in ((123, 1, 3000), (4567, 2, 777), (0, 1, 1)):
        d, c = st.draw(a, n, step, stream, zero_dead)
        ref, total = mo.sample(op, n, 42, step, stream, 0.005, zero_dead)
        assert total > 0 and np.array_equal(d.long().cpu().numpy(), ref), (step, stream)
        assert torch.equal(c.long().cpu(), torch.bincount(d.long().cpu(), minlength=a.N))
        d2, c2 = st.draw(a, n, step, stream, zero_dead)  # two calls, identical output
        assert torch.equal(d, d2) and torch.equal(c, c2)
    if zero_dead:
        d, _ = st.draw(a, 20000, 9, 1, True)
        assert not bool(torch.isin(d.long(), torch.arange(0, a.N, 7, device=cuda)).any())  # dead rows never drawn


def test_zero_weight_rows_and_the_last_row(cuda):
    a = _arena(1000, cuda, seed=2)
    op = a.view(a.param, "opacities")
    op[500:] = -60.0  # weight 0, including the last rows: the search must stay below them
    op[:10] = -60.0
    d, c = mcmc.MCMCStrategy(cuda).draw(a, 100000, 5, 2, False)
    assert int(d.min()) >= 10 and int(d.max()) < 500 and int(c[500:].sum()) == 0 and int(c.sum()) == 100000


def test_chi_square_of_a_million_draws(cuda):
    from scipy.stats import chi2

    a = _arena(1000, cuda, seed=3)
    d, c = mcmc.MCMCStrategy(cuda).draw(a, 10**6, 11, 2, False)
    w = mo.weights(a.view(a.param, "opacities").cpu().numpy(), 0.005, False).astype(np.float64)
    exp = 10**6 * w / w.sum()
    stat = float(((c.double().cpu().numpy() - exp) ** 2 / exp).sum())
    assert chi2.sf(stat, df=999) > 1e-4, stat


def test_relocation_values_against_the_float64_loop(cuda):
    """Ratios 2..60 (counts 1..59, the 51 clamp included) on opacities from 0.006 (o' clamped up to min_opacity at large
    ratios) to exactly 1 (logit 30: o' = 1, clamped down to 1 - FLT_EPSILON).  The reference starts from torch's float32
    sigmoid on the device, so a last-bit difference of exp cannot move 1 - o.  At o = 1 the alternating sum of the
    denominator loses ~2^ratio float64 epsilons (1e-3 at ratio 51; gsplat's float32 loop loses far more), so those rows
    are checked up to ratio 20."""
    ops = np.array([0.006, 0.02, 0.3, 0.7, 0.99, 0.9999], np.float64)
    pairs = [(l, c) for l in np.log(ops / (1 - ops)) for c in range(1, 60)] + [(30.0, c) for c in range(1, 20)]
    logits = np.array([l for l, _ in pairs], np.float32)
    N = len(pairs)
    a = _arena(N, cuda, seed=4)
    a.view(a.param, "opacities").copy_(torch.from_numpy(logits))
    cnt = torch.tensor([c for _, c in pairs], dtype=torch.int32, device=cuda)
    o_dev = torch.sigmoid(a.view(a.param, "opacities")).double().cpu().numpy()
    s_dev = torch.exp(a.view(a.param, "scales")).double().cpu().numpy()
    st = mcmc.MCMCStrategy(cuda)
    starts = st._starts(a)
    _lib.check(st.lib.qed_mcmc_relocate(N, _lib.ptr(cnt), 0.005, 1, 0, None, None, _lib.ptr(a.param), _lib.ptr(a.exp_avg), _lib.ptr(a.exp_avg_sq),
                                        starts.data_ptr(), _lib.current_stream()), "qed_mcmc_relocate")
    o_new, s_new = mo.compute_relocation(o_dev, s_dev, cnt.cpu().numpy() + 1)
    o_ref = np.clip(o_new, 0.005, 1 - mo.FLT_EPS)
    assert (o_new < 0.005).any() and (o_new >= 1 - mo.FLT_EPS).any() and (cnt.cpu().numpy() + 1 > 51).any()
    o_got = torch.sigmoid(a.view(a.param, "opacities").double()).cpu().numpy()
    assert np.allclose(o_got, o_ref, rtol=1e-6, atol=0), float(np.abs(o_got / o_ref - 1).max())
    s_got = torch.exp(a.view(a.param, "scales").double()).cpu().numpy()
    assert np.allclose(s_got, s_new, rtol=1e-6, atol=0), float(np.abs(s_got / s_new - 1).max())
    for g in GROUPS:  # every row was drawn: moments zeroed
        assert float(a.view(a.exp_avg, g).abs().max()) == 0.0 and float(a.view(a.exp_avg_sq, g).abs().max()) == 0.0


def test_relocate_and_add_on_device_draws_match_the_oracle(cuda):
    a = _arena(4000, cuda, seed=5, dead_every=13)
    st = mcmc.MCMCStrategy(cuda, cap_max=10**6)
    P, M, V = _np(a, a.param), _np(a, a.exp_avg), _np(a, a.exp_avg_sq)
    dead, n_dead = st.dead_rows(a)
    assert dead.cpu().tolist() == list(range(0, 4000, 13))
    draws, counts = st.draw(a, n_dead, 600, mcmc.STREAM_RELOCATE, True)
    st.relocate(a, draws, dead, counts)
    mo.relocate(P, M, V, draws.cpu().numpy(), dead.cpu().numpy(), 0.005)
    _check_against(a, P, M, V, "relocate")
    n_new = mcmc.growth(a.N, st.cap_max)
    draws, counts = st.draw(a, n_new, 600, mcmc.STREAM_ADD, False)
    st.add(a, draws, counts)
    P, M, V = mo.sample_add(P, M, V, draws.cpu().numpy(), 0.005)
    assert a.N == 4000 + n_new == 4200
    _check_against(a, P, M, V, "add")


def test_fused_refine_equals_torch_on_the_same_draws(cuda):
    fa, ta = _arena(3000, cuda, seed=6, dead_every=11), _arena(3000, cuda, seed=6, dead_every=11)
    fs, ts = mcmc.MCMCStrategy(cuda, impl="fused"), mcmc.MCMCStrategy(cuda, impl="torch")
    dead, n_dead = fs.dead_rows(fa)
    assert torch.equal(dead, ts.dead_rows(ta)[0])
    draws, counts = fs.draw(fa, n_dead, 700, 1, True)
    fs.relocate(fa, draws, dead, counts)
    ts.relocate(ta, draws, dead)
    add, counts = fs.draw(fa, mcmc.growth(fa.N, 10**6), 700, 2, False)
    fs.add(fa, add, counts)
    ts.add(ta, add)
    assert fa.N == ta.N == 3150
    _check_against(fa, _np(ta, ta.param), _np(ta, ta.exp_avg), _np(ta, ta.exp_avg_sq), "fused vs torch")


def test_noise_against_the_oracle(cuda):
    a = _arena(20000, cuda, seed=7, dead_every=5)
    P = _np(a, a.param)
    st = mcmc.MCMCStrategy(cuda, seed=1234)
    before = _np(a, a.param)["means"]
    st.inject_noise(a, 77, 1.6e-4 * 5e5)
    mo.inject_noise(P, mo.normals(a.N, 1234, 77), 1.6e-4 * 5e5)
    got = a.view(a.param, "means").double().cpu().numpy()
    delta_got, delta_ref = got - before, P["means"] - before
    assert float(np.abs(delta_ref).max()) > 0
    err = np.abs(delta_got - delta_ref)
    assert float(err.max()) <= 1e-3 * float(np.abs(delta_ref).max()) + 1e-6, float(err.max())


def test_regularizers_against_autograd(cuda):
    a = _arena(30000, cuda, seed=8)
    a.grad.normal_()
    a.view(a.grad, "opacities").zero_()  # the added terms are ~1e-7: on top of O(1) values they would round away
    a.view(a.grad, "scales").zero_()
    g0 = a.grad.clone()
    st = mcmc.MCMCStrategy(cuda, opacity_reg=0.01, scale_reg=0.02)
    loss = st.regularize(a).clone()
    op = a.view(a.param, "opacities").detach().double().requires_grad_(True)
    ls = a.view(a.param, "scales").detach().double().requires_grad_(True)
    lo, lsc = mcmc.regularizers_torch(op, ls, 0.01, 0.02)
    go, gs = torch.autograd.grad(lo + lsc, (op, ls))
    lo, lsc = lo.detach(), lsc.detach()
    assert float(loss[0]) == pytest.approx(float(lo), rel=1e-6) and float(loss[1]) == pytest.approx(float(lsc), rel=1e-6)
    dg = a.grad - g0
    assert torch.allclose(a.view(dg, "opacities").double(), go, rtol=1e-4, atol=1e-12)
    assert torch.allclose(a.view(dg, "scales").double(), gs, rtol=1e-4, atol=1e-12)
    for g in ("means", "quats", "sh"):
        assert torch.equal(a.view(a.grad, g), a.view(g0, g))
    st.regularize(a)  # the ticket was left at zero: the second call reports the same loss
    assert torch.equal(st.reg_loss, loss)


def _gaussian_args(s, dev):
    return (s.means.to(dev), s.quats.to(dev), torch.log(s.scales).to(dev), torch.logit(s.opacities).to(dev), s.sh.to(dev))


def test_trainer_grows_to_the_cap_with_camera_optimizer_and_bilateral_grid(cuda):
    s = scene_s0(N=3000, C=2, size=96)
    t = s.to(cuda)
    bg = torch.tensor([0.3, 0.3, 0.3], device=cuda)
    cfg = TrainConfig(strategy="mcmc", max_gs_num=3500, warmup_length=2, refine_every=5, camera_optimizer="SO3xR3", use_bilateral_grid=True,
                      sh_degree_interval=10, ssim_lambda=0.2)
    tr = SplatTrainer(*_gaussian_args(s, cuda), cfg=cfg, num_cameras=2)
    c2w = camera_to_worlds(s.viewmats).to(cuda)
    ids = torch.tensor([0, 1])
    losses, Ns, infos = [], [], []
    for _ in range(80):
        loss, info = tr.step(None, t.Ks, s.width, s.height, t.gt_rgb, t.gt_depth, bg, camera_to_worlds=c2w, camera_ids=ids)
        losses.append(float(loss[0]))
        Ns.append(tr.arena.N)
        if info is not None:
            infos.append(info)
    print("mcmc trainer", dict(first=losses[0], last=losses[-1], N=Ns[-1], infos=infos[:3]))
    assert Ns[-1] == 3500 and Ns == sorted(Ns) and Ns.index(3500) < 60
    assert all(i["n"] <= 3500 for i in infos)
    assert infos[-1]["n_added"] == 0
    assert all(np.isfinite(losses)) and bool(torch.isfinite(tr.arena.param).all())
    assert np.mean(losses[-5:]) < 0.9 * np.mean(losses[:5])
    assert tr.mcmc_reg_loss is not None and bool((tr.mcmc_reg_loss > 0).all())
    assert float(tr.pose_adjustment.abs().max()) > 0 and float(tr.bilagrid_tv_loss) >= 0 and tr.bilagrid.grad.abs().max() > 0


def _exchange_worker(rank, port, out):
    """One process, an NCCL group of one: an MCMC trainer forced onto the exchange path next to the plain one."""
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    res = {}
    try:
        s = scene_s0(N=4000, C=2, size=96)
        cfg = dict(strategy="mcmc", max_gs_num=4500, warmup_length=1, refine_every=2, **FROZEN)
        xt = SplatTrainer(*_gaussian_args(s, dev), cfg=TrainConfig(comm="exchange", **cfg))
        xt.comm = "exchange"  # world 1 picks no collective; one rank runs the multi-GPU code path unchanged
        ref = SplatTrainer(*_gaussian_args(s, dev), cfg=TrainConfig(**cfg))
        bg = torch.tensor([0.2, 0.5, 0.8], device=dev)
        t = s.to(dev)
        res.update(grad_err=[], grad_scale=[], exchanges=[], N=[])
        for _ in range(8):
            infos = [tr.step(t.viewmats, t.Ks, s.width, s.height, t.gt_rgb, t.gt_depth, bg)[1] for tr in (xt, ref)]
            if infos[1] is None:  # a step that grew the set leaves fresh (zero) gradient arenas behind
                res["grad_err"].append(float((xt.arena.grad - ref.arena.grad).abs().max()))
                res["grad_scale"].append(float(ref.arena.grad.abs().max()))
            res["exchanges"].append(id(xt._xg))
            res["N"].append((xt.arena.N, ref.arena.N))
        res["comm"] = xt.comm
        res["capacity"] = xt._xg.capacity
        res["param_err"] = float((xt.arena.param - ref.arena.param).abs().max())  # same draws: the same sets
    except RuntimeError as e:  # no symmetric memory available
        res["error"] = str(e)
    torch.save(res, out)
    dist.destroy_process_group()


def test_trainer_exchange_path_on_one_gpu(cuda, tmp_path):
    out = str(tmp_path / "xchg.pt")
    mp.spawn(_exchange_worker, args=(29500 + (os.getpid() + 31) % 2000, out), nprocs=1, join=True)
    r = torch.load(out)
    if "error" in r and "symmetric memory" in r["error"]:
        pytest.skip(r["error"])
    assert "error" not in r, r
    assert r["comm"] == "exchange" and r["capacity"] >= 4500, r
    assert len(set(r["exchanges"])) == 1, r  # sized for max_gs_num once: never rebuilt while N grows
    assert r["N"][0][0] < r["N"][-1][0] and all(a == b for a, b in r["N"]), r
    assert len(r["grad_err"]) >= 4, r
    for err, scale in zip(r["grad_err"], r["grad_scale"]):
        assert scale > 0 and err <= 1e-4 * scale, r
    assert r["param_err"] <= 1e-6, r
