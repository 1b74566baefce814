"""-m gpu: tile lists in the regimes their sizes switch on -- tile-sort key widths of 15, 16 and 17 bits (two passes,
an exact two-pass fit, a third pass with a 1-bit mask), 64-bit prepare keys of up to 38 bits, and scenes of more than
1024 x 2048 (camera, Gaussian) entries, where the single-launch scan sums several tiles per block and the prepare
sort runs three kernels per pass with its count on the device.

Reference: the oracle's isect_tiles / isect_offset_encode on the CPU, fed with the CUDA projection's outputs (the
projection itself is checked bit for bit elsewhere).  Each test recomputes its regime from the formulas of
isect.cu / scan.cuh / radix.cuh and asserts that it is reached.
"""
import contextlib
import functools

import pytest
import torch

import oracle
from qed_splatter_b200 import _lib, ops
from qed_splatter_b200._lib import check, current_stream, ptr
from qed_splatter_b200.pipeline import FusedSplatStep
from qed_splatter_b200.scenes import scene_s1
from helpers import assert_close_frac

pytestmark = pytest.mark.gpu

SCAN_TILE, FLAT_SCAN_BLOCKS = 2048, 1024  # scan.cuh kScanTile, kFlatScanBlocks
SORT_TILE, ONESWEEP_MAX_BLOCKS = 4096, 3 * 148  # radix.cuh kSortTile, kOnesweepMaxBlocks

# name: C, width, height, N, focal length, what the case must reach (tile-sort key bits, prepare key bits, flat-scan
# tiles per block, prepare sort with three kernels per pass)
CASES = {
    "4k_c1": dict(C=1, W=3840, H=2160, N=300_000, f=2400.0, tile_key=15, prep_key=32, tpb=1, three=False),
    "1080p_c8": dict(C=8, W=1920, H=1080, N=100_000, f=1200.0, tile_key=16, prep_key=35, tpb=1, three=False),
    "1080p_c9": dict(C=9, W=1920, H=1080, N=100_000, f=1200.0, tile_key=17, prep_key=36, tpb=1, three=False),
    "1080p_c16": dict(C=16, W=1920, H=1080, N=100_000, f=1200.0, tile_key=17, prep_key=36, tpb=1, three=False),
    "4k_c3": dict(C=3, W=3840, H=2160, N=100_000, f=2400.0, tile_key=17, prep_key=34, tpb=1, three=False),
    "128_c64": dict(C=64, W=128, H=128, N=20_000, f=80.0, tile_key=13, prep_key=38, tpb=1, three=False),
    "flat2_c1": dict(C=1, W=1920, H=1080, N=2_097_153, f=1200.0, tile_key=13, prep_key=32, tpb=2, three=True),
    "1440_c4": dict(C=4, W=1440, H=1080, N=800_000, f=1000.0, tile_key=15, prep_key=34, tpb=2, three=True),
}


def regime(C, N, W, H):
    """The code paths isect.cu picks for these sizes, from its own formulas."""
    tw, th = ops.tile_grid(W, H, 16)
    tile_key = (tw * th).bit_length() + (C - 1).bit_length()  # qed_isect_fill: tile bits + camera bits
    prep_key = 32 + (C - 1).bit_length() if C > 1 else 32     # qed_isect_prepare: (camera, depth bits)
    CN = C * N
    tiles = -(-CN // SCAN_TILE)
    blocks = min(tiles, FLAT_SCAN_BLOCKS)
    tpb = -(-tiles // blocks)                                  # scan_flat_to: tiles per block
    three = -(-CN // SORT_TILE) > ONESWEEP_MAX_BLOCKS           # prepare sort: three kernels per pass
    passes = -(-tile_key // 8)
    return dict(tile_key=tile_key, prep_key=prep_key, tpb=tpb, three=three, passes=passes, last_mask_bits=tile_key - 8 * (passes - 1))


@functools.lru_cache(maxsize=1)
def scene(name):
    c = CASES[name]
    return scene_s1(N=c["N"], width=c["W"], height=c["H"], C=c["C"], f=c["f"], sh_degree=1, targets=False)


@functools.lru_cache(maxsize=1)
def projected(name, device):
    s = scene(name)
    g = s.to(device)
    with torch.no_grad():
        radii, means2d, depths, _, _, _, _, tiles, _, _ = ops.project_gaussians(g.means, g.quats, g.scales, g.opacities, g.sh, g.viewmats, g.Ks,
                                                                                g.width, g.height, sh_degree=1)
    return radii, means2d, depths, tiles


@contextlib.contextmanager
def hook(name, value):
    lib = _lib.load()
    fn = getattr(lib, name)
    old = fn(value)
    try:
        yield
    finally:
        fn(old)


def prepare_counts(C, N, depths, tiles):
    lib = _lib.load()
    pws_bytes = lib.qed_isect_prepare_workspace_bytes(C * N)
    pws = torch.empty(pws_bytes, dtype=torch.uint8, device=depths.device)
    counts = torch.full((2,), -1, dtype=torch.int64, device=depths.device)
    host = torch.full((2,), -1, dtype=torch.int64).pin_memory()
    check(lib.qed_isect_prepare(C, N, ptr(depths), ptr(tiles), ptr(pws), pws_bytes, ptr(counts), ptr(host), current_stream()), "qed_isect_prepare")
    torch.cuda.synchronize()
    return counts.cpu(), host.clone()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("name", list(CASES))
def test_tile_lists_match_oracle(cuda, name):
    c = CASES[name]
    C, N, W, H = c["C"], c["N"], c["W"], c["H"]
    r = regime(C, N, W, H)
    assert (r["tile_key"], r["prep_key"], r["tpb"], r["three"]) == (c["tile_key"], c["prep_key"], c["tpb"], c["three"]), r
    if r["tile_key"] == 17:
        assert r["passes"] == 3 and r["last_mask_bits"] == 1
    radii, means2d, depths, tiles = projected(name, cuda)
    tw, th = ops.tile_grid(W, H, 16)
    t_o, ids_o, flat_o = oracle.isect_tiles(means2d.cpu(), radii.cpu(), depths.cpu(), 16, tw, th)
    off_o = oracle.isect_offset_encode(ids_o, C, tw, th)
    assert torch.equal(tiles.cpu(), t_o)
    # every view has entries, so the top camera bit of the key is in use
    per_view = t_o.to(torch.int64).sum(1)
    assert bool((per_view > 1000).all()), per_view
    n_isects = ids_o.numel()
    if r["tpb"] > 1:
        assert C * N > 1024 * SCAN_TILE
    counts, host = prepare_counts(C, N, depths, tiles)
    want = torch.tensor([int((t_o > 0).sum()), n_isects])
    assert torch.equal(counts, want) and torch.equal(host, want), (counts, host, want)
    with hook("qed_debug_set_flat_scan", 0):
        counts0, _ = prepare_counts(C, N, depths, tiles)
    assert torch.equal(counts0, want)

    for impl in ops.SORT_IMPLS:
        t, ids, flat, off = ops.isect_tiles(means2d, radii, depths, 16, tw, th, tiles_per_gauss=tiles, impl=impl, return_offsets=True)
        assert ids.numel() == n_isects
        assert torch.equal(ids.cpu(), ids_o), f"isect_ids ({impl})"
        assert torch.equal(flat.cpu(), flat_o), f"flatten_ids ({impl})"
        assert torch.equal(off.cpu(), off_o), f"isect_offsets ({impl})"
        t2, ids2, flat2 = ops.isect_tiles(means2d, radii, depths, 16, tw, th, impl=impl)  # counts from qed_isect_count
        assert torch.equal(t2, tiles) and torch.equal(ids2, ids) and torch.equal(flat2, flat), impl
    # the kept alternatives of the two-level build (thread-local hooks, restored): the same bytes
    for hname, value in (("qed_debug_set_flat_scan", 0), ("qed_debug_set_radix_onesweep", 0), ("qed_debug_set_radix_onesweep", 2),
                         ("qed_debug_set_radix_small_tiles", 1)):
        with hook(hname, value):
            _, ids, flat, off = ops.isect_tiles(means2d, radii, depths, 16, tw, th, tiles_per_gauss=tiles, impl="two_level", return_offsets=True)
        assert torch.equal(ids.cpu(), ids_o) and torch.equal(flat.cpu(), flat_o) and torch.equal(off.cpu(), off_o), f"{hname}({value})"


def _step(fs, s, bg, **kw):
    out = fs.step(s.means, s.quats, s.scales, s.opacities, s.sh, s.viewmats, s.Ks, s.width, s.height, 1, s.gt_rgb, s.gt_depth, bg, **kw)
    return out


def _entry_tiles(offsets, n):
    """Range table [n_tiles] -> the (view, tile) index of each of the n entries."""
    return torch.searchsorted(offsets.to(torch.int64), torch.arange(n, device=offsets.device), right=True) - 1


@functools.lru_cache(maxsize=1)
def scene_with_targets(name):
    c = CASES[name]
    return scene_s1(N=c["N"], width=c["W"], height=c["H"], C=c["C"], f=c["f"], sh_degree=1, targets=True)


EXACT_CASES = ["4k_c1", "1080p_c8", "1080p_c16", "4k_c3", "128_c64", "flat2_c1", "1440_c4"]


@pytest.mark.timeout(400)
@pytest.mark.parametrize("name", EXACT_CASES)
def test_exact_lists_and_batched_views(cuda, name):
    """FusedSplatStep at these sizes: (1) the exact tile lists are, per tile, an ordered subset of the bounding-box
    lists, every dropped entry stays below alpha = 1/255 on its tile (sampled), and the images are bit-identical;
    (2) a batch of C views renders each view bit-identically to C single-view steps, and its gradients are the mean
    of theirs."""
    c = CASES[name]
    s = scene_with_targets(name).to(cuda)
    C, W, H = s.C, s.width, s.height
    bg = torch.tensor([0.3, 0.1, 0.6], device=cuda)
    res = {}
    for exact in (False, True):
        fs = FusedSplatStep(cuda, exact_tile_lists=exact, defer_sync=False)
        out = _step(fs, s, bg)
        f = fs._fwd
        n = fs.n_isects_exact()
        n_tiles = C * f["tw"] * f["th"]
        res[exact] = dict(render=out.render.clone(), alphas=out.alphas.clone(), grads={k: v.clone() for k, v in out.grads.items()},
                          flat=f["flat"][:n].clone(), off=f["offsets"][:n_tiles].clone(), n=n, M=out.n_isects, geom=f["geom"].clone(),
                          tw=f["tw"], th=f["th"])
        del fs
    a, b = res[False], res[True]
    assert a["n"] == a["M"] and b["n"] == b["M"] and 0 < b["n"] < a["n"]
    assert torch.equal(a["render"], b["render"]) and torch.equal(a["alphas"], b["alphas"])
    for k in a["grads"]:
        sc = float(a["grads"][k].abs().mean()) + 1e-12
        assert_close_frac(b["grads"][k], a["grads"][k], 1e-4, 1e-4 * sc, 1e-3, f"exact v_{k}")
    # ordered subset: a Gaussian appears at most once per tile, so (tile, Gaussian) identifies an entry
    CN = C * s.N
    code_a = _entry_tiles(a["off"], a["n"]) * CN + a["flat"].to(torch.int64)
    code_b = _entry_tiles(b["off"], b["n"]) * CN + b["flat"].to(torch.int64)
    sorted_a, order_a = torch.sort(code_a)
    assert bool((sorted_a[1:] != sorted_a[:-1]).all()), "a Gaussian listed twice in one tile"
    pos = torch.searchsorted(sorted_a, code_b).clamp(max=a["n"] - 1)
    assert torch.equal(sorted_a[pos], code_b), "an exact entry is not in the bounding-box lists"
    pos_in_a = order_a[pos]
    assert bool((pos_in_a[1:] > pos_in_a[:-1]).all()), "the exact lists are not an ordered subset"
    kept = torch.zeros(a["n"], dtype=torch.bool, device=cuda)
    kept[pos_in_a] = True
    dropped = torch.nonzero(~kept)[:, 0]
    assert dropped.numel() == a["n"] - b["n"]
    # dropped entries (a sample) stay below 1/255 at every pixel centre of their tile (float64)
    g = torch.Generator(device="cpu").manual_seed(0)
    sample = dropped[torch.randperm(dropped.numel(), generator=g)[:50_000].to(cuda)]
    tile = (code_a[sample] // CN) % (a["tw"] * a["th"])
    gid = a["flat"][sample].to(torch.int64)
    gg = a["geom"].view(-1, 8)[gid].double()  # mx, my, opacity, depth, a, b, c, -
    ty, tx = (tile // a["tw"]).double(), (tile % a["tw"]).double()
    off16 = torch.arange(16, device=cuda, dtype=torch.float64)
    xs = tx[:, None] * 16 + off16[None] + 0.5  # [S,16]
    ys = ty[:, None] * 16 + off16[None] + 0.5
    dx = gg[:, 0, None, None] - xs[:, None, :]
    dy = gg[:, 1, None, None] - ys[:, :, None]
    sigma = 0.5 * (gg[:, 4, None, None] * dx * dx + gg[:, 6, None, None] * dy * dy) + gg[:, 5, None, None] * dx * dy
    alpha = gg[:, 2, None, None] * torch.exp(-sigma)
    inside = (xs[:, None, :] < W) & (ys[:, :, None] < H)
    assert float(torch.where(inside, alpha, torch.zeros((), dtype=alpha.dtype, device=cuda)).max()) < 1.0 / 255.0

    # batched views == single views
    fs = FusedSplatStep(cuda, defer_sync=False)
    whole = _step(fs, s, bg)
    whole_r, whole_a = whole.render.clone(), whole.alphas.clone()
    whole_g = {k: v.clone() for k, v in whole.grads.items()}
    assert torch.equal(whole_r, b["render"])
    acc = {k: torch.zeros_like(v) for k, v in whole_g.items()}
    for v in range(C):
        sl = slice(v, v + 1)
        one = fs.step(s.means, s.quats, s.scales, s.opacities, s.sh, s.viewmats[sl].contiguous(), s.Ks[sl].contiguous(), W, H, 1,
                      s.gt_rgb[sl].contiguous(), s.gt_depth[sl].contiguous(), bg, grad_scale=1.0 / C)
        assert torch.equal(one.render[0], whole_r[v]) and torch.equal(one.alphas[0], whole_a[v]), f"view {v}"
        for k in acc:
            acc[k] += one.grads[k]
    for k in acc:
        scale = float(whole_g[k].abs().mean()) + 1e-12
        assert_close_frac(acc[k], whole_g[k], 1e-4, 1e-5 * scale, 1e-3, f"batched v_{k}")
    if c["tpb"] > 1:
        assert C * s.N > 1024 * SCAN_TILE


@pytest.mark.timeout(400)
@pytest.mark.parametrize("name", ["flat2_c1", "1440_c4"])
@pytest.mark.parametrize("exact", [True, False])
def test_deferred_sizes_beyond_the_flat_scan_limit(cuda, name, exact):
    """FusedSplatStep(defer_sync=True) at C*N > 1024 x 2048: lists built into buffers sized from earlier calls give the
    synchronous path's images, also when a call overflows the learnt capacity and is repeated."""
    small = scene_with_targets(name).to(cuda)
    assert regime(small.C, small.N, small.width, small.height)["tpb"] > 1
    big = scene_with_targets(name).to(cuda)
    big.scales = big.scales * 3.0
    bg = torch.tensor([0.1, 0.2, 0.3], device=cuda)

    def run(fs, s):
        out = _step(fs, s, bg)
        return out.render.clone(), out.alphas.clone(), out.loss.clone(), {k: v.clone() for k, v in out.grads.items()}, out.n_isects

    sync = FusedSplatStep(cuda, defer_sync=False, exact_tile_lists=exact)
    ref_small, ref_big = run(sync, small), run(sync, big)
    del sync
    defer = FusedSplatStep(cuda, defer_sync=True, exact_tile_lists=exact)
    first = run(defer, small)
    second = run(defer, small)
    assert defer._cap_isects > 0 and defer.overflow_repeats == 0
    third = run(defer, big)
    assert defer.overflow_repeats == 1 and ref_big[4] > ref_small[4] + ref_small[4] // 4 + 4096
    fourth = run(defer, big)
    assert defer.overflow_repeats == 1
    for got, ref in ((first, ref_small), (second, ref_small), (third, ref_big), (fourth, ref_big)):
        assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1]) and got[4] == ref[4]
        assert float(got[2][0]) == pytest.approx(float(ref[2][0]), rel=1e-6)
        for k in ref[3]:
            scale = float(ref[3][k].abs().mean()) + 1e-20
            assert_close_frac(got[3][k], ref[3][k], 1e-4, 1e-5 * scale, 1e-3, f"deferred v_{k}")
