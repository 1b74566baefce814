"""Op-level host wrappers over the C-ABI (one per stage of the hot path) with torch autograd.

Names and argument meaning follow gsplat 1.4.0's `gsplat/cuda/_wrapper.py`, which is what
`gsplat.rendering.rasterization` — the call at `/root/reference/qed_splatter/model.py:267-288` — is
built from: `fully_fused_projection`, `isect_tiles`, `isect_offset_encode`, `rasterize_to_pixels`.
`project_gaussians` is the fused projection + SH stage this library actually runs.

torch is used for device memory, streams and autograd bookkeeping only; every computation is a kernel
in `libqedsplat.so`.  CUDA tensors only — CPU tensors raise (no fallback).
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import check, current_stream, ptr

GRAD_FLOATS = 12
GEOM_FLOATS = 8
_SORT_IMPL = "two_level"  # "two_level" (product path) | "own" | "cub" — identical output
SORT_IMPLS = ("two_level", "own", "cub")


def set_sort_impl(name: str) -> str:
    """Select how isect_tiles builds the sorted intersection list:
    "two_level": depth-sort the visible Gaussians, emit in that order, stable radix on the tile bits (default);
    "own": gsplat's formulation (emit 64-bit keys, full radix sort) with this library's radix sort;
    "cub": the same with cub::DeviceRadixSort (the library baseline gsplat uses)."""
    global _SORT_IMPL
    assert name in SORT_IMPLS
    old, _SORT_IMPL = _SORT_IMPL, name
    return old


def _f32c(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        raise TypeError(f"expected float32, got {t.dtype}")
    return t.contiguous()


def tile_grid(width: int, height: int, tile_size: int) -> Tuple[int, int]:
    return math.ceil(width / tile_size), math.ceil(height / tile_size)


def ctypes_ptr(addr: Optional[int]):
    import ctypes

    return None if addr is None else ctypes.c_void_p(addr)


def _packed_record_of(v_means2d, v_conics, v_colors, v_opac, C: int, N: int, D: int) -> Optional[int]:
    """Address of the packed [C*N,12] gradient record if the four tensors are exactly the views
    `_RasterizeToPixels.backward` returns of one such record (same storage, slots 0:2 / 4:7 / 8:8+D / 7, row stride 12),
    else None (autograd summed or copied them: they are then ordinary tensors and are passed one by one)."""
    ts = (v_means2d, v_conics, v_colors, v_opac)
    if any(t is None or t.dtype != torch.float32 for t in ts):
        return None
    base = v_means2d.untyped_storage().data_ptr()
    if any(t.untyped_storage().data_ptr() != base for t in ts):
        return None
    o0 = v_means2d.storage_offset()
    want = ((v_means2d, (C, N, 2), o0), (v_conics, (C, N, 3), o0 + 4), (v_colors, (C, N, D), o0 + 8), (v_opac, (C, N), o0 + 7))
    for t, shape, off in want:
        if tuple(t.shape) != shape or t.storage_offset() != off:
            return None
        st = t.stride()
        if st[0] != N * GRAD_FLOATS or st[1] != GRAD_FLOATS or (len(st) == 3 and shape[2] > 1 and st[2] != 1):
            return None
    addr = base + 4 * o0
    return addr if addr % 16 == 0 else None


# --------------------------------------------------------------------------------------------- #
# (a) fused projection + SH
# --------------------------------------------------------------------------------------------- #
class _ProjectGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means, quats, scales, opacities, colors, viewmats, Ks, width, height, eps2d, near_plane,
                far_plane, radius_clip, calc_compensations, sh_degree, n_color, append_depth, tile_size):
        lib = _lib.load()
        _lib.require_cuda(means, quats, scales, opacities, colors, viewmats, Ks)
        means, quats, scales = _f32c(means), _f32c(quats), _f32c(scales)
        opacities, colors = _f32c(opacities), _f32c(colors)
        viewmats, Ks = _f32c(viewmats), _f32c(Ks)
        N, C = means.shape[0], viewmats.shape[0]
        D = n_color + append_depth
        dev = means.device
        K = 0
        per_cam = 0
        if n_color:
            if sh_degree >= 0:
                assert colors.dim() == 3 and colors.shape[0] == N and colors.shape[2] == 3, "SH coeffs must be [N,K,3]"
                K = colors.shape[1]
                assert (sh_degree + 1) ** 2 <= K, "sh_degree too large for the coefficient tensor"
            else:
                assert colors.shape[-1] == 3, "only 3 colour channels are supported on this path"
                per_cam = 1 if colors.dim() == 3 else 0
                if per_cam:
                    assert colors.shape[:2] == (C, N)
        radii = torch.empty(C, N, dtype=torch.int32, device=dev)
        means2d = torch.empty(C, N, 2, device=dev)
        depths = torch.empty(C, N, device=dev)
        conics = torch.empty(C, N, 3, device=dev)
        comps = torch.empty(C, N, device=dev) if calc_compensations else None
        colors_out = torch.empty(C, N, D, device=dev)
        opac_out = torch.empty(C, N, device=dev)
        tiles = torch.empty(C, N, dtype=torch.int32, device=dev)
        tiles_exact = torch.empty(C, N, dtype=torch.int32, device=dev) if tile_size == 16 else None
        geom = torch.empty(C, N, GEOM_FLOATS, device=dev)
        check(lib.qed_project_fwd(C, N, ptr(means), ptr(quats), ptr(scales), ptr(opacities), 0, ptr(colors) if n_color else None,
                                  K, sh_degree, per_cam, ptr(viewmats), ptr(Ks), width, height, eps2d, near_plane,
                                  far_plane, radius_clip, int(calc_compensations), tile_size, n_color, append_depth,
                                  ptr(radii), ptr(means2d), ptr(depths), ptr(conics), ptr(comps), ptr(colors_out),
                                  ptr(opac_out), ptr(tiles), ptr(tiles_exact), ptr(geom), current_stream()), "qed_project_fwd")
        ctx.save_for_backward(means, quats, scales, opacities, colors, viewmats, Ks, radii, conics, comps)
        ctx.cfg = (width, height, eps2d, calc_compensations, sh_degree, n_color, append_depth, K, per_cam)
        if tiles_exact is None:
            tiles_exact = torch.empty(0, dtype=torch.int32, device=dev)
        ctx.mark_non_differentiable(radii, tiles, geom, tiles_exact)
        if comps is None:
            comps_out = torch.empty(0, device=dev)
            ctx.mark_non_differentiable(comps_out)
        else:
            comps_out = comps
        return radii, means2d, depths, conics, comps_out, colors_out, opac_out, tiles, geom, tiles_exact

    @staticmethod
    def backward(ctx, _v_radii, v_means2d, v_depths, v_conics, v_comps, v_colors, v_opac, _v_tiles, _v_geom, _v_tiles_exact):
        lib = _lib.load()
        means, quats, scales, opacities, colors, viewmats, Ks, radii, conics, comps = ctx.saved_tensors
        width, height, eps2d, calc_comp, sh_degree, n_color, append_depth, K, per_cam = ctx.cfg
        N, C = means.shape[0], viewmats.shape[0]
        dev = means.device
        if calc_comp and v_comps is not None and v_comps.numel() and bool((v_comps != 0).any()):
            raise NotImplementedError("gradient through `compensations` itself is not on the reference path")
        v_means = torch.empty_like(means)
        v_quats = torch.empty_like(quats)
        v_scales = torch.empty_like(scales)
        v_opacities = torch.empty_like(opacities) if opacities is not None else None
        v_colors_in = torch.empty_like(colors) if n_color else None
        packed = _packed_record_of(v_means2d, v_conics, v_colors, v_opac, C, N, n_color + append_depth)
        if packed is not None:
            # the four gradients are the views _RasterizeToPixels.backward made of ONE packed record: the kernel reads it directly
            separate = (None, ptr(_f32c(v_depths)), None, None, None)
        else:
            separate = (ptr(_f32c(v_means2d)), ptr(_f32c(v_depths)), ptr(_f32c(v_conics)), ptr(_f32c(v_colors)), ptr(_f32c(v_opac)))
        args = (C, N, ptr(means), ptr(quats), ptr(scales), ptr(opacities), 0, ptr(colors) if n_color else None,
                K, sh_degree, per_cam, ptr(viewmats), ptr(Ks), width, height, eps2d, int(calc_comp),
                n_color, append_depth, ptr(radii), ptr(conics), ptr(comps),
                *separate, ctypes_ptr(packed), ptr(v_means), ptr(v_quats), ptr(v_scales), ptr(v_opacities), ptr(v_colors_in))
        v_viewmats = None
        if ctx.needs_input_grad[5]:  # camera poses (gsplat's v_viewmats)
            v_viewmats = torch.empty(C, 4, 4, device=dev)
            ws_bytes = lib.qed_project_bwd_pose_workspace_bytes(C, N)
            ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
            check(lib.qed_project_bwd_pose(*args, ptr(v_viewmats), ptr(ws), ws_bytes, current_stream()), "qed_project_bwd_pose")
        else:
            check(lib.qed_project_bwd(*args, current_stream()), "qed_project_bwd")
        return (v_means, v_quats, v_scales, v_opacities, v_colors_in, v_viewmats, None) + (None,) * 11


def project_gaussians(means: Tensor, quats: Tensor, scales: Tensor, opacities: Tensor, colors: Optional[Tensor],
                      viewmats: Tensor, Ks: Tensor, width: int, height: int, eps2d: float = 0.3,
                      near_plane: float = 0.01, far_plane: float = 1e10, radius_clip: float = 0.0,
                      calc_compensations: bool = False, sh_degree: Optional[int] = None, n_color: int = 3,
                      append_depth: bool = True, tile_size: int = 16):
    """Fused fully_fused_projection + spherical_harmonics (+ clamp_min(c+0.5), depth concat, opacity*comp).

    -> radii[C,N] i32, means2d[C,N,2], depths[C,N], conics[C,N,3], compensations[C,N]|None,
       colors[C,N,D], opacities[C,N], tiles_per_gauss[C,N] i32, geom[C,N,8], tiles_exact[C,N] i32 (the tiles each Gaussian
       can reach with alpha >= 1/255: what `isect_tiles_exact` builds the compositor's lists from)
    """
    if colors is None:
        colors = torch.empty(0, device=means.device)
        n_color = 0
    out = _ProjectGaussians.apply(means, quats, scales, opacities, colors, viewmats, Ks, int(width), int(height),
                                  float(eps2d), float(near_plane), float(far_plane), float(radius_clip),
                                  bool(calc_compensations), -1 if sh_degree is None else int(sh_degree), int(n_color),
                                  int(bool(append_depth)), int(tile_size))
    radii, means2d, depths, conics, comps, colors_out, opac_out, tiles, geom, tiles_exact = out
    return radii, means2d, depths, conics, (comps if calc_compensations else None), colors_out, opac_out, tiles, geom, tiles_exact


def fully_fused_projection(means: Tensor, covars, quats: Tensor, scales: Tensor, viewmats: Tensor, Ks: Tensor,
                           width: int, height: int, eps2d: float = 0.3, near_plane: float = 0.01,
                           far_plane: float = 1e10, radius_clip: float = 0.0, packed: bool = False,
                           sparse_grad: bool = False, calc_compensations: bool = False):
    """gsplat `fully_fused_projection` surface -> (radii, means2d, depths, conics, compensations)."""
    if covars is not None or packed or sparse_grad:
        raise NotImplementedError("covars / packed / sparse_grad are not reachable from qed_splatter/model.py:267-288")
    opac = torch.ones(means.shape[0], device=means.device)
    radii, means2d, depths, conics, comps, _, _, _, _, _ = project_gaussians(
        means, quats, scales, opac, None, viewmats, Ks, width, height, eps2d, near_plane, far_plane, radius_clip,
        calc_compensations, None, 0, True)
    return radii, means2d, depths, conics, comps


# --------------------------------------------------------------------------------------------- #
# (b) tile intersection
# --------------------------------------------------------------------------------------------- #
@torch.no_grad()
def isect_tiles(means2d: Tensor, radii: Tensor, depths: Tensor, tile_size: int, tile_width: int, tile_height: int,
                sort: bool = True, tiles_per_gauss: Optional[Tensor] = None, impl: Optional[str] = None,
                return_offsets: bool = False):
    """gsplat `isect_tiles` -> tiles_per_gauss[C,N] i32, isect_ids[M] i64, flatten_ids[M] i32 (sorted).
    `return_offsets=True` additionally returns isect_offsets[C,th,tw] (the two-level build produces the ranges in
    the same pass that composes the 64-bit ids, so `isect_offset_encode` need not re-read them)."""
    lib = _lib.load()
    _lib.require_cuda(means2d, radii, depths)
    means2d, depths = _f32c(means2d.detach()), _f32c(depths.detach())
    radii = radii.contiguous()
    assert radii.dtype == torch.int32
    C, N = radii.shape
    dev = means2d.device
    stream = current_stream()
    impl = impl or _SORT_IMPL
    if tiles_per_gauss is None:
        tiles_per_gauss = torch.empty(C, N, dtype=torch.int32, device=dev)
        check(lib.qed_isect_count(C, N, ptr(means2d), ptr(radii), tile_size, tile_width, tile_height,
                                  ptr(tiles_per_gauss), stream), "qed_isect_count")
    CN = C * N
    if impl == "two_level" and sort:
        pws_bytes = lib.qed_isect_prepare_workspace_bytes(CN)
        pws = torch.empty(pws_bytes, dtype=torch.uint8, device=dev)
        counts = torch.zeros(2, dtype=torch.int64, device=dev)
        check(lib.qed_isect_prepare(C, N, ptr(depths), ptr(tiles_per_gauss), ptr(pws), pws_bytes, ptr(counts), None, stream),
              "qed_isect_prepare")
        n_visible, n_isects = (int(v) for v in counts.tolist())  # the one host sync of the forward (gsplat has the same one)
        isect_ids = torch.empty(n_isects, dtype=torch.int64, device=dev)
        flatten_ids = torch.empty(n_isects, dtype=torch.int32, device=dev)
        offsets = torch.empty(C, tile_height, tile_width, dtype=torch.int32, device=dev) if return_offsets else None
        fws_bytes = lib.qed_isect_fill_workspace_bytes(n_isects)
        fws = torch.empty(fws_bytes, dtype=torch.uint8, device=dev)
        # geom = NULL: gsplat's lists bit for bit (the exact tile lists are the fused pipeline's business)
        check(lib.qed_isect_fill(C, N, n_visible, n_isects, ptr(means2d), ptr(radii), ptr(depths), None, 0, 0, tile_size, tile_width,
                                 tile_height, ptr(pws), ptr(fws), fws_bytes, None, ptr(isect_ids) if n_isects else None,
                                 ptr(flatten_ids) if n_isects else None, ptr(offsets), None, stream), "qed_isect_fill")
        if return_offsets:
            return tiles_per_gauss, isect_ids, flatten_ids, offsets
        return tiles_per_gauss, isect_ids, flatten_ids
    cum = torch.empty(CN, dtype=torch.int64, device=dev)
    total = torch.zeros(1, dtype=torch.int64, device=dev)
    ws_bytes = lib.qed_isect_scan_workspace_bytes(CN)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    check(lib.qed_isect_scan(CN, ptr(tiles_per_gauss), ptr(cum), ptr(total), None, ptr(ws), ws_bytes, stream), "qed_isect_scan")
    n_isects = int(total.item())
    isect_ids = torch.empty(n_isects, dtype=torch.int64, device=dev)
    flatten_ids = torch.empty(n_isects, dtype=torch.int32, device=dev)
    if n_isects:
        check(lib.qed_isect_emit(C, N, ptr(means2d), ptr(radii), ptr(depths), ptr(cum), tile_size, tile_width,
                                 tile_height, ptr(isect_ids), ptr(flatten_ids), stream), "qed_isect_emit")
        if sort:
            tile_n_bits = (tile_width * tile_height).bit_length()
            cam_n_bits = C.bit_length()
            isect_ids, flatten_ids = sort_pairs(isect_ids, flatten_ids, 32 + tile_n_bits + cam_n_bits,
                                                impl="cub" if impl == "cub" else "own")
    if return_offsets:
        return tiles_per_gauss, isect_ids, flatten_ids, isect_offset_encode(isect_ids, C, tile_width, tile_height)
    return tiles_per_gauss, isect_ids, flatten_ids


@torch.no_grad()
def sort_pairs(keys: Tensor, vals: Tensor, end_bit: int = 64, impl: Optional[str] = None):
    """Stable ascending radix sort of (int64 key, int32 value) pairs on key bits [0, end_bit)."""
    lib = _lib.load()
    _lib.require_cuda(keys, vals)
    impl = impl or ("cub" if _SORT_IMPL == "cub" else "own")
    n = keys.numel()
    keys_out = torch.empty_like(keys)
    vals_out = torch.empty_like(vals)
    if n == 0:
        return keys_out, vals_out
    if impl == "cub":
        ws_bytes = lib.qed_sort_pairs_cub_workspace_bytes(n)
        fn, name = lib.qed_sort_pairs_cub, "qed_sort_pairs_cub"
    else:
        ws_bytes = lib.qed_sort_pairs_workspace_bytes(n)
        fn, name = lib.qed_sort_pairs, "qed_sort_pairs"
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=keys.device)
    check(fn(n, ptr(keys), ptr(vals), ptr(keys_out), ptr(vals_out), end_bit, ptr(ws), ws_bytes, current_stream()), name)
    return keys_out, vals_out


# Sizing hints for `isect_tiles_exact(defer=True)`: largest intersection count seen per (device, C, N, width, height), + 25 %.
# Only buffer SIZES come from here; a list that does not fit is detected and rebuilt, results never depend on the hint.
_CAPACITY_HINT = {}


@torch.no_grad()
def isect_tiles_exact(means2d: Tensor, radii: Tensor, depths: Tensor, geom: Tensor, width: int, height: int, tile_size: int,
                      tile_width: int, tile_height: int, tiles_exact: Tensor, defer: bool = False):
    """EXACT tile lists for the compositor (not gsplat's `info` lists): only the (Gaussian, tile) pairs that can reach
    alpha = 1/255 at a pixel centre of the tile -- `tiles_exact` = their per-Gaussian counts from `project_gaussians`
    (DESIGN.md section 5).  -> flatten_ids[M] i32 (M = capacity >= n_exact; the first n_exact entries are filled),
    isect_offsets[C*th*tw + 1] i32 (last element = n_exact = end of the last range), n_exact[1] i64 on the device,
    resolve.

    The list sizes are only known on the device.  defer=False: the host reads them between the two phases (the one
    host sync gsplat has too) and `resolve` is None.  defer=True: when an earlier call with the same shapes left a size
    hint, the lists are built into buffers of that capacity without waiting, and `resolve()` -- call it AFTER queueing
    the work that consumes the lists, so the device never idles on the read -- returns False if they did not fit (the
    device then built empty lists): build them again with defer=False."""
    lib = _lib.load()
    _lib.require_cuda(means2d, radii, depths, geom)
    means2d, depths = _f32c(means2d.detach()), _f32c(depths.detach())
    C, N = radii.shape
    dev = means2d.device
    stream = current_stream()
    pws_bytes = lib.qed_isect_prepare_workspace_bytes(C * N)
    pws = torch.empty(pws_bytes, dtype=torch.uint8, device=dev)
    counts = torch.zeros(3, dtype=torch.int64, device=dev)
    key = (dev.index, C, N, int(width), int(height))
    cap = _CAPACITY_HINT.get(key, 0) if defer else 0
    deferred = cap > 0 and C * N > 0
    counts_host = torch.empty(2, dtype=torch.int64, pin_memory=True) if deferred else None
    check(lib.qed_isect_prepare(C, N, ptr(depths), ptr(tiles_exact), ptr(pws), pws_bytes, ptr(counts), ptr(counts_host), stream),
          "qed_isect_prepare")
    resolve = None
    if deferred:
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream())
        n_visible, n_isects = C * N, cap  # capacities; the real counts stay on the device

        def resolve() -> bool:
            ready.synchronize()
            real = int(counts_host[1])
            _CAPACITY_HINT[key] = max(_CAPACITY_HINT.get(key, 0), real + real // 4 + 4096)
            return real <= cap
    else:
        n_visible, n_isects, _ = (int(v) for v in counts.tolist())  # the one host sync of the forward (gsplat has the same one)
        if defer:
            _CAPACITY_HINT[key] = max(_CAPACITY_HINT.get(key, 0), n_isects + n_isects // 4 + 4096)
    flatten_ids = torch.empty(n_isects, dtype=torch.int32, device=dev)
    offsets = torch.empty(C * tile_height * tile_width + 1, dtype=torch.int32, device=dev)
    fws_bytes = lib.qed_isect_fill_workspace_bytes(n_isects)
    fws = torch.empty(fws_bytes, dtype=torch.uint8, device=dev)
    check(lib.qed_isect_fill(C, N, n_visible, n_isects, ptr(means2d), ptr(radii), ptr(depths), ptr(geom), width, height, tile_size,
                             tile_width, tile_height, ptr(pws), ptr(fws), fws_bytes, ptr(counts) if deferred else None, None,
                             ptr(flatten_ids) if n_isects else None, ptr(offsets), ptr(counts[2:]), stream), "qed_isect_fill")
    return flatten_ids, offsets, counts[2:], resolve


@torch.no_grad()
def isect_offset_encode(isect_ids: Tensor, C: int, tile_width: int, tile_height: int) -> Tensor:
    """gsplat `isect_offset_encode` -> isect_offsets[C,tile_height,tile_width] i32."""
    lib = _lib.load()
    _lib.require_cuda(isect_ids)
    offsets = torch.empty(C, tile_height, tile_width, dtype=torch.int32, device=isect_ids.device)
    check(lib.qed_tile_ranges(isect_ids.numel(), ptr(isect_ids.contiguous()), C, tile_width, tile_height, ptr(offsets),
                              current_stream()), "qed_tile_ranges")
    return offsets


# --------------------------------------------------------------------------------------------- #
# (c)/(d) compositing
# --------------------------------------------------------------------------------------------- #
class _RasterizeToPixels(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means2d, conics, colors, opacities, backgrounds, geom, width, height, tile_size, isect_offsets,
                flatten_ids, absgrad, normalize_last):
        lib = _lib.load()
        _lib.require_cuda(means2d, conics, colors, opacities, isect_offsets, flatten_ids)
        C, N = opacities.shape
        D = colors.shape[-1]
        dev = means2d.device
        colors = _f32c(colors)
        backgrounds = _f32c(backgrounds)
        if geom is None:
            geom = torch.empty(C, N, GEOM_FLOATS, device=dev)
            check(lib.qed_pack_geom(C * N, ptr(_f32c(means2d)), ptr(_f32c(conics)), ptr(_f32c(opacities)), None, ptr(geom),
                                    current_stream()), "qed_pack_geom")
        has_end = isect_offsets.dim() == 1  # exact tile lists: [C*th*tw + 1], last element = end of the last range
        tile_width, tile_height = tile_grid(width, height, tile_size)
        assert isect_offsets.numel() == C * tile_height * tile_width + int(has_end), isect_offsets.shape
        n_isects = flatten_ids.numel()
        render = torch.empty(C, height, width, D, device=dev)
        alphas = torch.empty(C, height, width, 1, device=dev)
        last_ids = torch.empty(C, height, width, dtype=torch.int32, device=dev)
        check(lib.qed_raster_fwd(C, N, n_isects, D, ptr(geom), ptr(colors), ptr(backgrounds), width, height, tile_size,
                                 tile_width, tile_height, ptr(isect_offsets), int(has_end), ptr(flatten_ids), int(normalize_last),
                                 ptr(render), ptr(alphas), ptr(last_ids), current_stream()), "qed_raster_fwd")
        ctx.save_for_backward(means2d, conics, colors, opacities, backgrounds, geom, isect_offsets, flatten_ids, render,
                              alphas, last_ids)
        ctx.cfg = (width, height, tile_size, absgrad, normalize_last)
        ctx.mark_non_differentiable(last_ids)
        return render, alphas, last_ids

    @staticmethod
    def backward(ctx, v_render, v_alphas, _v_last):
        lib = _lib.load()
        means2d, conics, colors, opacities, backgrounds, geom, isect_offsets, flatten_ids, render, alphas, last_ids = ctx.saved_tensors
        width, height, tile_size, absgrad, normalize_last = ctx.cfg
        C, N = opacities.shape
        D = colors.shape[-1]
        dev = means2d.device
        tile_width, tile_height = tile_grid(width, height, tile_size)
        packed = torch.zeros(C * N, GRAD_FLOATS, device=dev)
        v_render = _f32c(v_render) if v_render is not None else torch.zeros_like(render)
        check(lib.qed_raster_bwd(C, N, flatten_ids.numel(), D, ptr(geom), ptr(colors), ptr(backgrounds), width, height,
                                 tile_size, tile_width, tile_height, ptr(isect_offsets), ptr(flatten_ids),
                                 int(normalize_last), ptr(render), ptr(alphas), ptr(last_ids), ptr(v_render),
                                 ptr(_f32c(v_alphas)), ptr(packed), current_stream()), "qed_raster_bwd")
        # the gradients leave as strided VIEWS of the packed [C*N,12] record (no unpack pass, no five allocations);
        # _ProjectGaussians.backward recognises them and hands the record to the kernel as it is (qed_project_bwd's
        # `packed_grads`), anything else that consumes them sees ordinary [C,N,k] tensors
        P = packed.view(C, N, GRAD_FLOATS)
        v_means2d, v_conics, v_opac, v_colors = P[..., 0:2], P[..., 4:7], P[..., 7], P[..., 8:8 + D]
        if absgrad:
            means2d.absgrad = P[..., 2:4]  # side channel read by gsplat's DefaultStrategy (model.py:284 absgrad=True)
        v_bg = None
        if backgrounds is not None and ctx.needs_input_grad[4]:
            g = v_render
            if normalize_last:
                g = g.clone()
                g[..., -1:] = g[..., -1:] / alphas.clamp(min=1e-10)
            v_bg = (g * (1.0 - alphas)).sum(dim=(1, 2))
        return v_means2d, v_conics, v_colors, v_opac, v_bg, None, None, None, None, None, None, None, None


def rasterize_to_pixels(means2d: Tensor, conics: Tensor, colors: Tensor, opacities: Tensor, image_width: int,
                        image_height: int, tile_size: int, isect_offsets: Tensor, flatten_ids: Tensor,
                        backgrounds: Optional[Tensor] = None, packed: bool = False, absgrad: bool = False,
                        geom: Optional[Tensor] = None, normalize_last: bool = False, return_last_ids: bool = False):
    """gsplat `rasterize_to_pixels` -> (render[C,H,W,D], alphas[C,H,W,1]) (+ last_ids when asked)."""
    if packed:
        raise NotImplementedError("packed mode is not reachable from qed_splatter/model.py:267-288")
    if colors.shape[-1] not in (1, 3, 4):
        raise NotImplementedError("channel count must be 1, 3 or 4 (D, RGB, RGB+D) on this path")
    if tile_size != 16:
        raise NotImplementedError("tile_size is 16 on this path (qed_splatter/model.py:243)")
    render, alphas, last_ids = _RasterizeToPixels.apply(
        means2d, conics, colors, opacities, backgrounds, geom, int(image_width), int(image_height), int(tile_size),
        isect_offsets.contiguous(), flatten_ids.contiguous(), bool(absgrad), bool(normalize_last))
    if return_last_ids:
        return render, alphas, last_ids
    return render, alphas


def set_raster_cull(enabled: bool) -> bool:
    """Test hook: disable/enable the exact warp-level culling in the compositor (results are identical)."""
    return bool(_lib.load().qed_debug_set_raster_cull(int(enabled)))


def set_raster_px(px_fwd: int = 0, px_bwd: int = 0) -> int:
    """Test/tuning hook: pixels per lane (1, 2 or 4; 0 = keep) of the forward / backward compositor.
    Returns 10*px_fwd + px_bwd now in effect."""
    return int(_lib.load().qed_debug_set_raster_px(int(px_fwd), int(px_bwd)))


def set_raster_packed(enabled: bool) -> bool:
    """Test/tuning hook: use the two-wide fp32 (FFMA2) compositor kernels where they exist (default on).
    Returns the previous setting."""
    return bool(_lib.load().qed_debug_set_raster_packed(1 if enabled else 0))
