"""Fused render + loss + backward pipeline (no autograd graph): the train-step hot path.

This is what the reference does per iteration between `get_outputs` (model.py:199-321), `get_loss_dict`
(model.py:73-118) and `loss.backward()`, restated as one straight sequence of C-ABI launches:

    project+SH fwd -> tile count scan -> emit keys -> radix sort -> tile ranges -> composite fwd
      -> loss + loss-gradient (background composite, clamp, depth fill, masked depth-L1, RGB-L1)
      -> composite bwd (packed per-Gaussian gradient records) -> project+SH bwd

Nothing is unpacked or re-laid-out between the two backward kernels: the compositor's backward writes
the [C*N,12] packed record that the projection backward reads.  `rasterization()` in rendering.py is
the autograd drop-in for the unchanged QEDSplatterModel; this class is the same kernels without the
autograd bookkeeping, used by the trainer and the benchmark.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import torch
from torch import Tensor

from . import _lib, ops
from ._lib import check, current_stream, ptr


@dataclass
class StepOutput:
    loss: Tensor  # [3] float32 device: total, rgb term, depth term
    grads: Dict[str, Tensor]  # v_means, v_quats, v_scales, v_opacities, v_sh
    packed_grads: Tensor  # [C*N,12] (absgrad in slots 2,3) for the strategy statistics
    radii: Tensor  # [C,N] i32
    render: Tensor  # [C,H,W,4]
    alphas: Tensor  # [C,H,W,1]
    n_isects: int
    n_visible: Optional[int] = None
    v_viewmats: Optional[Tensor] = None  # [C,4,4] d loss / d viewmats, step(pose_gradients=True) only


ACT_LOG_SCALES, ACT_LOGIT_OPACITIES = 1, 2  # `activations` bits (include/qed_splat.h)


def _pose_capable(exchange) -> bool:
    """No exchange, or one with a pose-gradient buffer (comm.ViewShardedGradients(num_cameras > 0))."""
    return exchange is None or getattr(exchange, "num_cameras", 0) > 0


class FusedSplatStep:
    """Holds reusable device buffers; `forward()` renders, `step()` renders + loss + full backward."""

    def __init__(self, device, sort_impl: str = "two_level", want_isect_ids: bool = False, exact_tile_lists: bool = True,
                 defer_sync: bool = True):
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.sort_impl = sort_impl
        self.want_isect_ids = want_isect_ids  # the compositor does not need the 64-bit keys; only `info` does
        # exact tile lists (two_level only): (Gaussian, tile) candidates that cannot reach alpha >= 1/255 at any pixel
        # centre of the tile are dropped before the tile sort (about half of gsplat's bounding-box lists); pixels are
        # unchanged.  The public `rasterization()` keeps gsplat's lists bit for bit (`info` contract).
        self.exact_tile_lists = exact_tile_lists
        # The sizes of the intersection lists are only known on the device.  defer_sync (two_level only): from the second
        # call on, the lists are built into buffers sized from the largest count seen so far (+25 %) and the counts are
        # read by the host AFTER the rest of the forward (and, in step(), the loss and the compositor's backward) has been
        # queued -- the device never idles on that read.  A count above the capacity builds an empty list on the device
        # (memory-safe); the host sees it, grows the buffers and repeats the pass (rare: first steps, new viewpoints).
        self.defer_sync = defer_sync and sort_impl == "two_level"
        self._cap_isects = 0
        self.overflow_repeats = 0
        self._n_exact = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._total = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._counts = torch.zeros(2, dtype=torch.int64, device=self.device)
        self._counts_host = torch.zeros(2, dtype=torch.int64).pin_memory()
        self._stats = None
        self._loss = torch.zeros(3, device=self.device)
        self._buf: Dict[str, Tensor] = {}
        self._prezero = False
        self._prezeroed = False
        self._counts_ready = torch.cuda.Event()
        self.marks = None  # set to [] to record (name, cuda event) after every stage (bench.py stage timing)

    def _mark(self, name: str) -> None:
        if self.marks is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(torch.cuda.current_stream())
            self.marks.append((name, ev))

    # -- buffers ------------------------------------------------------------------------------
    def _get(self, name: str, shape, dtype=torch.float32) -> Tensor:
        n = 1
        for s in shape:
            n *= int(s)
        t = self._buf.get(name)
        if t is None or t.dtype != dtype or t.numel() < n:
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._buf[name] = t
        return t[:n].view(*shape)

    # -- forward ------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, means, quats, scales, opacities, sh, viewmats, Ks, width: int, height: int, sh_degree: int,
                render_mode: str = "RGB+ED", rasterize_mode: str = "classic", near_plane: float = 0.01,
                far_plane: float = 1e10, eps2d: float = 0.3, backgrounds: Optional[Tensor] = None, activations: int = 0,
                _resolve: bool = True, _force_sync: bool = False):
        """`activations` (ACT_LOG_SCALES | ACT_LOGIT_OPACITIES): `scales` / `opacities` are the stored parameters; exp /
        sigmoid (qed_splatter/model.py:269-271) and their chain rule run inside the projection kernels."""
        self._call = dict(args=(means, quats, scales, opacities, sh, viewmats, Ks, width, height, sh_degree),
                          kw=dict(render_mode=render_mode, rasterize_mode=rasterize_mode, near_plane=near_plane, far_plane=far_plane, eps2d=eps2d,
                                  backgrounds=backgrounds, activations=activations))
        lib, stream = self.lib, current_stream()
        _lib.require_cuda(means, quats, scales, opacities, sh, viewmats, Ks)
        self._mark("begin")
        C, N = viewmats.shape[0], means.shape[0]
        want_rgb = render_mode in ("RGB", "RGB+D", "RGB+ED")
        want_depth = render_mode in ("D", "ED", "RGB+D", "RGB+ED")
        n_color, append = (3 if want_rgb else 0), int(want_depth)
        D = n_color + append
        normalize = int(render_mode in ("ED", "RGB+ED"))
        comp = rasterize_mode == "antialiased"
        K = sh.shape[1] if (want_rgb and sh_degree is not None) else 0
        deg = -1 if (sh_degree is None or not want_rgb) else int(sh_degree)
        tile = 16
        tw, th = ops.tile_grid(width, height, tile)

        radii = self._get("radii", (C, N), torch.int32)
        means2d = self._get("means2d", (C, N, 2))
        depths = self._get("depths", (C, N))
        conics = self._get("conics", (C, N, 3))
        comps = self._get("comps", (C, N)) if comp else None
        colors = self._get("colors", (C, N, D))
        opac = self._get("opac", (C, N))
        tiles = self._get("tiles", (C, N), torch.int32)
        exact = self.exact_tile_lists and self.sort_impl == "two_level"
        # exact tile lists: the projection counts the tiles each Gaussian can reach with alpha >= 1/255, the intersection
        # stage enumerates exactly those (its sizes / capacities then refer to the exact lists)
        tiles_exact = self._get("tiles_exact", (C, N), torch.int32) if exact else None
        geom = self._get("geom", (C, N, 8))
        check(lib.qed_project_fwd(C, N, ptr(means), ptr(quats), ptr(scales), ptr(opacities), int(activations), ptr(sh) if want_rgb else None, K, deg,
                                  int(want_rgb and sh_degree is None and sh.dim() == 3), ptr(viewmats), ptr(Ks), width, height, eps2d, near_plane,
                                  far_plane, 0.0, int(comp), tile, n_color, append, ptr(radii), ptr(means2d), ptr(depths),
                                  ptr(conics), ptr(comps), ptr(colors), ptr(opac), ptr(tiles), ptr(tiles_exact), ptr(geom), stream), "qed_project_fwd")
        self._mark("project_fwd")
        CN = C * N
        # exact tile lists / deferred sizes: one more element (the end of the last range)
        offsets = self._get("offsets", (C * th * tw + 1,), torch.int32)
        if self.sort_impl == "two_level":
            pws_bytes = lib.qed_isect_prepare_workspace_bytes(CN)
            pws = self._get("prep_ws", (pws_bytes,), torch.uint8)
            check(lib.qed_isect_prepare(C, N, ptr(depths), ptr(tiles_exact if exact else tiles), ptr(pws), pws_bytes, ptr(self._counts), ptr(self._counts_host), stream),
                  "qed_isect_prepare")
            self._mark("isect_prepare")
            # the single host sync of the step (output sizes) waits on an EVENT behind the counts' copy, not on the
            # stream: work that does not depend on the counts is queued behind the event and keeps the GPU busy while
            # the host reads the counts and launches the rest (here: clearing the gradient record of the backward)
            self._counts_ready.record(torch.cuda.current_stream())
            if self._prezero:
                self._get("packed", (C * N, 12)).zero_()
            deferred = self.defer_sync and not _force_sync and self._cap_isects > 0 and CN > 0
            if deferred:
                n_vis, M = CN, self._cap_isects  # capacities; the real counts stay on the device until _resolve_counts()
            else:
                self._counts_ready.synchronize()
                n_vis, M = int(self._counts_host[0]), int(self._counts_host[1])
                self._cap_isects = max(self._cap_isects, M + M // 4 + 4096)
                self._mark("sync")
            cap = max(M, 1)
            ids = self._get("ids", (cap,), torch.int64)[:M]
            flat = self._get("flat", (cap,), torch.int32)[:M]
            fws_bytes = lib.qed_isect_fill_workspace_bytes(M)
            fws = self._get("fill_ws", (fws_bytes,), torch.uint8)
            check(lib.qed_isect_fill(C, N, n_vis, M, ptr(means2d), ptr(radii), ptr(depths), ptr(geom) if exact else None, width, height,
                                     tile, tw, th, ptr(pws), ptr(fws), fws_bytes, ptr(self._counts) if deferred else None,
                                     ptr(ids) if (M and self.want_isect_ids) else None, ptr(flat) if M else None, ptr(offsets),
                                     ptr(self._n_exact) if exact else None, stream), "qed_isect_fill")
            self._mark("isect_fill")
        else:
            deferred = False
            cum = self._get("cum", (CN,), torch.int64)
            ws_bytes = lib.qed_isect_scan_workspace_bytes(CN)
            ws = self._get("scan_ws", (ws_bytes,), torch.uint8)
            check(lib.qed_isect_scan(CN, ptr(tiles), ptr(cum), ptr(self._total), None, ptr(ws), ws_bytes, stream), "qed_isect_scan")
            M = int(self._total.item())  # the single host sync of the step
            self._mark("scan+sync")
            cap = max(M, 1)
            ids_u = self._get("ids_u", (cap,), torch.int64)[:M]
            flat_u = self._get("flat_u", (cap,), torch.int32)[:M]
            ids = self._get("ids", (cap,), torch.int64)[:M]
            flat = self._get("flat", (cap,), torch.int32)[:M]
            if M:
                check(lib.qed_isect_emit(C, N, ptr(means2d), ptr(radii), ptr(depths), ptr(cum), tile, tw, th, ptr(ids_u), ptr(flat_u),
                                         stream), "qed_isect_emit")
                self._mark("emit")
                end_bit = 32 + (tw * th).bit_length() + C.bit_length()
                if self.sort_impl == "cub":
                    sb = lib.qed_sort_pairs_cub_workspace_bytes(M)
                    sws = self._get("sort_ws", (sb,), torch.uint8)
                    check(lib.qed_sort_pairs_cub(M, ptr(ids_u), ptr(flat_u), ptr(ids), ptr(flat), end_bit, ptr(sws), sb, stream), "qed_sort_pairs_cub")
                else:
                    sb = lib.qed_sort_pairs_workspace_bytes(M)
                    sws = self._get("sort_ws", (sb,), torch.uint8)
                    check(lib.qed_sort_pairs(M, ptr(ids_u), ptr(flat_u), ptr(ids), ptr(flat), end_bit, ptr(sws), sb, stream), "qed_sort_pairs")
            self._mark("sort")
            check(lib.qed_tile_ranges(M, ptr(ids) if M else None, C, tw, th, ptr(offsets), stream), "qed_tile_ranges")
            self._mark("ranges")
        render = self._get("render", (C, height, width, D))
        alphas = self._get("alphas", (C, height, width, 1))
        last_ids = self._get("last_ids", (C, height, width), torch.int32)
        check(lib.qed_raster_fwd(C, N, M, D, ptr(geom), ptr(colors), ptr(backgrounds), width, height, tile, tw, th, ptr(offsets), int(exact or deferred),
                                 ptr(flat) if M else None, normalize, ptr(render), ptr(alphas), ptr(last_ids), stream), "qed_raster_fwd")
        self._mark("raster_fwd")
        self._fwd = dict(C=C, N=N, D=D, M=M, exact=exact, deferred=deferred, has_end=int(exact or deferred), n_visible=None if deferred else n_vis, activations=int(activations), K=K, deg=deg, n_color=n_color, append=append, normalize=normalize, comp=comp, tw=tw,
                         th=th, width=width, height=height, eps2d=eps2d, radii=radii, conics=conics, comps=comps, colors=colors,
                         geom=geom, offsets=offsets, flat=flat, render=render, alphas=alphas, last_ids=last_ids, backgrounds=backgrounds,
                         inputs=(means, quats, scales, opacities, sh, viewmats, Ks))
        if _resolve and not self._resolve_counts():
            # the lists did not fit the buffers: repeat with the sizes read from the device (buffers grow, never shrink)
            self.overflow_repeats += 1
            return self.forward(*self._call["args"], **self._call["kw"], _force_sync=True)
        return render, alphas

    def _resolve_counts(self) -> bool:
        """Deferred mode: read the counts of the last forward (the copy was queued right behind the intersection build, the
        device is busy with what was queued after it).  False = the real entry count exceeded the capacity (the device built
        an empty list): the caller repeats the pass."""
        f = self._fwd
        if not f.get("deferred"):
            return True
        self._counts_ready.synchronize()
        n_vis, M = int(self._counts_host[0]), int(self._counts_host[1])
        ok = M <= f["M"]
        self._cap_isects = max(self._cap_isects, M + M // 4 + 4096)
        if ok:
            # M stays the capacity the flat buffers were sliced with (an upper bound for the compositors, whose ranges end at
            # the device-side count); the real count is kept for reporting
            f["deferred"], f["n_visible"], f["n_isects_real"] = False, n_vis, M
        return ok

    # -- backward from explicit output gradients ------------------------------------------------
    @torch.no_grad()
    def backward(self, v_render: Tensor, v_alphas: Optional[Tensor], grad_out: Optional[Dict[str, Tensor]] = None,
                 n_chunks: int = 1, on_chunk=None, exchange=None, v_viewmats: Optional[Tensor] = None, _redo=None):
        """`grad_out`: optional preallocated {means,quats,scales,opacities,sh} (e.g. views into a flat
        all-reduce arena) that the projection backward writes straight into.

        `n_chunks` > 1 (single-camera calls only) launches the projection backward over `n_chunks` Gaussian
        ranges and calls `on_chunk(k, n0, n1)` after each launch, so a caller can start the all-reduce of a
        finished range while the next one is still being computed (view-sharded training).

        `exchange` (comm.ViewShardedGradients, world_size > 1): the gradients are SUMMED OVER ALL RANKS' views before this
        returns (in stream order): the projection backward stores its per-view colour gradients into every rank's exchange
        buffer, one all-reduce kernel sums the 11 non-SH floats per Gaussian and every rank rebuilds the SH coefficient
        gradient locally.  Returns views into the exchange's arena.

        `v_viewmats` ([C,4,4] float32, optional): receives the gradient with respect to the camera poses (overwritten; with
        `exchange`, this rank's views only).  Not with `n_chunks` > 1, nor with an exchange built without pose capacity
        (comm.ViewShardedGradients(num_cameras=...))."""
        lib, stream = self.lib, current_stream()
        if v_viewmats is not None and (n_chunks > 1 or not _pose_capable(exchange)):
            raise ValueError("pose gradients (v_viewmats) are not available with n_chunks > 1 or an exchange without pose capacity")

        def composite_backward(v_r, v_a):
            f = self._fwd
            C, N, D, M = f["C"], f["N"], f["D"], f["M"]
            packed = self._get("packed", (C * N, 12))
            if not self._prezeroed:
                packed.zero_()
            self._prezeroed = False
            self._mark("zero_grads")
            if M:
                check(lib.qed_raster_bwd(C, N, M, D, ptr(f["geom"]), ptr(f["colors"]), ptr(f["backgrounds"]), f["width"], f["height"], 16,
                                         f["tw"], f["th"], ptr(f["offsets"]), ptr(f["flat"]), f["normalize"], ptr(f["render"]),
                                         ptr(f["alphas"]), ptr(f["last_ids"]), ptr(v_r), ptr(v_a), ptr(packed), stream), "qed_raster_bwd")
            self._mark("raster_bwd")
            return packed

        packed = composite_backward(v_render, v_alphas)
        if not self._resolve_counts():
            # deferred sizes (step() only): the intersection lists did not fit; everything queued so far ran on an empty
            # list.  Repeat forward + loss with the sizes now known, then the compositor's backward.
            if _redo is None:
                raise RuntimeError("intersection capacity exceeded and no way to repeat the forward pass")
            v_render, v_alphas = _redo()
            packed = composite_backward(v_render, v_alphas)
        f = self._fwd
        C, N, D, M = f["C"], f["N"], f["D"], f["M"]
        means, quats, scales, opacities, sh, viewmats, Ks = f["inputs"]
        if exchange is not None:
            if not f["n_color"] or f["deg"] < 0:
                raise ValueError("the view-colour exchange needs SH colours (render_mode RGB / RGB+D / RGB+ED with sh_degree)")
            ws = None
            if v_viewmats is not None:
                ws_bytes = lib.qed_project_bwd_pose_workspace_bytes(C, N)
                ws = self._get("pose_ws", (max(ws_bytes, 16),), torch.uint8)
            exchange.project_bwd(lib, C, means, quats, scales, opacities, f["activations"], sh, f["K"], f["deg"], viewmats, Ks, f["width"], f["height"],
                                 f["eps2d"], f["comp"], f["append"], f["radii"], f["conics"], f["comps"], packed, stream, v_viewmats=v_viewmats, pose_ws=ws)
            self._mark("project_bwd")
            exchange.finish(lib, means, f["K"], f["deg"], stream)
            self._mark("grad_exchange")
            return exchange.views(), packed
        if grad_out is not None:
            v_means, v_quats, v_scales, v_opac = grad_out["means"], grad_out["quats"], grad_out["scales"], grad_out["opacities"]
            v_sh = grad_out["sh"] if f["n_color"] else None
        else:
            v_means = torch.empty_like(means)
            v_quats = torch.empty_like(quats)
            v_scales = torch.empty_like(scales)
            v_opac = torch.empty_like(opacities)
            v_sh = torch.empty_like(sh) if f["n_color"] else None
        if C != 1 or n_chunks <= 1 or N < 4 * n_chunks:
            bounds = [(0, N)]
        else:
            step_n = ((N + n_chunks - 1) // n_chunks + 3) // 4 * 4  # multiples of 4 keep every slice 16-byte aligned
            bounds = [(a, min(a + step_n, N)) for a in range(0, N, step_n)]
        has_sh = bool(f["n_color"])
        for k, (n0, n1) in enumerate(bounds):
            # C == 1 when chunked: flat index == n, so a range is just a pointer offset on every [N,...] / [1,N,...] array
            sl = slice(n0, n1)
            args = (C, n1 - n0, ptr(means[sl]), ptr(quats[sl]), ptr(scales[sl]), ptr(opacities[sl]), f["activations"],
                    ptr(sh[sl]) if has_sh else None, f["K"], f["deg"], 0, ptr(viewmats), ptr(Ks), f["width"], f["height"],
                    f["eps2d"], int(f["comp"]), f["n_color"], f["append"],
                    ptr(f["radii"][:, sl] if len(bounds) > 1 else f["radii"]),
                    ptr(f["conics"][:, sl] if len(bounds) > 1 else f["conics"]),
                    ptr((f["comps"][:, sl] if len(bounds) > 1 else f["comps"]) if f["comps"] is not None else None),
                    None, None, None, None, None, ptr(packed[n0:n1] if len(bounds) > 1 else packed),
                    ptr(v_means[sl]), ptr(v_quats[sl]), ptr(v_scales[sl]), ptr(v_opac[sl]), ptr(v_sh[sl]) if has_sh else None)
            if v_viewmats is None:
                check(lib.qed_project_bwd(*args, stream), "qed_project_bwd")
            else:  # one range (n_chunks > 1 is refused above)
                ws_bytes = lib.qed_project_bwd_pose_workspace_bytes(C, N)
                ws = self._get("pose_ws", (max(ws_bytes, 16),), torch.uint8)
                check(lib.qed_project_bwd_pose(*args, ptr(v_viewmats), ptr(ws), ws_bytes, stream), "qed_project_bwd_pose")
            if on_chunk is not None:
                on_chunk(k, n0, n1)
        self._mark("project_bwd")
        grads = dict(means=v_means, quats=v_quats, scales=v_scales, opacities=v_opac, sh=v_sh)
        return grads, packed

    # -- full step: render + qed-splatter loss + backward -----------------------------------------
    @torch.no_grad()
    def step(self, means, quats, scales, opacities, sh, viewmats, Ks, width: int, height: int, sh_degree: int,
             gt_rgb: Tensor, gt_depth: Tensor, background: Tensor, render_mode: str = "RGB+ED", rgb_weight: float = 0.8,
             depth_lambda: float = 0.2, grad_scale: float = 1.0, rasterize_mode: str = "classic",
             grad_out: Optional[Dict[str, Tensor]] = None, ssim_lambda: float = 0.0, n_chunks: int = 1, on_chunk=None,
             activations: int = 0, mask: Optional[Tensor] = None, exchange=None, depth_unit_scale: float = 0.001,
             pose_gradients: bool = False, bilateral_grid=None, gt_downscale: int = 1) -> StepOutput:
        """`render_mode` RGB+ED (north_star) or RGB+D (what qed_splatter/model.py:257 passes).
        loss = rgb_weight * L1 + ssim_lambda * (1 - SSIM) + depth_lambda * masked depth-L1 (splatfacto: 0.8 / 0.2 / 0.2).
        `mask` [C,H,W(,1)] float32 / uint8 / bool = `batch["mask"]` (model.py:93-97), see losses.depth_supervised_loss.
        The returned StepOutput aliases buffers this object reuses: the next step() overwrites loss / render / alphas /
        packed_grads / radii / v_viewmats in place -- clone() what must outlive the step.
        `pose_gradients=True`: StepOutput.v_viewmats [C,4,4] = d loss / d viewmats (camera optimisation); not with
        `n_chunks` > 1, and with `exchange` only when it was built with pose capacity (num_cameras > 0).
        `bilateral_grid=(grids, grid_ids, v_grid_rows)`: splatfacto's bilateral grid on every view before the RGB loss
        (qed_loss_fwd_bwd_bilagrid): grids [G,12,L,Y,X] float32, grid_ids [C] int32 on the device (validated by the caller),
        v_grid_rows [C,12,L,Y,X] overwritten with each view's grid gradient.  Only the loss stage changes, so it combines
        with `n_chunks` and `exchange`.
        `gt_downscale` d > 1 (splatfacto's resolution schedule): the camera (Ks, width, height) is the rescaled one and
        gt_rgb [C,H,W,3] / gt_depth / mask are at full resolution with H // d == height and W // d == width; they are
        box-downscaled into buffers of this object (data_side.downscale_ground_truth) before the projection is queued."""
        assert render_mode in ("RGB+D", "RGB+ED")
        if pose_gradients and (n_chunks > 1 or not _pose_capable(exchange)):
            raise ValueError("pose_gradients=True is not available with n_chunks > 1 or an exchange without pose capacity")
        lib, stream = self.lib, current_stream()
        # raw pointers cross the C-ABI: wrong device / dtype must raise here, not fault in the kernel
        _lib.require_cuda(means, gt_rgb, gt_depth, background, mask)
        _lib.require_dtype(gt_rgb, (torch.float32, torch.uint8), "gt_rgb")
        _lib.require_dtype(gt_depth, (torch.float32, torch.uint16, torch.int16), "gt_depth")  # raw uint16: scaled in-kernel by depth_unit_scale
        _lib.require_dtype(background, (torch.float32,), "background")
        _lib.require_dtype(mask, (torch.float32, torch.uint8, torch.bool), "mask")
        C_, HW_ = viewmats.shape[0], width * height
        if gt_downscale != 1:
            from .data_side import downscale_ground_truth, downscaled_size

            if gt_rgb.dim() != 4 or gt_rgb.shape[0] != C_:
                raise ValueError("gt_downscale: full-resolution gt_rgb [C,H,W,3] expected")
            C_, H_, W_, _ = gt_rgb.shape
            if downscaled_size(W_, H_, gt_downscale) != (width, height):
                raise ValueError(f"gt_downscale={gt_downscale}: {W_}x{H_} ground truth does not downscale to the {width}x{height} render")
            # queued ahead of the projection: the loss then reads float32 ground truth at render size
            gt_rgb, gt_depth, mask = downscale_ground_truth(gt_rgb, gt_depth, mask, gt_downscale, depth_unit_scale,
                                                            out=(self._get("gt_rgb_ds", (C_, height, width, 3)), self._get("gt_depth_ds", (C_, height, width, 1)),
                                                                 self._get("mask_ds", (C_, height, width, 1)) if mask is not None else None))
        if gt_rgb.numel() != C_ * HW_ * 3 or gt_depth.numel() != C_ * HW_ or background.numel() != 3 or (mask is not None and mask.numel() != C_ * HW_):
            raise ValueError("shapes: gt_rgb [C,H,W,3], gt_depth [C,H,W(,1)], background [3], mask [C,H,W(,1)]")
        gt_rgb, gt_depth, background = gt_rgb.contiguous(), gt_depth.contiguous(), background.contiguous()
        if mask is not None:
            mask = mask.contiguous()
            if mask.dtype == torch.bool:
                mask = mask.view(torch.uint8)
        C = viewmats.shape[0]
        if self._stats is None or self._stats.numel() < C * 8:
            self._stats = torch.zeros(C * 8, dtype=torch.float64, device=self.device)

        def forward_and_loss(force_sync: bool):
            self._prezero = self.sort_impl == "two_level"
            render, alphas = self.forward(means, quats, scales, opacities, sh, viewmats, Ks, width, height, sh_degree, render_mode,
                                          rasterize_mode, activations=activations, _resolve=False, _force_sync=force_sync)
            self._prezeroed, self._prezero = self._prezero, False
            v_render = self._get("v_render", (C, height, width, 4))
            v_alphas = self._get("v_alphas", (C, height, width, 1))
            if bilateral_grid is None:
                lws_bytes = lib.qed_loss_workspace_bytes(C, width, height, ssim_lambda)
                lws = self._get("loss_ws", (lws_bytes,), torch.uint8) if lws_bytes else None
                check(lib.qed_loss_fwd_bwd(C, width, height, ptr(render), ptr(alphas), ptr(gt_rgb), int(gt_rgb.dtype == torch.uint8), ptr(gt_depth), int(gt_depth.dtype != torch.float32),
                                           float(depth_unit_scale), ptr(mask), int(mask is not None and mask.dtype == torch.uint8), ptr(background), rgb_weight,
                                           depth_lambda, ssim_lambda, grad_scale, ptr(self._stats), ptr(self._loss), ptr(v_render), ptr(v_alphas),
                                           ptr(lws), lws_bytes, stream), "qed_loss_fwd_bwd")
            else:
                grids, ids, rows = bilateral_grid
                G, _, L, Y, X = grids.shape
                lws_bytes = lib.qed_loss_bilagrid_workspace_bytes(C, width, height, ssim_lambda)
                lws = self._get("loss_ws", (lws_bytes,), torch.uint8)
                check(lib.qed_loss_fwd_bwd_bilagrid(C, width, height, ptr(render), ptr(alphas), ptr(gt_rgb), int(gt_rgb.dtype == torch.uint8), ptr(gt_depth),
                                                    int(gt_depth.dtype != torch.float32), float(depth_unit_scale), ptr(mask),
                                                    int(mask is not None and mask.dtype == torch.uint8), ptr(background), rgb_weight, depth_lambda, ssim_lambda,
                                                    grad_scale, ptr(self._stats), ptr(self._loss), ptr(v_render), ptr(v_alphas), ptr(grids), ptr(ids), G, X,
                                                    Y, L, ptr(rows), ptr(lws), lws_bytes, stream), "qed_loss_fwd_bwd_bilagrid")
            self._mark("loss")
            return render, alphas, v_render, v_alphas

        def redo():
            self.overflow_repeats += 1
            return forward_and_loss(True)[2:]

        render, alphas, v_render, v_alphas = forward_and_loss(False)
        v_viewmats = self._get("v_viewmats", (C, 4, 4)) if pose_gradients else None
        grads, packed = self.backward(v_render, v_alphas, grad_out, n_chunks=n_chunks, on_chunk=on_chunk, exchange=exchange, v_viewmats=v_viewmats,
                                      _redo=redo)
        self._last_v = (v_render, v_alphas)
        f = self._fwd
        return StepOutput(loss=self._loss, grads=grads, packed_grads=packed, radii=f["radii"], render=f["render"], alphas=f["alphas"],
                          n_isects=f.get("n_isects_real", f["M"]), n_visible=f.get("n_visible"), v_viewmats=v_viewmats)

    # -- instrumentation (never inside a timed region) --------------------------------------------
    def n_isects_exact(self) -> int:
        """Entries of the exact tile lists of the last forward (device -> host read: not for timed regions);
        equals StepOutput.n_isects (gsplat's bounding-box count) when exact_tile_lists is off."""
        f = self._fwd
        return int(self._n_exact.item()) if (f.get("exact") and f["M"]) else int(f.get("n_isects_real", f["M"]))

    @property
    def launches_per_step(self) -> int:
        """Launches of THIS library's kernels in one step() (memsets and torch's own fill kernels not counted):
        project 1; intersections two_level: flag scan 1 (single launch; its last phase compacts) + Gaussian sort + gather scan 1 +
        emit boundaries 1 + emit 1 + tile sort + compose/ranges 1 (a radix sort is 1 histogram + 1 kernel per 8-bit
        pass when it fits 444 blocks of 4096 pairs, else 3 kernels per pass); own/cub: scan 3 + emit 1 + sort + ranges 1; composite fwd 1, loss 3 (+2 with SSIM),
        composite bwd 1, project bwd 1.  Cross-checked against the ncu launch list (profiles/r02_step_ncu_summary.txt)."""
        f = self._fwd
        tile_bits = (f["tw"] * f["th"]).bit_length()
        cam_bits = (f["C"] - 1).bit_length()

        def radix(capacity: int, bits: int, segmented: bool = False) -> int:
            passes = (bits + 7) // 8
            one_kernel_passes = (not segmented) and (capacity + 4095) // 4096 <= 444
            return 1 + passes if one_kernel_passes else 3 * passes

        if self.sort_impl == "two_level":
            isect = 1 + radix(f["C"] * f["N"], 32 + cam_bits) + 1 + 1 + 1 + radix(f["M"], tile_bits + cam_bits) + 1
        else:
            end_bit = 32 + tile_bits + f["C"].bit_length()
            isect = 3 + 1 + (radix(f["M"], end_bit) if self.sort_impl == "own" else 8) + 1
        return 1 + isect + 1 + 3 + 1 + 1

    @torch.no_grad()
    def count_pairs(self, which=("fwd", "bwd")) -> Dict[str, int]:
        """Re-run the compositing kernels of the last step() (or, which=("fwd",), of the last forward()) with the
        instrumented (STATS) variants and return the work counters used for the FP32 roofline."""
        lib, stream, f = self.lib, current_stream(), self._fwd
        out = {}
        if not f["M"]:
            return out
        names = ("entries_loaded", "entries_staged", "warp_candidates", "pairs_evaluated", "pairs_contributing", "reduction_groups")
        for which in which:
            cnt = torch.zeros(6, dtype=torch.int64, device=self.device)
            check(lib.qed_debug_set_raster_counters(ptr(cnt)), "set counters")
            try:
                if which == "fwd":
                    check(lib.qed_raster_fwd(f["C"], f["N"], f["M"], f["D"], ptr(f["geom"]), ptr(f["colors"]), ptr(f["backgrounds"]),
                                             f["width"], f["height"], 16, f["tw"], f["th"], ptr(f["offsets"]), int(f["has_end"]), ptr(f["flat"]),
                                             f["normalize"], ptr(f["render"]), ptr(f["alphas"]), ptr(f["last_ids"]), stream), "qed_raster_fwd(stats)")
                else:
                    v_render, v_alphas = self._last_v
                    scratch = torch.zeros(f["C"] * f["N"], 12, device=self.device)
                    check(lib.qed_raster_bwd(f["C"], f["N"], f["M"], f["D"], ptr(f["geom"]), ptr(f["colors"]), ptr(f["backgrounds"]),
                                             f["width"], f["height"], 16, f["tw"], f["th"], ptr(f["offsets"]), ptr(f["flat"]), f["normalize"],
                                             ptr(f["render"]), ptr(f["alphas"]), ptr(f["last_ids"]), ptr(v_render), ptr(v_alphas),
                                             ptr(scratch), stream), "qed_raster_bwd(stats)")
                torch.cuda.synchronize()
            finally:
                lib.qed_debug_set_raster_counters(None)
            for n, v in zip(names, cnt.tolist()):
                out[f"{which}_{n}"] = int(v)
        return out
