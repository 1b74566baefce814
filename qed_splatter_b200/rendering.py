"""`rasterization` — the drop-in for `gsplat.rendering.rasterization` on the qed-splatter hot path.

The reference calls it at `/root/reference/qed_splatter/model.py:267-288` and uses the result at
`:289-306` (`info["means2d"].retain_grad()`, `info["radii"][0]`, `render[..., :3]`, `render[..., 3:4]`,
`alpha`).  Same keyword names, same return triple, same `info` keys as gsplat 1.4.0.  Arguments that
the reference never passes away from their defaults and that would need another code path
(`packed=True`, `sparse_grad=True`, `covars`, non-pinhole cameras, `distributed=True`) raise
NotImplementedError instead of silently doing something else.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from . import ops

RENDER_MODES = ("RGB", "D", "ED", "RGB+D", "RGB+ED")


class _Pending:
    """Placeholder of an `info` entry that is computed on first access."""


class LazyInfo(dict):
    """gsplat's `info` dict.  The compositor runs on EXACT tile lists (DESIGN.md section 5), so gsplat's own
    bounding-box lists -- `isect_ids`, `flatten_ids`, `isect_offsets`, which neither qed_splatter/model.py nor
    gsplat's strategies read -- are built, bit for bit, the first time one of them is looked up."""

    LAZY = ("isect_ids", "flatten_ids", "isect_offsets")

    def __init__(self, eager: Dict, build_lists):
        super().__init__(eager)
        self._build_lists = build_lists
        for k in self.LAZY:
            dict.__setitem__(self, k, _Pending)

    def _resolve(self) -> None:
        if self._build_lists is not None:
            build, self._build_lists = self._build_lists, None
            for k, v in zip(self.LAZY, build()):
                if dict.__getitem__(self, k) is _Pending:
                    dict.__setitem__(self, k, v)

    def __getitem__(self, key):
        v = dict.__getitem__(self, key)
        if v is _Pending:
            self._resolve()
            v = dict.__getitem__(self, key)
        return v

    def get(self, key, default=None):
        return self[key] if key in self else default

    def __iter__(self):  # (also keeps dict(info) / {**info} off CPython's raw-storage fast path)
        return iter(list(dict.keys(self)))

    def values(self):
        self._resolve()
        return dict.values(self)

    def items(self):
        self._resolve()
        return dict.items(self)

    def copy(self):
        self._resolve()
        return dict(dict.items(self))


def rasterization(
    means: Tensor,  # [N,3]
    quats: Tensor,  # [N,4] wxyz
    scales: Tensor,  # [N,3]
    opacities: Tensor,  # [N]
    colors: Tensor,  # [N,K,3] SH coefficients (sh_degree given) or [N,3] / [C,N,3] colours
    viewmats: Tensor,  # [C,4,4]
    Ks: Tensor,  # [C,3,3]
    width: int,
    height: int,
    near_plane: float = 0.01,
    far_plane: float = 1e10,
    radius_clip: float = 0.0,
    eps2d: float = 0.3,
    sh_degree: Optional[int] = None,
    packed: bool = False,
    tile_size: int = 16,
    backgrounds: Optional[Tensor] = None,
    render_mode: str = "RGB",
    sparse_grad: bool = False,
    absgrad: bool = False,
    rasterize_mode: str = "classic",
    channel_chunk: int = 32,
    distributed: bool = False,
    camera_model: str = "pinhole",
    covars: Optional[Tensor] = None,
    pose_gradients: bool = False,
) -> Tuple[Tensor, Tensor, Dict]:
    """-> (render_colors[C,H,W,D], render_alphas[C,H,W,1], info).

    `pose_gradients=True`: `viewmats` may require grad and receives d loss / d viewmats (gsplat's v_viewmats, what
    splatfacto's camera optimizer trains the poses with; row 3 is zero).  Bind it for the reference model with
    `functools.partial(rasterization, pose_gradients=True)` (INTEGRATION.md section 2b).  Off by default: a viewmat that
    requires grad then raises, as before."""
    if render_mode not in RENDER_MODES:
        raise ValueError(f"render_mode must be one of {RENDER_MODES}, got {render_mode!r}")
    if rasterize_mode not in ("classic", "antialiased"):
        raise ValueError(f"rasterize_mode must be 'classic' or 'antialiased', got {rasterize_mode!r}")
    if packed or sparse_grad or distributed or covars is not None or camera_model != "pinhole":
        raise NotImplementedError(
            "packed / sparse_grad / distributed / covars / non-pinhole cameras are not reachable from "
            "qed_splatter/model.py:267-288 and are out of scope for this path")
    if tile_size != 16:
        raise NotImplementedError("tile_size is 16 on this path (qed_splatter/model.py:243)")
    if torch.is_grad_enabled() and Ks.requires_grad:
        raise NotImplementedError("gradients with respect to Ks (intrinsics) are not implemented on this path: pass Ks.detach()")
    if torch.is_grad_enabled() and viewmats.requires_grad and not pose_gradients:
        # With splatfacto's camera_optimizer mode "off" (the default, and what qed_splatter/config.py keeps) the viewmat
        # built at model.py:212,246 carries no gradient.  A viewmat that does is refused unless pose gradients were asked
        # for, so that a camera optimizer never trains silently with zero pose gradients.
        raise NotImplementedError(
            "viewmats requires grad (camera optimisation): pass pose_gradients=True to compute v_viewmats, "
            "or pass viewmats.detach()")
    N = means.shape[0]
    C = viewmats.shape[0]
    assert means.shape == (N, 3), means.shape
    assert quats.shape == (N, 4), quats.shape
    assert scales.shape == (N, 3), scales.shape
    assert opacities.shape == (N,), opacities.shape
    assert viewmats.shape == (C, 4, 4), viewmats.shape
    assert Ks.shape == (C, 3, 3), Ks.shape
    if sh_degree is None:
        assert (colors.dim() == 2 and colors.shape == (N, 3)) or (colors.dim() == 3 and colors.shape == (C, N, 3)), colors.shape
    else:
        assert colors.dim() == 3 and colors.shape[0] == N and colors.shape[2] == 3, colors.shape
        assert (sh_degree + 1) ** 2 <= colors.shape[1], colors.shape

    want_rgb = render_mode in ("RGB", "RGB+D", "RGB+ED")
    want_depth = render_mode in ("D", "ED", "RGB+D", "RGB+ED")
    normalize = render_mode in ("ED", "RGB+ED")

    radii, means2d, depths, conics, comps, cols, opac, tiles_per_gauss, geom, tiles_exact = ops.project_gaussians(
        means, quats, scales, opacities, colors if want_rgb else None, viewmats, Ks, width, height, eps2d=eps2d,
        near_plane=near_plane, far_plane=far_plane, radius_clip=radius_clip,
        calc_compensations=(rasterize_mode == "antialiased"), sh_degree=sh_degree, n_color=3 if want_rgb else 0,
        append_depth=want_depth, tile_size=tile_size)

    tile_width, tile_height = ops.tile_grid(width, height, tile_size)
    # the compositor's lists (exact: about half of gsplat's entries, no pixel changes); gsplat's own lists are built
    # on demand by LazyInfo from the same projection outputs
    # (sizes of the lists live on the device: from the second call with these shapes on they are read only after the
    # compositor has been queued -- `resolve` -- so the device does not idle on the host)
    flatten_ids, isect_offsets, _, resolve = ops.isect_tiles_exact(means2d, radii, depths, geom, width, height, tile_size, tile_width,
                                                                   tile_height, tiles_exact, defer=True)

    def gsplat_lists(m=means2d.detach(), r=radii, d=depths.detach(), t=tiles_per_gauss):
        return ops.isect_tiles(m, r, d, tile_size, tile_width, tile_height, tiles_per_gauss=t, return_offsets=True)[1:]

    if backgrounds is not None:
        if want_rgb and want_depth:  # gsplat: the depth channel gets no background
            backgrounds = torch.cat([backgrounds, torch.zeros(C, 1, device=backgrounds.device, dtype=backgrounds.dtype)], dim=-1)
        elif not want_rgb:  # "D" / "ED": gsplat replaces the colour background by zeros(C, 1)
            backgrounds = torch.zeros(C, 1, device=backgrounds.device, dtype=backgrounds.dtype)
        n_channels = (3 if want_rgb else 0) + int(want_depth)
        if backgrounds.shape != (C, n_channels):
            raise ValueError(f"backgrounds must be [C, 3] = [{C}, 3], got {tuple(backgrounds.shape)}")

    render_colors, render_alphas = ops.rasterize_to_pixels(
        means2d, conics, cols, opac, width, height, tile_size, isect_offsets, flatten_ids, backgrounds=backgrounds,
        absgrad=absgrad, geom=geom, normalize_last=normalize)
    if resolve is not None and not resolve():
        # the lists did not fit the buffers sized from earlier calls (the device built empty ones): rebuild with the sizes
        # now known and composite again (rare: first frames of a new viewpoint / after densification)
        flatten_ids, isect_offsets, _, _ = ops.isect_tiles_exact(means2d, radii, depths, geom, width, height, tile_size, tile_width,
                                                                 tile_height, tiles_exact, defer=False)
        render_colors, render_alphas = ops.rasterize_to_pixels(
            means2d, conics, cols, opac, width, height, tile_size, isect_offsets, flatten_ids, backgrounds=backgrounds,
            absgrad=absgrad, geom=geom, normalize_last=normalize)

    info = LazyInfo({
        "camera_ids": None,
        "gaussian_ids": None,
        "radii": radii,
        "means2d": means2d,
        "depths": depths,
        "conics": conics,
        "opacities": opac,
        "tile_width": tile_width,
        "tile_height": tile_height,
        "tiles_per_gauss": tiles_per_gauss,
        "width": width,
        "height": height,
        "tile_size": tile_size,
        "n_cameras": C,
    }, gsplat_lists)
    return render_colors, render_alphas, info
