"""ctypes binding of the C-ABI library (`include/qed_splat.h`).

No torch types cross this boundary: tensors are passed as `data_ptr()`s plus extents, the stream as
`torch.cuda.current_stream().cuda_stream`.  There is NO fallback: if `libqedsplat.so` is missing or a
call fails, this raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint32, c_uint64, c_void_p
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("QED_SPLAT_LIB", _PKG / "libqedsplat.so"))

P = c_void_p  # every device pointer / stream
ABI_VERSION = 3  # QED_ABI_VERSION of include/qed_splat.h this binding was written against

# name -> (restype, argtypes); must match include/qed_splat.h exactly (tests/test_abi.py checks the names)
SIGNATURES = {
    "qed_abi_version": (c_int, []),
    "qed_error_string": (ctypes.c_char_p, [c_int]),
    "qed_project_fwd": (c_int, [c_int, c_int, P, P, P, P, c_int, P, c_int, c_int, c_int, P, P, c_int, c_int,
                                c_float, c_float, c_float, c_float, c_int, c_int, c_int, c_int,
                                P, P, P, P, P, P, P, P, P, P, P]),
    "qed_project_bwd": (c_int, [c_int, c_int, P, P, P, P, c_int, P, c_int, c_int, c_int, P, P, c_int, c_int,
                                c_float, c_int, c_int, c_int, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P]),
    "qed_project_bwd_pose_workspace_bytes": (c_size_t, [c_int, c_int]),
    "qed_project_bwd_pose": (c_int, [c_int, c_int, P, P, P, P, c_int, P, c_int, c_int, c_int, P, P, c_int, c_int,
                                     c_float, c_int, c_int, c_int, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P, c_size_t, P]),
    "qed_pack_geom": (c_int, [c_int, P, P, P, P, P, P]),
    "qed_isect_count": (c_int, [c_int, c_int, P, P, c_int, c_int, c_int, P, P]),
    "qed_isect_scan_workspace_bytes": (c_size_t, [c_int64]),
    "qed_isect_scan": (c_int, [c_int64, P, P, P, P, P, c_size_t, P]),
    "qed_isect_emit": (c_int, [c_int, c_int, P, P, P, P, c_int, c_int, c_int, P, P, P]),
    "qed_sort_pairs_workspace_bytes": (c_size_t, [c_int64]),
    "qed_sort_pairs": (c_int, [c_int64, P, P, P, P, c_int, P, c_size_t, P]),
    "qed_sort_pairs_cub_workspace_bytes": (c_size_t, [c_int64]),
    "qed_sort_pairs_cub": (c_int, [c_int64, P, P, P, P, c_int, P, c_size_t, P]),
    "qed_isect_prepare_workspace_bytes": (c_size_t, [c_int64]),
    "qed_isect_prepare": (c_int, [c_int, c_int, P, P, P, c_size_t, P, P, P]),
    "qed_isect_fill_workspace_bytes": (c_size_t, [c_int64]),
    "qed_isect_fill": (c_int, [c_int, c_int, c_int64, c_int64, P, P, P, P, c_int, c_int, c_int, c_int, c_int, P, P, c_size_t, P, P, P, P, P, P]),
    "qed_tile_ranges": (c_int, [c_int64, P, c_int, c_int, c_int, P, P]),
    "qed_raster_fwd": (c_int, [c_int, c_int, c_int64, c_int, P, P, P, c_int, c_int, c_int, c_int, c_int, P, c_int, P,
                               c_int, P, P, P, P]),
    "qed_raster_bwd": (c_int, [c_int, c_int, c_int64, c_int, P, P, P, c_int, c_int, c_int, c_int, c_int, P, P,
                               c_int, P, P, P, P, P, P, P]),
    "qed_unpack_grads": (c_int, [c_int, c_int, P, P, P, P, P, P, P]),
    "qed_loss_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_float]),
    "qed_loss_fwd_bwd": (c_int, [c_int, c_int, c_int, P, P, P, c_int, P, c_int, c_double, P, c_int, P, c_float, c_float, c_float, c_float, P, P, P, P, P, c_size_t, P]),
    "qed_loss_bilagrid_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_float]),
    "qed_loss_fwd_bwd_bilagrid": (c_int, [c_int, c_int, c_int, P, P, P, c_int, P, c_int, c_double, P, c_int, P, c_float, c_float, c_float, c_float,
                                          P, P, P, P, P, P, c_int, c_int, c_int, c_int, P, P, c_size_t, P]),
    "qed_downscale_ground_truth": (c_int, [c_int, c_int, c_int, c_int, P, c_int, P, c_int, c_double, P, c_int, P, P, P, P]),
    "qed_bilagrid_tv": (c_int, [c_int, c_int, c_int, c_int, P, c_float, P, P, P, P]),
    "qed_bilagrid_accumulate": (c_int, [c_int, P, P, c_int, c_int, c_int, c_int, P, P]),
    "qed_adam_arena": (c_int, [c_int64, P, P, P, P, c_int, P, P, P, P, P, c_double, c_double, c_double, c_int, P]),
    "qed_strategy_update": (c_int, [c_int, c_int, P, c_int, P, c_int, c_int, c_int, P, P, P, P]),
    "qed_project_bwd_exchange": (c_int, [c_int, c_int, P, P, P, P, c_int, P, c_int, c_int, P, P, c_int, c_int, c_float, c_int, c_int, P, P, P, P,
                                         P, P, P, P, P, P, c_int, c_int, c_int, c_float, P]),
    "qed_project_bwd_exchange_pose": (c_int, [c_int, c_int, P, P, P, P, c_int, P, c_int, c_int, P, P, c_int, c_int, c_float, c_int, c_int, P, P,
                                              P, P, P, P, P, P, P, P, c_int, c_int, c_int, c_float, P, P, c_size_t, P]),
    "qed_sh_grad_from_view_colors": (c_int, [c_int, c_int, c_int, c_int, P, P, c_float, P, P]),
    "qed_comm_flag_words": (c_int, []),
    "qed_comm_barrier": (c_int, [P, c_int, c_int, ctypes.c_uint32, P]),
    "qed_comm_allreduce_f32": (c_int, [P, P, P, c_int, c_int, c_int64, c_int64, ctypes.c_uint32, c_int, P]),
    "qed_arena_gather": (c_int, [c_int64, P, P, P, P, P, P, P, P, P, P, P, P, P, P]),
    "qed_mcmc_workspace_bytes": (c_size_t, [c_int64]),
    "qed_mcmc_census": (c_int, [c_int64, P, c_float, P, P, P, c_size_t, P]),
    "qed_mcmc_sample": (c_int, [c_int64, P, c_float, c_int, c_int64, c_uint64, c_uint32, c_uint32, P, P, P, P, c_size_t, P]),
    "qed_mcmc_relocate": (c_int, [c_int64, P, c_float, c_int, c_int64, P, P, P, P, P, P, P]),
    "qed_mcmc_noise": (c_int, [c_int64, P, P, c_float, c_uint64, c_uint32, P]),
    "qed_mcmc_reg_workspace_bytes": (c_size_t, []),
    "qed_mcmc_reg": (c_int, [c_int64, P, P, c_float, c_float, P, P, P, c_size_t, P]),
    "qed_viewmat_from_c2w": (c_int, [c_int, c_int, P, P, P]),
    "qed_viewmat_from_c2w_bwd": (c_int, [c_int, c_int, P, P, P, P]),
    "qed_camera_opt_apply": (c_int, [c_int, c_int, c_int, P, P, P, P, P]),
    "qed_camera_opt_bwd": (c_int, [c_int, c_int, c_int, P, P, P, P, P, P]),
    "qed_camera_opt_reg": (c_int, [c_int, P, c_float, c_float, P, P, P]),
    "qed_backproject_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "qed_backproject_depth": (c_int, [c_int, c_int, P, c_int, c_double, c_float, c_int, P, P, P, P, P, c_size_t, P]),
    "qed_voxel_downsample_workspace_bytes": (c_size_t, [c_int64]),
    "qed_voxel_downsample": (c_int, [c_int64, P, P, c_float, P, P, P, c_size_t, P]),
}
# test hooks, not part of the reference-facing surface
DEBUG_SIGNATURES = {
    "qed_debug_set_raster_cull": (c_int, [c_int]),
    "qed_debug_set_raster_counters": (c_int, [P]),
    "qed_debug_set_raster_px": (c_int, [c_int, c_int]),
    "qed_debug_set_raster_packed": (c_int, [c_int]),
    "qed_debug_set_raster_bwd_minb": (c_int, [c_int]),
    "qed_debug_set_raster_fwd_minb": (c_int, [c_int]),
    "qed_debug_set_radix_onesweep": (c_int, [c_int]),
    "qed_debug_set_flat_scan": (c_int, [c_int]),
    "qed_debug_set_radix_small_tiles": (c_int, [c_int]),
    "qed_debug_set_project_bwd_one": (c_int, [c_int]),
    "qed_debug_set_project_fwd_one": (c_int, [c_int]),
}


class QedLibraryError(RuntimeError):
    pass


_lib = None


def load() -> ctypes.CDLL:
    """Load the library (once).  Raises QedLibraryError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise QedLibraryError(
            f"{LIB_PATH} not found: the sm_100a CUDA library has not been built "
            f"(run `python -m qed_splatter_b200.build`).  There is no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in {**SIGNATURES, **DEBUG_SIGNATURES}.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise QedLibraryError(f"{LIB_PATH} does not export {name}; rebuild it") from e
        fn.restype = res
        fn.argtypes = args
    if lib.qed_abi_version() != ABI_VERSION:
        raise QedLibraryError(f"ABI version mismatch: library {lib.qed_abi_version()} != binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().qed_error_string(code).decode()
        raise RuntimeError(f"{what} failed with code {code}: {msg}")


def ptr(t) -> c_void_p:
    """Device pointer of a contiguous tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), "C-ABI takes contiguous tensors"
    return c_void_p(t.data_ptr())


def current_stream() -> c_void_p:
    """Raw handle of torch's current stream on the current device.  (torch.cuda.current_stream() builds a Stream
    object and costs ~20 us per call -- seven calls per step were 8 % of the host side of a 1080p step.)"""
    import torch

    try:
        return c_void_p(torch._C._cuda_getCurrentRawStream(torch.cuda.current_device()))
    except AttributeError:  # private binding moved: fall back to the public, slower path
        return c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors) -> None:
    """Every tensor handed to the C-ABI must live on ONE CUDA device, and that device must be the current one: the
    kernels are launched on `torch.cuda.current_stream()` of the current device (gsplat guards with the tensors'
    device; here a mismatch raises instead of launching on the wrong device).  None entries are skipped."""
    import torch

    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                "qed_splatter_b200 runs on CUDA (sm_100a) only: got a CPU tensor.  "
                "There is no CPU fallback; the CPU oracle lives in oracle/ and is test infrastructure.")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"qed_splatter_b200: tensors on different devices ({dev} and {t.device})")
    if dev is not None and dev.index != torch.cuda.current_device():
        raise RuntimeError(
            f"qed_splatter_b200: tensors live on {dev} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
            f"call torch.cuda.set_device({dev.index}) (or wrap the call in `with torch.cuda.device({dev.index})`)")


def require_dtype(t, dtypes, what: str) -> None:
    if t is not None and t.dtype not in dtypes:
        raise TypeError(f"{what}: expected {' or '.join(str(d) for d in dtypes)}, got {t.dtype}")
