"""Gradient reduction of the view-sharded step over NVLink 5 / NVSwitch, without NCCL on the data path.

`SymmetricArena` owns a float32 buffer in symmetric memory (torch.distributed._symmetric_memory is used for the
allocation and the address exchange only: the same allocation on every rank, mapped into every peer and -- with
NVSwitch multicast -- into one multicast address range) plus a small symmetric flag block.  `all_reduce_()` launches
ONE kernel of this library (`qed_comm_allreduce_f32`, csrc/comm.cu): a two-shot all-reduce whose sums are formed inside
the switch (multimem.ld_reduce / multimem.st), ordered against the other ranks by epoch flags.  The trainer and
bench.py keep their gradient arena in such a buffer, so the projection backward writes straight into memory the
reduction reads -- no staging copy, no host synchronisation.

SURVEY.md section 8e / section 5 "Distributed comm backend"; the reference has no collective (model.py:211: one camera per step).
"""
from __future__ import annotations

import ctypes
from typing import Optional

import torch

from . import _lib


class SymmetricArena:
    def __init__(self, n_floats: int, device, group=None, blocks: int = 32, force_peer_path: bool = False):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem

        self.lib = _lib.load()
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        self.device = torch.device(device)
        n_floats = (int(n_floats) + 3) // 4 * 4
        self.buf = symm_mem.empty(n_floats, dtype=torch.float32, device=self.device)
        self.buf.zero_()
        self.hdl = symm_mem.rendezvous(self.buf, self.group)
        self.flags = symm_mem.empty(self.lib.qed_comm_flag_words(), dtype=torch.int32, device=self.device)
        self.flags.zero_()
        self.fhdl = symm_mem.rendezvous(self.flags, self.group)
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)  # every rank's flags are zero before anybody raises one
        mc = int(self.hdl.multicast_ptr) if (self.hdl.has_multicast_support and not force_peer_path) else 0
        self.multicast_ptr = mc
        PtrArray = ctypes.c_void_p * self.world
        self._bases = PtrArray(*[int(p) for p in self.hdl.buffer_ptrs])
        self._flags = PtrArray(*[int(p) for p in self.fhdl.buffer_ptrs])
        self.epoch = 1
        self.blocks = blocks
        # two GPUs: the peer path moves S bytes per direction, the in-switch reduction 1.5 S (measured on 2 B200, 236 MB:
        # 0.39 ms with 256 blocks vs 0.59 ms); from 4 GPUs on the switch wins (8 B200: 0.54 ms vs 0.74 ms)
        self.reduce_in_switch = bool(mc) and self.world > 2

    @property
    def path(self) -> str:
        if self.reduce_in_switch:
            return "nvls-multimem"
        return "peer-load-store" + (" (multicast stores available)" if self.multicast_ptr else "")

    def all_reduce_(self, begin: int = 0, end: Optional[int] = None, blocks: Optional[int] = None) -> None:
        """Sum elements [begin, end) of the buffer over the ranks, in place, on the current stream.  Collective: every
        rank calls it with the same range in the same order."""
        end = self.buf.numel() if end is None else end
        if blocks is None:
            blocks = self.blocks if self.reduce_in_switch else 256
        _lib.check(self.lib.qed_comm_allreduce_f32(ctypes.c_void_p(self.multicast_ptr) if self.reduce_in_switch else None, self._bases, self._flags,
                                                   self.rank, self.world, int(begin), int(end), self.epoch, int(blocks),
                                                   _lib.current_stream()), "qed_comm_allreduce_f32")
        self.epoch += 2

    def barrier(self) -> None:
        """Everything every rank enqueued before this call (on its current stream) is complete and visible to all ranks
        for work enqueued after it.  One tiny kernel; collective."""
        _lib.check(self.lib.qed_comm_barrier(self._flags, self.rank, self.world, self.epoch, _lib.current_stream()), "qed_comm_barrier")
        self.epoch += 2


class ViewShardedGradients:
    """Everything the view-sharded step needs to end with the SUMMED gradient arena on every rank
    (include/qed_splat.h, "View-colour exchange"):

      * `arena`  : the flat gradient arena (trainer.GaussianArena layout for N Gaussians) in symmetric memory;
        `views()` are the [N,...] gradient tensors the projection backward writes into;
      * two exchange buffers (alternating by step) for the per-view colour gradients;
      * `project_bwd(...)` : the projection backward of the fused path with the exchange stores fused in;
      * `finish(...)`      : one all-reduce kernel over the 11 non-SH floats per Gaussian + the local rebuild of the SH
        coefficient gradient from all views.  After it the arena holds the sum over all ranks' views, bit-identical on
        every rank.
      * with `num_cameras` > 0 (camera_opt.CameraPoseOptimizer): `project_bwd` also returns the pose gradient of the rank's
        views, and `pose` is a small SymmetricArena for the [num_cameras, 6] table gradient, summed over the ranks by its
        `all_reduce_()`.
      * with `bilagrid_row` > 0 (bilateral_grid.BilateralGridOptimizer, one grid = `bilagrid_row` floats): `bilagrid`, a
        SymmetricArena of one grid-gradient row per view of the whole batch followed by the views' grid ids (as exact
        floats).  Each rank writes its own slots, leaves the others zero, and `bilagrid.all_reduce_()` makes every rank hold
        all rows and ids, bit-identical, without all-reducing the dense [num_grids, row] gradient.

    No NCCL call, no host synchronisation; collective: every rank makes the same calls in the same order."""

    def __init__(self, N: int, views_per_rank: int, device, group=None, force_peer_path: bool = False, headroom: float = 0.0,
                 num_cameras: int = 0, bilagrid_row: int = 0):
        """`headroom`: allocate for N * (1 + headroom) Gaussians so that `resize()` after a densification step usually
        needs no new symmetric allocation (a collective).  `num_cameras` > 0: pose-gradient capacity for a camera table of
        that many rows."""
        from .trainer import GaussianArena

        self.views_per_rank = int(views_per_rank)
        self.capacity = int(N * (1.0 + headroom)) + 4
        _, total = GaussianArena.layout(self.capacity)
        self.arena = SymmetricArena(total, device, group, force_peer_path=force_peer_path)
        self.rank, self.world = self.arena.rank, self.arena.world
        self.slots = self.world * self.views_per_rank
        n_xch = (self.slots * self.capacity + self.slots) * 4
        self.xch = [SymmetricArena(n_xch, device, group, force_peer_path=force_peer_path) for _ in range(2)]
        self.num_cameras = int(num_cameras)
        self.pose = SymmetricArena(self.num_cameras * 6, device, group, force_peer_path=force_peer_path) if self.num_cameras > 0 else None
        n_bg = self.slots * (int(bilagrid_row) + 1)
        self.bilagrid = SymmetricArena(n_bg, device, group, force_peer_path=force_peer_path) if bilagrid_row > 0 else None
        self.step = 0
        self._side = torch.cuda.Stream(device=self.arena.device)
        self._fork, self._join = torch.cuda.Event(), torch.cuda.Event()
        self.resize(N)

    def resize(self, N: int) -> bool:
        """Use the buffers for N Gaussians (N <= capacity; same N on every rank).  False = does not fit: build a new object."""
        from .trainer import GaussianArena

        if N > self.capacity:
            return False
        if getattr(self, "N", None) not in (None, int(N)):
            self.arena.buf.zero_()  # the group boundaries move: padding floats between the groups must read as zero gradients
        self.N = int(N)
        self.offsets, self.total = GaussianArena.layout(self.N)
        return True

    @property
    def grad(self) -> torch.Tensor:
        return self.arena.buf[:self.total]

    def views(self):
        from .trainer import GROUP_SHAPES

        return {g: self.arena.buf[a:b].view(self.N, *GROUP_SHAPES[g]) for g, (a, b) in self.offsets.items()}

    def _tag(self) -> float:
        return float(self.step % 8_000_000 + 1)  # exactly representable, never 0 (the buffers start zeroed)

    def project_bwd(self, lib, C, means, quats, scales, opacities, activations, sh, K, deg, viewmats, Ks, width, height, eps2d, comp, append,
                    radii, conics, comps, packed, stream, v_viewmats=None, pose_ws=None) -> None:
        """`v_viewmats` [C,4,4] (pose capacity only): also the pose gradient of this rank's views, with `pose_ws` of
        qed_project_bwd_pose_workspace_bytes(C, N) bytes."""
        assert C == self.views_per_rank and means.shape[0] == self.N
        x = self.xch[self.step & 1]
        g = self.views()
        ptr = _lib.ptr
        args = (C, self.N, ptr(means), ptr(quats), ptr(scales), ptr(opacities), int(activations), ptr(sh), K, deg, ptr(viewmats), ptr(Ks), width, height,
                eps2d, int(comp), int(append), ptr(radii), ptr(conics), ptr(comps), ptr(packed), ptr(g["means"]), ptr(g["quats"]), ptr(g["scales"]),
                ptr(g["opacities"]), ctypes.c_void_p(x.multicast_ptr) if x.multicast_ptr else None, x._bases, self.world, self.rank * C, self.slots,
                self._tag())
        if v_viewmats is None:
            _lib.check(lib.qed_project_bwd_exchange(*args, stream), "qed_project_bwd_exchange")
        else:
            assert self.num_cameras > 0
            _lib.check(lib.qed_project_bwd_exchange_pose(*args, ptr(v_viewmats), ptr(pose_ws), pose_ws.numel(), stream), "qed_project_bwd_exchange_pose")

    def finish(self, lib, means, K: int, deg: int, stream) -> None:
        x = self.xch[self.step & 1]
        sh0 = self.offsets["sh"][0]
        main = torch.cuda.current_stream()
        self.arena.barrier()  # every rank's exchange stores (and small gradients) have landed
        # the all-reduce is NVLink-bound and needs few SMs, the SH rebuild is HBM-bound and local: run them side by side
        self._fork.record(main)
        self._side.wait_event(self._fork)
        _lib.check(lib.qed_sh_grad_from_view_colors(self.slots, self.N, K, deg, _lib.ptr(means), _lib.ptr(x.buf), self._tag(),
                                                    _lib.ptr(self.arena.buf[sh0:self.total]), ctypes.c_void_p(self._side.cuda_stream)),
                   "qed_sh_grad_from_view_colors")
        self._join.record(self._side)
        self.arena.all_reduce_(0, sh0)  # means | quats | scales | opacities (+ padding, zero)
        main.wait_event(self._join)
        self.step += 1
