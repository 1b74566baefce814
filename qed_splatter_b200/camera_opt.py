"""Splatfacto's camera pose optimizer, mode SO3xR3 (nerfstudio `CameraOptimizer`, applied at qed_splatter/model.py:212/246).

A table `pose_adjustment[num_cameras, 6]` (zero at init; columns [:3] translation, [3:] rotation log) corrects the
training poses, e.g. robot odometry drift:

    theta^2 = max(|omega|^2, 1e-4),  R = I + (sin theta / theta) [omega]x + ((1 - cos theta) / theta^2) [omega]x^2
    c2w' = c2w[:3,:4] @ [[R, t], [0, 1]]   (SO3 x R3: the translation is not rotated)
    viewmat = get_viewmat(c2w')

Loss term (splatfacto's get_loss_dict while training, weight 1, once per step):
    trans_weight * mean_rows |t| + rot_weight * mean_rows |omega|   over all num_cameras rows.
Optimizer: Adam (torch semantics, dense: rows without a view this step still move by momentum) with an exponential
decay schedule after a sine warm-up from 0.  Evaluation uses the unadjusted pose.

`backend="cuda"`: the kernels of csrc/camera.cu and `qed_adam_arena`.  `backend="torch"`: the same arithmetic in torch,
for the CPU tests of the trainer's host logic.
"""
from __future__ import annotations

import math
import torch
from torch import Tensor

CAMERA_OPTIMIZER_MODES = ("off", "SO3xR3")


def exp_map_so3xr3(adj: Tensor) -> Tensor:
    """[n,6] -> [n,3,4] {R | t} (nerfstudio exp_map_SO3xR3), in the dtype of `adj`."""
    w = adj[:, 3:]
    theta = torch.clamp((w * w).sum(1), min=1e-4).sqrt()
    fac1 = torch.sin(theta) / theta
    fac2 = (1.0 - torch.cos(theta)) / (theta * theta)
    z = torch.zeros_like(w[:, 0])
    K = torch.stack([z, -w[:, 2], w[:, 1], w[:, 2], z, -w[:, 0], -w[:, 1], w[:, 0], z], dim=1).view(-1, 3, 3)
    eye = torch.eye(3, dtype=adj.dtype, device=adj.device)[None]
    R = eye + fac1[:, None, None] * K + fac2[:, None, None] * torch.bmm(K, K)
    return torch.cat([R, adj[:, :3, None]], dim=2)


def viewmats_torch(c2w: Tensor, camera_ids: Tensor, adj: Tensor) -> Tensor:
    """The apply step in torch: exp map -> c2w[:3,:4] @ [[R, t], [0, 1]] -> get_viewmat (model.py:22-38)."""
    T = exp_map_so3xr3(adj[camera_ids])
    Rc, tc = c2w[:, :3, :3], c2w[:, :3, 3:]
    R = torch.bmm(Rc, T[:, :, :3]) * torch.tensor([1.0, -1.0, -1.0], dtype=c2w.dtype, device=c2w.device)
    t = torch.bmm(Rc, T[:, :, 3:]) + tc
    Rinv = R.transpose(1, 2)
    out = torch.zeros(c2w.shape[0], 4, 4, dtype=c2w.dtype, device=c2w.device)
    out[:, 3, 3] = 1.0
    out[:, :3, :3] = Rinv
    out[:, :3, 3:] = -torch.bmm(Rinv, t)
    return out


def regularizer_torch(adj: Tensor, trans_weight: float, rot_weight: float) -> Tensor:
    return trans_weight * adj[:, :3].norm(dim=-1).mean() + rot_weight * adj[:, 3:].norm(dim=-1).mean()


def lr_at(step: int, lr: float, lr_final: float, warmup_steps: int, max_steps: int) -> float:
    """nerfstudio ExponentialDecayScheduler with lr_pre_warmup = 0 and its default cosine ramp: lr sin(pi/2 step / warmup)
    during the warm-up, then log-linear from lr to lr_final over the remaining steps.  lr = 0 freezes the table."""
    if lr == 0.0:
        return 0.0
    if step < warmup_steps:
        return lr * math.sin(0.5 * math.pi * step / warmup_steps)
    t = min(max((step - warmup_steps) / max(max_steps - warmup_steps, 1), 0.0), 1.0)
    return math.exp(math.log(lr) * (1 - t) + math.log(lr_final) * t)


def check_camera_ids(camera_ids: Tensor, n_views: int, num_cameras: int, device) -> Tensor:
    """Validation on the host before any pointer crosses the C-ABI -> contiguous int32 ids on `device`.  Ids on the CPU
    (what a data loader hands out) are checked there and copied without waiting for the device; ids already on the
    device cost one synchronisation for the check."""
    if not isinstance(camera_ids, Tensor) or camera_ids.dtype not in (torch.int32, torch.int64) or camera_ids.dim() != 1:
        raise TypeError("camera_ids must be a 1-D int32 or int64 tensor")
    if camera_ids.numel() != n_views:
        raise ValueError(f"camera_ids has {camera_ids.numel()} entries for {n_views} views")
    host = camera_ids.cpu()
    if n_views and (int(host.min()) < 0 or int(host.max()) >= num_cameras):
        raise ValueError(f"camera_ids must lie in [0, {num_cameras})")
    ids = camera_ids.to(torch.int32).contiguous()
    if ids.device != device:
        ids = (ids.pin_memory() if device.type == "cuda" else ids).to(device, non_blocking=True)
    return ids


class AdamTable:
    """A flat table trained by Adam (torch semantics, dense) with the `lr_at` schedule: `param`, `grad`, `exp_avg` and
    `exp_avg_sq` of `n` floats, padded to 4, zero at init.  `backend="cuda"`: `qed_adam_arena` as a one-group call;
    `backend="torch"`: the same arithmetic in torch."""

    def __init__(self, n: int, device, what: str, lr: float, lr_final: float, warmup_steps: int, max_steps: int, betas, eps: float,
                 backend: str):
        if lr < 0 or lr_final <= 0 or warmup_steps < 0:
            raise ValueError(f"{what}: lr >= 0, lr_final > 0 and warmup_steps >= 0 expected")
        self.backend = backend
        self.lr, self.lr_final, self.warmup_steps, self.max_steps = lr, lr_final, warmup_steps, max_steps
        self.betas, self.eps = betas, eps
        self.padded = (n + 3) // 4 * 4
        self.param, self.grad, self.exp_avg, self.exp_avg_sq = (torch.zeros(self.padded, device=device) for _ in range(4))
        self.device = self.param.device  # with its index
        self._lr = torch.zeros(1, device=self.device)
        self._ends = torch.tensor([self.padded], dtype=torch.int64, device=self.device)
        self.lib = None
        if backend == "cuda":
            from . import _lib

            self.lib = _lib.load()

    def use_grad_buffer(self, buf: Tensor) -> None:
        """Let the gradient live in `buf` (e.g. the symmetric buffer the ranks all-reduce)."""
        assert buf.numel() == self.padded and buf.dtype == torch.float32
        self.grad = buf

    def lr_at(self, step: int) -> float:
        return lr_at(step, self.lr, self.lr_final, self.warmup_steps, self.max_steps)

    def step(self, step: int) -> None:
        """Adam on the whole table with the scheduled lr of 0-based iteration `step` (bias corrections use step + 1)."""
        lr, t = self.lr_at(step), step + 1
        b1, b2 = self.betas
        if self.backend != "cuda":
            self.exp_avg.mul_(b1).add_(self.grad, alpha=1 - b1)
            self.exp_avg_sq.mul_(b2).addcmul_(self.grad, self.grad, value=1 - b2)
            denom = self.exp_avg_sq.sqrt() / math.sqrt(1.0 - b2 ** t) + self.eps
            self.param.sub_(lr / (1.0 - b1 ** t) * (self.exp_avg / denom))
            return
        from . import _lib

        self._lr.fill_(lr)
        _lib.check(self.lib.qed_adam_arena(self.padded, _lib.ptr(self.param), _lib.ptr(self.grad), _lib.ptr(self.exp_avg), _lib.ptr(self.exp_avg_sq),
                                           1, _lib.ptr(self._ends), _lib.ptr(self._lr), None, None, None, b1, b2, self.eps, t,
                                           _lib.current_stream()), "qed_adam_arena")


class CameraPoseOptimizer(AdamTable):
    """The pose table [num_cameras * 6] (zero at init), its gradient and its Adam moments.

    Per training step: `viewmats(c2w, ids)` -> render / backward with pose gradients -> `backward(v_viewmats, ids, c2w)`
    (data term, overwrites `grad`) -> sum `grad` over the ranks -> `regularize()` -> `step(t)`."""

    def __init__(self, num_cameras: int, device, lr: float = 1e-4, lr_final: float = 5e-7, warmup_steps: int = 1000,
                 max_steps: int = 30000, trans_weight: float = 1e-2, rot_weight: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-15,
                 backend: str = "cuda"):
        if num_cameras < 1:
            raise ValueError("the camera optimizer needs num_cameras >= 1")
        self.num_cameras = int(num_cameras)
        super().__init__(self.num_cameras * 6, device, "camera optimizer", lr, lr_final, warmup_steps, max_steps, betas, eps, backend)
        self.trans_weight, self.rot_weight = trans_weight, rot_weight
        self.reg_loss = torch.zeros(1, device=self.device)

    @property
    def pose_adjustment(self) -> Tensor:
        """[num_cameras, 6] view of the table: translation [:3], rotation log [3:]."""
        return self.param[:self.num_cameras * 6].view(self.num_cameras, 6)

    @property
    def pose_grad(self) -> Tensor:
        return self.grad[:self.num_cameras * 6].view(self.num_cameras, 6)

    def prepare(self, c2w: Tensor, camera_ids: Tensor):
        """Validated inputs of one step: -> (contiguous c2w, int32 ids on the table's device)."""
        if c2w.dim() != 3 or c2w.shape[1] not in (3, 4) or c2w.shape[2] != 4 or c2w.dtype != torch.float32:
            raise ValueError("camera_to_worlds must be float32 [C,3,4] or [C,4,4]")
        if c2w.device != self.device:
            raise ValueError(f"camera_to_worlds must live on {self.device}")
        return c2w.contiguous(), check_camera_ids(camera_ids, c2w.shape[0], self.num_cameras, self.device)

    def viewmats(self, c2w: Tensor, camera_ids: Tensor) -> Tensor:
        """[C,4,4] world-to-camera matrices of the adjusted poses (a fresh tensor)."""
        return self._viewmats(*self.prepare(c2w, camera_ids))

    def _viewmats(self, c2w: Tensor, ids: Tensor) -> Tensor:
        if self.backend != "cuda":
            return viewmats_torch(c2w, ids.long(), self.pose_adjustment)
        from . import _lib

        out = torch.empty(c2w.shape[0], 4, 4, device=self.device)
        _lib.check(self.lib.qed_camera_opt_apply(c2w.shape[0], c2w.shape[1], self.num_cameras, _lib.ptr(ids), _lib.ptr(c2w),
                                                 _lib.ptr(self.param), _lib.ptr(out), _lib.current_stream()), "qed_camera_opt_apply")
        return out

    def backward(self, v_viewmats: Tensor, camera_ids: Tensor, c2w: Tensor) -> None:
        """Data term of d loss / d table from d loss / d viewmats [C,4,4] of the same views; overwrites `grad`."""
        c2w, ids = self.prepare(c2w, camera_ids)
        self._backward(v_viewmats, ids, c2w)

    def _backward(self, v_viewmats: Tensor, ids: Tensor, c2w: Tensor) -> None:
        if v_viewmats.shape != (c2w.shape[0], 4, 4) or v_viewmats.dtype != torch.float32 or v_viewmats.device != self.device:
            raise ValueError("v_viewmats must be float32 [C,4,4] for the C views of camera_to_worlds")
        v_viewmats = v_viewmats.contiguous()
        if self.backend != "cuda":
            adj = self.pose_adjustment.detach().double().requires_grad_(True)
            vm = viewmats_torch(c2w.double(), ids.long(), adj)
            (g,) = torch.autograd.grad(vm, adj, v_viewmats.double())
            self.grad.zero_()
            self.pose_grad.copy_(g)
            return
        from . import _lib

        _lib.check(self.lib.qed_camera_opt_bwd(c2w.shape[0], c2w.shape[1], self.num_cameras, _lib.ptr(ids), _lib.ptr(c2w), _lib.ptr(self.param),
                                               _lib.ptr(v_viewmats), _lib.ptr(self.grad), _lib.current_stream()), "qed_camera_opt_bwd")

    def regularize(self) -> Tensor:
        """Adds the regulariser's gradient to `grad` (call once per step, after the cross-rank sum); returns its value (device)."""
        if self.backend != "cuda":
            adj = self.pose_adjustment.detach().clone().requires_grad_(True)
            r = regularizer_torch(adj, self.trans_weight, self.rot_weight)
            (g,) = torch.autograd.grad(r, adj)
            self.pose_grad.add_(g)
            self.reg_loss.copy_(r.detach().reshape(1))
            return self.reg_loss
        from . import _lib

        _lib.check(self.lib.qed_camera_opt_reg(self.num_cameras, _lib.ptr(self.param), self.trans_weight, self.rot_weight, _lib.ptr(self.grad),
                                               _lib.ptr(self.reg_loss), _lib.current_stream()), "qed_camera_opt_reg")
        return self.reg_loss
