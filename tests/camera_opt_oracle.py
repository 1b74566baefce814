"""Reference restatement of splatfacto's SO3xR3 camera optimizer (nerfstudio 1.1.5 CameraOptimizer, recalled) for the tests.

Written independently of qed_splatter_b200.camera_opt: the exp map is expanded entry by entry and the viewmat comes from
oracle.get_viewmat.  tests/test_camera_opt_cpu.py checks its autograd against finite differences of the whole render."""
import torch

import oracle


def exp_map(adj: torch.Tensor) -> torch.Tensor:
    """[n,6] {t, omega} -> [n,3,3] rotation: theta^2 = max(|omega|^2, 1e-4), I + (sin t / t) [w]x + ((1 - cos t) / t^2) [w]x^2."""
    x, y, z = adj[:, 3], adj[:, 4], adj[:, 5]
    th2 = torch.clamp(x * x + y * y + z * z, min=1e-4)
    th = th2.sqrt()
    a, b = torch.sin(th) / th, (1 - torch.cos(th)) / th2
    n2 = x * x + y * y + z * z
    rows = [[1 + b * (x * x - n2), -a * z + b * x * y, a * y + b * x * z],
            [a * z + b * x * y, 1 + b * (y * y - n2), -a * x + b * y * z],
            [-a * y + b * x * z, a * x + b * y * z, 1 + b * (z * z - n2)]]
    return torch.stack([torch.stack(r, dim=-1) for r in rows], dim=-2)


def adjusted_c2w(c2w: torch.Tensor, camera_ids: torch.Tensor, adj: torch.Tensor) -> torch.Tensor:
    """apply_to_camera: c2w[:3,:4] @ [[R, t], [0, 1]] -> [C,3,4]."""
    a = adj[camera_ids.long()]
    R = exp_map(a)
    Rc, tc = c2w[:, :3, :3], c2w[:, :3, 3]
    return torch.cat([Rc @ R, (tc + (Rc @ a[:, :3, None])[..., 0])[..., None]], dim=-1)


def viewmats(c2w: torch.Tensor, camera_ids: torch.Tensor, adj: torch.Tensor) -> torch.Tensor:
    return oracle.get_viewmat(adjusted_c2w(c2w, camera_ids, adj))


def regularizer(adj: torch.Tensor, trans_weight: float = 1e-2, rot_weight: float = 1e-3) -> torch.Tensor:
    return trans_weight * adj[:, :3].norm(dim=-1).mean() + rot_weight * adj[:, 3:].norm(dim=-1).mean()
