"""qed_splatter_b200 — B200-native (sm_100a) depth-supervised Gaussian-splat render/train hot path.

Drop-in for the one call leggedrobotics/qed-splatter makes into gsplat
(`gsplat.rendering.rasterization`, /root/reference/qed_splatter/model.py:267-288) plus the fused
loss-gradient / trainer step built on the same kernels.  Hand-written CUDA behind a C-ABI
(`include/qed_splat.h`, `libqedsplat.so`); no CPU fallback.
"""
from .rendering import rasterization  # noqa: F401
from .losses import bilateral_grid_tv_loss, depth_supervised_loss  # noqa: F401
from .data_side import get_viewmat  # noqa: F401
from .metrics import image_metrics, summarize  # noqa: F401
from . import data_side, metrics, ops, scenes  # noqa: F401

__version__ = "0.1.0"
