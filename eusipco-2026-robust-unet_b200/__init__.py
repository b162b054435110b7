"""B200-native (sm_100a) Robust U-Net hot path behind the reference's torch.nn.Module API.

Drop-in surface (reference: /root/reference/Main_Final.py):
  RobustUNet(n_channels=3, n_classes=1, base_channels=64)   Main_Final.py:226-321 (1 <= n_classes <= 32)
  ResidualBlock / AttentionGate / DilatedBlock (standalone)  Main_Final.py:120-223
  RobustBCEDiceLoss()  (defaults == nn.BCELoss())           Main_Final.py:551,580
  calculate_metrics(pred, target, threshold=0.5)            Main_Final.py:519-547
  predict_tiled(model, scene, tile, overlap)                whole scene at full resolution (predict_coastline.py:386-392)
  PatchSampler(images, masks, size, ...).sample(B)          training patches of whole scenes at native resolution
Everything below that surface is hand-written CUDA in csrc/ reached through the C ABI of
librbunet.so (include/rbunet.h).  There is no CPU fallback.
"""
from . import _lib  # noqa: F401
from .loss import (METRIC_KEYS, RobustBCEDiceLoss, batch_metrics, calculate_metrics,  # noqa: F401
                   class_confusion_counts, class_metrics, confusion_counts, metrics_from_counts)
from .model import AttentionGate, DilatedBlock, ResidualBlock, RobustUNet  # noqa: F401
from .ops import View, coastline_mask, enhance_image, preprocess, resize  # noqa: F401
from .optim import FusedAdam  # noqa: F401
from .parallel import DataParallel, GradBucketer  # noqa: F401
from .patches import PatchSampler  # noqa: F401
from .tiled import predict_tiled  # noqa: F401
from .unet import CrossEntropyArgmaxLoss, UNet  # noqa: F401

__all__ = ["RobustUNet", "ResidualBlock", "AttentionGate", "DilatedBlock", "RobustBCEDiceLoss", "calculate_metrics", "batch_metrics", "confusion_counts", "class_confusion_counts", "class_metrics",
           "metrics_from_counts", "METRIC_KEYS", "View", "preprocess", "resize", "enhance_image", "coastline_mask", "predict_tiled", "PatchSampler", "DataParallel", "GradBucketer", "FusedAdam", "UNet", "CrossEntropyArgmaxLoss"]
