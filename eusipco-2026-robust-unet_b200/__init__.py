"""B200-native (sm_100a) Robust U-Net hot path behind the reference's torch.nn.Module API.

Drop-in surface (reference: /root/reference/Main_Final.py):
  RobustUNet(n_channels=3, n_classes=1, base_channels=64)   Main_Final.py:226-321 (1 <= n_classes <= 32)
  ResidualBlock / AttentionGate / DilatedBlock (standalone)  Main_Final.py:120-223
  RobustBCEDiceLoss()  (defaults == nn.BCELoss())           Main_Final.py:551,580
  calculate_metrics(pred, target, threshold=0.5)            Main_Final.py:519-547
  predict_tiled(model, scene, tile, overlap)                whole scene at full resolution (predict_coastline.py:386-392)
  PatchSampler(images, masks, size, ...).sample(B)          training patches of whole scenes at native resolution
  coastline_metrics(pred, target, tolerances, pixel_size)   coastline position errors (mean distance, HD95, surface Dice)
  distance_transform(features)                              exact squared Euclidean distance transform
  remove_small_regions(mask, min_water, min_land)           drop small water blobs, fill small land specks
  label_components(mask, connectivity) / component_stats    connected components (scipy / OpenCV numbering and stats)
  find_contours(mask, approx)                               outer contours, bit for bit with cv2.findContours(RETR_EXTERNAL)
Everything below that surface is hand-written CUDA in csrc/ reached through the C ABI of
librbunet.so (include/rbunet.h).  There is no CPU fallback.
"""
from . import _lib  # noqa: F401
from .components import component_stats, label_components, remove_small_regions  # noqa: F401
from .contours import find_contours  # noqa: F401
from .distance import coastline_metrics, coastline_stats, distance_transform  # noqa: F401
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
           "metrics_from_counts", "METRIC_KEYS", "View", "preprocess", "resize", "enhance_image", "coastline_mask", "predict_tiled", "PatchSampler", "distance_transform", "coastline_stats", "coastline_metrics", "label_components", "component_stats", "remove_small_regions", "find_contours", "DataParallel", "GradBucketer", "FusedAdam", "UNet", "CrossEntropyArgmaxLoss"]
