"""B200-native prompted 3D shifted-window attention (drop-in for the reference's src/modules hot path).

Importing this package loads libpwa_b200.so (hand-written sm_100a kernels behind the C ABI of
include/pwa.h) and fails loudly if it is not built.  The directory name contains hyphens; import it as
`import pwa_b200` (shim at the repo root) or via importlib.
"""
from . import _lib
from .geometry import Geometry, get_geometry
from . import functional
from . import graphs
from . import trainer
from .graphs import GraphedStep
from . import inference
from .inference import sliding_window_inference, segmentation_counts, dice_iou
from .modules import (ConsecutiveSwinBlocks, SwinTransformerBlock, PatchMerging, WindowAttention, RelativePE,
                      BiasTables, window_partition, window_reverse, get_attn_mask, SwinUnetR, SwinUnetRConfig, SwinUpBlock)

__all__ = ['ConsecutiveSwinBlocks', 'SwinTransformerBlock', 'PatchMerging', 'WindowAttention', 'RelativePE',
           'BiasTables', 'window_partition', 'window_reverse', 'get_attn_mask', 'Geometry', 'get_geometry',
           'functional', 'graphs', 'trainer', 'GraphedStep', 'inference', 'sliding_window_inference',
           'segmentation_counts', 'dice_iou', 'SwinUnetR', 'SwinUnetRConfig', 'SwinUpBlock']
