"""B200-native multi-scale deformable attention hot path of
bharathikannann/Depth-Fusion-in-Transformer-Based-Video-Object-Detection.

Layout (only what the hot path needs):
  csrc/                                  hand-written sm_100a kernels + the C ABI (include/msda_b200.h)
  libmsda_b200.so                        built in-tree by ``make`` / ``__graft_entry__.build()``
  _lib.py                                ctypes binding of that ABI
  MultiScaleDeformableAttention.py       drop-in for the reference's pybind extension module
  ops/functions, ops/modules             mirror of the reference's models/ops (MSDeformAttnFunction, MSDeformAttn)
  transformer_layers.py                  encoder / decoder / Late Fusion / Encoder Cross Fusion layer classes
  backbone_fusion.py                     Backbone Cross Fusion (U-DF) layer + fuse_layers
  deformable_transformer.py              single-frame DeformableTransformer (baseline / Late Fusion / Encoder Cross Fusion)
  position_encoding.py                   PositionEmbeddingSine written token-major (lvl_pos_embed_flatten in one pass)
  temporal_stage.py                      TransVOD++ multi-frame transformer: RoIAlign, QRF head, TQE, TDTD
  criterion.py                           Deformable DETR's HungarianMatcher / SetCriterion, assignment solved on the GPU

The directory name carries hyphens; import it through the alias module ``dfvod_b200`` at the
repository root (``import dfvod_b200``), or put ``ops`` in place of the reference's ``models/ops``.
"""
from . import MultiScaleDeformableAttention
from .criterion import HungarianMatcher, SetCriterion, pad_targets
from .ops.functions import MSDeformAttnFunction
from .ops.modules import MSDeformAttn

__all__ = ["MultiScaleDeformableAttention", "MSDeformAttnFunction", "MSDeformAttn", "HungarianMatcher", "SetCriterion",
           "pad_targets"]
