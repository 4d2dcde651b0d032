"""Backbone Cross Fusion (U-DF) -- host-side mirror of the MSDeformAttn-bearing part of
/root/reference/models/dformer_crossfusion_backbone.py:

  DepthDeformableTransformerEncoderLayer   :120-181   (ReLU/GELU honoured here, unlike single.py)
  FusionBackboneBase.fuse_layers           :387-428   -> :func:`fuse_layers`
  FusionBackboneBase.get_valid_ratio       :360-368   -> :func:`get_valid_ratio`
  FusionBackboneBase.get_reference_points  :370-385   -> :func:`get_reference_points`

The RGB stage map (queries, Lq = h*w) deformably attends to the depth stage map (values,
S = h_d*w_d): the one place in the reference where the query grid and the value grid differ.
``FusionBackboneBase.forward`` itself is not mirrored: it cannot run as shipped (channel table
off by one stage, SURVEY.md section 9.2) and the convolutional stems are outside the path.
"""
import torch
from torch import nn

from .ops.functions import add_layer_norm, dropout, linear
from .ops.modules import MSDeformAttn
from .transformer_layers import _add_pos, _get_activation_fn, encoder_reference_points


class DepthDeformableTransformerEncoderLayer(nn.Module):
    """Transformer encoder layer for depth fusion (backbone variant)."""

    def __init__(self, d_model=256, d_ffn=1024, dropout=0.1, activation='relu', n_depth_levels=1, n_heads=8,
                 dpth_n_points=4, depth_self_attn=True):
        super().__init__()
        self.depth_self_attn = depth_self_attn
        self.cross_attn = MSDeformAttn(d_model, n_depth_levels, n_heads, dpth_n_points)
        self.dropout1 = nn.Dropout(dropout)
        self.norm1 = nn.LayerNorm(d_model)
        self.linear1 = nn.Linear(d_model, d_model)
        self.activation = _get_activation_fn(activation)
        self._activation_name = activation
        self.dropout4 = nn.Dropout(dropout)
        self.norm3 = nn.LayerNorm(d_model)
        self.depth_scale_adapt = nn.Linear(d_model, d_model)
        self.norm_depth_scale = nn.LayerNorm(d_model)
        self.cross_scale_adapt = nn.Linear(d_model, d_model)

    def with_pos_embed(self, tensor, pos):
        return _add_pos(tensor, pos)

    def forward_ffn(self, tgt):
        if self._activation_name not in ("relu", "gelu"):
            return add_layer_norm(self.norm3, dropout(self.dropout4, self.activation(linear(self.linear1, tgt))), tgt)
        return add_layer_norm(self.norm3, linear(self.linear1, tgt), tgt, self._activation_name, dropout=self.dropout4)

    def forward(self, tgt, query_pos, src_pos, tgt_spatial_shapes, reference_points, depth_reference_points,
                src, src_spatial_shapes, frame_start_index, tgt_padding_mask=None, src_padding_mask=None):
        src = add_layer_norm(self.norm_depth_scale, linear(self.depth_scale_adapt, src))
        sampled = self.cross_attn(_add_pos(tgt, query_pos), reference_points, src, src_spatial_shapes,
                                  frame_start_index, src_padding_mask)
        tgt = add_layer_norm(self.norm1, linear(self.cross_scale_adapt, sampled), tgt, dropout=self.dropout1)
        return self.forward_ffn(tgt)


def get_valid_ratio(mask):
    """Fraction of each map that is not padding, (w, h) per batch element.  mask [N,H,W] bool."""
    _, H, W = mask.shape
    valid_h = torch.sum(~mask[:, :, 0], dim=1).float() / H
    valid_w = torch.sum(~mask[:, 0, :], dim=1).float() / W
    return torch.stack([valid_w, valid_h], -1)


get_reference_points = encoder_reference_points


def fuse_layers(src, target, pos_src, pos_target, mask_src, mask_target, fusion_layer):
    """src [N,C,h,w] (RGB stage map, queries) and target [N,C,hd,wd] (depth stage map, values)
    -> fused src [N,C,h,w].  As in the reference, the reference points are the src pixel centres
    scaled by the TARGET's valid ratio (:414-416)."""
    n, c, h, w = src.shape
    hd, wd = target.shape[-2:]
    flat = lambda t: t.flatten(2).transpose(1, 2)
    shapes_src = torch.as_tensor([(h, w)], dtype=torch.long, device=src.device)
    shapes_target = torch.as_tensor([(hd, wd)], dtype=torch.long, device=target.device)
    start_target = shapes_target.new_zeros((1,))
    ratios_src = get_valid_ratio(mask_src)[:, None]
    ratios_target = get_valid_ratio(mask_target)[:, None]
    ref_for_queries = encoder_reference_points([(h, w)], ratios_target, target.device)
    ref_for_values = encoder_reference_points([(hd, wd)], ratios_src, src.device)      # unused by the layer
    fused = fusion_layer(flat(src), flat(pos_src), flat(pos_target), shapes_src, ref_for_queries, ref_for_values,
                         flat(target), shapes_target, start_target, mask_src.flatten(1), mask_target.flatten(1))
    return fused.transpose(1, 2).view(src.shape)
