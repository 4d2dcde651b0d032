"""Layer classes of the reference transformers that own an ``MSDeformAttn`` -- host-side mirror.

Same class names, constructor signatures, forward signatures, attribute names (hence state_dict
keys) and arithmetic as the reference, so a reference model can take these classes instead of
its own and load its checkpoints:

  DeformableTransformerEncoderLayer / DeformableTransformerEncoder
        /root/reference/models/deformable_transformer_single.py:520-593
        (dups: deformable_transformer_multi_plusplus.py:903-973, deformable_transformer_multi.py:675-746)
  DeformableTransformerDecoderLayer / DeformableTransformerDecoder      single.py:596-648, :703-748
  DepthDeformableTransformerEncoderLayer   (Late Fusion)                single.py:341-402
  DeformableTransformerFusionLayerV2       (Encoder Cross Fusion)       single.py:406-461
  RGBDDeformableTransformerEncoderV2                                    single.py:465-518
  TemporalDeformableTransformerEncoderLayer (frames as levels)          single.py:650-700
  TemporalDeformableTransformerDecoder     (TransVOD++ TDTD)            multi_plusplus.py:1030-1076

Every deformable attention inside them is the sm_100a op (ops/modules/ms_deform_attn.py).  The
element-wise chains around it -- residual add + LayerNorm, the "+ pos" that forms the next
query, bias + activation -- run as the fused layer-epilogue kernels of csrc/layer_epilogue.cu
(ops/functions/layer_epilogue_func.py); Linear / MultiheadAttention stay library GEMMs.
"""
import copy

import torch
import torch.nn.functional as F
from torch import nn

from .ops.functions import (add_layer_norm, dropout, ffn_layer_norm, ffn_layer_norm_supported, linear, linear_relu,
                            proj_layer_norm)
from .ops.modules import MSDeformAttn, project_values
from .ops.modules.ms_deform_attn import host_shape_list


def inverse_sigmoid(x, eps=1e-5):
    """/root/reference/util/misc.py:531-535."""
    x = x.clamp(min=0, max=1)
    return torch.log(x.clamp(min=eps) / (1 - x).clamp(min=eps))


def _get_clones(module, N):
    return nn.ModuleList([copy.deepcopy(module) for _ in range(N)])


def _get_activation_fn(activation):
    """Return an activation function given a string (single.py:755-763)."""
    table = {"relu": F.relu, "gelu": F.gelu, "glu": F.glu}
    if activation not in table:
        raise RuntimeError(F"activation should be relu/gelu, not {activation}.")
    return table[activation]


def mha_batch_first(mha, query, key, value):
    """``nn.MultiheadAttention`` (no masks, attention weights not needed) on BATCH-FIRST ``[N, L, E]`` tensors, computed
    from the module's own parameters: the reference hands ``[L, N, E]`` transposes to the module
    (deformable_transformer_single.py:621-623), which then copies them into head-major layouts and back -- here the
    heads are strided views of the projection outputs, q and k share one GEMM when they are the same tensor, and the
    fused scaled-dot-product kernel reads the views in place.  Same arithmetic, same parameters / state-dict keys."""
    e, heads = mha.embed_dim, mha.num_heads
    w, b = mha.in_proj_weight, mha.in_proj_bias
    bias = (lambda lo, hi: None) if b is None else (lambda lo, hi: b[lo:hi])
    if query is key:
        qk = F.linear(query, w[:2 * e], bias(0, 2 * e))
        q, k = qk[..., :e], qk[..., e:]
    else:
        q = F.linear(query, w[:e], bias(0, e))
        k = F.linear(key, w[e:2 * e], bias(e, 2 * e))
    v = F.linear(value, w[2 * e:], bias(2 * e, 3 * e))
    n, lq, lk = q.shape[0], q.shape[1], k.shape[1]
    split = lambda t, length: t.view(n, length, heads, e // heads).transpose(1, 2)         # [N, heads, L, head_dim] view
    out = F.scaled_dot_product_attention(split(q, lq), split(k, lk), split(v, lk),
                                         dropout_p=mha.dropout if mha.training else 0.0)
    out = out.transpose(1, 2).reshape(n, lq, e)
    return F.linear(out, mha.out_proj.weight, mha.out_proj.bias)


def _add_pos(tensor, pos):
    return tensor if pos is None else tensor + pos


def encoder_reference_points(spatial_shapes, valid_ratios, device):
    """Pixel-centre reference grid of every level, replicated to every level and scaled by the
    valid ratios: [N, sum_l H_l*W_l, L, 2] (x, y).  single.py:164-177 / :573-585 / :483-495."""
    per_level = []
    for lvl, (H_, W_) in enumerate(host_shape_list(spatial_shapes)):
        ys = torch.linspace(0.5, H_ - 0.5, H_, dtype=torch.float32, device=device)
        xs = torch.linspace(0.5, W_ - 0.5, W_, dtype=torch.float32, device=device)
        ref_y, ref_x = torch.meshgrid(ys, xs, indexing="ij")
        ref_y = ref_y.reshape(-1)[None] / (valid_ratios[:, None, lvl, 1] * H_)
        ref_x = ref_x.reshape(-1)[None] / (valid_ratios[:, None, lvl, 0] * W_)
        per_level.append(torch.stack((ref_x, ref_y), -1))
    points = torch.cat(per_level, 1)
    return points[:, :, None] * valid_ratios[:, None]


# ------------------------------------------------------------------------------------------
# encoder
# ------------------------------------------------------------------------------------------
class DeformableTransformerEncoderLayer(nn.Module):
    def __init__(self, d_model=256, d_ffn=1024, dropout=0.1, activation="relu",
                 n_levels=4, n_heads=8, n_points=4):
        super().__init__()
        # deformable self attention over the multi-scale map
        self.self_attn = MSDeformAttn(d_model, n_levels, n_heads, n_points)
        self.dropout1 = nn.Dropout(dropout)
        self.norm1 = nn.LayerNorm(d_model)
        # feed-forward
        self.linear1 = nn.Linear(d_model, d_ffn)
        self.activation = _get_activation_fn(activation)
        self._activation_name = activation
        self.dropout2 = nn.Dropout(dropout)
        self.linear2 = nn.Linear(d_ffn, d_model)
        self.dropout3 = nn.Dropout(dropout)
        self.norm2 = nn.LayerNorm(d_model)

    use_fused_ffn = True      # bf16 inference at d_model 256: the whole feed-forward block in one kernel
    with_pos_embed = staticmethod(_add_pos)

    def forward_ffn(self, src, pos=None):
        """norm2(src + linear2(act(linear1(src)))); with ``pos`` also returns that + pos."""
        if self._activation_name == "relu" and not (self.training and (self.dropout2.p > 0 or self.dropout3.p > 0)) \
                and self.use_fused_ffn and ffn_layer_norm_supported(src, self.linear1, self.linear2, self.norm2):
            return ffn_layer_norm(self.linear1, self.linear2, self.norm2, src, pos)     # one tcgen05 kernel
        hidden = linear_relu(self.linear1, src, self.dropout2) if self._activation_name == "relu" \
            else dropout(self.dropout2, self.activation(linear(self.linear1, src)))
        return add_layer_norm(self.norm2, linear(self.linear2, hidden), src, None, pos, dropout=self.dropout3)

    def forward(self, src, pos, reference_points, spatial_shapes, level_start_index, padding_mask=None,
                rgbd_src=None, query=None, emit_query=False):
        """Reference signature plus two private keywords used by the encoder loops: ``query`` is a
        precomputed ``src + pos`` and ``emit_query=True`` makes the call return
        ``(out, out + pos)`` so the next layer's query costs no extra pass."""
        if query is None:
            query = rgbd_src if rgbd_src is not None else _add_pos(src, pos)
        if self.training and self.dropout1.p > 0:
            attended = self.self_attn(query, reference_points, src, spatial_shapes, level_start_index, padding_mask)
            src = add_layer_norm(self.norm1, attended, src, dropout=self.dropout1)
        else:       # output projection + residual + LayerNorm as one kernel (bf16 inference), else GEMM + fused norm
            heads = self.self_attn(query, reference_points, src, spatial_shapes, level_start_index, padding_mask,
                                   project_output=False)
            src = proj_layer_norm(self.self_attn.output_proj, self.norm1, heads, src)
        if not emit_query:
            return self.forward_ffn(src)
        if pos is None:
            out = self.forward_ffn(src)
            return out, out
        return self.forward_ffn(src, pos)


class DeformableTransformerEncoder(nn.Module):
    def __init__(self, encoder_layer, num_layers):
        super().__init__()
        self.layers = _get_clones(encoder_layer, num_layers)
        self.num_layers = num_layers

    get_reference_points = staticmethod(encoder_reference_points)

    def forward(self, src, spatial_shapes, level_start_index, valid_ratios, pos=None, padding_mask=None,
                rgbd_src=None):
        reference_points = self.get_reference_points(spatial_shapes, valid_ratios, device=src.device)
        output = src
        if rgbd_src is not None:
            for layer in self.layers:
                output = layer(output, pos, reference_points, spatial_shapes, level_start_index, padding_mask,
                               rgbd_src=rgbd_src)
            return output
        query = None                  # layer i hands layer i+1 its query (output + pos) from its last kernel
        for i, layer in enumerate(self.layers):
            if i + 1 < len(self.layers):
                output, query = layer(output, pos, reference_points, spatial_shapes, level_start_index,
                                      padding_mask, query=query, emit_query=True)
            else:
                output = layer(output, pos, reference_points, spatial_shapes, level_start_index, padding_mask,
                               query=query)
        return output


# ------------------------------------------------------------------------------------------
# depth fusion: RGB queries sample depth-feature values
# ------------------------------------------------------------------------------------------
class _CrossModalFusion(nn.Module):
    """Shared body of the Late Fusion and Encoder Cross Fusion layers (single.py:341-461):
        src  = LN(Linear(depth))
        t    = Linear(MSDeformAttn(rgb + pos, ref, src))
        tgt  = LN(tgt + drop(t));  tgt = LN(tgt + drop(GELU(Linear(tgt))))
    The two reference classes differ only in the names of their last dropout / norm."""

    def _build(self, d_model, dropout, n_levels, n_heads, n_points, ffn_dropout_name, ffn_norm_name):
        self.cross_attn = MSDeformAttn(d_model, n_levels, n_heads, n_points)
        self.dropout1 = nn.Dropout(dropout)
        self.norm1 = nn.LayerNorm(d_model)
        self.linear1 = nn.Linear(d_model, d_model)
        self.activation = _get_activation_fn('gelu')          # hard-coded in the reference (:358, :418)
        setattr(self, ffn_dropout_name, nn.Dropout(dropout))
        setattr(self, ffn_norm_name, nn.LayerNorm(d_model))
        self.depth_scale_adapt = nn.Linear(d_model, d_model)
        self.norm_depth_scale = nn.LayerNorm(d_model)
        self.cross_scale_adapt = nn.Linear(d_model, d_model)
        self._ffn_dropout, self._ffn_norm = ffn_dropout_name, ffn_norm_name

    with_pos_embed = staticmethod(_add_pos)

    def forward_ffn(self, tgt):
        drop, norm = getattr(self, self._ffn_dropout), getattr(self, self._ffn_norm)
        # GELU (and the dropout, when training) inside the norm kernel
        return add_layer_norm(norm, linear(self.linear1, tgt), tgt, "gelu", dropout=drop)

    def _fuse(self, tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index, src_padding_mask,
              query=None):
        # Linear + (residual +) LayerNorm pairs: one tcgen05 kernel each for bf16 inference, else GEMM + fused norm
        src = proj_layer_norm(self.depth_scale_adapt, self.norm_depth_scale, src)
        if query is None:
            query = _add_pos(tgt, query_pos)
        sampled = self.cross_attn(query, reference_points, src, src_spatial_shapes, level_start_index,
                                  src_padding_mask)
        if self.training and self.dropout1.p > 0:
            tgt = add_layer_norm(self.norm1, linear(self.cross_scale_adapt, sampled), tgt, dropout=self.dropout1)
        else:
            tgt = proj_layer_norm(self.cross_scale_adapt, self.norm1, sampled, tgt)
        return self.forward_ffn(tgt)


class DepthDeformableTransformerEncoderLayer(_CrossModalFusion):
    """Late Fusion layer (single.py:341-402).  ``src_pos``, ``tgt_spatial_shapes``,
    ``depth_reference_points`` and ``tgt_padding_mask`` are accepted and ignored, as in the
    reference."""

    def __init__(self, d_model=256, d_ffn=1024, dropout=0.1, activation='relu', n_depth_levels=1, n_heads=8,
                 dpth_n_points=4, depth_self_attn=False, gate=True, adaptation_layers=True):
        super().__init__()
        self.depth_self_attn = depth_self_attn
        self.adaptation_layers = adaptation_layers
        self._build(d_model, dropout, n_depth_levels, n_heads, dpth_n_points, "dropout4", "norm3")

    def forward(self, tgt, query_pos, src_pos, tgt_spatial_shapes, reference_points, depth_reference_points,
                src, src_spatial_shapes, frame_start_index, tgt_padding_mask=None, src_padding_mask=None):
        return self._fuse(tgt, query_pos, reference_points, src, src_spatial_shapes, frame_start_index,
                          src_padding_mask)


class DeformableTransformerFusionLayerV2(_CrossModalFusion):
    """Encoder Cross Fusion layer (single.py:406-461)."""

    def __init__(self, d_model=256, d_ffn=1024, dropout=0.1, activation="gelu", n_levels=4, n_heads=8,
                 n_points=4):
        super().__init__()
        self._build(d_model, dropout, n_levels, n_heads, n_points, "dropout3", "norm2")

    def forward(self, tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                src_padding_mask=None, query=None):
        return self._fuse(tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                          src_padding_mask, query=query)


class RGBDDeformableTransformerEncoderV2(nn.Module):
    """Encoder of the Encoder-Cross-Fusion model (single.py:465-518): after RGB encoder layer i
    (i < depth_num_layers, i in fusion_layers_order) a fusion layer lets the RGB tokens sample
    the running fusion stream, and the result is added back.  Note the reference feeds the
    previous fusion OUTPUT (RGB length) as the next fusion's value and passes the RGB padding
    mask for it (:515) -- reproduced."""

    def __init__(self, encoder_layer, fusion_encoder_layer, num_layers, depth_num_layers, fusion_num_layers,
                 fusion_layers_order=[]):
        super().__init__()
        self.layers = _get_clones(encoder_layer, num_layers)
        self.fusion_layers = _get_clones(fusion_encoder_layer, fusion_num_layers)
        self.num_layers = num_layers
        self.depth_num_layers = depth_num_layers
        self.fusion_num_layers = fusion_num_layers
        self.fusion_layers_order = list(fusion_layers_order) if len(fusion_layers_order) > 0 \
            else list(range(fusion_num_layers))
        assert len(self.fusion_layers_order) == self.fusion_num_layers, \
            "The number of fusion layers should match the fusion layer count"

    get_reference_points = staticmethod(encoder_reference_points)

    def forward(self, src, spatial_shapes, level_start_index, valid_ratios, pos=None, padding_mask=None,
                rgbd_src=None, depth_src=None, depth_spatial_shapes=None, depth_level_start_index=None,
                depth_valid_ratios=None, depth_pos=None, depth_padding_mask=None):
        reference_points = self.get_reference_points(spatial_shapes, valid_ratios, device=src.device)
        output, fusion_stream = src, depth_src
        query = None
        for i, layer in enumerate(self.layers):
            fuse = i < self.depth_num_layers and i in self.fusion_layers_order
            if fuse or i + 1 < len(self.layers):
                output, query = layer(output, pos, reference_points, spatial_shapes, level_start_index,
                                      padding_mask, query=query, emit_query=True)
            else:
                output = layer(output, pos, reference_points, spatial_shapes, level_start_index, padding_mask,
                               query=query)
            if fuse:
                fusion_layer = self.fusion_layers[self.fusion_layers_order.index(i)]
                fusion_stream = fusion_layer(output, pos, reference_points, fusion_stream, depth_spatial_shapes,
                                             depth_level_start_index, padding_mask, query=query)
                output = output + fusion_stream
                query = None          # output changed: the next layer forms its own query
        return output


# ------------------------------------------------------------------------------------------
# decoder
# ------------------------------------------------------------------------------------------
class DeformableTransformerDecoderLayer(nn.Module):
    def __init__(self, d_model=256, d_ffn=1024, dropout=0.1, activation="relu",
                 n_levels=4, n_heads=8, n_points=4):
        super().__init__()
        # deformable cross attention into the encoder memory
        self.cross_attn = MSDeformAttn(d_model, n_levels, n_heads, n_points)
        self.dropout1 = nn.Dropout(dropout)
        self.norm1 = nn.LayerNorm(d_model)
        # dense self attention among the object queries
        self.self_attn = nn.MultiheadAttention(d_model, n_heads, dropout=dropout)
        self.dropout2 = nn.Dropout(dropout)
        self.norm2 = nn.LayerNorm(d_model)
        # feed-forward
        self.linear1 = nn.Linear(d_model, d_ffn)
        self.activation = _get_activation_fn(activation)
        self._activation_name = activation
        self.dropout3 = nn.Dropout(dropout)
        self.linear2 = nn.Linear(d_ffn, d_model)
        self.dropout4 = nn.Dropout(dropout)
        self.norm3 = nn.LayerNorm(d_model)

    with_pos_embed = staticmethod(_add_pos)

    def forward_ffn(self, tgt, pos=None):
        hidden = linear_relu(self.linear1, tgt, self.dropout3) if self._activation_name == "relu" \
            else dropout(self.dropout3, self.activation(linear(self.linear1, tgt)))
        return add_layer_norm(self.norm3, linear(self.linear2, hidden), tgt, None, pos, dropout=self.dropout4)

    def forward(self, tgt, query_pos, reference_points, src, src_spatial_shapes, level_start_index,
                src_padding_mask=None, qk=None, emit_qk=False, value=None):
        """Reference signature plus private keywords used by the decoder loop: ``qk`` is a precomputed
        ``tgt + query_pos``; ``emit_qk=True`` returns ``(out, out + query_pos)``; ``value`` is this layer's
        ``cross_attn.value_proj(src)`` computed together with the other layers' (ops.modules.project_values)."""
        if qk is None:
            qk = _add_pos(tgt, query_pos)
        mixed = mha_batch_first(self.self_attn, qk, qk, tgt)
        if query_pos is not None:
            tgt, query = add_layer_norm(self.norm2, mixed, tgt, None, query_pos, dropout=self.dropout2)
        else:
            tgt = query = add_layer_norm(self.norm2, mixed, tgt, dropout=self.dropout2)
        sampled = self.cross_attn(query, reference_points, src, src_spatial_shapes, level_start_index,
                                  src_padding_mask, precomputed_value=value)
        tgt = add_layer_norm(self.norm1, sampled, tgt, dropout=self.dropout1)
        if not emit_qk:
            return self.forward_ffn(tgt)
        if query_pos is None:
            out = self.forward_ffn(tgt)
            return out, out
        return self.forward_ffn(tgt, query_pos)


class TemporalDeformableTransformerEncoderLayer(DeformableTransformerDecoderLayer):
    """Frames-as-levels layer (single.py:650-700): identical computation to the decoder layer
    with ``n_levels = n_frames`` and the value built from the reference frames' memories.
    Disabled in every shipped path of the reference; kept for API completeness."""

    def __init__(self, d_model=256, d_ffn=1024, dropout=0.1, activation='relu', n_frames=4, h_heads=8,
                 n_points=4):
        super().__init__(d_model, d_ffn, dropout, activation, n_frames, h_heads, n_points)

    def forward(self, tgt, query_pos, reference_points, src, src_spatial_shapes, frame_start_index,
                src_padding_mask=None):
        return super().forward(tgt, query_pos, reference_points, src, src_spatial_shapes, frame_start_index,
                               src_padding_mask)


class DeformableTransformerDecoder(nn.Module):
    _refine_boxes = True

    def __init__(self, decoder_layer, num_layers, return_intermediate=False):
        super().__init__()
        self.layers = _get_clones(decoder_layer, num_layers)
        self.num_layers = num_layers
        self.return_intermediate = return_intermediate
        # set by the detector for iterative box refinement / two-stage (deformable_detr_single.py)
        self.bbox_embed = None
        self.class_embed = None

    def forward(self, tgt, reference_points, src, src_spatial_shapes, src_level_start_index, src_valid_ratios,
                query_pos=None, src_padding_mask=None):
        output = tgt
        qk = None
        intermediate, intermediate_reference_points = [], []
        # every layer re-projects the same memory with its own value_proj: one GEMM for all of them (inference)
        values = project_values([layer.cross_attn for layer in self.layers], src, src_padding_mask)
        for lid, layer in enumerate(self.layers):
            if reference_points.shape[-1] == 4:
                scale = torch.cat([src_valid_ratios, src_valid_ratios], -1)
            else:
                assert reference_points.shape[-1] == 2
                scale = src_valid_ratios
            reference_points_input = reference_points[:, :, None] * scale[:, None]
            if lid + 1 < len(self.layers):
                output, qk = layer(output, query_pos, reference_points_input, src, src_spatial_shapes,
                                   src_level_start_index, src_padding_mask, qk=qk, emit_qk=True,
                                   value=None if values is None else values[lid])
            else:
                output = layer(output, query_pos, reference_points_input, src, src_spatial_shapes,
                               src_level_start_index, src_padding_mask, qk=qk,
                               value=None if values is None else values[lid])

            if self._refine_boxes and self.bbox_embed is not None:       # single.py:729-739
                delta = self.bbox_embed[lid](output)
                if reference_points.shape[-1] == 4:
                    refined = delta + inverse_sigmoid(reference_points)
                else:
                    assert reference_points.shape[-1] == 2
                    refined = delta
                    refined[..., :2] = delta[..., :2] + inverse_sigmoid(reference_points)
                reference_points = refined.sigmoid().detach()

            if self.return_intermediate:
                intermediate.append(output)
                intermediate_reference_points.append(reference_points)

        if self.return_intermediate:
            return torch.stack(intermediate), torch.stack(intermediate_reference_points)
        return output, reference_points


class TemporalDeformableTransformerDecoder(DeformableTransformerDecoder):
    """TransVOD++ temporal decoder (multi_plusplus.py:1030-1076): the decoder loop with box
    refinement switched off (the reference resets ``self.bbox_embed = None`` inside the loop,
    :1055).  NOTE: TransVOD++ calls it with ``valid_ratios`` expanded to ``num_ref_frames``
    pseudo-levels against a one-level memory (:425,:539); the reference CUDA op then mis-indexes
    silently (SURVEY.md 9.1).  Here that shape mismatch raises; pass ``valid_ratios[:, 0:1]``."""
    _refine_boxes = False
