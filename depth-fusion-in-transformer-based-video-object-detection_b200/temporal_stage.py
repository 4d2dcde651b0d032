"""TransVOD++ temporal query stage (SURVEY.md 8f rank 3): what the multi-frame transformer does after
the per-frame encoder + decoder -- RoIAlign of every decoder box out of its frame's memory, the
query / RoI fusion head (QRF = SparseRCNN ``RCNNHead`` with ``DynamicConv``), three rounds of the
temporal query encoder (TQE) over the top-k reference-frame queries, each followed by the temporal
deformable decoder (TDTD).  Host-side mirror of

    /root/reference/models/deformable_transformer_multi_plusplus.py
        bbox2roi :48-67, DeformableTransformer.__init__ :70-172, forward :262-603,
        TemporalQueryEncoderLayer :787-837, TemporalQueryEncoder :840-850
    /root/reference/models/sparse_roi_head/head.py  RCNNHead :31-91, DynamicConv :134-173

with the same class names, constructor arguments, forward signatures and parameter names
(``temporal_query_layer{1,2,3}``, ``dynamic_layer_for_current_query{1,2,3}``,
``temporal_decoder{1,2,3}``, ``temporal_roi_layers1``), so reference checkpoints load.

B200-native differences (results unchanged):
  * ``RoIAlign`` replaces ``mmcv.ops.RoIAlign`` with the token-major CUDA kernel of
    csrc/roi_align.cu (C ABI ``msda_roi_align_forward/backward``): it pools straight out of the
    encoder memory ``[frames, H*W, C]`` and writes ``[rois, 49, C]``, the layout the dynamic
    convolution consumes, so the reference's permute-to-NCHW (:498, :512) and permute-back
    (head.py:66) copies do not exist;
  * the per-reference-frame python loops (class / box heads :457-483, RoIAlign + QRF :507-517) are
    one batched call over all frames of the clip -- every frame is an independent batch element of
    those modules;
  * the temporal decoder receives ``valid_ratios[:, 0:1]`` instead of the reference's
    ``[1, num_ref_frames, 2]`` expansion (:425), which only "works" in the reference because its CUDA
    op never checks the level count (SURVEY.md 9.1); all copies are identical, so the numbers are
    those of a correctly indexed call.
"""
import math

import torch
import torch.nn.functional as F
from torch import nn

from . import _lib
from .deformable_transformer import DeformableTransformer as _SingleFrameTransformer
from .ops.functions import norm_act
from .transformer_layers import (DeformableTransformerDecoderLayer, TemporalDeformableTransformerDecoder,
                                 _get_activation_fn, _get_clones, inverse_sigmoid, mha_batch_first)

_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.float64: _lib.DTYPE_F64, torch.bfloat16: _lib.DTYPE_BF16,
           torch.float16: _lib.DTYPE_F16}


def bbox2roi(bbox_list):
    """List of per-image ``[n_i, 4]`` boxes -> ``[sum n_i, 5]`` rows (batch index, x1, y1, x2, y2)
    (reference :48-67)."""
    rois = []
    for img_id, boxes in enumerate(bbox_list):
        boxes = getattr(boxes, "tensor", boxes)
        rois.append(torch.cat([boxes.new_full((boxes.size(0), 1), img_id), boxes], dim=-1))
    return torch.cat(rois, 0)


def box_cxcywh_to_xyxy(x):
    """/root/reference/util/box_ops.py:15-19."""
    cx, cy, w, h = x.unbind(-1)
    return torch.stack([cx - 0.5 * w, cy - 0.5 * h, cx + 0.5 * w, cy + 0.5 * h], dim=-1)


class _RoIAlignTokens(torch.autograd.Function):
    """tokens [N, H*W, C] , rois [K, 5] -> pooled [K, PH*PW, C]; gradient w.r.t. the tokens only (mmcv's
    RoIAlignFunction.backward returns None for the rois as well)."""

    @staticmethod
    def forward(ctx, tokens, rois, height, width, pooled, scale, sampling_ratio, aligned):
        if not tokens.is_cuda:
            raise RuntimeError("Not implemented on the CPU")      # same refusal as the deformable attention op
        if tokens.dtype not in _DTYPES:
            raise RuntimeError(f"roi_align: unsupported dtype {tokens.dtype}")
        n, hw, c = tokens.shape
        if hw != height * width:
            raise RuntimeError(f"roi_align: {hw} tokens do not form a {height} x {width} map")
        if rois.dim() != 2 or rois.size(1) != 5:
            raise RuntimeError("roi_align: rois must be [K, 5] rows of (batch index, x1, y1, x2, y2)")
        tokens = tokens.contiguous()
        rois = rois.detach().to(device=tokens.device,
                                dtype=torch.float64 if tokens.dtype == torch.float64 else torch.float32).contiguous()
        ph, pw = pooled
        out = torch.empty((rois.size(0), ph * pw, c), dtype=tokens.dtype, device=tokens.device)
        with torch.cuda.device(tokens.device):
            code = _lib.load().msda_roi_align_forward(
                _DTYPES[tokens.dtype], tokens.data_ptr(), rois.data_ptr(), n, height, width, c, rois.size(0), ph, pw,
                float(scale), int(sampling_ratio), int(bool(aligned)), out.data_ptr(),
                torch.cuda.current_stream().cuda_stream)
        _lib.check(code, "msda_roi_align_forward")
        ctx.save_for_backward(rois)
        ctx.geom = (n, height, width, c, ph, pw, float(scale), int(sampling_ratio), int(bool(aligned)), tokens.dtype)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        (rois,) = ctx.saved_tensors
        n, height, width, c, ph, pw, scale, sampling_ratio, aligned, dtype = ctx.geom
        grad_out = grad_out.contiguous()
        args = (_DTYPES[dtype], grad_out.data_ptr(), rois.data_ptr(), n, height, width, c, rois.size(0), ph, pw,
                scale, sampling_ratio, aligned)
        with torch.cuda.device(grad_out.device):
            stream = torch.cuda.current_stream().cuda_stream
            if torch.are_deterministic_algorithms_enabled():
                # fixed-point accumulation, bitwise reproducible (DESIGN.md section 3.15), written in the dtype
                grad = torch.empty((n, height * width, c), dtype=dtype, device=grad_out.device)
                scratch = _lib.deterministic_scratch(grad_out.device, grad.numel())
                code = _lib.load().msda_roi_align_backward_deterministic(*args, grad.data_ptr(), scratch.data_ptr(),
                                                                         scratch.numel(), stream)
                _lib.check(code, "msda_roi_align_backward_deterministic")
                return grad, None, None, None, None, None, None, None
            acc_dtype = torch.float64 if dtype == torch.float64 else torch.float32
            accum = torch.zeros((n, height * width, c), dtype=acc_dtype, device=grad_out.device)
            code = _lib.load().msda_roi_align_backward(*args, accum.data_ptr(), stream)
        _lib.check(code, "msda_roi_align_backward")
        return accum.to(dtype), None, None, None, None, None, None, None


def roi_align_tokens(tokens, rois, height, width, output_size, spatial_scale=1.0, sampling_ratio=0, aligned=True):
    """RoIAlign ('avg') of token-major maps: ``tokens [N, H*W, C]`` -> ``[K, PH*PW, C]``."""
    pooled = (output_size, output_size) if isinstance(output_size, int) else tuple(output_size)
    return _RoIAlignTokens.apply(tokens, rois, int(height), int(width), pooled, spatial_scale, sampling_ratio, aligned)


class RoIAlign(nn.Module):
    """Drop-in for ``mmcv.ops.RoIAlign`` as the reference builds it (:129-132): same constructor, same
    ``forward(input [N,C,H,W], rois [K,5]) -> [K,C,PH,PW]``.  ``forward_tokens`` is the copy-free entry the
    temporal stage uses.  pool_mode 'max' is not part of the reference's use and raises."""

    def __init__(self, output_size, spatial_scale=1.0, sampling_ratio=0, pool_mode="avg", aligned=True,
                 use_torchvision=False):
        super().__init__()
        if pool_mode != "avg":
            raise NotImplementedError("RoIAlign: only pool_mode='avg' (the mode the reference uses) is implemented")
        self.output_size = (output_size, output_size) if isinstance(output_size, int) else tuple(output_size)
        self.spatial_scale = float(spatial_scale)
        self.sampling_ratio = int(sampling_ratio)
        self.pool_mode = pool_mode
        self.aligned = aligned
        self.use_torchvision = use_torchvision

    def pooling_args(self):
        return self.output_size, self.spatial_scale, self.sampling_ratio, self.aligned

    def forward_tokens(self, tokens, rois, height, width):
        return roi_align_tokens(tokens, rois, height, width, *self.pooling_args())

    def forward(self, input, rois):
        n, c, h, w = input.shape
        tokens = input.permute(0, 2, 3, 1).reshape(n, h * w, c)       # free when input is a view of token-major memory
        out = self.forward_tokens(tokens, rois, h, w)
        return out.view(-1, self.output_size[0], self.output_size[1], c).permute(0, 3, 1, 2)

    def __repr__(self):
        return (f"{self.__class__.__name__}(output_size={self.output_size}, spatial_scale={self.spatial_scale}, "
                f"sampling_ratio={self.sampling_ratio}, pool_mode={self.pool_mode}, aligned={self.aligned})")


class DynamicConv(nn.Module):
    """head.py:134-173: two per-box 1x1 'convolutions' whose weights are generated from the box's query."""

    def __init__(self, cfg):
        super().__init__()
        self.hidden_dim = cfg['MODEL']['SparseRCNN']['HIDDEN_DIM']
        self.dim_dynamic = cfg['MODEL']['SparseRCNN']['DIM_DYNAMIC']
        self.num_dynamic = cfg['MODEL']['SparseRCNN']['NUM_DYNAMIC']
        self.num_params = self.hidden_dim * self.dim_dynamic
        self.dynamic_layer = nn.Linear(self.hidden_dim, self.num_dynamic * self.num_params)
        self.norm1 = nn.LayerNorm(self.dim_dynamic)
        self.norm2 = nn.LayerNorm(self.hidden_dim)
        self.activation = nn.ReLU(inplace=True)
        pooler_resolution = cfg['MODEL']['ROI_BOX_HEAD']['POOLER_RESOLUTION']
        self.out_layer = nn.Linear(self.hidden_dim * pooler_resolution ** 2, self.hidden_dim)
        self.norm3 = nn.LayerNorm(self.hidden_dim)

    def forward(self, pro_features, roi_features):
        """pro_features [1, K, C]; roi_features [49, K, C] (the reference's layout) -- see ``forward_tokens``."""
        return self.forward_tokens(pro_features, roi_features.permute(1, 0, 2))

    def forward_tokens(self, pro_features, pooled):
        """pooled [K, 49, C]: what ``RoIAlign.forward_tokens`` writes."""
        parameters = self.dynamic_layer(pro_features).permute(1, 0, 2)
        param1 = parameters[:, :, :self.num_params].view(-1, self.hidden_dim, self.dim_dynamic)
        param2 = parameters[:, :, self.num_params:].view(-1, self.dim_dynamic, self.hidden_dim)
        # normalise + ReLU as one in-place kernel each when no gradient is needed (ops/functions: norm_act)
        features = norm_act(self.norm1, torch.bmm(pooled, param1), "relu", inplace=True)
        features = norm_act(self.norm2, torch.bmm(features, param2), "relu", inplace=True)
        features = self.out_layer(features.flatten(1))
        return norm_act(self.norm3, features, "relu", inplace=True)


_DEFAULT_SCALE_CLAMP = math.log(100000.0 / 16)


class RCNNHead(nn.Module):
    """head.py:31-91 (QRF): self-attention over a frame's queries, dynamic interaction with each query's pooled
    patch, feed-forward.  ``forward(roi_features, pro_features)`` accepts the reference's ``[K, C, 7, 7]`` patches
    or the token-major ``[K, 49, C]`` ones."""

    def __init__(self, cfg, d_model, num_classes, dim_feedforward=2048, nhead=8, dropout=0.1, activation="relu",
                 scale_clamp=_DEFAULT_SCALE_CLAMP, bbox_weights=(2.0, 2.0, 1.0, 1.0)):
        super().__init__()
        self.d_model = d_model
        self.self_attn = nn.MultiheadAttention(d_model, nhead, dropout=dropout)
        self.inst_interact = DynamicConv(cfg)
        self.linear1 = nn.Linear(d_model, dim_feedforward)
        self.dropout = nn.Dropout(dropout)
        self.linear2 = nn.Linear(dim_feedforward, d_model)
        self.norm1 = nn.LayerNorm(d_model)
        self.norm2 = nn.LayerNorm(d_model)
        self.norm3 = nn.LayerNorm(d_model)
        self.dropout1 = nn.Dropout(dropout)
        self.dropout2 = nn.Dropout(dropout)
        self.dropout3 = nn.Dropout(dropout)
        self.activation = _get_activation_fn(activation)
        self.scale_clamp = scale_clamp
        self.bbox_weights = bbox_weights

    def forward(self, roi_features, pro_features):
        N, nr_boxes = pro_features.shape[:2]
        if roi_features.dim() == 4:                                    # [K, C, 7, 7] (reference layout)
            pooled = roi_features.flatten(2).transpose(1, 2)
        else:                                                          # [K, 49, C]
            pooled = roi_features
        pro = pro_features.reshape(N, nr_boxes, self.d_model)                 # batch-first: no [boxes, N, C] round trip
        pro = self.norm1(pro + self.dropout1(mha_batch_first(self.self_attn, pro, pro, pro)))
        pro = pro.reshape(1, N * nr_boxes, self.d_model)
        obj = self.norm2(pro + self.dropout2(self.inst_interact.forward_tokens(pro, pooled)))
        obj2 = self.linear2(self.dropout(self.activation(self.linear1(obj))))
        return self.norm3(obj + self.dropout3(obj2))

    def apply_deltas(self, deltas, boxes):
        """head.py:93-131 (box decoding of SparseRCNN; kept for API completeness, unused by the reference)."""
        boxes = boxes.to(deltas.dtype)
        widths = boxes[:, 2] - boxes[:, 0]
        heights = boxes[:, 3] - boxes[:, 1]
        ctr_x = boxes[:, 0] + 0.5 * widths
        ctr_y = boxes[:, 1] + 0.5 * heights
        wx, wy, ww, wh = self.bbox_weights
        dx, dy = deltas[:, 0::4] / wx, deltas[:, 1::4] / wy
        dw = torch.clamp(deltas[:, 2::4] / ww, max=self.scale_clamp)
        dh = torch.clamp(deltas[:, 3::4] / wh, max=self.scale_clamp)
        pred_ctr_x = dx * widths[:, None] + ctr_x[:, None]
        pred_ctr_y = dy * heights[:, None] + ctr_y[:, None]
        pred_w = torch.exp(dw) * widths[:, None]
        pred_h = torch.exp(dh) * heights[:, None]
        pred = torch.zeros_like(deltas)
        pred[:, 0::4] = pred_ctr_x - 0.5 * pred_w
        pred[:, 1::4] = pred_ctr_y - 0.5 * pred_h
        pred[:, 2::4] = pred_ctr_x + 0.5 * pred_w
        pred[:, 3::4] = pred_ctr_y + 0.5 * pred_h
        return pred


class TemporalQueryEncoderLayer(nn.Module):
    """:787-837 (TQE): self-attention over the current frame's queries, cross-attention to the selected
    reference-frame queries, feed-forward."""

    def __init__(self, d_model=256, d_ffn=1024, dropout=0.1, activation="relu", n_heads=8):
        super().__init__()
        self.self_attn = nn.MultiheadAttention(d_model, n_heads, dropout=dropout)
        self.dropout2 = nn.Dropout(dropout)
        self.norm2 = nn.LayerNorm(d_model)
        self.cross_attn = nn.MultiheadAttention(d_model, n_heads, dropout=dropout)
        self.dropout1 = nn.Dropout(dropout)
        self.norm1 = nn.LayerNorm(d_model)
        self.linear1 = nn.Linear(d_model, d_ffn)
        self.activation = _get_activation_fn(activation)
        self.dropout3 = nn.Dropout(dropout)
        self.linear2 = nn.Linear(d_ffn, d_model)
        self.dropout4 = nn.Dropout(dropout)
        self.norm3 = nn.LayerNorm(d_model)

    @staticmethod
    def with_pos_embed(tensor, pos):
        return tensor if pos is None else tensor + pos

    def forward_ffn(self, tgt):
        tgt2 = self.linear2(self.dropout3(self.activation(self.linear1(tgt))))
        return self.norm3(tgt + self.dropout4(tgt2))

    def forward(self, query, ref_query, query_pos=None, ref_query_pos=None):
        q = self.with_pos_embed(query, query_pos)
        tgt2 = mha_batch_first(self.self_attn, q, q, query)
        tgt = self.norm2(query + self.dropout2(tgt2))
        tgt2 = mha_batch_first(self.cross_attn, self.with_pos_embed(tgt, query_pos),
                               self.with_pos_embed(ref_query, ref_query_pos), ref_query)
        tgt = self.norm1(tgt + self.dropout1(tgt2))
        return self.forward_ffn(tgt)


class TemporalQueryEncoder(nn.Module):
    """:840-850."""

    def __init__(self, encoder_layer, num_layers):
        super().__init__()
        self.layers = _get_clones(encoder_layer, num_layers)
        self.num_layers = num_layers

    def forward(self, query, ref_query, query_pos=None, ref_query_pos=None):
        output = query
        for layer in self.layers:
            output = layer(output, ref_query, query_pos, ref_query_pos)
        return output


class DeformableTransformer(_SingleFrameTransformer):
    """TransVOD++ multi-frame transformer (:70-603).  The frames of a clip -- current frame first, then
    ``num_ref_frames`` reference frames -- are the batch dimension of the per-frame encoder / decoder (inherited,
    identical to the single-frame transformer); the temporal query stage then refines the CURRENT frame's queries.

    forward(...) -> (hs[:, 0:1], init_reference[0:1], inter_references[:, 0:1], None, None, final_hs,
                     final_references, {'aux_outputs': [...]})                                         (:593)
    """

    TOPK_PER_REF_FRAME = (80, 50, 30)          # :531, :556, :579

    def __init__(self, d_model=256, nhead=8, num_encoder_layers=6, num_decoder_layers=6, dim_feedforward=1024,
                 dropout=0.1, activation="relu", return_intermediate_dec=False, num_feature_levels=4,
                 dec_n_points=4, enc_n_points=4, two_stage=False, two_stage_num_proposals=300, num_query=300,
                 n_temporal_decoder_layers=1, num_ref_frames=3, fixed_pretrained_model=False, args=None,
                 use_depth=False, depth_type='', dpth_feature_levels=1, dpth_n_points=4):
        self._temporal_cfg = dict(d_model=d_model, nhead=nhead, dim_feedforward=dim_feedforward, dropout=dropout,
                                  activation=activation, num_feature_levels=num_feature_levels,
                                  dec_n_points=dec_n_points, n_temporal_decoder_layers=n_temporal_decoder_layers)
        self.num_ref_frames = num_ref_frames
        self.fixed_pretrained_model = fixed_pretrained_model
        self.n_temporal_query_layers = 3
        self.num_query = num_query
        super().__init__(d_model, nhead, num_encoder_layers, num_decoder_layers, dim_feedforward, dropout, activation,
                         return_intermediate_dec, num_feature_levels, dec_n_points, enc_n_points, two_stage,
                         two_stage_num_proposals, use_depth, depth_type, dpth_feature_levels, dpth_n_points)

    def _build_extra_modules(self):
        """Called by the base constructor before ``_reset_parameters`` so that the temporal modules get the same
        xavier / LayerNorm / MSDeformAttn initialisation pass as in the reference (:174-188)."""
        t = self._temporal_cfg
        d_model, nhead, dff, dropout, activation = t["d_model"], t["nhead"], t["dim_feedforward"], t["dropout"], t["activation"]
        self.temporal_roi_layers1 = nn.ModuleList(
            [RoIAlign(output_size=7, sampling_ratio=2, spatial_scale=1 / s) for s in [32]])              # :129-132
        self.cfg = {"MODEL": {"SparseRCNN": {"NHEADS": 8, "DROPOUT": 0.0, "DIM_FEEDFORWARD": 2048, "ACTIVATION": 'relu',
                                             "HIDDEN_DIM": d_model, "NUM_CLS": 1, "NUM_REG": 3, "NUM_HEADS": 6,
                                             "NUM_DYNAMIC": 2, "DIM_DYNAMIC": 64},
                              "ROI_BOX_HEAD": {'POOLER_RESOLUTION': 7}}}                                   # :138-145
        for i in (1, 2, 3):
            setattr(self, f"temporal_query_layer{i}", TemporalQueryEncoderLayer(d_model, dff, dropout, activation, nhead))
        for i in (1, 2, 3):
            setattr(self, f"dynamic_layer_for_current_query{i}",
                    RCNNHead(self.cfg, d_model, 3, dff, nhead, dropout, activation))
        decoder_layer = DeformableTransformerDecoderLayer(d_model, dff, dropout, activation, t["num_feature_levels"],
                                                          nhead, t["dec_n_points"])
        for i in (1, 2, 3):
            setattr(self, f"temporal_decoder{i}",
                    TemporalDeformableTransformerDecoder(decoder_layer, t["n_temporal_decoder_layers"], False))

    # ------------------------------------------------------------------------------------------
    def forward(self, srcs, masks, pos_embeds, depth_srcs, depth_masks, depth_pos_embeds, imgs_whwh_shape,
                query_embed=None, class_embed=None, cur_bbox_embed=None, temp_class_embed_list=None,
                temp_bbox_embed_list=None, rgbd_query=[]):
        """The batch is one clip -- current frame first, then ``num_ref_frames`` reference frames -- exactly as in the
        reference, or SEVERAL clips laid out clip-major (``[clip0 cur, clip0 refs..., clip1 cur, ...]``): every
        module of the temporal stage treats clips as independent batch elements, so a GPU's share of clips runs as
        one set of launches.  With several clips every returned "current frame" tensor has one entry per clip where
        the reference has exactly one, and ``imgs_whwh_shape`` may hold one (w, h, w, h) row per clip."""
        hs, init_reference_out, inter_references, enc_cls, enc_coord, state = super().forward(
            srcs, masks, pos_embeds, depth_srcs, depth_masks, depth_pos_embeds, query_embed, rgbd_query,
            _return_state=True)
        if self.two_stage:                                                                              # :394-395
            return hs, init_reference_out, inter_references, enc_cls, enc_coord
        memory, lvl_pos, spatial_shapes, level_start_index, valid_ratios, shapes = state
        if self.fixed_pretrained_model:                                                                 # :397-401
            memory, hs, inter_references = memory.detach(), hs.detach(), inter_references.detach()

        frames = self.num_ref_frames + 1
        batch, tokens, c = memory.shape
        if batch % frames != 0:
            raise RuntimeError(f"batch of {batch} frames is not a whole number of {frames}-frame clips")
        clips = batch // frames
        h, w = shapes[-1]                                   # the reference keeps the LAST level's (h, w) (:270-276)
        if tokens != h * w:
            raise RuntimeError("TransVOD++ temporal stage needs ONE feature level: the reference views the whole "
                               "memory as a single (h, w) map (deformable_transformer_multi_plusplus.py:498)")
        device = memory.device
        imgs_whwh = torch.as_tensor(imgs_whwh_shape, dtype=torch.long, device=device).reshape(-1, 1, 4)   # :287-288
        if imgs_whwh.shape[0] not in (1, clips):
            raise RuntimeError("imgs_whwh_shape must hold one (w, h, w, h) row, or one per clip")
        if imgs_whwh.shape[0] == clips and clips > 1:
            imgs_whwh = imgs_whwh.repeat_interleave(frames, 0)

        last_hs = hs[-1]                                    # [clips*frames, Q, C]
        last_ref = inter_references[-1]                     # [clips*frames, Q, 2|4]
        nq = last_hs.shape[1]
        by_clip = lambda t: t.view(clips, frames, *t.shape[1:])
        cur_memory = by_clip(memory)[:, 0]                  # [clips, HW, C]
        cur_reference_out = by_clip(last_ref)[:, 0]         # [clips, Q, 2|4]

        # class scores of the reference-frame queries (:457-470) and boxes of every frame (:475-491): one batched
        # call each instead of a python loop per frame
        ref_prob = class_embed(by_clip(last_hs)[:, 1:]).sigmoid().reshape(clips, self.num_ref_frames * nq, -1)
        boxes = (cur_bbox_embed(last_hs) + inverse_sigmoid(last_ref)).sigmoid()            # (cx, cy, w, h)
        boxes_xyxy = box_cxcywh_to_xyxy(boxes) * imgs_whwh                                 # image units

        # RoI features + query / RoI fusion.  Current frame: memory (:498-501); reference frames: memory + position
        # embedding (:418-423, :511-517).  Each frame pools from its own map: roi batch index = frame.
        if frames > 1:              # one fused multiply-add: position embedding on the reference frames only
            is_ref = (torch.arange(batch, device=device) % frames != 0).to(memory.dtype).view(batch, 1, 1)
            maps = torch.addcmul(memory, lvl_pos, is_ref)
        else:
            maps = memory
        frame_index = torch.arange(batch, device=device, dtype=boxes_xyxy.dtype).repeat_interleave(nq)
        rois = torch.cat([frame_index[:, None], boxes_xyxy.reshape(batch * nq, 4)], -1)    # = bbox2roi per frame
        pooled = roi_align_tokens(maps, rois, h, w, *self.temporal_roi_layers1[0].pooling_args())   # [batch*Q, 49, C]
        enhanced = self.dynamic_layer_for_current_query1(pooled, last_hs).view(clips, frames * nq, c)
        cur_hs = enhanced[:, :nq]
        ref_hs_concat = enhanced[:, nq:]

        vr = by_clip(valid_ratios)[:, 0, 0:1]                                              # see module docstring
        # one level (checked above), so the reference's spatial_shapes[0:1] / level_start_index[0:1] (:539) are the
        # tensors themselves; passing them unsliced keeps the per-tensor host-shape cache (no D2H copy, graph-safe)
        scores = ref_prob[:, :, 1]
        out = {"aux_outputs": []}
        final_hs = final_references_out = None
        for stage, per_frame in enumerate(self.TOPK_PER_REF_FRAME):
            topk_indexes = torch.topk(scores, per_frame * self.num_ref_frames, dim=1)[1]
            ref_in = torch.gather(ref_hs_concat, 1, topk_indexes.unsqueeze(-1).expand(-1, -1, c))
            cur_hs = getattr(self, f"temporal_query_layer{stage + 1}")(cur_hs, ref_in)
            cur_hs, refs_out = getattr(self, f"temporal_decoder{stage + 1}")(
                cur_hs, cur_reference_out, cur_memory, spatial_shapes, level_start_index, vr, None, None)
            if stage < 2:                                                                  # :544-553, :567-576
                reference = inverse_sigmoid(refs_out if stage == 0 else cur_reference_out)
                tmp = temp_bbox_embed_list[stage](cur_hs)
                if reference.shape[-1] == 4:
                    tmp = tmp + reference
                else:
                    assert reference.shape[-1] == 2
                    tmp = torch.cat([tmp[..., :2] + reference, tmp[..., 2:]], -1)
                out["aux_outputs"].append({"pred_logits": temp_class_embed_list[stage](cur_hs),
                                           "pred_boxes": tmp.sigmoid()})
            else:
                final_hs, final_references_out = cur_hs, refs_out
        cur = slice(0, batch, frames)                       # the current frame of every clip (0:1 for one clip)
        return (hs[:, cur], init_reference_out[cur], inter_references[:, cur], None, None, final_hs,
                final_references_out, out)


class TransVODDeformableTransformer(_SingleFrameTransformer):
    """TransVOD multi-frame transformer (the reference's ``DeformableTransformer`` of
    /root/reference/models/deformable_transformer_multi.py:24-379; TransVOD++ above adds RoIAlign + QRF to it).
    Frames of a clip -- current first -- are the batch of the per-frame encoder / decoder; then three temporal query
    encoder rounds over the top 80 / 50 / 30 (x num_ref_frames) reference-frame queries ranked by their best
    non-background class score (:352-368), and ONE temporal deformable decoder over the current frame's memory (:371).
    Same constructor, forward signature and parameter names (``temporal_encoder_layer`` -- the frames-as-levels
    layer, built but unused because the reference hard-codes ``self.TDAM = False`` (:46) --,
    ``temporal_query_layer{1,2,3}``, ``temporal_decoder``).  Clips batch clip-major like the TransVOD++ class, and
    the temporal decoder gets ``valid_ratios[:, 0:1]`` (SURVEY.md 9.1).

    forward(...) -> (hs[:, 0:1], init_reference[0:1], inter_references[:, 0:1], None, None, final_hs,
                     final_references)                                                                 (:374)
    """

    TOPK_PER_REF_FRAME = (80, 50, 30)

    def __init__(self, d_model=256, nhead=8, num_encoder_layers=6, num_decoder_layers=6, dim_feedforward=1024,
                 dropout=0.1, activation="relu", return_intermediate_dec=False, num_feature_levels=4,
                 dec_n_points=4, enc_n_points=4, two_stage=False, two_stage_num_proposals=300,
                 n_temporal_decoder_layers=1, num_ref_frames=3, fixed_pretrained_model=False, args=None,
                 use_depth=False, depth_type='', dpth_feature_levels=1, dpth_n_points=4):
        self._temporal_cfg = dict(d_model=d_model, nhead=nhead, dim_feedforward=dim_feedforward, dropout=dropout,
                                  activation=activation, num_feature_levels=num_feature_levels,
                                  dec_n_points=dec_n_points, enc_n_points=enc_n_points,
                                  n_temporal_decoder_layers=n_temporal_decoder_layers)
        self.num_ref_frames = num_ref_frames
        self.fixed_pretrained_model = fixed_pretrained_model
        self.n_temporal_query_layers = 3
        self.TDAM = False                                                                                # :46
        super().__init__(d_model, nhead, num_encoder_layers, num_decoder_layers, dim_feedforward, dropout, activation,
                         return_intermediate_dec, num_feature_levels, dec_n_points, enc_n_points, two_stage,
                         two_stage_num_proposals, use_depth, depth_type, dpth_feature_levels, dpth_n_points)

    def _build_extra_modules(self):
        from .transformer_layers import TemporalDeformableTransformerEncoderLayer
        t = self._temporal_cfg
        d_model, nhead, dff, dropout, activation = t["d_model"], t["nhead"], t["dim_feedforward"], t["dropout"], t["activation"]
        self.temporal_encoder_layer = TemporalDeformableTransformerEncoderLayer(
            d_model, dff, dropout, activation, self.num_ref_frames, nhead, t["enc_n_points"])            # :84-86
        for i in (1, 2, 3):
            setattr(self, f"temporal_query_layer{i}", TemporalQueryEncoderLayer(d_model, dff, dropout, activation, nhead))
        decoder_layer = DeformableTransformerDecoderLayer(d_model, dff, dropout, activation, t["num_feature_levels"],
                                                          nhead, t["dec_n_points"])
        self.temporal_decoder = TemporalDeformableTransformerDecoder(decoder_layer, t["n_temporal_decoder_layers"], False)

    def forward(self, srcs, masks, pos_embeds, depth_srcs, depth_masks, depth_pos_embeds, query_embed=None,
                class_embed=None, rgbd_query=[]):
        hs, init_reference_out, inter_references, enc_cls, enc_coord, state = super().forward(
            srcs, masks, pos_embeds, depth_srcs, depth_masks, depth_pos_embeds, query_embed, rgbd_query,
            _return_state=True)
        if self.two_stage:                                                                              # :318-319
            return hs, init_reference_out, inter_references, enc_cls, enc_coord
        memory, lvl_pos, spatial_shapes, level_start_index, valid_ratios, shapes = state
        if self.fixed_pretrained_model:                                                                 # :321-325
            memory, hs, inter_references = memory.detach(), hs.detach(), inter_references.detach()

        frames = self.num_ref_frames + 1
        batch, tokens, c = memory.shape
        if batch % frames != 0:
            raise RuntimeError(f"batch of {batch} frames is not a whole number of {frames}-frame clips")
        clips = batch // frames
        by_clip = lambda t: t.view(clips, frames, *t.shape[1:])
        cur_memory = by_clip(memory)[:, 0]
        if self.TDAM:                                       # frames-as-levels attention of the current frame (:328-343)
            if len(shapes) != 1:
                raise RuntimeError("the temporal encoder layer treats the reference FRAMES as levels: one feature level")
            ref_memory = (by_clip(memory)[:, 1:] + by_clip(lvl_pos)[:, 1:]).reshape(clips, self.num_ref_frames * tokens, c)
            ref_shapes = spatial_shapes.expand(self.num_ref_frames, 2).contiguous()
            frame_start = torch.cat((ref_shapes.new_zeros((1,)), ref_shapes.prod(1).cumsum(0)[:-1])).contiguous()
            # the current frame's pixel grid, once per reference frame (the reference gets there by expanding the
            # valid ratios to num_ref_frames pseudo-levels, :336-338)
            ref_points = self.get_reference_points([shapes[0]], by_clip(valid_ratios)[:, 0, 0:1], device=memory.device)
            ref_points = ref_points.expand(-1, -1, self.num_ref_frames, -1).contiguous()
            cur_memory = self.temporal_encoder_layer(cur_memory, by_clip(lvl_pos)[:, 0], ref_points, ref_memory,
                                                     ref_shapes, frame_start)

        last_hs, last_ref = by_clip(hs[-1]), by_clip(inter_references[-1])
        nq = last_hs.shape[2]
        cur_hs, cur_reference_out = last_hs[:, 0], last_ref[:, 0]
        ref_hs = last_hs[:, 1:].reshape(clips, self.num_ref_frames * nq, c)
        prob = class_embed(ref_hs).sigmoid()
        n_cls = prob.shape[2] - 1                                                   # the last class is left out (:353)
        scores = prob[:, :, :-1].reshape(clips, -1)
        for stage, per_frame in enumerate(self.TOPK_PER_REF_FRAME):
            topk_indexes = torch.topk(scores, per_frame * self.num_ref_frames, dim=1)[1] // n_cls
            ref_in = torch.gather(ref_hs, 1, topk_indexes.unsqueeze(-1).expand(-1, -1, c))
            cur_hs = getattr(self, f"temporal_query_layer{stage + 1}")(cur_hs, ref_in)
        vr = by_clip(valid_ratios)[:, 0, 0:1]
        final_hs, final_references_out = self.temporal_decoder(
            cur_hs, cur_reference_out, cur_memory, spatial_shapes[0:1] if len(shapes) > 1 else spatial_shapes,
            level_start_index[0:1] if len(shapes) > 1 else level_start_index, vr, None, None)
        cur = slice(0, batch, frames)
        return (hs[:, cur], init_reference_out[cur], inter_references[:, cur], None, None, final_hs,
                final_references_out)


def build_deforamble_transformer(args):
    """Same (misspelt) name and argument mapping as the reference builder (:1145-1170)."""
    return DeformableTransformer(
        d_model=args.hidden_dim, nhead=args.nheads, num_encoder_layers=args.enc_layers,
        num_decoder_layers=args.dec_layers, dim_feedforward=args.dim_feedforward, dropout=args.dropout,
        activation="relu", return_intermediate_dec=True, num_feature_levels=args.num_feature_levels,
        dec_n_points=args.dec_n_points, enc_n_points=args.enc_n_points, two_stage=args.two_stage,
        two_stage_num_proposals=args.num_queries, num_query=args.num_queries,
        n_temporal_decoder_layers=args.n_temporal_decoder_layers, num_ref_frames=args.num_ref_frames,
        fixed_pretrained_model=args.fixed_pretrained_model, args=args, use_depth=args.use_depth,
        depth_type=args.depth_type, dpth_n_points=args.dpth_n_points)
