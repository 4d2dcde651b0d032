"""Deformable DETR's Hungarian matcher and set criterion, with the assignment solved on the device.

Mirrors the reference's ``models/matcher.py`` (``HungarianMatcher``) and ``SetCriterion`` in
``models/deformable_detr_single.py``: same class names, constructor arguments, ``forward`` and loss-dict keys.  The
cost matrix is computed with the reference's torch ops in the reference's order; the reference then calls ``.cpu()``
and ``scipy.optimize.linear_sum_assignment`` per image and head, and ``.item()`` on the box count.  Here every
(image, head) problem goes to one launch of the batched solver in ``csrc/hungarian.cu`` (DESIGN.md section 3.17) and
the box count stays on the device, so the criterion issues no device-to-host copy and can be captured in a CUDA graph
(``data_parallel.GraphedTrainStep``) when the targets come in the padded form of ``pad_targets``.

Deviations from the reference:
  * ``HungarianMatcher.forward`` returns the ``(i, j)`` int64 pairs on the device of the predictions, not on the CPU.
  * An image may not have more boxes than a head has queries (scipy would leave the extra boxes unmatched).
  * A NaN or infinite matching cost does not raise (scipy's ``ValueError`` needs a sync): every loss of the head it
    occurs in, and its gradient, becomes NaN.
  * The ``masks`` loss (segmentation head) is not provided.
"""
import collections

import torch
import torch.distributed as dist
import torch.nn.functional as F
from torch import nn

from . import _lib

__all__ = ["HungarianMatcher", "SetCriterion", "PaddedTargets", "pad_targets", "linear_assignment",
           "sigmoid_focal_loss", "generalized_box_iou", "box_cxcywh_to_xyxy"]

PaddedTargets = collections.namedtuple("PaddedTargets", ["labels", "boxes", "counts"])
PaddedTargets.__doc__ = """Targets of a batch in static shapes: ``labels`` [B, T_max] int64, ``boxes`` [B, T_max, 4]
(normalised cx, cy, w, h), ``counts`` [B] int64.  Entries at and after ``counts[b]`` are padding."""

Matching = collections.namedtuple("Matching", ["query_of_target", "target_of_query", "status"])

# padding box: the whole image, so that GIoU against any prediction is finite and so is its (unused) gradient
_DUMMY_BOX = (0.5, 0.5, 1.0, 1.0)


def pad_targets(targets, max_boxes):
    """Pack the reference's list of ``{"labels": [T_b], "boxes": [T_b, 4]}`` dicts into ``PaddedTargets`` with
    ``T_max = max_boxes``.  A graphed training step captured once on such buffers takes batches of any box counts
    up to ``max_boxes`` (images without boxes too) by copying new ``pad_targets`` results into them.  Checks the
    shapes, that labels are non-negative integers and that boxes are finite with non-negative width and height;
    the value checks read the tensors, so call it where the data is prepared, outside the captured step."""
    padded = _pack(targets, max_boxes)
    for b, t in enumerate(targets):
        if len(t["labels"]):
            if bool((t["labels"] < 0).any()):
                raise ValueError(f"image {b}: negative label")
            box = t["boxes"]
            if not bool(torch.isfinite(box).all()) or bool((box[:, 2:] < 0).any()):
                raise ValueError(f"image {b}: boxes must be finite with non-negative width and height")
    return padded


def _pack(targets, max_boxes):
    """pad_targets without the value checks: shapes only, nothing read from the device."""
    max_boxes = int(max_boxes)
    if max_boxes < 1:
        raise ValueError(f"max_boxes must be at least 1, got {max_boxes}")
    if len(targets) == 0:
        raise ValueError("pad_targets needs at least one image")
    device = targets[0]["boxes"].device
    dtype = targets[0]["boxes"].dtype
    labels = torch.zeros(len(targets), max_boxes, dtype=torch.int64, device=device)
    boxes = torch.tensor(_DUMMY_BOX, dtype=dtype, device=device).repeat(len(targets), max_boxes, 1)
    counts = []
    for b, t in enumerate(targets):
        lab, box = t["labels"], t["boxes"]
        if lab.dim() != 1 or lab.dtype.is_floating_point or lab.dtype == torch.bool or lab.is_complex():
            raise ValueError(f"image {b}: labels must be a 1-D integer tensor, got {tuple(lab.shape)} {lab.dtype}")
        if box.dim() != 2 or box.shape[1] != 4 or box.shape[0] != lab.shape[0] or not box.dtype.is_floating_point:
            raise ValueError(f"image {b}: boxes must be a floating [{lab.shape[0]}, 4] tensor, got "
                             f"{tuple(box.shape)} {box.dtype}")
        n = lab.shape[0]
        if n > max_boxes:
            raise ValueError(f"image {b} has {n} boxes, more than max_boxes = {max_boxes}")
        labels[b, :n] = lab
        boxes[b, :n] = box
        counts.append(n)
    return PaddedTargets(labels, boxes, torch.tensor(counts, dtype=torch.int64, device=device))


def linear_assignment(cost, counts):
    """Solve ``cost[p, :, :counts[p]]`` ([P, Q, T_max], queries x targets) for every problem p in one launch of the
    sm_100a solver.  Every target is matched to a distinct query at the least total cost (scipy's
    ``linear_sum_assignment`` on the transposed matrix).  Returns ``Matching(query_of_target [P, T_max],
    target_of_query [P, Q], status [P])``, int32 on the device, -1 where nothing is matched; a non-zero status
    (NaN or Inf cost, count out of range) writes -1 for the whole problem.  Reads nothing back to the host."""
    if not cost.is_cuda:
        raise RuntimeError("linear_assignment: Not implemented on the CPU (the solver is an sm_100a kernel)")
    if cost.dim() != 3 or counts.shape != cost.shape[:1]:
        raise ValueError(f"cost must be [P, Q, T_max] and counts [P], got {tuple(cost.shape)} and "
                         f"{tuple(counts.shape)}")
    cost = cost.float()
    if cost.shape[2] > 1 and cost.stride(2) != 1:
        cost = cost.contiguous()
    counts = counts.to(device=cost.device, dtype=torch.int64).contiguous()
    p, q, t = cost.shape
    qot = torch.empty(p, t, dtype=torch.int32, device=cost.device)
    toq = torch.empty(p, q, dtype=torch.int32, device=cost.device)
    status = torch.empty(p, dtype=torch.int32, device=cost.device)
    lib = _lib.load()
    nbytes = lib.msda_linear_assignment_scratch_bytes(p, q, t)
    if nbytes < 0:
        raise _lib.MSDAError(f"msda_linear_assignment_scratch_bytes({p}, {q}, {t}) failed")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=cost.device)
    with torch.cuda.device(cost.device):
        _lib.check(lib.msda_linear_assignment(
            cost.data_ptr(), cost.stride(0), cost.stride(1), counts.data_ptr(), p, q, t, qot.data_ptr(),
            toq.data_ptr(), status.data_ptr(), scratch.data_ptr() if nbytes else None, nbytes,
            torch.cuda.current_stream().cuda_stream), "msda_linear_assignment")
    return Matching(qot, toq, status)


def box_cxcywh_to_xyxy(x):
    x_c, y_c, w, h = x.unbind(-1)
    return torch.stack([(x_c - 0.5 * w), (y_c - 0.5 * h), (x_c + 0.5 * w), (y_c + 0.5 * h)], dim=-1)


def _box_area(boxes):
    return (boxes[..., 2] - boxes[..., 0]) * (boxes[..., 3] - boxes[..., 1])


def generalized_box_iou(boxes1, boxes2):
    """GIoU of every pair, ``[..., N, 4] x [..., M, 4] -> [..., N, M]`` (xyxy), with the reference's ops
    (util/box_ops.py) but without its host-side degenerate-box asserts, which would sync."""
    return _giou(boxes1.unsqueeze(-2), boxes2.unsqueeze(-3))


def _giou(b1, b2):
    """GIoU of broadcast box pairs, elementwise in the reference's order of operations."""
    area1, area2 = _box_area(b1), _box_area(b2)
    lt = torch.max(b1[..., :2], b2[..., :2])
    rb = torch.min(b1[..., 2:], b2[..., 2:])
    wh = (rb - lt).clamp(min=0)
    inter = wh[..., 0] * wh[..., 1]
    union = area1 + area2 - inter
    iou = inter / union
    lt = torch.min(b1[..., :2], b2[..., :2])
    rb = torch.max(b1[..., 2:], b2[..., 2:])
    wh = (rb - lt).clamp(min=0)
    area = wh[..., 0] * wh[..., 1]
    return iou - (area - union) / area


def sigmoid_focal_loss(inputs, targets, num_boxes, alpha: float = 0.25, gamma: float = 2):
    """The reference's focal loss (RetinaNet), summed over classes, averaged over queries, divided by num_boxes."""
    prob = inputs.sigmoid()
    ce_loss = F.binary_cross_entropy_with_logits(inputs, targets, reduction="none")
    p_t = prob * targets + (1 - prob) * (1 - targets)
    loss = ce_loss * ((1 - p_t) ** gamma)
    if alpha >= 0:
        alpha_t = alpha * targets + (1 - alpha) * (1 - targets)
        loss = alpha_t * loss
    return loss.mean(1).sum() / num_boxes


def _pairs(target_of_query, lengths):
    """The reference's per-image ``(i, j)``: matched queries ascending and their targets, as int64 device tensors.
    Image b has exactly ``lengths[b]`` matches, so the split needs nothing from the device."""
    q = target_of_query.shape[1]
    ar = torch.arange(q, device=target_of_query.device)
    order = torch.where(target_of_query >= 0, ar, ar + q).argsort(dim=1)
    out = []
    for b, n in enumerate(lengths):
        i = order[b, :n]
        out.append((i, target_of_query[b].gather(0, i).long()))
    return out


class HungarianMatcher(nn.Module):
    """Optimal one-to-one matching of predictions to targets (reference: models/matcher.py).  The cost of matching
    query q to target t is ``cost_bbox * L1 + cost_class * focal-class-cost + cost_giou * (-GIoU)``."""

    def __init__(self, cost_class: float = 1, cost_bbox: float = 1, cost_giou: float = 1):
        super().__init__()
        self.cost_class = cost_class
        self.cost_bbox = cost_bbox
        self.cost_giou = cost_giou
        assert cost_class != 0 or cost_bbox != 0 or cost_giou != 0, "all costs cant be 0"

    @torch.no_grad()
    def cost(self, outputs, labels, boxes):
        """``[B, Q, T_max]`` matching costs of ``outputs`` against padded ``labels`` / ``boxes``; element by
        element the reference's values (the same ops on the same operands)."""
        out_prob = outputs["pred_logits"].sigmoid()
        out_bbox = outputs["pred_boxes"]
        alpha = 0.25
        gamma = 2.0
        neg_cost_class = (1 - alpha) * (out_prob ** gamma) * (-(1 - out_prob + 1e-8).log())
        pos_cost_class = alpha * ((1 - out_prob) ** gamma) * (-(out_prob + 1e-8).log())
        ids = labels.unsqueeze(1).expand(-1, out_prob.shape[1], -1)
        cost_class = pos_cost_class.gather(2, ids) - neg_cost_class.gather(2, ids)
        cost_bbox = torch.cdist(out_bbox, boxes.to(out_bbox.dtype), p=1)
        cost_giou = -generalized_box_iou(box_cxcywh_to_xyxy(out_bbox), box_cxcywh_to_xyxy(boxes.to(out_bbox.dtype)))
        return self.cost_bbox * cost_bbox + self.cost_class * cost_class + self.cost_giou * cost_giou

    @torch.no_grad()
    def match_padded(self, heads):
        """Match several heads at once: ``heads`` is a list of ``(outputs, labels, padded)``.  Heads with the same
        number of queries share one solver launch.  Returns one ``Matching`` per head."""
        groups = collections.OrderedDict()
        for h, (outputs, labels, padded) in enumerate(heads):
            q = outputs["pred_logits"].shape[1]
            if padded.labels.shape[1] > q:
                raise ValueError(f"{padded.labels.shape[1]} target slots for {q} queries: every target needs a "
                                 "query of its own (pad_targets max_boxes must not exceed the number of queries)")
            groups.setdefault(q, []).append(h)
        result = [None] * len(heads)
        for idx in groups.values():
            cost = torch.cat([self.cost(heads[h][0], heads[h][1], heads[h][2].boxes) for h in idx])
            counts = torch.cat([heads[h][2].counts for h in idx])
            m = linear_assignment(cost, counts)
            for k, h in enumerate(idx):
                b = heads[h][2].counts.shape[0]
                result[h] = Matching(*(x[k * b:(k + 1) * b] for x in m))
        return result

    @torch.no_grad()
    def forward(self, outputs, targets):
        """The reference's interface: ``targets`` is a list of ``{"labels", "boxes"}`` dicts; returns per image
        ``(index_i, index_j)`` int64 tensors on the predictions' device, ``index_i`` ascending."""
        lengths = [len(v["boxes"]) for v in targets]
        padded = _pack(targets, max(1, max(lengths)))
        padded = PaddedTargets(*(x.to(outputs["pred_logits"].device) for x in padded))
        m, = self.match_padded([(outputs, padded.labels, padded)])
        return _pairs(m.target_of_query, lengths)


class SetCriterion(nn.Module):
    """Deformable DETR's loss (reference: ``SetCriterion`` in models/deformable_detr_single.py): Hungarian
    matching of every head, then sigmoid focal classification, L1 and GIoU box losses per matched pair.

    ``forward(outputs, targets, num_boxes=None)`` takes the reference's list of target dicts, or ``PaddedTargets``
    (see ``pad_targets``), which keeps every shape static: with it the call reads nothing back to the host and a
    CUDA graph can capture it.  ``num_boxes`` is the box count the losses are divided by; by default the batch's
    count, summed over the ranks when ``torch.distributed`` is initialised, divided by the world size and clamped
    to at least 1, as in the reference, but kept on the device."""

    def __init__(self, num_classes, matcher, weight_dict, losses, focal_alpha=0.25):
        super().__init__()
        self.num_classes = num_classes
        self.matcher = matcher
        self.weight_dict = weight_dict
        self.losses = losses
        self.focal_alpha = focal_alpha
        for loss in losses:
            if loss not in ("labels", "cardinality", "boxes"):
                raise ValueError(f"unsupported loss {loss!r} (the masks loss is not provided)")

    def loss_labels(self, outputs, labels, padded, m, num_boxes, log=True):
        src_logits = outputs["pred_logits"]
        toq = m.target_of_query.long()
        matched = toq >= 0
        target_classes = torch.where(matched, labels.gather(1, toq.clamp(min=0)), self.num_classes)
        target_classes_onehot = torch.zeros([src_logits.shape[0], src_logits.shape[1], src_logits.shape[2] + 1],
                                            dtype=src_logits.dtype, layout=src_logits.layout,
                                            device=src_logits.device)
        target_classes_onehot.scatter_(2, target_classes.unsqueeze(-1), 1)
        target_classes_onehot = target_classes_onehot[:, :, :-1]
        loss_ce = sigmoid_focal_loss(src_logits, target_classes_onehot, num_boxes, alpha=self.focal_alpha,
                                     gamma=2) * src_logits.shape[1]
        losses = {"loss_ce": loss_ce}
        if log:
            with torch.no_grad():
                pred = src_logits.topk(1, -1, True, True)[1][..., 0]
                n = matched.sum()
                correct = (matched & (pred == target_classes)).sum().float()
                accuracy = correct * (100.0 / n.clamp(min=1).float())
                losses["class_error"] = torch.where(n > 0, 100 - accuracy, 100.0)
        return losses

    @torch.no_grad()
    def loss_cardinality(self, outputs, labels, padded, m, num_boxes):
        pred_logits = outputs["pred_logits"]
        card_pred = (pred_logits.argmax(-1) != pred_logits.shape[-1] - 1).sum(1)
        return {"cardinality_error": F.l1_loss(card_pred.float(), padded.counts.float())}

    def loss_boxes(self, outputs, labels, padded, m, num_boxes):
        qot = m.query_of_target.long()
        valid = qot >= 0
        src_boxes = outputs["pred_boxes"].gather(1, qot.clamp(min=0).unsqueeze(-1).expand(-1, -1, 4))
        target_boxes = padded.boxes.to(src_boxes.dtype)
        loss_bbox = torch.where(valid.unsqueeze(-1), F.l1_loss(src_boxes, target_boxes, reduction="none"), 0)
        giou = _giou(box_cxcywh_to_xyxy(src_boxes), box_cxcywh_to_xyxy(target_boxes))
        loss_giou = torch.where(valid, 1 - giou, 0)
        return {"loss_bbox": loss_bbox.sum() / num_boxes, "loss_giou": loss_giou.sum() / num_boxes}

    def _head_losses(self, outputs, labels, padded, m, num_boxes, suffix, log):
        losses = {}
        for loss in self.losses:
            fn = {"labels": self.loss_labels, "cardinality": self.loss_cardinality, "boxes": self.loss_boxes}[loss]
            kwargs = {"log": log} if loss == "labels" else {}
            losses.update(fn(outputs, labels, padded, m, num_boxes, **kwargs))
        # a problem the solver refused (non-finite cost) poisons the head's losses and their gradients
        poison = torch.where(m.status.ne(0).any(), float("nan"), 1.0)
        return {k + suffix: v * poison.to(v.dtype) for k, v in losses.items()}

    def forward(self, outputs, targets, num_boxes=None):
        device = outputs["pred_logits"].device
        if isinstance(targets, PaddedTargets):
            padded = targets
        else:
            padded = _pack(targets, max(1, max(len(t["labels"]) for t in targets)))
        padded = PaddedTargets(*(x.to(device) for x in padded))
        if num_boxes is None:
            num_boxes = padded.counts.sum().float()
            world = 1
            if dist.is_available() and dist.is_initialized():
                dist.all_reduce(num_boxes)
                world = dist.get_world_size()
            num_boxes = torch.clamp(num_boxes / world, min=1)
        else:
            num_boxes = torch.as_tensor(num_boxes, dtype=torch.float32, device=device)

        outputs_without_aux = {k: v for k, v in outputs.items() if k != "aux_outputs" and k != "enc_outputs"}
        heads = [(outputs_without_aux, padded.labels, "", True)]
        for i, aux_outputs in enumerate(outputs.get("aux_outputs", ())):
            heads.append((aux_outputs, padded.labels, f"_{i}", False))
        if "enc_outputs" in outputs:
            heads.append((outputs["enc_outputs"], torch.zeros_like(padded.labels), "_enc", False))
        matchings = self.matcher.match_padded([(o, lab, padded) for o, lab, _, _ in heads])
        losses = {}
        for (o, lab, suffix, log), m in zip(heads, matchings):
            losses.update(self._head_losses(o, lab, padded, m, num_boxes, suffix, log))
        return losses
