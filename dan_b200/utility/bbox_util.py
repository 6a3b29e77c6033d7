"""Drop-in mirror of the reference's ``utility/bbox_util.py`` on CUDA tensors.

Same function names, argument order and return values as
/root/reference/utility/bbox_util.py:24-119.  ``parse_by_class`` runs the fused
filter -> radix-select/sort -> bitmask-NMS pipeline of libdan_b200.so; the small
helpers are one elementwise kernel each."""
from __future__ import annotations

import torch

from .. import _lib as L
from .. import functional as F


def select_bboxes(scores_pred, bboxes_pred, num_classes, select_threshold, name=None):
    """bbox_util.py:24-36."""
    scores_pred = L.as_f32(scores_pred)
    bboxes_pred = L.as_f32(bboxes_pred)
    selected_bboxes = {}
    selected_scores = {}
    for class_ind in range(1, num_classes):
        selected_bboxes[class_ind], selected_scores[class_ind] = F.select_bboxes_class(
            scores_pred, bboxes_pred, class_ind, select_threshold)
    return selected_bboxes, selected_scores


def _stack4(ymin, xmin, ymax, xmax):
    return torch.stack([L.as_f32(ymin), L.as_f32(xmin), L.as_f32(ymax), L.as_f32(xmax)], dim=-1).contiguous()


def clip_bboxes(ymin, xmin, ymax, xmax, height, width, name=None):
    """bbox_util.py:38-48."""
    out = F.clip_boxes(_stack4(ymin, xmin, ymax, xmax), height, width)
    return out[..., 0], out[..., 1], out[..., 2], out[..., 3]


def filter_bboxes(scores_pred, ymin, xmin, ymax, xmax, min_size, name=None):
    """bbox_util.py:50-59."""
    s, b = F.filter_boxes(L.as_f32(scores_pred), _stack4(ymin, xmin, ymax, xmax), min_size)
    return s, b[..., 0], b[..., 1], b[..., 2], b[..., 3]


def sort_bboxes(scores_pred, ymin, xmin, ymax, xmax, keep_topk, name=None):
    """bbox_util.py:61-72: tf.nn.top_k (descending, ties -> lower index) + zero pad to keep_topk."""
    s, b, _ = F.sort_boxes(L.as_f32(scores_pred), _stack4(ymin, xmin, ymax, xmax), keep_topk)
    return s, b[..., 0], b[..., 1], b[..., 2], b[..., 3]


def nms_bboxes(scores_pred, bboxes_pred, nms_topk, nms_threshold, name=None):
    """bbox_util.py:75-78 (variable-length result; reading the count synchronises the stream)."""
    s, b, _, cnt = F.nms_boxes(L.as_f32(scores_pred), L.as_f32(bboxes_pred), nms_topk, nms_threshold)
    n = int(cnt.item())
    return s[:n], b[:n]


def nms_bboxes_with_padding(scores_pred, bboxes_pred, nms_topk, nms_threshold, name=None):
    """bbox_util.py:80-90 (zero padded to nms_topk)."""
    s, b, _, _ = F.nms_boxes(L.as_f32(scores_pred), L.as_f32(bboxes_pred), nms_topk, nms_threshold)
    return s, b


def bbox_point2center(bboxes, name=None):
    """bbox_util.py:92-96."""
    return F.bbox_convert(L.as_f32(bboxes), 0)


def bbox_center2point(bboxes, name=None):
    """bbox_util.py:98-101."""
    return F.bbox_convert(L.as_f32(bboxes), 1)


def parse_by_class(image_shape, cls_pred, bboxes_pred, num_classes, select_threshold, min_size, keep_topk, nms_topk,
                   nms_threshold):
    """bbox_util.py:103-119 -> ({class: boxes [nms_topk,4]}, {class: scores [nms_topk]}).  fp16 / bf16 CUDA predictions
    of ONE dtype on one device are read as they are (fp32 results, bit-identical to the call on the widened values);
    any other pair, e.g. half logits with the fp32 boxes of decode_anchors, goes through as_f32 as a whole."""
    if not (L.is_half_cuda(cls_pred) and L.is_half_cuda(bboxes_pred) and cls_pred.dtype == bboxes_pred.dtype
            and cls_pred.device == bboxes_pred.device):
        cls_pred = L.as_f32(cls_pred)
        bboxes_pred = L.as_f32(bboxes_pred)
    params = F.postprocess_params(num_classes, image_shape, select_threshold, min_size, keep_topk, nms_topk,
                                  nms_threshold)
    det = F.postprocess_batch(params, cls_pred.unsqueeze(0), boxes_pred=bboxes_pred.unsqueeze(0), want_index=False)
    selected_bboxes = {}
    selected_scores = {}
    for class_ind in range(1, num_classes):
        selected_bboxes[class_ind] = det.boxes[0, class_ind - 1]
        selected_scores[class_ind] = det.scores[0, class_ind - 1]
    return selected_bboxes, selected_scores


def parse_by_class_batch(image_shape, cls_pred, num_classes, select_threshold, min_size, keep_topk, nms_topk,
                         nms_threshold, loc_pred=None, bboxes_pred=None, anchors=None,
                         prior_scaling=(0.1, 0.1, 0.2, 0.2), out=None, want_index=True):
    """Batched addition: cls_pred [B,N,C] and either loc_pred [B,N,4] (+ anchors; decoded in-kernel like
    decode_anchors) or bboxes_pred [B,N,4].  -> functional.Detections indexed [b, class-1]."""
    params = F.postprocess_params(num_classes, image_shape, select_threshold, min_size, keep_topk, nms_topk,
                                  nms_threshold, prior_scaling)
    return F.postprocess_batch(params, cls_pred, loc_pred=loc_pred, boxes_pred=bboxes_pred, anchors=anchors, out=out,
                               want_index=want_index)
