"""Drop-in mirror of the reference's ``utility/anchor_manipulator.py`` on CUDA tensors.

Same module-level functions, same class, same method names, positional order,
defaults and return-tuple order as /root/reference/utility/anchor_manipulator.py;
symbolic ``tf.Tensor`` arguments become ``torch.Tensor`` on a CUDA device and every
computation runs in the sm_100a kernels of libdan_b200.so (no TF graph ops, no
Triton, no CPU fallback).  Additions that have no analogue in the reference are
the batched entry points (``encode_anchors_batch`` ...) -- the reference encodes one
image per call inside its CPU input queue (dataset/dataset_common.py:150,178).
"""
from __future__ import annotations

import math

import torch

from .. import _lib as L
from .. import functional as F
from . import custom_op


def _soa(boxes):
    """[N,4] AoS -> four contiguous [N] vectors (layout hand-off only)."""
    boxes = L.as_f32(boxes).view(-1, 4)
    return [boxes[:, i].contiguous() for i in range(4)]


def areas(gt_bboxes):
    """anchor_manipulator.py:24-27 -> [N, 1]."""
    b = L.as_f32(gt_bboxes).view(-1, 4)
    return F.bbox_convert(b, 2)[:, 0:1]


def intersection(gt_bboxes, default_bboxes):
    """anchor_manipulator.py:29-43 -> [N, M] (first argument: the anchors, see :285-287)."""
    return F.intersection_matrix(*_soa(gt_bboxes), L.as_f32(default_bboxes).view(-1, 4))


def iou_matrix(gt_bboxes, default_bboxes):
    """anchor_manipulator.py:44-52 -> [N, M] fp32."""
    return F.iou_matrix(*_soa(gt_bboxes), L.as_f32(default_bboxes).view(-1, 4))


def do_dual_max_match(overlap_matrix, low_thres, high_thres, ignore_between=True, gt_max_first=True):
    """anchor_manipulator.py:54-105 -> (match_indices int64 [N], selected_scores fp32 [N])."""
    return F.dual_max_match(L.as_f32(overlap_matrix), low_thres, high_thres, ignore_between, gt_max_first)


class AnchorEncoder(object):
    """Mirror of anchor_manipulator.py:107 ``AnchorEncoder``."""

    def __init__(self, positive_threshold, ignore_threshold, prior_scaling):
        super(AnchorEncoder, self).__init__()
        self._all_anchors = None
        self._positive_threshold = positive_threshold
        self._ignore_threshold = ignore_threshold
        self._prior_scaling = prior_scaling
        self._pyramid = None

    # ---- :125-132 ------------------------------------------------------------------
    def center2point(self, center_y, center_x, height, width):
        c = torch.stack(torch.broadcast_tensors(*[L.as_f32(v) for v in (center_y, center_x, height, width)]), dim=-1)
        out = F.bbox_convert(c.contiguous(), 1)
        return out[..., 0], out[..., 1], out[..., 2], out[..., 3]

    def point2center(self, ymin, xmin, ymax, xmax):
        c = torch.stack(torch.broadcast_tensors(*[L.as_f32(v) for v in (ymin, xmin, ymax, xmax)]), dim=-1)
        out = F.bbox_convert(c.contiguous(), 0)
        return out[..., 0], out[..., 1], out[..., 2], out[..., 3]

    # ---- :134-161 ------------------------------------------------------------------
    def get_anchors_width_height(self, anchor_scale, extra_anchor_scale, anchor_ratio, name=None):
        """Heights / widths of the anchors of one layer, in depth order: first one square anchor per extra scale, then
        for every scale each aspect ratio r as (s / sqrt(r), s * sqrt(r)).  Computed in python doubles and rounded to
        fp32 once, which is what the reference's tf.constant(float32) of python floats does.

        -> (heights [depth], widths [depth], depth)"""
        squares = [(float(s), float(s)) for s in extra_anchor_scale]
        shaped = [(float(s) / math.sqrt(r), float(s) * math.sqrt(r)) for s in anchor_scale for r in anchor_ratio]
        sizes = squares + shaped
        heights = torch.tensor([h for h, _ in sizes], dtype=torch.float32)
        widths = torch.tensor([w for _, w in sizes], dtype=torch.float32)
        return heights, widths, len(sizes)

    # ---- :163-198 ------------------------------------------------------------------
    def generate_anchors_by_offset(self, anchors_height, anchors_width, anchor_depth, image_shape, layer_shape,
                                   feat_stride, offset=0.5, name=None):
        pyr = F.make_pyramid(image_shape, [anchors_height], [anchors_width], [anchor_depth], [offset], [layer_shape],
                             [feat_stride], [0.], [False])
        ymin, xmin, ymax, xmax, _ = F.generate_anchors(pyr)
        return (ymin.view(-1, anchor_depth), xmin.view(-1, anchor_depth), ymax.view(-1, anchor_depth),
                xmax.view(-1, anchor_depth))

    # ---- :200-211 ------------------------------------------------------------------
    def get_anchors_count(self, anchors_depth, layer_shape, name=None):
        """-> (cells of the layer, anchors of the layer = cells * depth)."""
        cells = int(layer_shape[0]) * int(layer_shape[1])
        return cells, cells * anchors_depth

    # ---- :213-273 ------------------------------------------------------------------
    def get_all_anchors(self, image_shape, anchors_height, anchors_width, anchors_depth, anchors_offsets, layer_shapes,
                        feat_strides, allowed_borders, should_clips, name=None):
        self._pyramid = F.make_pyramid(image_shape, anchors_height, anchors_width, anchors_depth, anchors_offsets,
                                       layer_shapes, feat_strides, allowed_borders, should_clips)
        self._generated = F.generate_anchors(self._pyramid)
        return self._generated

    @property
    def pyramid(self):
        """dan_pyramid POD of the last get_all_anchors call (None before): functional.encode_params(pyramid=...) turns
        it into the layout hint of the encode kernels."""
        return getattr(self, "_pyramid", None)

    def _hint_for(self, anchors):
        """The layout hint is only used for the very tensors get_all_anchors returned (any other anchor set is encoded
        without it: same results, strips instead of tiles)."""
        gen = getattr(self, "_generated", None)
        if gen is None or any(a is not g for a, g in zip(anchors, gen[:4])):
            return None
        return self._pyramid

    # ---- :275-387 ------------------------------------------------------------------
    def _params(self, ignore_threshold, positive_threshold, match_mining, pa_scale, debug, anchors=None):
        return F.encode_params(positive_threshold, ignore_threshold, self._prior_scaling, match_mining,
                               pa_scale=pa_scale, debug=debug,
                               pyramid=self._hint_for(anchors) if anchors is not None else None)

    def _encode_one(self, bboxes, anchors, inside_mask, params):
        bboxes = L.as_f32(bboxes).view(-1, 4)
        offsets = torch.tensor([0, bboxes.shape[0]], dtype=torch.int32, device=bboxes.device)
        r = F.encode_batch(params, *anchors, inside_mask, bboxes, offsets)
        return r.targets[0], r.labels[0], r.scores[0], r.matched_gt[0]

    def encode_anchors(self, bboxes, anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax, inside_mask,
                       match_mining=False, debug=False):
        """encode anchors with ground truth on the fly (one image), anchor_manipulator.py:275-326.

        -> (gt_targets [N,4], gt_labels int64 [N], gt_scores [N], matched_gt_bbox*pos [N,4])"""
        anchors = (anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax)
        params = self._params(self._ignore_threshold, self._positive_threshold, match_mining, 0.0, debug, anchors)
        return self._encode_one(bboxes, anchors, inside_mask, params)

    def encode_pa_anchors(self, bboxes, anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax, inside_mask,
                          ignore_threshold, positive_threshold, match_mining=True, scale=1., debug=False):
        """PyramidBox face/head/body encode, anchor_manipulator.py:328-387."""
        if not scale > 0:
            raise L.DanError(-1, "scale must be > 0")
        anchors = (anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax)
        params = self._params(ignore_threshold, positive_threshold, match_mining, float(scale), debug, anchors)
        return self._encode_one(bboxes, anchors, inside_mask, params)

    # ---- batched additions (no analogue in the reference) ---------------------------
    def encode_anchors_batch(self, gt_boxes, gt_offsets, anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax,
                             inside_mask, match_mining=False, debug=False, want_match=False, out=None):
        """All images of a batch in one launch sequence.  gt_boxes [sum M,4], gt_offsets int32 [B+1] (CSR).

        -> EncodeResult(targets [B,N,4], labels [B,N], scores [B,N], matched_gt [B,N,4], match [B,N]|None)"""
        params = self._params(self._ignore_threshold, self._positive_threshold, match_mining, 0.0, debug,
                              (anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax))
        return F.encode_batch(params, anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax, inside_mask, gt_boxes,
                              gt_offsets, out=out, want_match=want_match)

    def encode_pa_anchors_batch(self, gt_boxes, gt_offsets, anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax,
                                inside_mask, ignore_threshold, positive_threshold, match_mining=True, scale=1.,
                                debug=False, want_match=False, out=None):
        params = self._params(ignore_threshold, positive_threshold, match_mining, float(scale), debug,
                              (anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax))
        return F.encode_batch(params, anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax, inside_mask, gt_boxes,
                              gt_offsets, out=out, want_match=want_match)

    # BASELINE.json's north_star names this entry point `encode_all_anchors`
    encode_all_anchors = encode_anchors_batch

    # ---- :389-424 ------------------------------------------------------------------
    def batch_decode_anchors(self, pred_location, anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax):
        """pred_location [batch, num_preds, 4] in yxhw format -> boxes [batch, num_preds, 4] (fp32; fp16 / bf16 CUDA
        predictions are widened inside the kernel)."""
        pred = pred_location if L.is_half_cuda(pred_location) else L.as_f32(pred_location)
        return F.decode_batch(pred, anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax, self._prior_scaling)

    def decode_anchors(self, pred_location, anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax):
        """pred_location [num_preds, 4] in yxhw format -> boxes [num_preds, 4] (fp32, as batch_decode_anchors)."""
        pred = pred_location if L.is_half_cuda(pred_location) else L.as_f32(pred_location)
        return F.decode_batch(pred.unsqueeze(0), anchors_ymin, anchors_xmin, anchors_ymax, anchors_xmax,
                              self._prior_scaling)[0]

    # north_star alias
    decode_all_anchors = batch_decode_anchors


class AnchorCreator(object):
    """north_star alias: owns one stride pyramid and generates its anchors.

    The reference has no such class (SURVEY.md 0.3); the work is
    AnchorEncoder.get_anchors_width_height + get_all_anchors."""

    def __init__(self, image_shape, layer_shapes, anchor_scales, extra_anchor_scales, anchor_ratios, layer_strides,
                 offsets=None, allowed_borders=None, should_clips=None):
        n = len(layer_shapes)
        self.image_shape = image_shape
        self.layer_shapes = layer_shapes
        self.anchor_scales = anchor_scales
        self.extra_anchor_scales = extra_anchor_scales
        self.anchor_ratios = anchor_ratios
        self.layer_strides = layer_strides
        self.offsets = offsets if offsets is not None else [0.5] * n
        self.allowed_borders = allowed_borders if allowed_borders is not None else [0.] * n
        self.should_clips = should_clips if should_clips is not None else [False] * n
        self._encoder = AnchorEncoder(None, None, [0.1, 0.1, 0.2, 0.2])

    def get_all_anchors(self):
        hs, ws, ds = [], [], []
        for i in range(len(self.layer_shapes)):
            h, w, d = self._encoder.get_anchors_width_height(self.anchor_scales[i], self.extra_anchor_scales[i],
                                                             self.anchor_ratios[i])
            hs.append(h)
            ws.append(w)
            ds.append(d)
        self.anchors_depth = ds
        return self._encoder.get_all_anchors(self.image_shape, hs, ws, ds, self.offsets, self.layer_shapes,
                                             self.layer_strides, self.allowed_borders, self.should_clips)
