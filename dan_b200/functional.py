"""Tensor-level entry points: one python function per C-ABI call of include/dan_b200.h.

Every function takes / returns CUDA ``torch.Tensor`` objects, allocates only the
outputs (and a caller-owned workspace) with torch, and enqueues the kernels on
torch's current stream.  No arithmetic of the hot path is done in PyTorch."""
from __future__ import annotations

import ctypes
import os
from collections import namedtuple

import torch

from . import _lib as L

_ws = L.StreamWorkspaces()

EncodeResult = namedtuple("EncodeResult", ["targets", "labels", "scores", "matched_gt", "match"])
Detections = namedtuple("Detections", ["boxes", "scores", "counts", "anchor_index", "keep_pos"])
HardNegatives = namedtuple("HardNegatives", ["cls_pred", "loc_pred", "cls_targets", "loc_targets", "counts", "final_mask",
                                             "n_neg_select", "score_at_k"])


def _dev(t):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError("dan_b200 operates on CUDA torch.Tensors only (no CPU fallback)")
    return t.device


# ----------------------------------------------------------------------------------
# anchors
# ----------------------------------------------------------------------------------
def make_pyramid(image_shape, anchors_height, anchors_width, anchors_depth, anchors_offsets, layer_shapes,
                 feat_strides, allowed_borders, should_clips):
    """Pack the arguments of AnchorEncoder.get_all_anchors (anchor_manipulator.py:213) into the
    dan_pyramid POD.  Heights / widths are rounded to fp32 once, like tf.constant(float32)."""
    p = L.Pyramid()
    nl = len(anchors_depth)
    if nl < 1 or nl > L.DAN_MAX_LAYERS:
        raise L.DanError(-1, "num_layers must be in [1, %d], got %d" % (L.DAN_MAX_LAYERS, nl))
    p.num_layers = nl
    p.image_h, p.image_w = int(image_shape[0]), int(image_shape[1])
    dpos = 0
    for i in range(nl):
        p.layer_h[i], p.layer_w[i] = int(layer_shapes[i][0]), int(layer_shapes[i][1])
        p.depth[i] = int(anchors_depth[i])
        p.clip[i] = 1 if should_clips[i] else 0
        p.stride[i] = float(feat_strides[i])
        off = anchors_offsets[i]
        if isinstance(off, (list, tuple)):
            p.offset_h[i], p.offset_w[i] = float(off[0]), float(off[1])
        else:
            p.offset_h[i] = p.offset_w[i] = float(off)
        p.border[i] = float(allowed_borders[i])
        hs = [float(v) for v in (anchors_height[i].tolist() if hasattr(anchors_height[i], "tolist") else anchors_height[i])]
        ws = [float(v) for v in (anchors_width[i].tolist() if hasattr(anchors_width[i], "tolist") else anchors_width[i])]
        if len(hs) != p.depth[i] or len(ws) != p.depth[i]:
            raise L.DanError(-1, "layer %d: %d heights / %d widths for depth %d" % (i, len(hs), len(ws), p.depth[i]))
        if dpos + p.depth[i] > L.DAN_MAX_DEPTH_TOTAL:
            raise L.DanError(-4, "sum of anchor depths exceeds %d" % L.DAN_MAX_DEPTH_TOTAL)
        for d in range(p.depth[i]):
            p.anchor_h[dpos + d] = hs[d]
            p.anchor_w[dpos + d] = ws[d]
        dpos += p.depth[i]
    return p


def anchor_count(pyramid):
    n = L.lib().dan_anchor_count(ctypes.byref(pyramid))
    if n < 0:
        L.check(-1)
    return int(n)


def generate_anchors(pyramid, device=None):
    """-> (ymin, xmin, ymax, xmax) fp32 [N] and inside_mask bool [N]."""
    L.require_device()
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    n = anchor_count(pyramid)
    out = [torch.empty(n, dtype=torch.float32, device=device) for _ in range(4)]
    mask = torch.empty(n, dtype=torch.bool, device=device)
    with torch.cuda.device(device):
        L.check(L.lib().dan_generate_anchors(ctypes.byref(pyramid), *[L.dev_ptr(t) for t in out], L.dev_ptr(mask),
                                             L.stream_ptr()))
    return out[0], out[1], out[2], out[3], mask


def _anchor_ptrs(ymin, xmin, ymax, xmax):
    n = ymin.numel()
    for name, t in (("anchors_ymin", ymin), ("anchors_xmin", xmin), ("anchors_ymax", ymax), ("anchors_xmax", xmax)):
        if t.numel() != n:
            raise ValueError("anchor vectors differ in length")
    return [L.dev_ptr(t, torch.float32, name) for name, t in
            (("anchors_ymin", ymin), ("anchors_xmin", xmin), ("anchors_ymax", ymax), ("anchors_xmax", xmax))]


def _mask_u8(inside_mask):
    if inside_mask is None:
        return None
    if inside_mask.dtype not in (torch.bool, torch.uint8):
        raise TypeError("inside_mask must be bool or uint8")
    return inside_mask.contiguous()


# ----------------------------------------------------------------------------------
# matching on a dense overlaps matrix (the custom-op boundary)
# ----------------------------------------------------------------------------------
def iou_matrix(ymin, xmin, ymax, xmax, gt_boxes, inside_mask=None):
    L.require_device()
    gt_boxes = gt_boxes.contiguous()
    n, m = ymin.numel(), gt_boxes.shape[0]
    out = torch.empty((n, m), dtype=torch.float32, device=_dev(ymin))
    mask = _mask_u8(inside_mask)
    with torch.cuda.device(_dev(ymin)):
        L.check(L.lib().dan_iou_matrix(*_anchor_ptrs(ymin, xmin, ymax, xmax), L.dev_ptr(mask), n,
                                       L.dev_ptr(gt_boxes, torch.float32, "gt_boxes"), m, L.dev_ptr(out), L.stream_ptr()))
    return out


def intersection_matrix(ymin, xmin, ymax, xmax, gt_boxes):
    L.require_device()
    gt_boxes = gt_boxes.contiguous()
    n, m = ymin.numel(), gt_boxes.shape[0]
    out = torch.empty((n, m), dtype=torch.float32, device=_dev(ymin))
    with torch.cuda.device(_dev(ymin)):
        L.check(L.lib().dan_intersection_matrix(*_anchor_ptrs(ymin, xmin, ymax, xmax), n,
                                                L.dev_ptr(gt_boxes, torch.float32, "gt_boxes"), m, L.dev_ptr(out),
                                                L.stream_ptr()))
    return out


def small_mining_match(overlaps, negative_low_thres, negative_high_thres, positive_thres, min_match,
                       stop_positive_thres):
    """SmallMiningMatch op (cpp/ExtraLib/small_mining_match.cc:31-54) -> (int32 [N], fp32 [N])."""
    L.require_device()
    if overlaps.dim() != 2:
        raise L.DanError(-1, "inputs must be in 'num_anchors x num_ground_truth' format.")
    overlaps = overlaps.contiguous()
    n, m = overlaps.shape
    match = torch.empty(n, dtype=torch.int32, device=_dev(overlaps))
    scores = torch.empty(n, dtype=torch.float32, device=_dev(overlaps))
    nbytes = L.lib().dan_match_workspace_bytes(n, m)
    ws = _ws.get(nbytes, _dev(overlaps))
    with torch.cuda.device(_dev(overlaps)):
        L.check(L.lib().dan_small_mining_match(L.dev_ptr(overlaps, torch.float32, "overlaps"), n, m, negative_low_thres,
                                               negative_high_thres, positive_thres, int(min_match), stop_positive_thres,
                                               L.dev_ptr(match), L.dev_ptr(scores), L.dev_ptr(ws), nbytes, L.stream_ptr()))
    return match, scores


def dual_max_match(overlaps, low_thres, high_thres, ignore_between=True, gt_max_first=True):
    """do_dual_max_match (anchor_manipulator.py:54-105) -> (int64 [N], fp32 [N])."""
    L.require_device()
    if overlaps.dim() != 2:
        raise L.DanError(-1, "overlap_matrix must be num_anchors x num_gt")
    overlaps = overlaps.contiguous()
    n, m = overlaps.shape
    match = torch.empty(n, dtype=torch.int64, device=_dev(overlaps))
    scores = torch.empty(n, dtype=torch.float32, device=_dev(overlaps))
    nbytes = L.lib().dan_match_workspace_bytes(n, m)
    ws = _ws.get(nbytes, _dev(overlaps))
    with torch.cuda.device(_dev(overlaps)):
        L.check(L.lib().dan_dual_max_match(L.dev_ptr(overlaps, torch.float32, "overlaps"), n, m, low_thres, high_thres,
                                           1 if ignore_between else 0, 1 if gt_max_first else 0, L.dev_ptr(match),
                                           L.dev_ptr(scores), L.dev_ptr(ws), nbytes, L.stream_ptr()))
    return match, scores


# ----------------------------------------------------------------------------------
# fused batched encode
# ----------------------------------------------------------------------------------
def encode_params(positive_threshold, ignore_threshold, prior_scaling, match_mining, pa_scale=0.0, debug=False,
                  negative_low_thres=0.0, min_match=6, stop_positive_thres=0.3, ignore_between=True,
                  gt_max_first=True, pyramid=None):
    """dan_encode_params.  pyramid (optional, the dan_pyramid POD of make_pyramid / AnchorEncoder.get_all_anchors): fills
    the LAYOUT HINT of the params - which stretches of the flat anchor arrays are row-major grids with one anchor per
    cell - so that the encode kernels can give every warp a compact tile of cells.  Performance only: the results do
    not depend on it.  The anchors passed to encode_batch must then be the ones that pyramid generates."""
    p = L.EncodeParams()
    if pyramid is not None:
        for start, w, h in grid_hint(pyramid):
            if p.num_grids < L.DAN_MAX_GRIDS:
                p.grid_start[p.num_grids], p.grid_w[p.num_grids], p.grid_h[p.num_grids] = start, w, h
                p.num_grids += 1
    p.matcher = L.DAN_MATCH_MINING if match_mining else L.DAN_MATCH_DUAL
    p.ignore_threshold = float(ignore_threshold)
    p.positive_threshold = float(positive_threshold)
    for i in range(4):
        p.prior_scaling[i] = float(prior_scaling[i])
    p.pa_scale = float(pa_scale)
    p.debug = 1 if debug else 0
    p.negative_low_thres = float(negative_low_thres)
    p.min_match = int(min_match)
    p.stop_positive_thres = float(stop_positive_thres)
    p.ignore_between = 1 if ignore_between else 0
    p.gt_max_first = 1 if gt_max_first else 0
    return p


def grid_hint(pyramid):
    """[(first anchor, cells per row, rows)] of the pyramid levels the layout hint can describe: one anchor per cell,
    level start a multiple of 32, width a multiple of 8, height a multiple of 4 (include/dan_b200.h)."""
    out, start = [], 0
    for i in range(pyramid.num_layers):
        h, w, d = int(pyramid.layer_h[i]), int(pyramid.layer_w[i]), int(pyramid.depth[i])
        if d == 1 and start % 32 == 0 and w > 0 and h > 0 and w % 8 == 0 and h % 4 == 0:
            out.append((start, w, h))
        start += h * w * d
    return out


def encode_batch(params, ymin, xmin, ymax, xmax, inside_mask, gt_boxes, gt_offsets, out=None, want_match=False,
                 want_matched_gt=True, workspace=None, profile=False):
    """Fused IoU + match + encode for a batch (anchor_manipulator.py:275-387 per image).

    gt_boxes [sum M, 4] fp32, gt_offsets [B+1] int32 (CSR).  Returns EncodeResult with
    targets [B,N,4] f32, labels [B,N] int64, scores [B,N] f32, matched_gt [B,N,4] f32."""
    L.require_device()
    dev = _dev(ymin)
    n = ymin.numel()
    if gt_offsets.dtype != torch.int32:
        raise TypeError("gt_offsets must be int32")
    batch = gt_offsets.numel() - 1
    gt_boxes = gt_boxes.contiguous().view(-1, 4)
    total_gt = gt_boxes.shape[0]
    if out is None:
        targets = torch.empty((batch, n, 4), dtype=torch.float32, device=dev)
        labels = torch.empty((batch, n), dtype=torch.int64, device=dev)
        scores = torch.empty((batch, n), dtype=torch.float32, device=dev)
        matched = torch.empty((batch, n, 4), dtype=torch.float32, device=dev) if want_matched_gt else None
        match = torch.empty((batch, n), dtype=torch.int32, device=dev) if want_match else None
    else:
        targets, labels, scores, matched, match = out
    mask = _mask_u8(inside_mask)
    if os.environ.get("DAN_B200_DEBUG"):
        # the CSR contract of dan_encode_batch (costs a device synchronisation, hence debug only)
        offs = gt_offsets.cpu()
        if int(offs[0]) != 0 or int(offs[-1]) != total_gt or bool((offs[1:] < offs[:-1]).any()):
            raise ValueError("gt_offsets must rise from 0 to len(gt_boxes) = %d, got %s ... %s" % (total_gt, int(offs[0]), int(offs[-1])))
    nbytes = L.lib().dan_encode_workspace_bytes(n, batch, total_gt)
    ws = (workspace or _ws).get(nbytes, dev)
    args = [ctypes.byref(params), *_anchor_ptrs(ymin, xmin, ymax, xmax), L.dev_ptr(mask), n,
            L.dev_ptr(gt_boxes, torch.float32, "gt_boxes") if total_gt else ctypes.c_void_p(0),
            L.dev_ptr(gt_offsets, torch.int32, "gt_offsets"), batch, total_gt,
            L.dev_ptr(targets, torch.float32), L.dev_ptr(labels, torch.int64),
            L.dev_ptr(scores, torch.float32), L.dev_ptr(matched), L.dev_ptr(match),
            L.dev_ptr(ws), nbytes, L.stream_ptr()]
    with torch.cuda.device(dev):
        if profile:   # CUDA-event duration of each pass, [pass1, pass2, pass3] in ms (synchronises)
            ms = (ctypes.c_float * 3)()
            L.check(L.lib().dan_encode_batch_profile(*args, ms))
            return EncodeResult(targets, labels, scores, matched, match), list(ms)
        L.check(L.lib().dan_encode_batch(*args))
    return EncodeResult(targets, labels, scores, matched, match)


# ----------------------------------------------------------------------------------
# decode
# ----------------------------------------------------------------------------------
def decode_batch(pred_location, ymin, xmin, ymax, xmax, prior_scaling):
    """pred_location [batch, num_preds, 4] in fp32, fp16 or bf16 -> fp32 boxes [batch, num_preds, 4]."""
    L.require_device()
    pred = pred_location.contiguous()
    if pred.dtype not in L.PRED_DTYPES or pred.dim() != 3 or pred.shape[-1] != 4:
        raise TypeError("pred_location must be fp32, fp16 or bf16 [batch, num_preds, 4]")
    batch, n = pred.shape[0], pred.shape[1]
    if n != ymin.numel():
        raise ValueError("pred_location has %d rows but there are %d anchors" % (n, ymin.numel()))
    out = torch.empty(pred.shape, dtype=torch.float32, device=_dev(pred))
    ps = (ctypes.c_float * 4)(*[float(v) for v in prior_scaling])
    with torch.cuda.device(_dev(pred)):
        L.check(L.lib().dan_decode_batch_typed(L.pred_dtype(pred), L.dev_ptr(pred), *_anchor_ptrs(ymin, xmin, ymax, xmax), n,
                                               batch, ps, L.dev_ptr(out), L.stream_ptr()))
    return out


# ----------------------------------------------------------------------------------
# bbox_util pieces
# ----------------------------------------------------------------------------------
def softmax(logits):
    L.require_device()
    x = logits.contiguous()
    c = x.shape[-1]
    rows = x.numel() // max(c, 1)
    out = torch.empty_like(x)
    with torch.cuda.device(_dev(x)):
        L.check(L.lib().dan_softmax(L.dev_ptr(x, torch.float32, "logits"), rows, c, L.dev_ptr(out), L.stream_ptr()))
    return out


def select_bboxes_class(scores_pred, bboxes_pred, class_ind, select_threshold):
    L.require_device()
    s = scores_pred.contiguous()
    b = bboxes_pred.contiguous()
    n, c = s.shape
    ob = torch.empty_like(b)
    osc = torch.empty(n, dtype=torch.float32, device=_dev(s))
    with torch.cuda.device(_dev(s)):
        L.check(L.lib().dan_select_bboxes(L.dev_ptr(s, torch.float32, "scores_pred"), c, class_ind,
                                          L.dev_ptr(b, torch.float32, "bboxes_pred"), n, float(select_threshold),
                                          L.dev_ptr(ob), L.dev_ptr(osc), L.stream_ptr()))
    return ob, osc


def clip_boxes(boxes, height, width):
    L.require_device()
    b = boxes.contiguous()
    out = torch.empty_like(b)
    with torch.cuda.device(_dev(b)):
        L.check(L.lib().dan_clip_bboxes(L.dev_ptr(b, torch.float32, "boxes"), b.numel() // 4, float(height), float(width),
                                        L.dev_ptr(out), L.stream_ptr()))
    return out


def filter_boxes(scores, boxes, min_size):
    L.require_device()
    s = scores.contiguous()
    b = boxes.contiguous()
    os_, ob = torch.empty_like(s), torch.empty_like(b)
    import numpy as np
    thr = float(np.float32(float(min_size) + 1.0))
    with torch.cuda.device(_dev(b)):
        L.check(L.lib().dan_filter_bboxes(L.dev_ptr(s, torch.float32, "scores"), L.dev_ptr(b, torch.float32, "boxes"),
                                          s.numel(), thr, L.dev_ptr(os_), L.dev_ptr(ob), L.stream_ptr()))
    return os_, ob


def bbox_convert(boxes, mode):
    L.require_device()
    b = boxes.contiguous()
    out = torch.empty_like(b)
    with torch.cuda.device(_dev(b)):
        L.check(L.lib().dan_bbox_convert(L.dev_ptr(b, torch.float32, "boxes"), b.numel() // 4, int(mode), L.dev_ptr(out),
                                         L.stream_ptr()))
    return out


def sort_boxes(scores, boxes, keep_topk):
    """tf.nn.top_k + gather + zero pad -> (scores [keep_topk], boxes [keep_topk,4], index int32 [keep_topk])."""
    L.require_device()
    s = scores.contiguous()
    b = boxes.contiguous()
    n = s.numel()
    dev = _dev(s)
    os_ = torch.empty(keep_topk, dtype=torch.float32, device=dev)
    ob = torch.empty((keep_topk, 4), dtype=torch.float32, device=dev)
    oi = torch.empty(keep_topk, dtype=torch.int32, device=dev)
    nbytes = L.lib().dan_sort_workspace_bytes(n, keep_topk)
    ws = _ws.get(nbytes, dev)
    with torch.cuda.device(dev):
        L.check(L.lib().dan_sort_bboxes(L.dev_ptr(s, torch.float32, "scores"), L.dev_ptr(b, torch.float32, "boxes"), n,
                                        int(keep_topk), L.dev_ptr(os_), L.dev_ptr(ob), L.dev_ptr(oi), L.dev_ptr(ws), nbytes,
                                        L.stream_ptr()))
    return os_, ob, oi


def nms_boxes(scores, boxes, nms_topk, nms_threshold):
    """tf.image.non_max_suppression + gather + zero pad.
    -> (scores [nms_topk], boxes [nms_topk,4], keep int32 [nms_topk] (-1 padded), count int32 [1])."""
    L.require_device()
    s = scores.contiguous()
    b = boxes.contiguous()
    n = s.numel()
    dev = _dev(s)
    os_ = torch.empty(nms_topk, dtype=torch.float32, device=dev)
    ob = torch.empty((nms_topk, 4), dtype=torch.float32, device=dev)
    keep = torch.empty(nms_topk, dtype=torch.int32, device=dev)
    cnt = torch.empty(1, dtype=torch.int32, device=dev)
    nbytes = L.lib().dan_nms_workspace_bytes(n, nms_topk)
    ws = _ws.get(nbytes, dev)
    with torch.cuda.device(dev):
        L.check(L.lib().dan_nms_bboxes(L.dev_ptr(s, torch.float32, "scores"), L.dev_ptr(b, torch.float32, "boxes"), n,
                                       int(nms_topk), float(nms_threshold), L.dev_ptr(os_), L.dev_ptr(ob), L.dev_ptr(keep),
                                       L.dev_ptr(cnt), L.dev_ptr(ws), nbytes, L.stream_ptr()))
    return os_, ob, keep, cnt


def postprocess_params(num_classes, image_shape, select_threshold, min_size, keep_topk, nms_topk, nms_threshold,
                       prior_scaling=(0.1, 0.1, 0.2, 0.2)):
    p = L.PostprocessParams()
    p.num_classes = int(num_classes)
    p.image_h, p.image_w = int(image_shape[0]), int(image_shape[1])
    p.select_threshold = float(select_threshold)
    p.min_size = float(min_size)
    p.keep_topk = int(keep_topk)
    p.nms_topk = int(nms_topk)
    p.nms_threshold = float(nms_threshold)
    for i in range(4):
        p.prior_scaling[i] = float(prior_scaling[i])
    return p


def postprocess_batch(params, cls_pred, loc_pred=None, boxes_pred=None, anchors=None, out=None, want_index=True,
                      workspace=None, profile=False, peers=None):
    """Batched fused parse_by_class (bbox_util.py:103-119).  cls_pred [B,N,C]; give loc_pred [B,N,4]
    (+ anchors = (ymin,xmin,ymax,xmax)) or boxes_pred [B,N,4].  Returns Detections indexed [b, c-1].
    The predictions are fp32, fp16 or bf16, one dtype for all of them; the outputs are fp32 and bit-identical to the
    fp32 call on the widened predictions.
    loc_pred / boxes_pred may be PINNED HOST tensors: the kernels then read only the rows of the anchors that pass the
    score threshold, in place over PCIe (host-resident geometry, include/dan_b200.h)."""
    L.require_device()
    cls_pred = cls_pred.contiguous()
    if cls_pred.dim() != 3:
        raise TypeError("cls_pred must be [batch, num_anchors, num_classes]")
    dtype = L.pred_dtype(cls_pred, "cls_pred")
    geo_name, geo = ("loc_pred", loc_pred) if loc_pred is not None else ("boxes_pred", boxes_pred)
    if isinstance(geo, torch.Tensor) and geo.dtype != cls_pred.dtype:
        raise TypeError("cls_pred is %s but %s is %s: the predictions must share one dtype" % (cls_pred.dtype, geo_name, geo.dtype))
    batch, n, c = cls_pred.shape
    if c != params.num_classes:
        raise ValueError("cls_pred has %d classes, params say %d" % (c, params.num_classes))
    dev = _dev(cls_pred)
    lists = c - 1
    if out is None:
        boxes = torch.empty((batch, lists, params.nms_topk, 4), dtype=torch.float32, device=dev)
        scores = torch.empty((batch, lists, params.nms_topk), dtype=torch.float32, device=dev)
        counts = torch.empty((batch, lists), dtype=torch.int32, device=dev)
        aidx = torch.empty((batch, lists, params.nms_topk), dtype=torch.int32, device=dev) if want_index else None
        kpos = torch.empty((batch, lists, params.nms_topk), dtype=torch.int32, device=dev) if want_index else None
    else:
        boxes, scores, counts, aidx, kpos = out
    if loc_pred is not None:
        loc_pred = loc_pred.contiguous()
        if anchors is None:
            raise ValueError("anchors are needed to decode loc_pred")
        aptr = _anchor_ptrs(*anchors)
    else:
        boxes_pred = boxes_pred.contiguous()
        aptr = [ctypes.c_void_p(0)] * 4
    nbytes = L.lib().dan_postprocess_workspace_bytes(n, batch, c, params.keep_topk)
    ws = (workspace or _ws).get(nbytes, dev)
    ms = (ctypes.c_float * 2)() if profile else None          # [filter, top-k/sort + NMS] in ms (synchronises)
    # peers (L.PeerExchangeArgs): the NMS kernel also stores the slab rows into the other ranks' buffers; a profiling
    # call takes no part in the exchange
    exchange = ctypes.byref(peers) if peers is not None and not profile else None
    with torch.cuda.device(dev):
        L.check(L.lib().dan_postprocess_batch_typed(
            ctypes.byref(params), dtype, L.dev_ptr(cls_pred, cls_pred.dtype, "cls_pred"),
            L.dev_ptr(loc_pred, cls_pred.dtype, "loc_pred", allow_pinned=True),
            L.dev_ptr(boxes_pred, cls_pred.dtype, "boxes_pred", allow_pinned=True), *aptr, n, batch,
            L.dev_ptr(boxes), L.dev_ptr(scores), L.dev_ptr(counts), L.dev_ptr(aidx), L.dev_ptr(kpos), L.dev_ptr(ws), nbytes,
            exchange, L.stream_ptr(), ms))
    if profile:
        return Detections(boxes, scores, counts, aidx, kpos), list(ms)
    return Detections(boxes, scores, counts, aidx, kpos)


# ----------------------------------------------------------------------------------
# hard-negative mining (SURVEY.md 8(f3))
# ----------------------------------------------------------------------------------
def hard_negative_mining(cls_pred, loc_pred, cls_targets, loc_targets, rows, negative_ratio, num_classes,
                         at_least_one=True, strict_greater=False, out=None, workspace=None):
    """dan_hard_negative_mining: everything stays on the device and nothing synchronises.

    cls_pred [rows*n, C] (or [rows, n, C]), loc_pred / loc_targets [rows*n, 4], cls_targets [rows, n] int64.
    Returns HardNegatives whose four compacted tensors have CAPACITY rows*n; their valid lengths are
    counts = int32 [2] = (selected rows, positive rows) on the device."""
    L.require_device()
    dev = _dev(cls_pred)
    total = cls_targets.numel()
    rows = int(rows)
    n = total // rows if rows > 0 else 0
    if rows * n != total:
        raise ValueError("cls_targets has %d elements, not a multiple of rows=%d" % (total, rows))
    c = cls_pred.numel() // total if total else int(cls_pred.shape[-1])
    cp = cls_pred.contiguous()
    lp = loc_pred.contiguous()
    tg = cls_targets.contiguous()
    lt = loc_targets.contiguous()
    if out is None:
        out = (torch.empty((total, c), dtype=torch.float32, device=dev), torch.empty((total, 4), dtype=torch.float32, device=dev),
               torch.empty(total, dtype=torch.int64, device=dev), torch.empty((total, 4), dtype=torch.float32, device=dev),
               torch.empty(2, dtype=torch.int32, device=dev), torch.empty(total, dtype=torch.uint8, device=dev),
               torch.empty(rows, dtype=torch.int32, device=dev), torch.empty(rows, dtype=torch.float32, device=dev))
    o_cls, o_lp, o_tg, o_lt, o_cnt, o_mask, o_nsel, o_cut = out
    nbytes = L.lib().dan_hard_negative_workspace_bytes(rows, n)
    ws = (workspace or _ws).get(nbytes, dev)
    with torch.cuda.device(dev):
        L.check(L.lib().dan_hard_negative_mining(
            L.dev_ptr(cp, torch.float32, "cls_pred"), int(c), L.dev_ptr(tg, torch.int64, "cls_targets"),
            L.dev_ptr(lp, torch.float32, "location_pred"), L.dev_ptr(lt, torch.float32, "loc_targets"), rows, n,
            float(negative_ratio), int(num_classes), int(bool(at_least_one)), int(bool(strict_greater)),
            L.dev_ptr(o_mask, torch.uint8, "final_mask"), L.dev_ptr(o_nsel, torch.int32, "n_neg_select"),
            L.dev_ptr(o_cut, torch.float32, "score_at_k"), L.dev_ptr(o_cls, torch.float32, "out cls_pred"),
            L.dev_ptr(o_tg, torch.int64, "out cls_targets"), L.dev_ptr(o_lp, torch.float32, "out location_pred"),
            L.dev_ptr(o_lt, torch.float32, "out loc_targets"), L.dev_ptr(o_cnt, torch.int32, "counts"),
            L.dev_ptr(ws), nbytes, L.stream_ptr()))
    return HardNegatives(o_cls, o_lp, o_tg, o_lt, o_cnt, o_mask, o_nsel, o_cut)


# ----------------------------------------------------------------------------------
# DynamicAnchorRouting, evaluation branch (SURVEY.md 8(f1))
# ----------------------------------------------------------------------------------
def routing_layers(feat_heights, feat_widths, anchor_depths, feat_strides):
    n = len(feat_heights)
    if not (len(feat_widths) == len(anchor_depths) == len(feat_strides) == n):
        raise ValueError("per-layer lists must have the same length")
    if not 1 <= n <= 16:
        raise ValueError("1..16 layers")
    lay = L.RoutingLayers()
    lay.num_layers = n
    for i in range(n):
        lay.feat_height[i], lay.feat_width[i] = int(feat_heights[i]), int(feat_widths[i])
        lay.anchor_depth[i], lay.feat_strides[i] = int(anchor_depths[i]), int(feat_strides[i])
    return lay


def dynamic_anchor_routing_eval(layers, anchors, gt_targets, labels, mask_in, workspace=None):
    """dan_dynamic_anchor_routing_eval: anchors / gt_targets [B, N, 4] (or [N, 4]), labels / mask_in [B, N] (or [N]).
    -> (mask_out int32, decode_out fp32) shaped like the inputs."""
    Lib = L.lib()
    L.require_device()
    dev = _dev(anchors)
    a = anchors.contiguous()
    t = gt_targets.contiguous()
    lb = labels.contiguous()
    m = mask_in.contiguous()
    n = sum(layers.feat_height[i] * layers.feat_width[i] * layers.anchor_depth[i] for i in range(layers.num_layers))
    total = lb.numel()
    if n <= 0 or total % n != 0:
        raise ValueError("labels has %d elements, the layers hold %d anchors" % (total, n))
    batch = total // n
    if a.numel() != total * 4 or t.numel() != total * 4 or m.numel() != total:
        raise ValueError("anchors and gt_targets must be [.., 4] and mask_in like labels")
    mask_out = torch.empty(lb.shape, dtype=torch.int32, device=dev)
    decode_out = torch.empty(a.shape, dtype=torch.float32, device=dev)
    nbytes = Lib.dan_routing_workspace_bytes(n, batch)
    ws = (workspace or _ws).get(nbytes, dev)
    with torch.cuda.device(dev):
        L.check(Lib.dan_dynamic_anchor_routing_eval(
            ctypes.byref(layers), L.dev_ptr(a, torch.float32, "anchors"), L.dev_ptr(t, torch.float32, "gt_targets"),
            L.dev_ptr(lb, torch.float32, "labels"), L.dev_ptr(m, torch.int32, "mask_in"), n, batch, L.dev_ptr(mask_out),
            L.dev_ptr(decode_out), L.dev_ptr(ws), nbytes, L.stream_ptr()))
    return mask_out, decode_out


# ----------------------------------------------------------------------------------
# evaluation merge: detect_face top-k + bbox_vote (SURVEY.md 8(f2))
# ----------------------------------------------------------------------------------
def detect_face_select(bboxes, scores, shrink, top):
    """dan_detect_face_select -> (det [top, 5] zero padded, index int32 [top] (-1 padded), count int32 [1])."""
    L.require_device()
    dev = _dev(bboxes)
    b = bboxes.contiguous()
    s = scores.contiguous()
    n = s.numel()
    det = torch.empty((top, 5), dtype=torch.float32, device=dev)
    idx = torch.empty(top, dtype=torch.int32, device=dev)
    cnt = torch.empty(1, dtype=torch.int32, device=dev)
    nbytes = L.lib().dan_detect_face_workspace_bytes(n)
    ws = _ws.get(nbytes, dev)
    with torch.cuda.device(dev):
        L.check(L.lib().dan_detect_face_select(L.dev_ptr(b, torch.float32, "bboxes"), L.dev_ptr(s, torch.float32, "scores"), n,
                                               float(shrink), int(top), L.dev_ptr(det), L.dev_ptr(idx), L.dev_ptr(cnt),
                                               L.dev_ptr(ws), nbytes, L.stream_ptr()))
    return det, idx, cnt


def detect_face_batch(cls_pred, loc_pred, anchors, shrink, top, prior_scaling=(0.1, 0.1, 0.2, 0.2), workspace=None):
    """dan_detect_face_batch: softmax + decode + detect_face of B images from the head's raw outputs, fused.
    cls_pred [B, N, 2] logits and loc_pred [B, N, 4] offsets, one dtype out of fp32 / fp16 / bf16; anchors =
    (ymin, xmin, ymax, xmax) [N] each.  -> (det [B, top, 5] zero padded, index int32 [B, top] (-1 padded), k) where
    k = max(min(N - 1, top), 0) valid rows per image.  Nothing synchronises with the host."""
    L.require_device()
    cls_pred = cls_pred.contiguous()
    loc_pred = loc_pred.contiguous()
    dtype = L.pred_dtype(cls_pred, "cls_pred")
    if loc_pred.dtype != cls_pred.dtype:
        raise TypeError("cls_pred is %s but loc_pred is %s: the predictions must share one dtype" % (cls_pred.dtype, loc_pred.dtype))
    if cls_pred.dim() != 3 or cls_pred.shape[2] != 2:
        raise ValueError("cls_pred must be [batch, num_anchors, 2], got %s" % (tuple(cls_pred.shape),))
    batch, n = int(cls_pred.shape[0]), int(cls_pred.shape[1])
    if tuple(loc_pred.shape) != (batch, n, 4):
        raise ValueError("loc_pred must be [%d, %d, 4], got %s" % (batch, n, tuple(loc_pred.shape)))
    if any(a.numel() != n for a in anchors):
        raise ValueError("cls_pred has %d anchors per image but there are %d anchors" % (n, anchors[0].numel()))
    dev = _dev(cls_pred)
    _dev(loc_pred)
    top = int(top)
    det = torch.empty((batch, top, 5), dtype=torch.float32, device=dev)
    idx = torch.empty((batch, top), dtype=torch.int32, device=dev)
    nbytes = L.lib().dan_detect_face_batch_workspace_bytes(n, batch)
    ws = (workspace or _ws).get(nbytes, dev)
    ps = (ctypes.c_float * 4)(*[float(v) for v in prior_scaling])
    with torch.cuda.device(dev):
        L.check(L.lib().dan_detect_face_batch(dtype, L.dev_ptr(cls_pred, cls_pred.dtype, "cls_pred"),
                                              L.dev_ptr(loc_pred, cls_pred.dtype, "loc_pred"), *_anchor_ptrs(*anchors), n, batch,
                                              ps, float(shrink), top, L.dev_ptr(det), L.dev_ptr(idx), L.dev_ptr(ws), nbytes,
                                              L.stream_ptr()))
    return det, idx, max(min(n - 1, top), 0)


def bbox_vote_batch(det, counts, nms_threshold, max_per_image, details=False):
    """dan_bbox_vote: det [B, cap, 5], counts int32 [B] or None -> (out [B, max_per_image, 5], out_count int32 [B]
    [, order int32 [B, cap], assign int32 [B, cap]])."""
    L.require_device()
    dev = _dev(det)
    d = det.contiguous()
    if d.dim() != 3 or d.shape[2] != 5:
        raise ValueError("det must be [B, capacity, 5]")
    batch, cap = int(d.shape[0]), int(d.shape[1])
    out = torch.empty((batch, max_per_image, 5), dtype=torch.float32, device=dev)
    cnt = torch.empty(batch, dtype=torch.int32, device=dev)
    order = torch.full((batch, cap), -1, dtype=torch.int32, device=dev) if details else None
    assign = torch.full((batch, cap), -1, dtype=torch.int32, device=dev) if details else None
    c = counts.contiguous() if counts is not None else None
    with torch.cuda.device(dev):
        L.check(L.lib().dan_bbox_vote(L.dev_ptr(d, torch.float32, "det"), L.dev_ptr(c, torch.int32, "counts"), batch, cap,
                                      float(nms_threshold), int(max_per_image), L.dev_ptr(out), L.dev_ptr(cnt),
                                      L.dev_ptr(order), L.dev_ptr(assign), L.stream_ptr()))
    return (out, cnt, order, assign) if details else (out, cnt)


# ----------------------------------------------------------------------------------
# input hand-off (SURVEY.md 8(f4))
# ----------------------------------------------------------------------------------
def gt_handoff(gt_boxes, gt_offsets, patch_hw, out_shape, mirror=None, min_height=6., min_width=3.):
    """dan_gt_handoff -> (gt_boxes [total,4] capacity, gt_offsets int32 [B+1] capacity, image_index int32 [B],
    counts int32 [2] = (kept images, kept boxes)); nothing synchronises."""
    L.require_device()
    dev = _dev(gt_offsets)
    g = gt_boxes.contiguous()
    o = gt_offsets.contiguous()
    hw = patch_hw.contiguous()
    batch = o.numel() - 1
    total = g.numel() // 4
    m = None
    if mirror is not None:
        m = mirror.to(torch.uint8).contiguous()
        if m.numel() != batch:
            raise ValueError("mirror must have one entry per image")
    if hw.numel() != 2 * batch:
        raise ValueError("patch_hw must be [B, 2]")
    ob = torch.empty((total, 4), dtype=torch.float32, device=dev)
    oo = torch.zeros(batch + 1, dtype=torch.int32, device=dev)
    oi = torch.full((batch,), -1, dtype=torch.int32, device=dev)
    oc = torch.empty(2, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.lib().dan_gt_handoff(L.dev_ptr(g, torch.float32, "gt_boxes") if total else ctypes.c_void_p(0),
                                       L.dev_ptr(o, torch.int32, "gt_offsets"), L.dev_ptr(hw, torch.float32, "patch_hw"),
                                       L.dev_ptr(m, torch.uint8, "mirror"), batch, total, float(out_shape[0]), float(out_shape[1]),
                                       float(min_height), float(min_width), L.dev_ptr(ob) if total else ctypes.c_void_p(0),
                                       L.dev_ptr(oo), L.dev_ptr(oi), L.dev_ptr(oc), L.stream_ptr()))
    return ob, oo, oi, oc
