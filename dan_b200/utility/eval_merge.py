"""Drop-in for the detection merge of the reference's evaluation scripts (SURVEY.md 8(f2)).

    detect_face_select   the numpy part of detect_face, eval_sfd.py:101-112 (= eval_dan.py:101-118): after net.run
    detect_face_batch    softmax + decode_anchors + detect_face of a batch, from the head's logits and offsets
    bbox_vote            eval_sfd.py:170-210 (= eval_dan.py:201-241)

Detections are rows (xmin, ymin, xmax, ymax, score), float32, +1 pixel convention, like the reference's numpy arrays;
here they are CUDA tensors and stay on the device.  ``FLAGS.max_per_image`` / ``FLAGS.nms_threshold`` become keyword
arguments (750 / 0.3, eval_sfd.py:62-66)."""
from __future__ import annotations

import torch

from .. import _lib as L
from .. import functional as F


def detect_face_select(bboxes, scores, shrink, max_per_image=750):
    """bboxes [n, 4] (ymin, xmin, ymax, xmax) and scores [n] as returned by the network -> det [k, 5] with
    k = min(n - 1, int(max_per_image * 1.5)), sorted by descending score (equal scores: higher index first; the
    reference's default argsort leaves ties unspecified).  One host read (k)."""
    top = int(max_per_image * 1.5)
    det, _, cnt = F.detect_face_select(L.as_f32(bboxes), L.as_f32(scores), shrink, top)
    return det[:int(cnt)]


def detect_face_batch(cls_pred, loc_pred, anchors, shrink, max_per_image=750, prior_scaling=(0.1, 0.1, 0.2, 0.2)):
    """The evaluation scripts' whole per-pass chain - softmax (eval_sfd.py:279), decode_anchors (:283) and
    detect_face (:95-114) - for a batch, from the head's raw outputs: cls_pred [B, N, 2] logits and loc_pred [B, N, 4]
    offsets (fp32, fp16 or bf16, one dtype), anchors (ymin, xmin, ymax, xmax) -> det [B, k, 5] rows
    (xmin, ymin, xmax, ymax, score) with k = min(N - 1, int(max_per_image * 1.5)), sorted by descending score (equal
    scores: higher index first).  No host read: the passes of one batch (scales, flips) are stacked with
    torch.cat(dim=1) and go straight into bbox_vote_batch(det, None)."""
    det, _, k = F.detect_face_batch(cls_pred, loc_pred, anchors, shrink, int(max_per_image * 1.5), prior_scaling)
    return det[:, :k]


def bbox_vote(det, nms_threshold=0.3, max_per_image=750):
    """det [n, 5] -> merged detections [m, 5] (m <= max_per_image).  One host read (m)."""
    det = L.as_f32(det)
    if det.shape[0] == 0:
        return det.new_zeros((0, 5))
    out, cnt = F.bbox_vote_batch(det.reshape(1, -1, 5), None, nms_threshold, max_per_image)
    return out[0, :int(cnt[0])]


def bbox_vote_batch(det, counts, nms_threshold=0.3, max_per_image=750):
    """Many images at once, nothing synchronises: det [B, capacity, 5] (rows beyond counts[b] are ignored), counts
    int32 [B] -> (out [B, max_per_image, 5] zero padded, out_count int32 [B])."""
    return F.bbox_vote_batch(L.as_f32(det), None if counts is None else counts.to(torch.int32), nms_threshold, max_per_image)
