"""dan_detect_face_batch: softmax + decode + detect_face of a batch from the head's raw outputs, fused.

For fp32 the rows and indices must equal the composition softmax -> decode_batch -> detect_face_select per image BIT FOR
BIT (int32 views of the floats); fp16 / bf16 must equal the fp32 call on the widened tensors; one image at 1600^2 is
checked against the numpy oracle."""
import ctypes

import numpy as np
import pytest
import torch

from dan_b200 import synthetic

from conftest import to_dev

pytestmark = pytest.mark.gpu
PS = [0.1, 0.1, 0.2, 0.2]
HALF = [torch.float16, torch.bfloat16]
K_SORT_CAP = 8192


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _anchors_np(oracle, size):
    return synthetic.build_anchors(oracle.AnchorEncoder(None, None, PS), synthetic.pyramid_config("s3fd", size, border=0.))


def _predictions(a_np, size, B, seed, faces=80):
    an = np.stack(a_np[:4], -1)
    preds = [synthetic.gen_predictions(seed + i, an, size=size, max_faces=faces) for i in range(B)]
    return np.stack([p[0] for p in preds]), np.stack([p[1] for p in preds])


def _offset_view(t, elements):
    """t's values in a tensor whose storage starts `elements` elements before it (a misaligned view)."""
    store = torch.empty(t.numel() + elements, dtype=t.dtype, device=t.device)
    v = store[elements:].view(t.shape)
    v.copy_(t)
    return v


def _composition(cls, loc, anchors, shrink, top):
    """The chain the evaluation scripts run, one entry point per step: softmax, decode, per-image select."""
    from dan_b200 import functional as F
    scores = F.softmax(cls)[..., 1]
    boxes = F.decode_batch(loc, *anchors, PS)
    dets, idxs = [], []
    for b in range(cls.shape[0]):
        d, i, _ = F.detect_face_select(boxes[b], scores[b], shrink, top)
        dets.append(d)
        idxs.append(i)
    return torch.stack(dets), torch.stack(idxs)


def _assert_same(got, ref, what=""):
    det, idx = got[0], got[1]
    assert torch.equal(_bits(det), _bits(ref[0])), what + " det"
    assert torch.equal(idx, ref[1]), what + " index"


@pytest.mark.parametrize("size,B", [((640, 640), 8), ((1024, 768), 2)])
def test_fp32_equals_composition(cuda, oracle, size, B):
    from dan_b200 import functional as F
    a_np = _anchors_np(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np[:4]]
    cls, loc = _predictions(a_np, size, B, 300)
    cls, loc = to_dev(cls, cuda), to_dev(loc, cuda)
    n = cls.shape[1]
    for shrink in (0.5, 1.0, 1.75):
        det, idx, k = F.detect_face_batch(cls, loc, anchors, shrink, 1125, PS)
        assert k == 1125 and det.shape == (B, 1125, 5) and idx.shape == (B, 1125)
        _assert_same((det, idx), _composition(cls, loc, anchors, shrink, 1125), "shrink %g" % shrink)
        assert int(idx.min()) >= 0 and int(idx.max()) < n


def test_oracle_1600(cuda, oracle):
    from dan_b200.utility import eval_merge
    size = (1600, 1600)
    a_np = _anchors_np(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np[:4]]
    cls, loc = _predictions(a_np, size, 1, 910, faces=300)
    enc = oracle.AnchorEncoder(None, None, PS)
    scores = oracle.softmax(cls[0])[:, 1]
    boxes = enc.decode_anchors(loc[0], *a_np[:4])
    ref, keep = oracle.detect_face_select(boxes, scores, 1.25)
    det = eval_merge.detect_face_batch(to_dev(cls, cuda), to_dev(loc, cuda), anchors, 1.25)
    assert det.shape == (1,) + ref.shape
    np.testing.assert_array_equal(det[0].cpu().numpy().view(np.uint32), ref.view(np.uint32))
    from dan_b200 import functional as F
    _, idx, k = F.detect_face_batch(to_dev(cls, cuda), to_dev(loc, cuda), anchors, 1.25, 1125)
    np.testing.assert_array_equal(idx[0, :k].cpu().numpy(), keep)


@pytest.mark.parametrize("dtype", HALF)
def test_half_equals_widened(cuda, oracle, dtype):
    """NaN, +-inf, signed zeros and subnormals in the logits and the offsets; cls_pred views one element into their
    storage (no logit pair aligned for one load)."""
    from dan_b200 import functional as F
    size = (640, 640)
    a_np = _anchors_np(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np[:4]]
    B = 3
    cls, loc = _predictions(a_np, size, B, 520)
    rng = np.random.default_rng(8)
    n = cls.shape[1]
    sub = 1e-7 if dtype == torch.float16 else 1e-39
    special = [np.inf, -np.inf, 0.0, -0.0, np.nan, sub, -sub, 6e4]
    idx = rng.choice(n, 400, replace=False)
    for j, a in enumerate(idx):
        b = j % B
        cls[b, a, j % 2] = special[j % len(special)]
        if j % 3 == 0:
            cls[b, a] = [-20.0, 20.0]                             # a top score whose offset row carries the special value
            loc[b, a, (j // 3) % 4] = special[(j // 3) % len(special)]
    cls_h, loc_h = to_dev(cls, cuda).to(dtype), to_dev(loc, cuda).to(dtype)
    for shrink in (0.5, 1.75):
        ref = F.detect_face_batch(cls_h.float(), loc_h.float(), anchors, shrink, 1125, PS)
        got = F.detect_face_batch(cls_h, loc_h, anchors, shrink, 1125, PS)
        _assert_same(got, ref, "%s shrink %g" % (dtype, shrink))
        _assert_same(ref, _composition(cls_h.float(), loc_h.float(), anchors, shrink, 1125), "fp32 composition")
        off = _offset_view(cls_h, 1)
        assert off.data_ptr() % 4 == 2
        _assert_same(F.detect_face_batch(off, loc_h, anchors, shrink, 1125, PS), ref, "%s one element off" % dtype)
    # fp32 logits one element off (pairs 4-byte aligned only)
    cls32 = to_dev(cls, cuda)
    off32 = _offset_view(cls32, 1)
    assert off32.data_ptr() % 8 == 4
    _assert_same(F.detect_face_batch(off32, to_dev(loc, cuda), anchors, 1.0, 1125, PS),
                 F.detect_face_batch(cls32, to_dev(loc, cuda), anchors, 1.0, 1125, PS), "fp32 one element off")


def _random_case(rng, B, n):
    cls = rng.normal(0, 2, (B, n, 2)).astype(np.float32)
    loc = rng.normal(0, 0.5, (B, n, 4)).astype(np.float32)
    c = rng.uniform(0, 640, (n, 2))
    wh = rng.uniform(4, 80, (n, 2))
    a = np.concatenate([c - wh / 2, c + wh / 2], -1).astype(np.float32)
    return cls, loc, [a[:, i].copy() for i in range(4)]


def _check_vs_oracle(oracle, cls, loc, a_np, shrink, top, det, idx):
    enc = oracle.AnchorEncoder(None, None, PS)
    k = max(min(cls.shape[1] - 1, top), 0)
    for b in range(cls.shape[0]):
        ref, keep = oracle.detect_face_select(enc.decode_anchors(loc[b], *a_np), oracle.softmax(cls[b])[:, 1], shrink, 1 << 30)
        ref, keep = ref[:k], keep[:k]                             # (the full descending order, cut at k)
        np.testing.assert_array_equal(det[b, :k].cpu().numpy().view(np.uint32), ref.view(np.uint32))
        np.testing.assert_array_equal(idx[b, :k].cpu().numpy(), keep)
        assert not det[b, k:].any() and bool((idx[b, k:] == -1).all())


def test_ties_across_the_boundary(cuda, oracle):
    """Equal logits across the k-th row: the higher index comes first.  2 000 equal top scores fit the select's shared
    memory; 12 000 equal scores (one histogram bin beyond 8192 keys) take the radix select over all keys."""
    from dan_b200 import functional as F
    rng = np.random.default_rng(21)
    B, n = 2, 30000
    cls, loc, a_np = _random_case(rng, B, n)
    anchors = [to_dev(v, cuda) for v in a_np]
    for ties in (2000, 12000):
        c = cls.copy()
        for b in range(B):
            c[b, rng.choice(n, ties, replace=False)] = [-10.0, 10.0]  # p rounds to 1.0: above every random anchor
        det, idx, k = F.detect_face_batch(to_dev(c, cuda), to_dev(loc, cuda), anchors, 1.0, 1125, PS)
        _check_vs_oracle(oracle, c, loc, a_np, 1.0, 1125, det, idx)
        i = idx.cpu().numpy()
        assert (np.diff(i, axis=1) < 0).all()                     # all 1125 rows are ties: descending indices
        _assert_same((det, idx), _composition(to_dev(c, cuda), to_dev(loc, cuda), anchors, 1.0, 1125), "ties %d" % ties)


@pytest.mark.parametrize("n,top", [(1, 1125), (2, 1125), (1125, 1125), (1126, 1125), (34125, K_SORT_CAP), (9000, 10)])
def test_edges(cuda, oracle, n, top):
    from dan_b200 import functional as F
    rng = np.random.default_rng(n)
    B = 3
    cls, loc, a_np = _random_case(rng, B, n)
    anchors = [to_dev(v, cuda) for v in a_np]
    det, idx, k = F.detect_face_batch(to_dev(cls, cuda), to_dev(loc, cuda), anchors, 0.75, top, PS)
    assert k == max(min(n - 1, top), 0) and det.shape == (B, top, 5)
    if k == 0:
        assert not det.any() and bool((idx == -1).all())
    _check_vs_oracle(oracle, cls, loc, a_np, 0.75, top, det, idx)
    _assert_same((det, idx), _composition(to_dev(cls, cuda), to_dev(loc, cuda), anchors, 0.75, top), "n %d" % n)


def test_merge_of_three_passes(cuda, oracle):
    """Three passes of one batch stacked with torch.cat(dim=1) and voted in one launch equal the per-image old chain
    (decoded boxes -> detect_face_select -> stack -> bbox_vote)."""
    from dan_b200 import functional as F
    from dan_b200.utility import eval_merge
    size = (640, 640)
    a_np = _anchors_np(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np[:4]]
    B = 3
    passes = []
    for p, shrink in enumerate((0.5, 1.0, 1.75)):
        cls, loc = _predictions(a_np, size, B, 40 + 10 * p, faces=30)
        passes.append((to_dev(cls, cuda), to_dev(loc, cuda), shrink))
    det = torch.cat([eval_merge.detect_face_batch(c, l, anchors, s) for c, l, s in passes], dim=1)
    assert det.shape == (B, 3 * 1125, 5)
    out, cnt = eval_merge.bbox_vote_batch(det, None)
    for b in range(B):
        rows = []
        for c, l, s in passes:
            scores = F.softmax(c[b])[:, 1]
            boxes = F.decode_batch(l[b:b + 1], *anchors, PS)[0]
            rows.append(eval_merge.detect_face_select(boxes, scores, s))
        ref = eval_merge.bbox_vote(torch.cat(rows, 0))
        m = int(cnt[b])
        assert m == ref.shape[0] and m > 0
        assert torch.equal(_bits(out[b, :m]), _bits(ref))


def test_cuda_graph(cuda, oracle):
    from dan_b200 import _lib as L, functional as F
    size = (640, 640)
    a_np = _anchors_np(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np[:4]]
    cls, loc = _predictions(a_np, size, 4, 70)
    cls, loc = to_dev(cls, cuda).to(torch.bfloat16), to_dev(loc, cuda).to(torch.bfloat16)
    ref = F.detect_face_batch(cls, loc, anchors, 1.5, 1125, PS)
    ws = L.Workspace()
    F.detect_face_batch(cls, loc, anchors, 1.5, 1125, PS, workspace=ws)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            out = F.detect_face_batch(cls, loc, anchors, 1.5, 1125, PS, workspace=ws)
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(2):
        out[0].fill_(-7.0)
        out[1].fill_(-7)
        g.replay()
        torch.cuda.synchronize()
        _assert_same(out, ref, "graph replay")
    del g


def test_errors(cuda):
    from dan_b200 import _lib as L, functional as F
    rng = np.random.default_rng(4)
    n, B = 777, 2
    cls_np, loc_np, a_np = _random_case(rng, B, n)
    cls, loc = to_dev(cls_np, cuda), to_dev(loc_np, cuda)
    anchors = [to_dev(v, cuda) for v in a_np]
    with pytest.raises(TypeError):
        F.detect_face_batch(cls.double(), loc.double(), anchors, 1.0, 1125)
    for c, l in ((cls.half(), loc), (cls, loc.bfloat16()), (cls.half(), loc.bfloat16())):
        with pytest.raises(TypeError, match=str(c.dtype)) as e:
            F.detect_face_batch(c, l, anchors, 1.0, 1125)
        assert str(l.dtype) in str(e.value)
    with pytest.raises(ValueError):
        F.detect_face_batch(to_dev(rng.normal(size=(B, n, 3)).astype(np.float32), cuda), loc, anchors, 1.0, 1125)
    with pytest.raises(ValueError):
        F.detect_face_batch(cls, loc, [a[:-1].contiguous() for a in anchors], 1.0, 1125)
    # the C ABI: every refusal before anything is enqueued (the outputs keep their sentinel)
    det = torch.full((B, K_SORT_CAP + 1, 5), 3.0, device=cuda)
    idx = torch.full((B, K_SORT_CAP + 1), 5, dtype=torch.int32, device=cuda)
    nb = L.lib().dan_detect_face_batch_workspace_bytes(n, B)
    ws = torch.empty(nb, dtype=torch.uint8, device=cuda)
    ps = (ctypes.c_float * 4)(*PS)
    aptr = [L.dev_ptr(a) for a in anchors]

    def call(dtype, c, l, top=1125, nbytes=nb):
        return L.lib().dan_detect_face_batch(dtype, ctypes.c_void_p(c.data_ptr()), ctypes.c_void_p(l.data_ptr()), *aptr, n, B, ps,
                                             1.0, top, L.dev_ptr(det), L.dev_ptr(idx), L.dev_ptr(ws), nbytes, L.stream_ptr())
    assert call(7, cls, loc) == -1
    assert call(L.DAN_DTYPE_F32, cls, _offset_view(loc, 1)) == -1             # 4 bytes into a 16-byte row
    lh = loc.half()
    assert call(L.DAN_DTYPE_F16, cls.half(), _offset_view(lh, 2)) == -1       # 4 bytes into an 8-byte row
    assert call(L.DAN_DTYPE_F32, cls, loc, nbytes=nb - 1) == -2
    assert call(L.DAN_DTYPE_F32, cls, loc, top=0) == -4
    assert call(L.DAN_DTYPE_F32, cls, loc, top=K_SORT_CAP + 1) == -4
    torch.cuda.synchronize()
    assert bool((det == 3.0).all()) and bool((idx == 5).all())
    assert call(L.DAN_DTYPE_F32, cls, loc, top=K_SORT_CAP) == 0              # the largest top is accepted
    torch.cuda.synchronize()
    assert not bool((det == 3.0).all())
