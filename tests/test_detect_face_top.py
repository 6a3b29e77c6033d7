"""detect_face with more than 8192 rows per image (dan_detect_face_batch_top, dan_detect_face_select_top): the rows, scores
and anchor indices must equal the numpy oracle's (softmax -> decode_anchors -> detect_face_select) BIT FOR BIT, fp16 /
bf16 must equal the fp32 call on the widened tensors, and for top <= 8192 the new entry points must give the bits of the
old ones."""
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
TOPS = [8193, 16384, 98302]                   # 98302 = int(1.5 * 65535), bbox_vote's largest max_per_image


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _assert_same(got, ref, what=""):
    assert torch.equal(_bits(got[0]), _bits(ref[0])), what + " det"
    assert torch.equal(got[1], ref[1]), what + " index"


def _anchors_np(oracle, size):
    return synthetic.build_anchors(oracle.AnchorEncoder(None, None, PS), synthetic.pyramid_config("s3fd", size, border=0.))[:4]


def _predictions(a_np, size, B, seed, faces=300):
    an = np.stack(a_np, -1)
    preds = [synthetic.gen_predictions(seed + i, an, size=size, max_faces=faces) for i in range(B)]
    return np.stack([p[0] for p in preds]), np.stack([p[1] for p in preds])


def _oracle_order(oracle, cls, loc, a_np, shrink):
    """per image: the oracle's rows and anchor indices of ALL anchors in descending score order"""
    enc = oracle.AnchorEncoder(None, None, PS)
    return [oracle.detect_face_select(enc.decode_anchors(loc[b], *a_np), oracle.softmax(cls[b])[:, 1], shrink, 1 << 30)
            for b in range(cls.shape[0])]


def _check(ref, det, idx, top):
    n1 = ref[0][0].shape[0]                   # N - 1 rows: the reference keeps at most N - 1
    k = min(n1, top)
    assert det.shape[1:] == (top, 5) and idx.shape[1:] == (top,)
    d, i = det.cpu().numpy(), idx.cpu().numpy()
    for b, (rows, keep) in enumerate(ref):
        np.testing.assert_array_equal(d[b, :k].view(np.uint32), rows[:k].view(np.uint32))
        np.testing.assert_array_equal(i[b, :k], keep[:k])
        assert not d[b, k:].any() and (i[b, k:] == -1).all()
    return k


@pytest.mark.parametrize("dtype", [torch.float32] + HALF)
@pytest.mark.parametrize("size,B", [((1024, 1024), 3), ((1600, 1600), 2)])
def test_vs_oracle(cuda, oracle, size, B, dtype):
    """S3FD anchors (N = 87 360 at 1024^2, 213 294 at 1600^2); at 1024^2 top = 98 302 keeps all N - 1 rows.  Half
    predictions: the oracle runs on the widened values."""
    from dan_b200 import functional as F
    a_np = _anchors_np(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np]
    cls, loc = _predictions(a_np, size, B, 700 + size[0])
    cls_d, loc_d = to_dev(cls, cuda).to(dtype), to_dev(loc, cuda).to(dtype)
    if dtype != torch.float32:
        cls, loc = cls_d.float().cpu().numpy(), loc_d.float().cpu().numpy()
    ref = _oracle_order(oracle, cls, loc, a_np, 1.25)
    for top in TOPS:
        det, idx, k = F.detect_face_batch(cls_d, loc_d, anchors, 1.25, top, PS)
        assert k == _check(ref, det, idx, top) and k > K_SORT_CAP
        if dtype != torch.float32:
            _assert_same((det, idx), F.detect_face_batch(cls_d.float(), loc_d.float(), anchors, 1.25, top, PS)[:2],
                         "%s top %d" % (dtype, top))


@pytest.mark.parametrize("dtype", HALF)
def test_half_specials_equal_widened(cuda, oracle, dtype):
    """NaN, +-inf, signed zeros and subnormals in the logits and offsets, rows beyond 8192 included; the logits one
    element into their storage (no pair aligned for one load): the fp32 call on the widened values, bit for bit."""
    from dan_b200 import functional as F
    size = (640, 640)
    a_np = _anchors_np(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np]
    B = 3
    cls, loc = _predictions(a_np, size, B, 520)
    rng = np.random.default_rng(9)
    n = cls.shape[1]
    sub = 1e-7 if dtype == torch.float16 else 1e-39
    special = [np.inf, -np.inf, 0.0, -0.0, np.nan, sub, -sub, 6e4]
    for j, a in enumerate(rng.choice(n, 3000, replace=False)):
        b = j % B
        cls[b, a, j % 2] = special[j % len(special)]
        if j % 3 == 0:
            loc[b, a, (j // 3) % 4] = special[(j // 3) % len(special)]
    cls_h, loc_h = to_dev(cls, cuda).to(dtype), to_dev(loc, cuda).to(dtype)
    store = torch.empty(cls_h.numel() + 1, dtype=dtype, device=cuda)
    off = store[1:].view(cls_h.shape)
    off.copy_(cls_h)
    for top in (16384, 30000):
        ref = F.detect_face_batch(cls_h.float(), loc_h.float(), anchors, 0.75, top, PS)
        got = F.detect_face_batch(cls_h, loc_h, anchors, 0.75, top, PS)
        assert ref[2] == top
        _assert_same(got, ref, "%s top %d" % (dtype, top))
        _assert_same(F.detect_face_batch(off, loc_h, anchors, 0.75, top, PS), ref, "%s one element off" % dtype)
        assert torch.isnan(ref[0][:, :, 4]).any()                # NaN scores are among the rows, with their payloads


def _random_case(rng, B, n):
    cls = rng.normal(0, 2, (B, n, 2)).astype(np.float32)
    loc = rng.normal(0, 0.5, (B, n, 4)).astype(np.float32)
    c = rng.uniform(0, 640, (n, 2))
    wh = rng.uniform(4, 80, (n, 2))
    a = np.concatenate([c - wh / 2, c + wh / 2], -1).astype(np.float32)
    return cls, loc, [a[:, i].copy() for i in range(4)]


@pytest.mark.parametrize("ties", [12000, 30000])
def test_ties_across_the_boundary(cuda, oracle, ties):
    """Equal top scores across the k-th row, k = 10 000: the higher index comes first.  12 000 ties fit the candidate
    area (2k keys); 30 000 keys in the k-th key's bin do not, and the select runs over all of the image's keys."""
    from dan_b200 import functional as F
    rng = np.random.default_rng(ties)
    B, n, top = 2, 60000, 10000
    cls, loc, a_np = _random_case(rng, B, n)
    for b in range(B):
        cls[b, rng.choice(n, ties, replace=False)] = [-10.0, 10.0]   # p rounds to 1.0: above every random anchor
    anchors = [to_dev(v, cuda) for v in a_np]
    det, idx, k = F.detect_face_batch(to_dev(cls, cuda), to_dev(loc, cuda), anchors, 1.0, top, PS)
    _check(_oracle_order(oracle, cls, loc, a_np, 1.0), det, idx, top)
    assert (np.diff(idx.cpu().numpy(), axis=1) < 0).all()         # all k rows are ties: descending indices


@pytest.mark.parametrize("n,top", [(34125, 1125), (34125, K_SORT_CAP), (5000, 98302)])
def test_small_k_same_as_old_entry_points(cuda, n, top):
    """k <= 8192 (also with top above 8192 and N - 1 below it): dan_detect_face_batch_top gives the bits of
    dan_detect_face_batch, dan_detect_face_select_top those of dan_detect_face_select (at top 8192 when top is larger:
    the rows beyond are padding)."""
    from dan_b200 import _lib as L, functional as F
    rng = np.random.default_rng(n + top)
    B = 2
    cls_np, loc_np, a_np = _random_case(rng, B, n)
    cls, loc = to_dev(cls_np, cuda), to_dev(loc_np, cuda)
    anchors = [to_dev(v, cuda) for v in a_np]
    det, idx, k = F.detect_face_batch(cls, loc, anchors, 0.75, top, PS)
    assert k == min(n - 1, top) <= K_SORT_CAP
    assert L.lib().dan_detect_face_top_workspace_bytes(n, B, top) == L.lib().dan_detect_face_batch_workspace_bytes(n, B)
    t0 = min(top, K_SORT_CAP)
    assert not det[:, t0:].any() and bool((idx[:, t0:] == -1).all())
    nb = L.lib().dan_detect_face_batch_workspace_bytes(n, B)
    ws = torch.empty(nb, dtype=torch.uint8, device=cuda)
    d0 = torch.full((B, t0, 5), 3.0, device=cuda)
    i0 = torch.full((B, t0), 5, dtype=torch.int32, device=cuda)
    ps = (ctypes.c_float * 4)(*PS)
    L.check(L.lib().dan_detect_face_batch(L.DAN_DTYPE_F32, L.dev_ptr(cls), L.dev_ptr(loc), *[L.dev_ptr(a) for a in anchors], n, B,
                                          ps, 0.75, t0, L.dev_ptr(d0), L.dev_ptr(i0), L.dev_ptr(ws), nb, L.stream_ptr()))
    _assert_same((det[:, :t0], idx[:, :t0]), (d0, i0), "batch n %d top %d" % (n, top))
    scores = F.softmax(cls[0])[:, 1].contiguous()
    boxes = F.decode_batch(loc[:1], *anchors, PS)[0].contiguous()
    d1, i1, c1 = F.detect_face_select(boxes, scores, 0.75, top)
    assert int(c1) == k
    _assert_same((d1[None], i1[None]), (det[:1], idx[:1]), "select_top vs batch_top")
    nb = L.lib().dan_detect_face_workspace_bytes(n)
    ws = torch.empty(nb, dtype=torch.uint8, device=cuda)
    d2 = torch.full((t0, 5), 3.0, device=cuda)
    i2 = torch.full((t0,), 5, dtype=torch.int32, device=cuda)
    c2 = torch.zeros(1, dtype=torch.int32, device=cuda)
    L.check(L.lib().dan_detect_face_select(L.dev_ptr(boxes), L.dev_ptr(scores), n, 0.75, t0, L.dev_ptr(d2), L.dev_ptr(i2),
                                           L.dev_ptr(c2), L.dev_ptr(ws), nb, L.stream_ptr()))
    _assert_same((d1[:t0], i1[:t0]), (d2, i2), "select n %d top %d" % (n, top))
    assert int(c2) == k


@pytest.mark.parametrize("max_per_image", [6000, 65535])
def test_select_top_on_decoded_boxes(cuda, oracle, max_per_image):
    """dan_detect_face_select_top (DAN's stage-2 path: boxes already decoded) with k > 8192, through eval_merge"""
    from dan_b200 import functional as F
    from dan_b200.utility import eval_merge
    size = (1024, 1024)
    a_np = _anchors_np(oracle, size)
    cls, loc = _predictions(a_np, size, 1, 41)
    enc = oracle.AnchorEncoder(None, None, PS)
    scores = oracle.softmax(cls[0])[:, 1]
    boxes = enc.decode_anchors(loc[0], *a_np)
    ref, keep = oracle.detect_face_select(boxes, scores, 1.5, max_per_image)
    assert ref.shape[0] > K_SORT_CAP
    got = eval_merge.detect_face_select(to_dev(boxes, cuda), to_dev(scores, cuda), 1.5, max_per_image)
    np.testing.assert_array_equal(got.cpu().numpy().view(np.uint32), ref.view(np.uint32))
    top = int(max_per_image * 1.5)
    _, idx, cnt = F.detect_face_select(to_dev(boxes, cuda), to_dev(scores, cuda), 1.5, top)
    assert int(cnt) == ref.shape[0]
    np.testing.assert_array_equal(idx[:int(cnt)].cpu().numpy(), keep)


def test_cuda_graph_replay_new_inputs(cuda, oracle):
    from dan_b200 import _lib as L, functional as F
    size = (640, 640)
    a_np = _anchors_np(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np]
    B, top = 3, 16384
    inputs = [tuple(to_dev(x, cuda).to(torch.bfloat16) for x in _predictions(a_np, size, B, seed)) for seed in (70, 80, 90)]
    cls, loc = (t.clone() for t in inputs[0])
    ws = L.Workspace()
    F.detect_face_batch(cls, loc, anchors, 1.5, top, PS, workspace=ws)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            out = F.detect_face_batch(cls, loc, anchors, 1.5, top, PS, workspace=ws)
    torch.cuda.current_stream().wait_stream(side)
    for c, l in inputs[1:] + inputs[:1]:
        cls.copy_(c)
        loc.copy_(l)
        out[0].fill_(-7.0)
        out[1].fill_(-7)
        g.replay()
        torch.cuda.synchronize()
        _assert_same(out, F.detect_face_batch(c, l, anchors, 1.5, top, PS), "graph replay")
    del g


def test_chain_two_passes_into_large_vote(cuda, oracle):
    """Two passes at max_per_image = 6000 (9 000 rows each) stacked with torch.cat(dim=1) into bbox_vote_batch, which
    takes its large path (18 000 rows per image), against the oracle chain per image."""
    from dan_b200.utility import eval_merge
    size = (640, 640)
    a_np = _anchors_np(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np]
    enc = oracle.AnchorEncoder(None, None, PS)
    B, mpi = 2, 6000
    passes = []
    for p, shrink in enumerate((0.5, 1.0)):
        cls, loc = _predictions(a_np, size, B, 60 + 10 * p, faces=30)
        passes.append((cls, loc, shrink))
    det = torch.cat([eval_merge.detect_face_batch(to_dev(c, cuda), to_dev(l, cuda), anchors, s, max_per_image=mpi)
                     for c, l, s in passes], dim=1)
    assert det.shape == (B, 2 * 9000, 5)
    out, cnt = eval_merge.bbox_vote_batch(det, None, max_per_image=mpi)
    for b in range(B):
        stack = np.concatenate([oracle.detect_face_select(enc.decode_anchors(l[b], *a_np), oracle.softmax(c[b])[:, 1], s, mpi)[0]
                                for c, l, s in passes])
        ref = oracle.bbox_vote(stack, max_per_image=mpi)
        m = int(cnt[b])
        assert m == ref.shape[0] and m > 0
        np.testing.assert_array_equal(out[b, :m].cpu().numpy().view(np.uint32), ref.view(np.uint32))
