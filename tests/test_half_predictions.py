"""fp16 / bf16 predictions in the batched postprocess and in decode (dan_postprocess_batch_typed,
dan_decode_batch_typed).  The kernels widen each prediction to fp32 as they load it, which is exact, and run the
fp32 code after the load, so every output must equal the fp32 call on `.float()` of the same half tensors BIT FOR BIT
(int32 views of the floats: NaN and signed zeros included)."""
import ctypes

import numpy as np
import pytest
import torch

from dan_b200 import synthetic

from conftest import to_dev

pytestmark = pytest.mark.gpu
PS = [0.1, 0.1, 0.2, 0.2]
HALF = [torch.float16, torch.bfloat16]
FIELDS = ("boxes", "scores", "counts", "anchor_index", "keep_pos")


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _assert_same(a, b, what=""):
    for name in FIELDS:
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None), name
        if x is not None:
            assert torch.equal(_bits(x), _bits(y)), "%s %s" % (what, name)


def _anchors(oracle, size):
    a_np = synthetic.build_anchors(oracle.AnchorEncoder(None, None, PS), synthetic.pyramid_config("s3fd", size, border=0.))
    return a_np


def _g3(a_np, size, B, seed, faces=80):
    an = np.stack(a_np[:4], -1)
    preds = [synthetic.gen_predictions(seed + i, an, size=size, max_faces=faces) for i in range(B)]
    return np.stack([p[0] for p in preds]), np.stack([p[1] for p in preds])


def _detector_logits(rng, B, N):
    """~5 % foreground anchors, the rest background: both sides of the quick reject."""
    x = np.stack([rng.normal(8, 1, (B, N)), rng.normal(0, 1, (B, N))], -1)
    fg = rng.random((B, N)) < 0.05
    x[fg] = np.stack([rng.normal(0, 1, fg.sum()), rng.normal(5, 1, fg.sum())], -1)
    return x.astype(np.float32)


def _random_boxes(rng, shape, extent):
    c = rng.uniform(0, extent, shape + (2,))
    wh = rng.uniform(4, 60, shape + (2,))
    return np.concatenate([c - wh / 2, c + wh / 2], -1).astype(np.float32)


def _offset_view(t, elements):
    """t's values in a tensor whose storage starts `elements` elements before it (a misaligned view)."""
    store = torch.empty(t.numel() + elements, dtype=t.dtype, device=t.device)
    v = store[elements:].view(t.shape)
    v.copy_(t)
    return v


@pytest.mark.parametrize("dtype", HALF)
def test_two_classes_fused_filter(cuda, oracle, dtype):
    from dan_b200.utility import bbox_util as bu
    size = (640, 640)
    a_np = _anchors(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np[:4]]
    cls, loc = _g3(a_np, size, 3, 700)
    cls_h, loc_h = to_dev(cls, cuda).to(dtype), to_dev(loc, cuda).to(dtype)
    args = (list(size), 2, 0.01, 0, 5000, 750, 0.3)
    ref = bu.parse_by_class_batch(args[0], cls_h.float(), *args[1:], loc_pred=loc_h.float(), anchors=anchors)
    det = bu.parse_by_class_batch(args[0], cls_h, *args[1:], loc_pred=loc_h, anchors=anchors)
    _assert_same(det, ref, "loc_pred")
    assert int(det.counts.min()) > 0
    # decoded boxes instead of offsets
    enc = oracle.AnchorEncoder(None, None, PS)
    boxes = np.stack([enc.decode_anchors(loc[b], *a_np[:4]) for b in range(3)]).astype(np.float32)
    boxes_h = to_dev(boxes, cuda).to(dtype)
    ref_b = bu.parse_by_class_batch(args[0], cls_h.float(), *args[1:], bboxes_pred=boxes_h.float())
    det_b = bu.parse_by_class_batch(args[0], cls_h, *args[1:], bboxes_pred=boxes_h)
    _assert_same(det_b, ref_b, "boxes_pred")
    # one image against the CPU oracle on the widened values
    cls_w = cls_h[1].float().cpu().numpy()
    boxes_w = enc.decode_anchors(loc_h[1].float().cpu().numpy(), *a_np[:4])
    sb, ss = oracle.parse_by_class(list(size), cls_w, boxes_w, 2, 0.01, 0, 5000, 750, 0.3)
    np.testing.assert_array_equal(det.scores[1, 0].cpu().numpy(), ss[1])
    np.testing.assert_array_equal(det.boxes[1, 0].cpu().numpy(), sb[1])
    # the single-image mirror passes half CUDA tensors through as they are
    sb1, ss1 = bu.parse_by_class(list(size), cls_h[1], boxes_h[1], 2, 0.01, 0, 5000, 750, 0.3)
    assert torch.equal(ss1[1], det_b.scores[1, 0]) and torch.equal(sb1[1], det_b.boxes[1, 0])


@pytest.mark.parametrize("dtype", HALF)
def test_parse_by_class_mixed_inputs(cuda, oracle, dtype):
    """The reference's evaluation sequence under autocast: decode_anchors(half offsets) returns fp32 boxes, which
    parse_by_class then takes with the half logits.  A pair that is not one half dtype on the device (half logits with
    fp32, numpy or other-half boxes) goes through as_f32 as a whole and equals the all-fp32 call."""
    from dan_b200.utility import anchor_manipulator as am, bbox_util as bu
    size = (640, 640)
    enc = am.AnchorEncoder(0.4, 0.4, PS)
    anchors = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd", size, border=0.))[:4]
    cls, loc = _g3(_anchors(oracle, size), size, 1, 900)
    cls_h, loc_h = to_dev(cls[0], cuda).to(dtype), to_dev(loc[0], cuda).to(dtype)
    boxes = enc.decode_anchors(loc_h, *anchors)
    assert boxes.dtype == torch.float32
    args = (2, 0.01, 0, 5000, 750, 0.3)
    other = torch.bfloat16 if dtype == torch.float16 else torch.float16
    cls_o = cls_h.to(other)
    cases = (((cls_h, boxes), (cls_h.float(), boxes)),                               # half logits, decoded fp32 boxes
             ((cls_h, boxes.cpu().numpy()), (cls_h.float(), boxes)),                 # ... boxes as numpy
             ((cls_h, boxes.cpu()), (cls_h.float(), boxes)),                         # ... boxes on the host
             ((cls_o, boxes.to(dtype)), (cls_o.float(), boxes.to(dtype).float())))   # fp16 with bf16, or back
    for (c, b), (c_ref, b_ref) in cases:
        sb, ss = bu.parse_by_class(list(size), c, b, *args)
        rb, rs = bu.parse_by_class(list(size), c_ref, b_ref, *args)
        assert int((rs[1] > 0).sum()) > 0
        assert torch.equal(_bits(sb[1]), _bits(rb[1])) and torch.equal(_bits(ss[1]), _bits(rs[1]))


@pytest.mark.parametrize("dtype", HALF)
def test_three_classes_filter_kernel(cuda, oracle, dtype):
    from dan_b200.utility import bbox_util as bu
    a_np = _anchors(oracle, (640, 640))
    anchors = [to_dev(v, cuda) for v in a_np[:4]]
    n = a_np[0].shape[0]
    rng = np.random.default_rng(41)
    cls_h = to_dev(rng.normal(0, 2.0, (2, n, 3)).astype(np.float32), cuda).to(dtype)
    loc_h = to_dev(rng.normal(0, 0.5, (2, n, 4)).astype(np.float32), cuda).to(dtype)
    for kw in ((0.2, 10, 400, 100, 0.45), (0.0, 0, 5000, 750, 0.3)):
        ref = bu.parse_by_class_batch([640, 640], cls_h.float(), 3, *kw, loc_pred=loc_h.float(), anchors=anchors)
        det = bu.parse_by_class_batch([640, 640], cls_h, 3, *kw, loc_pred=loc_h, anchors=anchors)
        _assert_same(det, ref, str(kw))


@pytest.mark.parametrize("dtype", HALF)
def test_beyond_shared_memory_limits(cuda, dtype):
    """candidates (and kept list) in the workspace: the WHERE = 1 and 2 instantiations."""
    from dan_b200.utility import bbox_util as bu
    rng = np.random.default_rng(77)
    n = 20000
    cls_h = to_dev(rng.normal(0, 2.0, (1, n, 2)).astype(np.float32), cuda).to(dtype)
    boxes_h = to_dev(_random_boxes(rng, (1, n), 2000), cuda).to(dtype)
    for keep_topk, nms_topk in ((12000, 9500), (9000, 400)):
        ref = bu.parse_by_class_batch([2000, 2000], cls_h.float(), 2, 0.05, 0, keep_topk, nms_topk, 0.5, bboxes_pred=boxes_h.float())
        det = bu.parse_by_class_batch([2000, 2000], cls_h, 2, 0.05, 0, keep_topk, nms_topk, 0.5, bboxes_pred=boxes_h)
        _assert_same(det, ref, str((keep_topk, nms_topk)))
        assert int(det.counts[0, 0]) > 0.8 * min(nms_topk, 9000)


@pytest.mark.parametrize("n", [777, 34125])
def test_alignment_and_tails(cuda, n):
    """N odd and not a multiple of 4 (per-image heads of 0-3 anchors, tails of 1-3); cls_pred views that start one
    anchor or one element into their storage, against contiguous aligned copies.  One element off leaves no aligned
    anchor pairs, for half and for fp32 alike: those go through the separate filter kernel."""
    from dan_b200.utility import bbox_util as bu
    rng = np.random.default_rng(n)
    B = 5
    cls_np = _detector_logits(rng, B, n)
    boxes_np = _random_boxes(rng, (B, n), 640)
    # the first and last 4 anchors of every image row (the head and tail of any alignment) become its 8 best, mutually
    # disjoint detections: a head or tail anchor that is dropped or misread changes counts, anchor_index and keep_pos
    edge = list(range(4)) + list(range(n - 4, n))
    for j, a in enumerate(edge):
        cls_np[:, a] = [-4.0, 12.0 - 0.25 * j]
        boxes_np[:, a] = [70.0 * j, 10.0, 70.0 * j + 50.0, 60.0]
    cls = to_dev(cls_np, cuda)
    boxes = to_dev(boxes_np, cuda)
    args = ([640, 640], 2, 0.01, 0, 5000, 750, 0.3)
    ref32 = bu.parse_by_class_batch(args[0], cls, *args[1:], bboxes_pred=boxes)
    for b in range(B):
        assert ref32.anchor_index[b, 0, :8].tolist() == edge
    off32 = _offset_view(cls, 1)
    assert off32.data_ptr() % 8 == 4
    _assert_same(bu.parse_by_class_batch(args[0], off32, *args[1:], bboxes_pred=boxes), ref32, "fp32 one element off")
    for dtype in HALF:
        cls_h, boxes_h = cls.to(dtype), boxes.to(dtype)
        ref = bu.parse_by_class_batch(args[0], cls_h.float(), *args[1:], bboxes_pred=boxes_h.float())
        aligned = bu.parse_by_class_batch(args[0], cls_h, *args[1:], bboxes_pred=boxes_h)
        _assert_same(aligned, ref, "%s aligned" % dtype)
        for elements in (2, 1):                  # one anchor (head path), one element (2-byte aligned)
            v = _offset_view(cls_h, elements)
            assert v.data_ptr() % 16 == 2 * elements
            _assert_same(bu.parse_by_class_batch(args[0], v, *args[1:], bboxes_pred=boxes_h), aligned,
                         "%s offset %d" % (dtype, elements))


@pytest.mark.parametrize("dtype", HALF)
def test_special_values(cuda, dtype):
    """logits beyond +-1e5 (the quick reject's guard), +-inf, signed zeros, fp16 subnormals and NaN, in the logits and
    in the box rows of passing anchors."""
    from dan_b200.utility import bbox_util as bu
    rng = np.random.default_rng(5)
    B, n = 2, 4099
    cls = _detector_logits(rng, B, n)
    boxes = _random_boxes(rng, (B, n), 640)
    big = [3e5, -3e5, 1e6, -1e6, 2e5] if dtype == torch.bfloat16 else [6e4, -6e4]
    special = [np.inf, -np.inf, 0.0, -0.0, np.nan, 1e-7, -3e-6, 6e-5] + big
    idx = rng.choice(n, 300, replace=False)
    for k, a in enumerate(idx):
        b = k % B
        cls[b, a, k % 2] = special[k % len(special)]
        if k % 3 == 0:
            cls[b, a, 1 - k % 2] = special[(k // 2) % len(special)]
        if k % 4 == 0:
            cls[b, a] = [-20.0, 20.0]            # passes: its box row carries the special value
            boxes[b, a, (k // 4) % 4] = special[(k // 4) % len(special)]
    cls_h, boxes_h = to_dev(cls, cuda).to(dtype), to_dev(boxes, cuda).to(dtype)
    for thr in (0.01, 0.0):
        ref = bu.parse_by_class_batch([640, 640], cls_h.float(), 2, thr, 0, 5000, 750, 0.3, bboxes_pred=boxes_h.float())
        det = bu.parse_by_class_batch([640, 640], cls_h, 2, thr, 0, 5000, 750, 0.3, bboxes_pred=boxes_h)
        _assert_same(det, ref, "thr %g" % thr)
    # the offsets path: inf / NaN offsets through the in-kernel decode
    loc = rng.normal(0, 0.5, (B, n, 4)).astype(np.float32)
    loc[0, idx[:40], 2] = np.resize(np.array(special), 40)
    anchors = [to_dev(v.astype(np.float32), cuda) for v in np.split(_random_boxes(rng, (n,), 640), 4, -1)]
    anchors = [a.reshape(-1).contiguous() for a in anchors]
    loc_h = to_dev(loc, cuda).to(dtype)
    ref = bu.parse_by_class_batch([640, 640], cls_h.float(), 2, 0.01, 0, 5000, 750, 0.3, loc_pred=loc_h.float(), anchors=anchors)
    det = bu.parse_by_class_batch([640, 640], cls_h, 2, 0.01, 0, 5000, 750, 0.3, loc_pred=loc_h, anchors=anchors)
    _assert_same(det, ref, "loc_pred")


@pytest.mark.parametrize("dtype", HALF)
def test_host_resident_geometry(cuda, oracle, dtype):
    """pinned half loc_pred / boxes_pred (8-byte rows read in place over PCIe) equal the device-resident half run, eagerly
    and replayed from a CUDA graph with new rows written into the same host buffer between replays."""
    from dan_b200 import _lib as L, functional as F
    from dan_b200.utility import bbox_util as bu
    size = (640, 640)
    a_np = _anchors(oracle, size)
    anchors = [to_dev(v, cuda) for v in a_np[:4]]
    cls, loc = _g3(a_np, size, 3, 520)
    cls_h, loc_h = to_dev(cls, cuda).to(dtype), to_dev(loc, cuda).to(dtype)
    loc_host = loc_h.cpu().pin_memory()
    args = (list(size), cls_h, 2, 0.01, 0, 5000, 750, 0.3)
    ref = bu.parse_by_class_batch(*args, loc_pred=loc_h, anchors=anchors)
    _assert_same(bu.parse_by_class_batch(*args, loc_pred=loc_host, anchors=anchors), ref, "pinned loc_pred")
    enc = oracle.AnchorEncoder(None, None, PS)
    boxes_h = to_dev(np.stack([enc.decode_anchors(loc[b], *a_np[:4]) for b in range(3)]).astype(np.float32), cuda).to(dtype)
    _assert_same(bu.parse_by_class_batch(*args, bboxes_pred=boxes_h.cpu().pin_memory()),
                 bu.parse_by_class_batch(*args, bboxes_pred=boxes_h), "pinned boxes_pred")
    # CUDA graph
    params = F.postprocess_params(2, size, 0.01, 0, 5000, 750, 0.3, prior_scaling=PS)
    ws = L.Workspace()
    out = F.postprocess_batch(params, cls_h, loc_pred=loc_host, anchors=anchors, workspace=ws)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            out = F.postprocess_batch(params, cls_h, loc_pred=loc_host, anchors=anchors, workspace=ws, out=tuple(out))
    torch.cuda.current_stream().wait_stream(side)
    g.replay()
    torch.cuda.synchronize()
    _assert_same(out, ref, "graph")
    loc_host.copy_(loc_h.flip(0).cpu())                                    # other offsets, same buffer
    ref2 = bu.parse_by_class_batch(*args, loc_pred=loc_h.flip(0).contiguous(), anchors=anchors)
    g.replay()
    torch.cuda.synchronize()
    _assert_same(out, ref2, "graph, new rows")
    del g


@pytest.mark.parametrize("dtype", HALF)
def test_hot_path_peer_exchange(cuda, oracle, dtype):
    """HotPath.step with a one-rank PeerExchange, half cls_pred and half loc_pred on the device or in pinned host memory:
    slab and received copy equal the run on the widened predictions, eagerly and in a CUDA graph."""
    from dan_b200 import functional as F, pipeline
    from dan_b200.utility import anchor_manipulator as am
    enc = am.AnchorEncoder(0.4, 0.4, PS)
    a_train = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd"))
    a_eval = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd", border=0.))
    ev_np = _anchors(oracle, (640, 640))
    B = 3
    gts = [synthetic.gen_faces(40 + i, 20) for i in range(B)]
    cls, loc = _g3(ev_np, (640, 640), B, 40, faces=30)
    cat, offs = synthetic.to_csr(gts)
    gt_d, offs_d = to_dev(cat, cuda), to_dev(offs, cuda)
    cls_h, loc_h = to_dev(cls, cuda).to(dtype), to_dev(loc, cuda).to(dtype)
    loc_host = loc_h.cpu().pin_memory()
    pp_params = F.postprocess_params(2, (640, 640), 0.01, 0, 5000, 750, 0.3, prior_scaling=PS)
    px = pipeline.PeerExchange(0, 1, cuda, pipeline.DetectionSlab.words_for(B, 1, 750), num_sets=1)
    hp = pipeline.HotPath(a_train[:4], a_train[4], F.encode_params(0.4, 0.4, PS, match_mining=True), pp_params,
                          anchors_eval=a_eval[:4], peer_exchange=px, peer_set=0)
    hp.step(gt_d, offs_d, cls_h.float(), loc_h.float())
    torch.cuda.synchronize()
    ref = [t.clone() for t in hp._slab.views()]           # counts, scores, boxes
    assert int(ref[0].sum()) > 0

    def same(buf=None):
        return all(torch.equal(_bits(a), _bits(b)) for a, b in zip(hp._slab.views(buf), ref))

    def clear():
        for t in hp._slab.views():
            t.fill_(-3)
        px.recv(0).zero_()
    for loc_in in (loc_h, loc_host):
        clear()
        hp.step(gt_d, offs_d, cls_h, loc_in)
        torch.cuda.synchronize()
        assert same() and same(px.recv(0))
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                hp.step(gt_d, offs_d, cls_h, loc_in)
        torch.cuda.current_stream().wait_stream(side)
        clear()
        graph.replay()
        torch.cuda.synchronize()
        assert same() and same(px.recv(0))
        del graph
    px.close()


@pytest.mark.parametrize("dtype", HALF)
def test_decode(cuda, dtype):
    from dan_b200.utility import anchor_manipulator as am
    enc = am.AnchorEncoder(0.4, 0.4, PS)
    a = synthetic.build_anchors(enc, synthetic.pyramid_config("s3fd", (1600, 1600), border=0.))
    n = a[0].numel()
    rng = np.random.default_rng(16)
    loc = rng.normal(0, 0.5, (2, n, 4)).astype(np.float32)
    loc[0, :8, 2] = [np.inf, -np.inf, np.nan, 0.0, -0.0, 1e-7, 60.0, -60.0]
    loc_h = to_dev(loc, cuda).to(dtype)
    out = enc.batch_decode_anchors(loc_h, *a[:4])
    assert out.dtype == torch.float32 and out.shape == (2, n, 4)
    assert torch.equal(_bits(out), _bits(enc.batch_decode_anchors(loc_h.float(), *a[:4])))
    assert torch.equal(_bits(enc.decode_all_anchors(loc_h, *a[:4])), _bits(out))
    one = enc.decode_anchors(loc_h[1], *a[:4])
    assert torch.equal(_bits(one), _bits(out[1]))


def test_errors(cuda, oracle):
    from dan_b200 import _lib as L, functional as F
    from dan_b200.utility import bbox_util as bu
    n = 777
    rng = np.random.default_rng(3)
    cls = to_dev(_detector_logits(rng, 1, n), cuda)
    boxes = to_dev(_random_boxes(rng, (1, n), 640), cuda)
    args = ([640, 640], 2, 0.01, 0, 100, 10, 0.3)
    for c, b in ((cls.half(), boxes.bfloat16()), (cls, boxes.half()), (cls.bfloat16(), boxes), (cls.double(), boxes.double()),
                 (cls.double(), boxes)):
        with pytest.raises(TypeError):
            bu.parse_by_class_batch(args[0], c, *args[1:], bboxes_pred=b)
    with pytest.raises(TypeError):
        F.decode_batch(boxes.double(), *[torch.zeros(n, device=cuda)] * 4, PS)
    # the C ABI
    params = F.postprocess_params(2, (640, 640), 0.01, 0, 100, 10, 0.3)
    nb = L.lib().dan_postprocess_workspace_bytes(n, 1, 2, 100)
    ws = torch.empty(nb, dtype=torch.uint8, device=cuda)
    ob = torch.empty((1, 1, 10, 4), device=cuda)
    osc = torch.empty((1, 1, 10), device=cuda)
    oc = torch.empty((1, 1), dtype=torch.int32, device=cuda)
    null = ctypes.c_void_p(0)

    def call(dtype, c, b, peers=None, ms=None):
        return L.lib().dan_postprocess_batch_typed(ctypes.byref(params), dtype, ctypes.c_void_p(c), ctypes.c_void_p(0), b,
                                                   null, null, null, null, n, 1, L.dev_ptr(ob), L.dev_ptr(osc), L.dev_ptr(oc),
                                                   null, null, L.dev_ptr(ws), nb, peers, L.stream_ptr(), ms)
    ch, bh = cls.half(), boxes.half()
    assert call(L.DAN_DTYPE_F16, ch.data_ptr(), L.dev_ptr(bh)) == 0
    torch.cuda.synchronize()
    for bad in (3, -1):
        assert call(bad, ch.data_ptr(), L.dev_ptr(bh)) == -1
    ms = (ctypes.c_float * 2)()
    assert call(L.DAN_DTYPE_F16, ch.data_ptr(), L.dev_ptr(bh), ctypes.byref(L.PeerExchangeArgs()), ms) == -1
    mis = _offset_view(bh, 2)                      # 4 bytes into an 8-byte row
    assert mis.data_ptr() % 8 == 4
    assert call(L.DAN_DTYPE_F16, ch.data_ptr(), L.dev_ptr(mis)) == -1
    pageable = bh.cpu()
    assert not pageable.is_pinned()
    assert call(L.DAN_DTYPE_BF16, cls.bfloat16().data_ptr(), ctypes.c_void_p(pageable.data_ptr())) == -1
    ps = (ctypes.c_float * 4)(*PS)
    a = torch.zeros(n, device=cuda)
    o = torch.empty((1, n, 4), device=cuda)
    assert L.lib().dan_decode_batch_typed(7, L.dev_ptr(bh), *[L.dev_ptr(a)] * 4, n, 1, ps, L.dev_ptr(o), L.stream_ptr()) == -1
    assert L.lib().dan_decode_batch_typed(L.DAN_DTYPE_F16, L.dev_ptr(mis), *[L.dev_ptr(a)] * 4, n, 1, ps, L.dev_ptr(o),
                                          L.stream_ptr()) == -1
    torch.cuda.synchronize()
