"""dan_bbox_vote_ws above 8192 detections per image: stacks of more passes than the small kernel holds, positions and
group sizes beyond 16 bits, the edge paths of test_bbox_vote_edges.py in such stacks, and both paths on the same images.

Every case compares the groups, their count, the sort order and the head assignment with the oracle BIT FOR BIT.  Rows
beyond an image's count are NaN, so a result that read one would differ."""
import os

import numpy as np
import pytest

from dan_b200 import synthetic

from conftest import to_dev

pytestmark = pytest.mark.gpu
F32 = np.float32
SMALL_CAP = 8192
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _np(t):
    return t.detach().cpu().numpy()


def _stack(dets, cap=None):
    cap = max([d.shape[0] for d in dets] + [cap or 0])
    batch = np.full((len(dets), cap, 5), np.nan, F32)
    for i, d in enumerate(dets):
        batch[i, :d.shape[0]] = d
    return batch, np.array([d.shape[0] for d in dets], np.int32)


def _run(cuda, dets, thr=0.3, max_out=750, cap=None):
    from dan_b200 import functional as F
    batch, counts = _stack(dets, cap)
    return [_np(t) for t in F.bbox_vote_batch(to_dev(batch, cuda), to_dev(counts, cuda), thr, max_out, details=True)]


def _check(got, i, d, oracle, thr, max_out):
    out, cnt, order, assign = got
    ref, aux = oracle.bbox_vote(d, nms_threshold=thr, max_per_image=max_out, return_details=True)
    k = int(cnt[i])
    assert k == ref.shape[0], (i, k, ref.shape)
    np.testing.assert_array_equal(out[i, :k].view(np.uint32), ref.view(np.uint32))
    assert not out[i, k:].any()
    n = d.shape[0]
    np.testing.assert_array_equal(order[i, :n], aux["order"])
    np.testing.assert_array_equal(assign[i, :n], aux["assign"])
    return ref, aux


def _vote_vs_oracle(cuda, oracle, dets, thr=0.3, max_out=750, cap=None):
    """one launch over the ragged batch `dets` (capacity: the largest image, at least `cap`), each image vs the oracle"""
    got = _run(cuda, dets, thr, max_out, cap)
    assert got[2].shape[1] > SMALL_CAP                               # the large path ran
    return [_check(got, i, d, oracle, thr, max_out) for i, d in enumerate(dets)]


def _dets(seed, n, bg=0.6):
    return synthetic.gen_vote_dets(seed, n, max(n // 56, 1), bg)


def _cluster(seed, n, box=(100., 120., 180., 220.), score_lo=0.3):
    """n near-identical boxes (jitter below a pixel) with distinct scores: one group of n members"""
    rng = np.random.default_rng(seed)
    b = np.asarray(box, np.float64) + rng.uniform(-0.5, 0.5, (n, 4))
    s = rng.permutation(np.linspace(score_lo, 1.0, n, endpoint=False))
    return np.column_stack([b, s]).astype(F32)


def test_realistic_stacks_ragged(cuda, oracle):
    """8, 10 and about 18 passes of 1125 rows, an image of the small kernel's size and an empty one, in one launch"""
    dets = [_dets(200, 9000), _dets(201, 11250), np.zeros((0, 5), F32), _dets(202, 20000), _dets(203, 3000)]
    assert dets[0].shape[0] > SMALL_CAP and dets[1].shape[0] > SMALL_CAP and dets[3].shape[0] > 19000
    refs = _vote_vs_oracle(cuda, oracle, dets)
    assert all(r.shape[0] > 10 for r, _ in refs[:2])


def test_positions_beyond_16_bits(cuda, oracle):
    """about 70 000 rows: positions and head positions above 65 535"""
    d = _dets(210, 70000)
    assert d.shape[0] > 65536
    (ref, aux), = _vote_vs_oracle(cuda, oracle, [d])
    assert aux["assign"].max() > 65535


def test_group_beyond_16_bits(cuda, oracle):
    """one group of 66 000 near-identical boxes: its count exceeds 16 bits and numpy's pairwise sum recurses deeper than
    the small kernel's stack holds (11 levels; it has 8)"""
    d = _cluster(211, 66000)
    (ref, aux), = _vote_vs_oracle(cuda, oracle, [d])
    assert ref.shape[0] == 1 and (aux["assign"] == 0).all()


@pytest.mark.parametrize("thr", [0.0, -0.5])
def test_threshold_not_positive(cuda, oracle, thr):
    dets = [_dets(220, 9000), _dets(221, 40)]
    for ref, aux in _vote_vs_oracle(cuda, oracle, dets, thr):
        assert ref.shape[0] == 1 and (aux["assign"] == 0).all()


@pytest.mark.filterwarnings("ignore:overflow encountered:RuntimeWarning")   # the oracle's areas and widths overflow on purpose
def test_huge_coordinates(cuda, oracle):
    huge = np.array([[-3e38, -3e38, 3e38, 3e38, 0.97],                # a head deleted alone (NaN IoU with itself)
                     [1e30, 1e30, 1e30, 1e30, 0.91],
                     [1e30, 1e30, 1e30, 1e30, 0.42],
                     [-2e30, 50., -2e30, 80., 0.88],
                     [-2e30, 52., -2e30, 81., 0.35],
                     [150., 1e31, 200., 1e31, 0.77],
                     [-1e36, 300., 1e36, 340., 0.66],
                     [100., 100., 3e38, 3e38, 0.55]], F32)
    rows = np.concatenate([_dets(230, 9500), huge])
    d = rows[np.random.default_rng(231).permutation(rows.shape[0])]
    (ref, aux), = _vote_vs_oracle(cuda, oracle, [d])
    row = int(np.nonzero(d[:, 0] == F32(-3e38))[0][0])
    assert aux["assign"][np.nonzero(aux["order"] == row)[0][0]] == -2
    assert (np.abs(ref[:, 0]) > 1e29).sum() == 2
    _vote_vs_oracle(cuda, oracle, [d], thr=0.5, max_out=100)


def test_equal_scores(cuda, oracle):
    """at most 8 score levels, all > 0 (a group of 0 scores gives a NaN whose bits differ from numpy's)"""
    d = _dets(240, 10000)
    d[:, 4] = np.ceil(d[:, 4] * 8) / 8
    assert np.unique(d[:, 4]).shape[0] <= 8 and d.shape[0] > SMALL_CAP
    _vote_vs_oracle(cuda, oracle, [d])


@pytest.mark.parametrize("max_out", [1, 65535])
def test_max_per_image_limits(cuda, oracle, max_out):
    dets = [_dets(250, 9000), _cluster(251, 300)]
    for ref, _ in _vote_vs_oracle(cuda, oracle, dets, max_out=max_out):
        assert ref.shape[0] <= max_out


def test_both_paths_agree(cuda, oracle):
    """the same images through the small kernel (capacity 8192) and the large one (capacity 8193, with counts), and the
    goldens of the reference's own function through the large kernel"""
    from test_oracle import VOTE_CASES
    dets = [_dets(260, 6750), _dets(261, 8192)[:8192], _cluster(262, 300), np.zeros((0, 5), F32)]
    dets += [synthetic.gen_vote_dets(i, n, faces, bg) for i, n, faces, bg in VOTE_CASES]
    small = _run(cuda, dets, cap=SMALL_CAP)
    large = _run(cuda, dets, cap=SMALL_CAP + 1)
    assert small[2].shape[1] == SMALL_CAP and large[2].shape[1] == SMALL_CAP + 1
    np.testing.assert_array_equal(small[0].view(np.uint32), large[0].view(np.uint32))
    np.testing.assert_array_equal(small[1], large[1])
    np.testing.assert_array_equal(small[2], large[2][:, :SMALL_CAP])
    np.testing.assert_array_equal(small[3], large[3][:, :SMALL_CAP])
    g = np.load(os.path.join(GOLD, "vote_reference.npz"))
    for j, (image_index, *_rest) in enumerate(VOTE_CASES):
        ref = g["vote_%d" % image_index]
        k = int(large[1][4 + j])
        assert k == ref.shape[0]
        np.testing.assert_array_equal(large[0][4 + j, :k].view(np.uint32), ref.view(np.uint32))
    for i in range(2):
        _check(large, i, dets[i], oracle, 0.3, 750)


def test_counts_none(cuda, oracle):
    """counts = NULL: every image has all capacity rows"""
    from dan_b200 import functional as F
    dets = [_dets(270, 9500)[:9000], _dets(271, 9500)[:9000]]
    batch, _ = _stack(dets)
    got = [_np(t) for t in F.bbox_vote_batch(to_dev(batch, cuda), None, 0.3, 750, details=True)]
    for i, d in enumerate(dets):
        _check(got, i, d, oracle, 0.3, 750)


def test_cuda_graph_replay(cuda, oracle):
    """one call captured in a CUDA graph, replayed twice with new inputs copied into the same buffers"""
    import torch
    from dan_b200 import _lib as L
    from dan_b200 import functional as F
    first = [_dets(280, 9000), _dets(281, 2000)]
    batch, counts = _stack(first, cap=10000)
    x, c = to_dev(batch, cuda), to_dev(counts, cuda)
    ws = L.Workspace()
    stream = torch.cuda.Stream(cuda)
    with torch.cuda.stream(stream):
        F.bbox_vote_batch(x, c, 0.3, 750, details=True, workspace=ws)                 # warm-up: loads, workspace
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            outs = F.bbox_vote_batch(x, c, 0.3, 750, details=True, workspace=ws)
    for r, dets in enumerate([[_dets(282, 9900), _dets(283, 500)], [_dets(284, 300), _dets(285, 9300)]]):
        batch, counts = _stack(dets, cap=10000)
        x.copy_(to_dev(batch, cuda))
        c.copy_(to_dev(counts, cuda))
        graph.replay()
        torch.cuda.synchronize()
        got = [_np(t) for t in outs]
        for i, d in enumerate(dets):
            _check(got, i, d, oracle, 0.3, 750)


def test_eval_merge_single_stack(cuda, oracle):
    """eval_merge.bbox_vote on one [n, 5] stack of more than 8192 rows"""
    from dan_b200.utility import eval_merge
    d = _dets(290, 12000)
    got = _np(eval_merge.bbox_vote(to_dev(d, cuda)))
    ref = oracle.bbox_vote(d)
    assert got.shape == ref.shape and ref.shape[0] > 10
    np.testing.assert_array_equal(got.view(np.uint32), ref.view(np.uint32))
