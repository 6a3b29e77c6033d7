"""dan_bbox_vote on the paths the synthetic detections of test_gpu_parity.py never reach: thresholds <= 0 (every pair
overlaps), finite coordinates of magnitude >= 1e30 (outside the stripe grid), groups of more than 128 and 256 members
(numpy's pairwise summation recurses), a full image of 8192 members, equal scores and max_per_image = 1.

Every case compares the groups, their count, the sort order and the head assignment with the oracle BIT FOR BIT."""
import numpy as np
import pytest

from dan_b200 import synthetic

from conftest import to_dev

pytestmark = pytest.mark.gpu
F32 = np.float32


def _np(t):
    return t.detach().cpu().numpy()


def _vote_vs_oracle(cuda, oracle, dets, thr=0.3, max_out=750):
    """one launch over the ragged batch `dets` (rows beyond an image's count are NaN), each image against the oracle"""
    from dan_b200 import functional as F
    cap = max(d.shape[0] for d in dets)
    batch = np.full((len(dets), cap, 5), np.nan, F32)
    for i, d in enumerate(dets):
        batch[i, :d.shape[0]] = d
    counts = np.array([d.shape[0] for d in dets], np.int32)
    out, cnt, order, assign = F.bbox_vote_batch(to_dev(batch, cuda), to_dev(counts, cuda), thr, max_out, details=True)
    refs = []
    for i, d in enumerate(dets):
        ref, aux = oracle.bbox_vote(d, nms_threshold=thr, max_per_image=max_out, return_details=True)
        k = int(cnt[i])
        assert k == ref.shape[0], (i, k, ref.shape)
        np.testing.assert_array_equal(_np(out[i, :k]).view(np.uint32), ref.view(np.uint32))
        assert not _np(out[i, k:]).any()
        n = d.shape[0]
        np.testing.assert_array_equal(_np(order[i, :n]), aux["order"])
        np.testing.assert_array_equal(_np(assign[i, :n]), aux["assign"])
        refs.append((ref, aux))
    return refs


def _cluster(seed, n, box=(100., 120., 180., 220.), score_lo=0.3):
    """n near-identical boxes (jitter below a pixel) with distinct scores: one group of n members"""
    rng = np.random.default_rng(seed)
    b = np.asarray(box, np.float64) + rng.uniform(-0.5, 0.5, (n, 4))
    s = rng.permutation(np.linspace(score_lo, 1.0, n, endpoint=False))
    return np.column_stack([b, s]).astype(F32)


def _group_sizes(aux):
    a = aux["assign"]
    return np.bincount(a[a >= 0])


@pytest.mark.parametrize("thr", [0.0, -0.5])
def test_bbox_vote_threshold_not_positive(cuda, oracle, thr):
    """thr <= 0: disjoint and degenerate boxes overlap too, every detection joins the first head (one group)"""
    dets = [synthetic.gen_vote_dets(80 + i, n, max(n // 25, 1), 0.5) for i, n in enumerate([2, 40, 700, 3000])]
    for (ref, aux), d in zip(_vote_vs_oracle(cuda, oracle, dets, thr), dets):
        assert ref.shape[0] == 1 and (aux["assign"] == 0).all()


@pytest.mark.filterwarnings("ignore:overflow encountered:RuntimeWarning")   # the oracle's areas and widths overflow on purpose
def test_bbox_vote_huge_coordinates(cuda, oracle):
    """finite coordinates of magnitude >= 1e30 (every head's exact test, not the stripe grid), mixed into ordinary rows;
    [-3e38, -3e38, 3e38, 3e38] has an infinite area and a NaN IoU with itself: a head that is deleted alone"""
    huge = np.array([[-3e38, -3e38, 3e38, 3e38, 0.97],
                     [1e30, 1e30, 1e30, 1e30, 0.91],                  # these two: a group of two far outside the grid
                     [1e30, 1e30, 1e30, 1e30, 0.42],
                     [-2e30, 50., -2e30, 80., 0.88],                  # one axis huge, the other ordinary
                     [-2e30, 52., -2e30, 81., 0.35],
                     [150., 1e31, 200., 1e31, 0.77],
                     [-1e36, 300., 1e36, 340., 0.66],                 # a finite area, far larger than any other box's
                     [100., 100., 3e38, 3e38, 0.55]], F32)            # an infinite area: deleted alone too
    dets = []
    for i, n in enumerate([300, 1500, 4000]):
        rows = np.concatenate([synthetic.gen_vote_dets(90 + i, n, max(n // 25, 1), 0.5), huge])
        dets.append(rows[np.random.default_rng(190 + i).permutation(rows.shape[0])])
    for (ref, aux), d in zip(_vote_vs_oracle(cuda, oracle, dets), dets):
        row = int(np.nonzero(d[:, 0] == F32(-3e38))[0][0])
        assert aux["assign"][np.nonzero(aux["order"] == row)[0][0]] == -2
        assert (np.abs(ref[:, 0]) > 1e29).sum() == 2                 # the two groups outside the grid
    _vote_vs_oracle(cuda, oracle, dets, thr=0.5, max_out=100)


def test_bbox_vote_large_groups(cuda, oracle):
    """a group of 300 members and more (the pairwise sum splits above 128 elements, then again above 256) among ordinary
    rows, which join it where they overlap; a group of 129 (the smallest split); two groups of 260 and 300"""
    base = synthetic.gen_vote_dets(100, 2000, 80, 0.5)
    big = _cluster(101, 300, score_lo=0.2)
    big[:, 4] += F32(1.5)                                             # above every ordinary score: distinct
    d0 = np.concatenate([base, big])
    d0 = d0[np.random.default_rng(102).permutation(d0.shape[0])]
    d1 = _cluster(103, 129)
    d2 = np.concatenate([_cluster(104, 260, box=(400., 400., 470., 480.)), _cluster(105, 300, box=(10., 10., 60., 70.), score_lo=1.1)])
    refs = _vote_vs_oracle(cuda, oracle, [d0, d1, d2])
    assert _group_sizes(refs[0][1]).max() >= 300
    assert sorted(_group_sizes(refs[2][1])[_group_sizes(refs[2][1]) > 0]) == [260, 300]


def test_bbox_vote_full_capacity_one_group(cuda, oracle):
    """one image of 8192 near-identical boxes: one group at the capacity, the deepest pairwise recursion"""
    d = _cluster(110, 8192)
    (ref, aux), = _vote_vs_oracle(cuda, oracle, [d])
    assert ref.shape[0] == 1 and (aux["assign"] == 0).all()


def test_bbox_vote_equal_scores(cuda, oracle):
    """scores rounded up to a few levels: equal scores are sorted higher row index first, in the order and in the groups.
    (No score is 0: a group whose scores are all 0 divides 0 by 0, and the NaN this gives on the GPU, 0x7fffffff, is not
    numpy's 0xffc00000.)"""
    dets = []
    for i, n in enumerate([50, 900, 5000]):
        d = synthetic.gen_vote_dets(120 + i, n, max(n // 25, 1), 0.5)
        d[:, 4] = np.ceil(d[:, 4] * 8) / 8                           # at most 8 distinct values, all > 0
        dets.append(d)
    big = _cluster(123, 300)
    big[:, 4] = np.round(big[:, 4] * 4) / 4
    dets.append(big)
    assert all(np.unique(d[:, 4]).shape[0] <= 8 for d in dets)
    _vote_vs_oracle(cuda, oracle, dets)


def test_bbox_vote_one_group_per_image(cuda, oracle):
    """max_per_image = 1: only the first group (in head order) is written"""
    dets = [synthetic.gen_vote_dets(130 + i, n, max(n // 25, 1), 0.5) for i, n in enumerate([3, 200, 6750])]
    dets.append(_cluster(133, 300))
    for thr in (0.3, 0.0):
        for ref, _ in _vote_vs_oracle(cuda, oracle, dets, thr=thr, max_out=1):
            assert ref.shape[0] <= 1
