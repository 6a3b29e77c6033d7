"""dan_detect_face_batch_top / dan_detect_face_select_top: the workspace size and the argument checks that need no device.
Every refusal happens on the host, before anything is enqueued (the pointers below are never dereferenced)."""
import ctypes

import pytest

K_SORT_CAP = 8192
TOP_CAP = 1 << 20
N1600 = 213294                                                    # S3FD anchors at 1600^2


@pytest.fixture(scope="module")
def lib():
    from dan_b200 import build, _lib
    build.build()
    return _lib.lib()


def _align(v):
    return (v + 255) // 256 * 256


def test_workspace_bytes(lib):
    for n, B in ((34125, 1), (N1600, 4)):
        base = lib.dan_detect_face_batch_workspace_bytes(n, B)
        for top in (1, 1125, K_SORT_CAP):
            assert lib.dan_detect_face_top_workspace_bytes(n, B, top) == base
        sizes = []
        for top in (K_SORT_CAP + 1, 16384, 30000, 98302, TOP_CAP):
            k = min(n - 1, top)
            got = lib.dan_detect_face_top_workspace_bytes(n, B, top)
            assert got == base + B * (2 * _align(8 * k) + _align(16 * k)), (n, B, top)
            sizes.append(got)
        assert sizes == sorted(sizes) and sizes[0] < sizes[1]                 # grows with top ...
        assert lib.dan_detect_face_top_workspace_bytes(n, B, n - 1) == lib.dan_detect_face_top_workspace_bytes(n, B, TOP_CAP)
    # k = N - 1 <= 8192 whatever the top: nothing beyond the small path's workspace
    assert lib.dan_detect_face_top_workspace_bytes(5000, 2, 98302) == lib.dan_detect_face_batch_workspace_bytes(5000, 2)
    assert lib.dan_detect_face_top_workspace_bytes(34125, 1, 16384) < lib.dan_detect_face_top_workspace_bytes(34125, 2, 16384)
    assert lib.dan_detect_face_top_workspace_bytes(-1, 1, 16384) == 0
    assert lib.dan_detect_face_top_workspace_bytes(34125, -1, 16384) == 0
    assert lib.dan_detect_face_top_workspace_bytes(34125, 1, TOP_CAP + 1) == 0


def test_batch_top_refusals(lib):
    from dan_b200 import _lib as L
    n, B = N1600, 2
    p = ctypes.c_void_p(1 << 20)                                  # 16-byte aligned, never dereferenced
    ps = (ctypes.c_float * 4)(0.1, 0.1, 0.2, 0.2)
    null = ctypes.c_void_p(0)

    def call(dtype=L.DAN_DTYPE_F32, cls=p, loc=p, num=n, batch=B, top=16384, ws=p, nbytes=None, out=p, prior=ps, fn=None):
        if nbytes is None:
            nbytes = lib.dan_detect_face_top_workspace_bytes(num, batch, top)
        f = fn or lib.dan_detect_face_batch_top
        return f(dtype, cls, loc, p, p, p, p, num, batch, prior, 1.0, top, out, null, ws, nbytes, null)

    for bad in (3, -1, 7):
        assert call(dtype=bad) == -1
    assert call(top=0) == -4
    assert call(top=-5) == -4
    assert call(top=TOP_CAP + 1) == -4
    assert call(top=TOP_CAP + 1, batch=0, ws=null, nbytes=0) == -4              # checked before batch == 0 returns
    assert call(num=1 << 31) == -1
    assert call(num=-1) == -1
    assert call(batch=-1) == -1
    for kw in (dict(cls=null), dict(loc=null), dict(out=null), dict(prior=None)):
        assert call(**kw) == -1, kw
    assert call(loc=ctypes.c_void_p((1 << 20) + 8)) == -1                                   # fp32 rows: 16 bytes
    assert call(dtype=L.DAN_DTYPE_BF16, loc=ctypes.c_void_p((1 << 20) + 4)) == -1          # half rows: 8 bytes
    assert call(num=(1 << 31) - 1, batch=1 << 20) == -4                                      # chunks x batch >= 2^31
    for top in (K_SORT_CAP + 1, 98302, TOP_CAP):
        need = lib.dan_detect_face_top_workspace_bytes(n, B, top)
        assert call(top=top, nbytes=need - 1) == -2
        assert call(top=top, nbytes=lib.dan_detect_face_batch_workspace_bytes(n, B)) == -2   # the small path's size
        assert call(top=top, ws=null) == -2
    assert call(top=1125, nbytes=lib.dan_detect_face_batch_workspace_bytes(n, B) - 1) == -2
    assert call(batch=0, ws=null, nbytes=0) == 0                                           # nothing to do
    assert call(batch=0, top=TOP_CAP, ws=null, nbytes=0) == 0


def test_select_top_refusals(lib):
    n = N1600
    p = ctypes.c_void_p(1 << 20)
    null = ctypes.c_void_p(0)

    def call(bboxes=p, scores=p, num=n, top=16384, out=p, count=p, ws=p, nbytes=None, fn=None):
        if nbytes is None:
            nbytes = lib.dan_detect_face_top_workspace_bytes(num, 1, top)
        f = fn or lib.dan_detect_face_select_top
        return f(bboxes, scores, num, 1.0, top, out, null, count, ws, nbytes, null)

    assert call(num=-1) == -1
    assert call(num=1 << 31) == -1
    assert call(top=0) == -4
    assert call(top=TOP_CAP + 1) == -4
    assert call(out=null) == -1
    assert call(count=null) == -1
    assert call(bboxes=null) == -1
    assert call(scores=null) == -1
    assert call(bboxes=ctypes.c_void_p((1 << 20) + 4)) == -1                                 # rows: 16 bytes
    for top in (K_SORT_CAP + 1, 98302, TOP_CAP):
        need = lib.dan_detect_face_top_workspace_bytes(n, 1, top)
        assert need > lib.dan_detect_face_workspace_bytes(n)
        assert call(top=top, nbytes=need - 1) == -2
        assert call(top=top, nbytes=lib.dan_detect_face_workspace_bytes(n)) == -2
        assert call(top=top, ws=null) == -2


def test_old_entry_points_keep_their_limit(lib):
    """dan_detect_face_batch and dan_detect_face_select still refuse top = 8193, with any workspace."""
    from dan_b200 import _lib as L
    n, B = N1600, 2
    p = ctypes.c_void_p(1 << 20)
    ps = (ctypes.c_float * 4)(0.1, 0.1, 0.2, 0.2)
    null = ctypes.c_void_p(0)
    big = lib.dan_detect_face_top_workspace_bytes(n, B, TOP_CAP)
    for top in (K_SORT_CAP + 1, 98302):
        assert lib.dan_detect_face_batch(L.DAN_DTYPE_F32, p, p, p, p, p, p, n, B, ps, 1.0, top, p, null, p, big, null) == -4
        assert lib.dan_detect_face_select(p, p, n, 1.0, top, p, null, p, p, big, null) == -4
    assert lib.dan_detect_face_batch(L.DAN_DTYPE_F32, p, p, p, p, p, p, n, 0, ps, 1.0, K_SORT_CAP + 1, p, null, null, 0, null) == -4
