"""dan_detect_face_batch's argument checks that need no device: every refusal happens on the host, before anything is
enqueued (the pointers below are never dereferenced)."""
import ctypes

import pytest

K_SORT_CAP = 8192


@pytest.fixture(scope="module")
def lib():
    from dan_b200 import build, _lib
    build.build()
    return _lib.lib()


def test_workspace_bytes(lib):
    one = lib.dan_detect_face_batch_workspace_bytes(34125, 1)
    assert one >= 34125 * 8 and one % 256 == 0
    assert lib.dan_detect_face_batch_workspace_bytes(34125, 32) >= 32 * 34125 * 8
    assert lib.dan_detect_face_batch_workspace_bytes(34125, 1) == lib.dan_detect_face_workspace_bytes(34125)
    assert lib.dan_detect_face_batch_workspace_bytes(-1, 1) == 0


def test_refusals(lib):
    from dan_b200 import _lib as L
    n, B = 1000, 2
    nb = lib.dan_detect_face_batch_workspace_bytes(n, B)
    p = ctypes.c_void_p(1 << 20)                                  # 16-byte aligned, never dereferenced
    ps = (ctypes.c_float * 4)(0.1, 0.1, 0.2, 0.2)
    null = ctypes.c_void_p(0)

    def call(dtype=L.DAN_DTYPE_F32, cls=p, loc=p, num=n, batch=B, top=1125, ws=p, nbytes=nb, out=p, prior=ps):
        return lib.dan_detect_face_batch(dtype, cls, loc, p, p, p, p, num, batch, prior, 1.0, top, out, null, ws, nbytes, null)

    for bad in (3, -1, 7):
        assert call(dtype=bad) == -1
    assert call(top=0) == -4
    assert call(top=K_SORT_CAP + 1) == -4
    assert call(num=1 << 31) == -1
    assert call(num=-1) == -1
    assert call(batch=-1) == -1
    for kw in (dict(cls=null), dict(loc=null), dict(out=null), dict(prior=None)):
        assert call(**kw) == -1, kw
    assert call(loc=ctypes.c_void_p((1 << 20) + 8)) == -1                                   # fp32 rows: 16 bytes
    assert call(dtype=L.DAN_DTYPE_BF16, loc=ctypes.c_void_p((1 << 20) + 4)) == -1          # half rows: 8 bytes
    assert call(nbytes=nb - 1) == -2
    assert call(ws=null) == -2
    assert call(batch=0, ws=null, nbytes=0) == 0                                           # nothing to do
