"""dan_bbox_vote_ws / dan_bbox_vote_workspace_bytes argument checks that need no device: every refusal happens on the
host, before anything is enqueued (the pointers below are never dereferenced)."""
import ctypes

import pytest

SMALL_CAP = 8192
LARGE_CAP = 1 << 20
OK, INVALID, WORKSPACE, UNSUPPORTED = 0, -1, -2, -4


@pytest.fixture(scope="module")
def lib():
    from dan_b200 import build, _lib
    build.build()
    return _lib.lib()


def test_workspace_bytes(lib):
    for cap in (0, 1, 750, SMALL_CAP):
        assert lib.dan_bbox_vote_workspace_bytes(32, cap) == 0
    one = lib.dan_bbox_vote_workspace_bytes(1, SMALL_CAP + 1)
    assert one >= (SMALL_CAP + 1) * 40 and one % 256 == 0
    assert lib.dan_bbox_vote_workspace_bytes(32, SMALL_CAP + 1) == 32 * one
    assert lib.dan_bbox_vote_workspace_bytes(1, 20000) > one
    assert lib.dan_bbox_vote_workspace_bytes(1, LARGE_CAP) >= LARGE_CAP * 40
    assert lib.dan_bbox_vote_workspace_bytes(0, 20000) == 0
    assert lib.dan_bbox_vote_workspace_bytes(-1, 20000) == 0
    assert lib.dan_bbox_vote_workspace_bytes(1, -1) == 0
    assert lib.dan_bbox_vote_workspace_bytes(1, LARGE_CAP + 1) == 0          # refused: no size


def test_refusals(lib):
    p = ctypes.c_void_p(1 << 20)                                  # 16-byte aligned, never dereferenced
    null = ctypes.c_void_p(0)
    B, cap = 2, 20000
    nb = lib.dan_bbox_vote_workspace_bytes(B, cap)

    def call(det=p, batch=B, capacity=cap, max_out=750, out=p, cnt=p, ws=p, nbytes=nb):
        return lib.dan_bbox_vote_ws(det, null, batch, capacity, 0.3, max_out, out, cnt, null, null, ws, nbytes, null)

    assert call(ws=null) == WORKSPACE
    assert call(nbytes=nb - 1) == WORKSPACE
    assert call(ws=null, nbytes=0) == WORKSPACE
    assert call(ws=ctypes.c_void_p((1 << 20) + 8)) == INVALID                # misaligned workspace
    assert call(capacity=LARGE_CAP + 1, nbytes=1 << 40) == UNSUPPORTED
    assert call(capacity=1 << 30) == UNSUPPORTED
    assert call(batch=-1) == INVALID
    assert call(capacity=-1) == INVALID
    for m in (0, -1, 65536):
        assert call(max_out=m) == INVALID, m
    for kw in (dict(det=null), dict(out=null), dict(cnt=null)):
        assert call(**kw) == INVALID, kw
    assert call(batch=0, ws=null, nbytes=0) == OK                            # nothing to do
    assert call(batch=0, capacity=LARGE_CAP, ws=null, nbytes=0) == OK


def test_dan_bbox_vote_keeps_its_limit(lib):
    p = ctypes.c_void_p(1 << 20)
    null = ctypes.c_void_p(0)

    def call(batch=2, capacity=SMALL_CAP, max_out=750, out=p):
        return lib.dan_bbox_vote(p, null, batch, capacity, 0.3, max_out, out, p, null, null, null)

    assert call(capacity=SMALL_CAP + 1) == UNSUPPORTED
    assert call(capacity=20000) == UNSUPPORTED
    assert call(batch=-1) == INVALID
    assert call(capacity=-1) == INVALID
    assert call(max_out=0) == INVALID
    assert call(out=null) == INVALID
    assert call(batch=0) == OK
