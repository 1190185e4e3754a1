"""CPU tests of the fused multiclass NMS's size limits: every call below is refused before any CUDA work is enqueued,
so the pointers are never dereferenced."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from s2anet_b200 import build
    build.build()
    from s2anet_b200 import _lib
    return _lib.load()


def _call(lib, n, nc, B, iou_thr=0.5):
    p = C.c_void_p(256)
    return lib.s2a_multiclass_nms_rotated(p, p, n, nc, B, 0.05, iou_thr, 100, p, p, p, 100, p, 1 << 40, None)


def test_boxes_per_image_limits(lib):
    assert _call(lib, 1 << 30, 1, 1) == -1
    assert b"out of range" in lib.s2a_last_error()
    assert _call(lib, 819201, 1, 1) == -4                      # the sweep's shared-memory bitmaps
    assert b"819200" in lib.s2a_last_error()
    assert _call(lib, 100000, 15, 2000) == -4                  # batch * classes * n above 2^31 - 256
    assert b"2^31" in lib.s2a_last_error()
    assert _call(lib, 8000, 15, 8, iou_thr=-0.5) == -4
    assert b"iou_thr" in lib.s2a_last_error()


def test_workspace_grows_by_the_sort_keys_above_6144_boxes(lib):
    ws = lib.s2a_multiclass_nms_rotated_workspace_bytes
    mask = lambda n, S: 8 * S * n * ((n + 63) // 64)          # noqa: E731
    assert ws(6144, 15, 8) - mask(6144, 120) < 51 * 120 * 6144
    assert ws(6145, 15, 8) - mask(6145, 120) >= (48 + 16) * 120 * 6145
    assert 0.67e9 < mask(6720, 120) < 0.69e9 and 7.1e9 < mask(21824, 120) < 7.2e9
