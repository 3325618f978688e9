"""Batched detection (nv_detect_multiscale_batch, nv_face_*_batch) at the C-ABI boundary without a device: the symbols are
exported, bad arguments are refused with NV_ERR_ARG before anything else, and the Python wrappers refuse inputs of the
wrong dtype or shape before calling the library."""
import ctypes as C
import os

import numpy as np
import pytest

import nubovca as nv

BATCH_SYMBOLS = ["nv_detect_multiscale_batch", "nv_face_submit_batch", "nv_face_collect_batch", "nv_face_detect_batch"]


def test_batch_symbols_exported():
    lib = C.CDLL(nv.LIB_PATH)
    for name in BATCH_SYMBOLS:
        assert hasattr(lib, name) and name in nv.EXPORTS
    hdr = open(os.path.join(os.path.dirname(nv.LIB_PATH), "..", "..", "include", "nubovca.h")).read()
    assert f"#define NV_BATCH_MAX {nv.BATCH_MAX}" in hdr


@pytest.fixture(scope="module")
def casc():
    return nv.Cascade("haarcascade_frontalface_alt.xml")


@pytest.mark.parametrize("n", [-1, 0, 1, 2, nv.BATCH_MAX + 1])
def test_batch_bad_arguments(casc, n):
    L = nv._lib
    frames = (C.c_void_p * 2)()
    counts = (C.c_int * 2)()
    out = (nv.Rect * 4)()
    fp = nv.FaceParams(160, 1.25, 3, -1, -1)
    dp = nv.DetectParams(1.1, 3, 0, 0, 0, 0, 0)
    total = C.c_int(0)
    # null context (no device is needed to get here)
    assert L.nv_face_submit_batch(None, casc.handle, frames, n, 640, 480, 1920, 0, C.byref(fp)) == -1
    assert L.nv_face_detect_batch(None, casc.handle, frames, n, 640, 480, 1920, 0, C.byref(fp), out, 4, counts, C.byref(total)) == -1
    assert L.nv_detect_multiscale_batch(None, casc.handle, frames, n, 160, 120, 160, 0, C.byref(dp), out, 4, counts) == -1
    assert L.nv_face_collect_batch(None, out, 4, counts, C.byref(total)) == -1
    # null cascade, frame table, parameters, counts
    assert L.nv_face_detect_batch(None, None, None, n, -640, 480, 1920, 0, None, out, -4, None, None) == -1
    assert L.nv_detect_multiscale_batch(None, None, None, n, 160, -120, 160, 0, None, None, 0, None) == -1


class _NoCtx(nv.Context):
    """A Context without a library context: the wrappers must refuse bad input before they use the handle."""
    def __init__(self):
        self.handle = None

    def close(self):
        pass


@pytest.mark.parametrize("bad", [
    np.zeros((2, 48, 64, 3), np.float32),           # dtype
    np.zeros((2, 48, 64, 3), np.int16),
    np.zeros((48, 64, 3), np.uint8),                # no batch dimension
    np.zeros((2, 48, 64), np.uint8),                # gray where BGR is expected
    np.zeros((2, 48, 64, 4), np.uint8),             # BGRA
    [np.zeros((48, 64, 3), np.uint8)],              # not an array
])
def test_face_batch_wrapper_refuses(casc, bad):
    ctx = _NoCtx()
    with pytest.raises((TypeError, ValueError)):
        ctx.face_detect_batch(casc, bad)
    with pytest.raises((TypeError, ValueError)):
        ctx.face_submit_batch(casc, bad)


@pytest.mark.parametrize("bad", [
    np.zeros((2, 48, 64), np.float64),
    np.zeros((48, 64), np.uint8),
    np.zeros((2, 48, 64, 3), np.uint8),
    np.zeros((2, 48, 64, 1, 1), np.uint8),
])
def test_gray_batch_wrapper_refuses(casc, bad):
    with pytest.raises((TypeError, ValueError)):
        _NoCtx().detect_multiscale_batch(casc, bad)


def test_batch_wrapper_frame_table():
    """Row and image strides of a non-packed array reach the library as they are; packed pixels are required per row."""
    a = np.zeros((3, 50, 70, 3), np.uint8)[:, 1:49, 2:66]       # rows further apart than packed, images too
    ptrs, n, w, h, stride, dev, keep = nv._batch_frames(a, 3)
    assert (n, w, h, stride, dev) == (3, 64, 48, 70 * 3, 0)
    assert [ptrs[i] for i in range(3)] == [a.ctypes.data + i * a.strides[0] for i in range(3)]
    g = np.zeros((2, 40, 60), np.uint8)[:, :, ::2]              # pixels not packed: a packed copy is made
    ptrs, n, w, h, stride, dev, keep = nv._batch_frames(g, 1)
    assert (n, w, h, stride) == (2, 30, 40, 30) and keep.flags["C_CONTIGUOUS"]
