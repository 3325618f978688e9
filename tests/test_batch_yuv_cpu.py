"""Batches of 4:2:0 frames (nv_face_*_batch_yuv) at the C-ABI boundary without a device: the symbols are exported, bad
arguments are refused with NV_ERR_ARG before anything else, and the Python wrapper refuses malformed batches and hands the
library the right plane pointers and strides for every format."""
import ctypes as C

import numpy as np
import pytest

import nubovca as nv

YUV_BATCH_SYMBOLS = ["nv_face_submit_batch_yuv", "nv_face_detect_batch_yuv"]


def test_yuv_batch_symbols_exported():
    lib = C.CDLL(nv.LIB_PATH)
    for name in YUV_BATCH_SYMBOLS:
        assert hasattr(lib, name) and name in nv.EXPORTS


@pytest.fixture(scope="module")
def casc():
    return nv.Cascade("haarcascade_frontalface_alt.xml")


@pytest.mark.parametrize("n", [-1, 0, 1, 2, nv.BATCH_MAX + 1])
def test_yuv_batch_bad_arguments(casc, n):
    L = nv._lib
    frames = (nv.YuvFrame * 2)()
    counts = (C.c_int * 2)()
    out = (nv.Rect * 4)()
    fp = nv.FaceParams(160, 1.25, 3, -1, -1)
    total = C.c_int(0)
    # null context (no device is needed to get here)
    assert L.nv_face_submit_batch_yuv(None, casc.handle, frames, n, C.byref(fp)) == -1
    assert L.nv_face_detect_batch_yuv(None, casc.handle, frames, n, C.byref(fp), out, 4, counts, C.byref(total)) == -1
    # null cascade, frame table, parameters, counts
    assert L.nv_face_submit_batch_yuv(None, None, None, n, None) == -1
    assert L.nv_face_detect_batch_yuv(None, None, None, n, None, out, -4, None, None) == -1


class _NoCtx(nv.Context):
    """A Context without a library context: the wrappers must refuse bad input before they use the handle."""
    def __init__(self):
        self.handle = None

    def close(self):
        pass


@pytest.mark.parametrize("bad,fmt", [
    (np.zeros((2, 72, 64), np.float32), "NV12"),           # dtype
    (np.zeros((2, 72, 64), np.int16), "I420"),
    (np.zeros((72, 64), np.uint8), "NV12"),                 # no batch dimension
    (np.zeros((2, 48, 64, 3), np.uint8), "NV12"),           # BGR frames
    (np.zeros((2, 73, 64), np.uint8), "NV12"),              # not H*3/2 rows
    (np.zeros((2, 72, 80), np.uint8)[:, :, :64], "I420"),   # I420 / YV12 rows not packed
    (np.zeros((2, 72, 80), np.uint8)[:, :, :64], "YV12"),
    (np.zeros((2, 72, 64), np.uint8), "BGR"),               # not a 4:2:0 format
    ([np.zeros((72, 64), np.uint8)], "NV12"),               # not an array
])
def test_yuv_batch_wrapper_refuses(casc, bad, fmt):
    ctx = _NoCtx()
    with pytest.raises((TypeError, ValueError)):
        ctx.face_detect_batch_yuv(casc, bad, fmt)
    with pytest.raises((TypeError, ValueError)):
        ctx.face_submit_batch_yuv(casc, bad, fmt)


@pytest.mark.parametrize("fmt", ["I420", "YV12", "NV12", "NV21"])
def test_yuv_batch_wrapper_plane_split(casc, fmt, monkeypatch):
    """The library sees, per image, the planes synth.yuv420_planes takes out of the packed buffer (YV12 in I420 order);
    NV12 / NV21 keep a pitched row stride, and images may be further apart than packed."""
    from nubovca import synth
    w, h, n = 64, 48, 3
    pad = 0 if fmt in ("I420", "YV12") else 16
    big = np.zeros((n + 1, h * 3 // 2, w + pad), np.uint8)
    a = big[1:, :, :w] if pad else big[1:]
    seen = {}

    def fake_submit(handle, casc_handle, table, k, params):
        seen["frames"] = [table[i] for i in range(k)]
        seen["n"] = k
        return 0

    monkeypatch.setattr(nv._lib, "nv_face_submit_batch_yuv", fake_submit)
    ctx = _NoCtx()
    ctx.face_submit_batch_yuv(casc, a, fmt)
    assert seen["n"] == n and ctx._batch_n == n
    assert ctx._batch_keep is a
    for i, f in enumerate(seen["frames"]):
        assert (f.format, f.width, f.height, f.on_device) == (nv._FMT[fmt], w, h, 0)
        img, packed = a[i], np.ascontiguousarray(a[i])
        exp = synth.yuv420_planes(packed, w, h, fmt)                       # plane offsets within a packed copy
        base, pbase = img.ctypes.data, packed.ctypes.data
        assert f.plane[0] == base and f.stride[0] == img.strides[0]
        if fmt in ("NV12", "NV21"):
            assert f.plane[1] == base + h * img.strides[0] and f.stride[1] == img.strides[0]
            assert exp[1].ctypes.data - pbase == h * w
        else:
            assert f.plane[1] - base == exp[1].ctypes.data - pbase and f.plane[2] - base == exp[2].ctypes.data - pbase
            assert f.stride[1] == f.stride[2] == w // 2
            if fmt == "YV12":
                assert f.plane[1] > f.plane[2]                                # V comes first in a YV12 buffer
