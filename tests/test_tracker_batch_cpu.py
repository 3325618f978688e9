"""The batched tracker (nv_tracker_process_batch / _yuv, nv_tracker_reset_batch) at the C-ABI boundary without a device: the
symbols are exported, bad arguments are refused with NV_ERR_ARG, and the Python wrappers refuse bad input before they call
the library."""
import ctypes as C

import numpy as np
import pytest

import nubovca as nv

SYMBOLS = ["nv_tracker_process_batch", "nv_tracker_process_batch_yuv", "nv_tracker_reset_batch"]
NV_ERR_ARG = -1


def test_tracker_batch_symbols_exported():
    lib = C.CDLL(nv.LIB_PATH)
    for name in SYMBOLS:
        assert hasattr(lib, name) and name in nv.EXPORTS


@pytest.mark.parametrize("n", [-1, 0, 1, 2, nv.BATCH_MAX + 1])
def test_tracker_batch_bad_arguments(n):
    L = nv._lib
    frames = (C.c_void_p * 2)()
    yuv = (nv.YuvFrame * 2)()
    ts = (C.c_double * 2)()
    params = (nv.TrackerParams * 2)()
    counts = (C.c_int * 2)()
    out = (nv.Rect * 4)()
    total = C.c_int(0)
    # null context (no device is needed to get here)
    assert L.nv_tracker_process_batch(None, frames, n, 64, 48, 256, 0, ts, params, out, 4, counts, C.byref(total)) == NV_ERR_ARG
    assert L.nv_tracker_process_batch_yuv(None, yuv, n, ts, params, out, 4, counts, C.byref(total)) == NV_ERR_ARG
    assert L.nv_tracker_reset_batch(None, -1) == NV_ERR_ARG
    assert L.nv_tracker_reset_batch(None, 0) == NV_ERR_ARG
    # null frame table, timestamps, parameters, counts; out null with a capacity
    assert L.nv_tracker_process_batch(None, None, n, 64, 48, 256, 0, None, None, None, 4, None, None) == NV_ERR_ARG
    assert L.nv_tracker_process_batch_yuv(None, None, n, None, None, None, 4, None, None) == NV_ERR_ARG


class _NoCtx(nv.Context):
    """A Context without a library context: the wrappers must refuse bad input before they use the handle."""
    def __init__(self):
        self.handle = None

    def close(self):
        pass


@pytest.mark.parametrize("bad", [
    np.zeros((2, 48, 64, 4), np.float32),           # dtype
    np.zeros((2, 48, 64, 4), np.int16),
    np.zeros((48, 64, 4), np.uint8),                # no batch dimension
    np.zeros((2, 48, 64, 3), np.uint8),             # BGR where BGRA is expected
    np.zeros((2, 48, 64), np.uint8),                # gray
    [np.zeros((48, 64, 4), np.uint8)],              # not an array
])
def test_tracker_batch_wrapper_refuses_frames(bad):
    with pytest.raises((TypeError, ValueError)):
        _NoCtx().tracker_process_batch(bad, [1.0, 2.0])


@pytest.mark.parametrize("kw", [
    dict(ts_ms=[1.0]),                              # len(ts) != N
    dict(ts_ms=[1.0, 2.0, 3.0]),
    dict(ts_ms=[1.0, 2.0], threshold=[20]),         # wrong-length parameter sequences
    dict(ts_ms=[1.0, 2.0], min_area=[50, 50, 50]),
    dict(ts_ms=[1.0, 2.0], max_area=[]),
    dict(ts_ms=[1.0, 2.0], distance=(35,)),
])
def test_tracker_batch_wrapper_refuses_arguments(kw):
    frames = np.zeros((2, 48, 64, 4), np.uint8)
    with pytest.raises(ValueError):
        _NoCtx().tracker_process_batch(frames, **kw)
    with pytest.raises(ValueError):
        _NoCtx().tracker_process_batch_yuv(np.zeros((2, 72, 64), np.uint8), "NV12", **kw)


@pytest.mark.parametrize("bad,fmt", [
    (np.zeros((2, 72, 64), np.float32), "NV12"),
    (np.zeros((72, 64), np.uint8), "NV12"),         # no batch dimension
    (np.zeros((2, 71, 64), np.uint8), "NV12"),      # not H*3/2 rows
    (np.zeros((2, 72, 64), np.uint8), "BGR"),       # not a 4:2:0 format
])
def test_tracker_batch_yuv_wrapper_refuses(bad, fmt):
    with pytest.raises((TypeError, ValueError)):
        _NoCtx().tracker_process_batch_yuv(bad, fmt, [1.0, 2.0])


def test_tracker_batch_wrapper_arguments():
    """Scalars apply to every slot, sequences per slot; a BGRA batch's row and image strides reach the library as they are."""
    ts, params = nv.Context._tracker_batch_args(3, [1, 2.5, 3], 20, [10, 20, 30], 30000, (5, 6, 7))
    assert list(ts) == [1.0, 2.5, 3.0]
    assert [(p.threshold, p.min_area, p.max_area, p.distance) for p in params] == [(20, 10, 30000, 5), (20, 20, 30000, 6),
                                                                                   (20, 30, 30000, 7)]
    a = np.zeros((3, 50, 70, 4), np.uint8)[:, 1:49, 2:66]
    ptrs, n, w, h, stride, dev, keep = nv._batch_frames(a, 4)
    assert (n, w, h, stride, dev) == (3, 64, 48, 70 * 4, 0)
    assert [ptrs[i] for i in range(3)] == [a.ctypes.data + i * a.strides[0] for i in range(3)]
