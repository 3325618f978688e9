"""CUDA-graph replay on every call path that graphs: the first call with a key runs plain launches, the second captures
them into a graph, every later one replays it.  Each of those calls must give the rectangles of a debug context (which
never graphs) and count the same launches; with profiling on, a replayed face block reports the stage times its capture
recorded, and a single detect (which never graphs with profiling on) reports them on every call."""
import ctypes as C
import os

import numpy as np
import pytest

import nubovca as nv
from nubovca import synth

pytestmark = pytest.mark.gpu
W, H = 640, 480                                   # BASELINE config 1: processed at 160 x 120
CALLS = 5                                         # plain, captured, three replays
# stages of the small-plan chain that hold a kernel; "hist_lut" (the LUT comes from face_prep's last block) and
# "cascade_tiles" (stage 0 queues the tail's windows itself) hold none and may read 0 or a few microseconds
DETECT_STAGES = ("pyramid_rowscan", "integral_colscan", "cascade_stage0", "cascade_tail", "group_rectangles")
FACE_STAGES = ("face_prep",) + DETECT_STAGES
EMPTY_STAGES = {"hist_lut", "cascade_tiles"}


@pytest.fixture(scope="module")
def casc(cascade_dir):
    return nv.Cascade(os.path.join(cascade_dir, "haarcascade_frontalface_alt.xml"))


@pytest.fixture(scope="module")
def frame():
    return synth.frame(W, H, 4, 1)


@pytest.fixture(scope="module")
def gray():
    return synth.frame(160, 120, 2, 77)[..., 1].copy()


def raw_counters(ctx):
    o = (C.c_longlong * 8)()
    assert nv._lib.nv_debug_get_counters(ctx.handle, o) == 0
    return list(o)


def same(a, b):
    return a.shape == b.shape and (a == b).all()


def run_path(path, casc, frame, gray):
    """One call on `path`, as a function of the context that returns its rectangles (a list of them for a batch)."""
    if path == "detect":
        return lambda c: c.detect_multiscale(casc, gray, 1.1, 3)
    if path == "face_host":
        return lambda c: c.face_detect(casc, frame, 160, 1.25, 3, None)
    if path == "face_device":
        import torch
        d = torch.from_numpy(frame).cuda()
        torch.cuda.synchronize()

        def face_device(c):
            c.face_submit_device(casc, d.data_ptr(), W, H, 3 * W, 160, 1.25, 3, None)
            return c.face_collect()
        return face_device
    batch = np.stack([frame, synth.frame(W, H, 2, 1003), np.full((H, W, 3), 128, np.uint8)])
    return lambda c: c.face_detect_batch(casc, batch, 160, 1.25, 3, None)


@pytest.mark.parametrize("path", ["detect", "face_host", "face_device", "batch"])
def test_plain_captured_replayed_calls_agree(casc, frame, gray, path):
    call = run_path(path, casc, frame, gray)
    ref_ctx = nv.Context(0, W, H, debug=True)
    ctx = nv.Context(0, W, H)
    try:
        ref = call(ref_ctx)
        got, launches = [], []
        for it in range(CALLS):
            before = ctx.counters()["launches"]
            got.append(call(ctx))
            c = raw_counters(ctx)
            if path == "batch":
                launches.append(c[3])                 # a batch reports the launches of the call itself
                assert c[4] == (it >= 2), it          # seen, captured, then replayed
            else:
                launches.append(c[3] - before)
        if path == "batch":
            assert any(len(g) for g in ref) and any(len(g) == 0 for g in ref)
            for it, g in enumerate(got):
                assert len(g) == len(ref) and all(same(a, b) for a, b in zip(g, ref)), it
        else:
            assert len(ref) > 0
            for it, g in enumerate(got):
                assert same(g, ref), (it, g, ref)
        assert launches[0] > 1 and launches == [launches[0]] * CALLS, launches
    finally:
        ctx.close()
        ref_ctx.close()


def nonzero(times):
    return {k for k, v in times.items() if v > 0}


def test_face_replay_reports_captured_stage_times(casc, frame):
    """What bench.py runs: the face block with profiling on, replayed from its graph from the third call on."""
    ctx = nv.Context(0, W, H)
    try:
        ctx.set_profile(True)
        times = []
        for _ in range(4):
            ctx.face_detect(casc, frame, 160, 1.25, 3, None)
            times.append(ctx.stage_times())
        first = nonzero(times[0])
        assert set(FACE_STAGES) <= first, times[0]
        for it in (2, 3):
            assert nonzero(times[it]) - EMPTY_STAGES == first - EMPTY_STAGES, (it, times[it], times[0])
    finally:
        ctx.close()


def test_detect_with_profiling_reports_stage_times_every_call(casc, gray):
    ctx = nv.Context(0, W, H)
    try:
        ctx.set_profile(True)
        ref = None
        for it in range(4):
            r = ctx.detect_multiscale(casc, gray, 1.1, 3)
            ref = r if ref is None else ref
            assert same(r, ref), it
            t = ctx.stage_times()
            assert set(DETECT_STAGES) <= nonzero(t), (it, t)
    finally:
        ctx.close()
