"""Batches of 4:2:0 frames on the GPU (nv_face_*_batch_yuv): every image of a batch gets exactly the rectangles of the
single 4:2:0 call on it and of the CPU oracle on the converted frame, whatever the format, the route (the batched chain or
the sequential fallback), the plane sources (pageable, page-locked, device, scattered), the row pitch and the batch size."""
import ctypes as C
import os

import numpy as np
import pytest

import nubovca as nv
import oracle as O
from cascade_xml_util import write_cascade
from nubovca import synth

pytestmark = pytest.mark.gpu
W, H = 640, 480                                   # BASELINE config 1: processed at 160 x 120
FMTS = ["I420", "YV12", "NV12", "NV21"]


@pytest.fixture(scope="module")
def face(cascade_dir):
    p = os.path.join(cascade_dir, "haarcascade_frontalface_alt.xml")
    return nv.Cascade(p), O.Cascade(p)


@pytest.fixture(scope="module")
def ctx():
    c = nv.Context(0, 1920, 1080)
    yield c
    c.close()


def config1_frame(seed):
    """seed 0: flat (every window variance-rejected), 1: no face, 2: many faces, else 1..4 faces."""
    if seed == 0:
        return np.full((H, W, 3), 128, np.uint8)
    if seed == 1:
        return synth.frame(W, H, 0, 1001)
    if seed == 2:
        return synth.frame(W, H, 14, 1002, smin=0.12, smax=0.16)
    return synth.frame(W, H, 1 + seed % 4, 1000 + seed)


_BGR, _POOL = {}, {}


def yuv_buf(seed, fmt):
    """The 4:2:0 buffer of config-1 frame `seed`.  All four formats carry the same samples, so they convert to one BGR frame."""
    if (seed, fmt) not in _POOL:
        if seed not in _BGR:
            _BGR[seed] = config1_frame(seed)
        _POOL[(seed, fmt)] = synth.to_yuv420(_BGR[seed], fmt)
    return _POOL[(seed, fmt)]


def yuv_batch(n, fmt, start=0):
    return np.stack([yuv_buf(start + i, fmt) for i in range(n)])


def ora_bgr(buf, fmt, w=W, h=H):
    return O.yuv420_to_bgr(*O.yuv420_planes(buf, w, h, fmt), fmt=fmt)


_ORACLE = {}


def oracle_faces(ocasc, seed, mn):
    if (seed, mn) not in _ORACLE:
        _ORACLE[(seed, mn)] = O.face_process(ora_bgr(yuv_buf(seed, "I420"), "I420"), ocasc, 160, 1.25, mn, None)[0]
    return _ORACLE[(seed, mn)]


def same(a, b):
    a = np.asarray(a, np.int32).reshape(-1, 4); b = np.asarray(b, np.int32).reshape(-1, 4)
    return a.shape == b.shape and bool((a == b).all())


def check(got, ocasc, mn, start=0):
    for i, g in enumerate(got):
        assert same(g, oracle_faces(ocasc, start + i, mn)), (i, g, oracle_faces(ocasc, start + i, mn))


def single_yuv(c, ncasc, buf, fmt, w=W, h=H, w2p=160, mn=3):
    return c.face_detect_yuv(ncasc, synth.yuv420_planes(np.ascontiguousarray(buf), w, h, fmt), fmt, w2p, 1.25, mn, None)


def raw_counters(c):
    o = (C.c_longlong * 8)()
    assert nv._lib.nv_debug_get_counters(c.handle, o) == 0
    return list(o)


def _pinned(shape):
    ptr = C.c_void_p()
    size = int(np.prod(shape))
    assert nv._lib.nv_host_alloc(size, C.byref(ptr)) == 0
    arr = np.ctypeslib.as_array((C.c_uint8 * size).from_address(ptr.value)).reshape(shape)
    return arr, ptr


@pytest.mark.parametrize("mn", [3, 0])
@pytest.mark.parametrize("n", [1, 7, 32, nv.BATCH_MAX])
@pytest.mark.parametrize("fmt", FMTS)
def test_yuv_batch_config1(ctx, face, fmt, n, mn):
    ncasc, ocasc = face
    b = yuv_batch(n, fmt)
    got = ctx.face_detect_batch_yuv(ncasc, b, fmt, 160, 1.25, mn, None)
    assert len(got) == n
    assert raw_counters(ctx)[3] == 6                  # the batched route: six launches for the whole batch
    check(got, ocasc, mn)
    if n >= 32:
        assert any(len(g) == 0 for g in got) and any(len(g) > 0 for g in got)
    if n <= 32:
        single = nv.Context(0, W, H)
        for i in range(n):
            assert same(single_yuv(single, ncasc, b[i], fmt, mn=mn), got[i]), i
        single.close()


SOURCE_CASES = [("NV12", 0), ("NV12", 36), ("I420", 0)]


@pytest.mark.parametrize("n", [9, 32])
@pytest.mark.parametrize("source", ["pageable", "pinned", "device"])
@pytest.mark.parametrize("fmt,pad", SOURCE_CASES, ids=[f"{f}-pad{p}" for f, p in SOURCE_CASES])
def test_yuv_batch_sources_strides_and_replay(face, fmt, pad, source, n):
    """New contents in new buffers on every call, the same shape: the graph replays (counter [4]) and every result stays
    exact.  Row padding: NV12 rows at a decoder's pitch (the chroma rows follow at the same pitch)."""
    import torch
    ncasc, ocasc = face
    pitch = W + pad
    c = nv.Context(0, W, H)
    for it in range(3):
        start = 3 + n * it
        b = yuv_batch(n, fmt, start)
        keep = None
        if source == "pinned":
            wide, keep = _pinned((n, H * 3 // 2, pitch))
        else:
            wide = np.zeros((n, H * 3 // 2, pitch), np.uint8)
        wide[:, :, :W] = b
        if source == "device":
            t = torch.from_numpy(wide).cuda()
            src = t[:, :, :W]
        else:
            src = wide[:, :, :W]
        got = c.face_detect_batch_yuv(ncasc, src, fmt, 160, 1.25, 3, None)
        check(got, ocasc, 3, start)
        k = raw_counters(c)
        assert k[3] == 6 and k[4] == (it == 2)         # seen, captured, replayed
        if keep is not None:
            del src, wide
            nv._lib.nv_host_free(keep)
    c.close()


def prep_kernels(fn):
    """fn()'s result and the names of the 4:2:0 prep kernels it launched (torch.profiler records every kernel of the
    process, the library's own stream included)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    return r, {e.name for e in prof.events() if "k_face_prep_yuv" in e.name}


# layout of a batch of n packed 4:2:0 buffers:
#   host         numpy array, images an odd number of bytes apart: the upload puts every plane into an aligned slot
#   device       CUDA tensor, contiguous: every plane of every image 4-byte aligned
#   device-odd   CUDA tensor, images an odd number of bytes apart: image 0 aligned, image 1 not
#   device-pitch CUDA tensor, NV12 / NV21 rows at an odd pitch (W + 1): aligned image starts, odd strides
STREAM_CASES = [(fmt, layout) for fmt in ("I420", "NV12", "NV21") for layout in ("host", "device", "device-odd", "device-pitch")
                if not (fmt == "I420" and layout == "device-pitch")]


@pytest.mark.parametrize("w,h", [(160, 120), (320, 240)], ids=["copy", "box2"])
@pytest.mark.parametrize("fmt,layout", STREAM_CASES, ids=[f"{f}-{l}" for f, l in STREAM_CASES])
def test_yuv_batch_streaming_modes(face, fmt, layout, w, h):
    """Frames of the processing size (copy) and of twice it (2x box): the vectorised prep kernel runs only when every plane
    pointer of every image the kernel reads, and every stride, is 4-byte aligned; otherwise the byte-per-lane kernel."""
    import torch
    ncasc, ocasc = face
    n = 10
    bgr = [np.full((h, w, 3), 90, np.uint8)] + [synth.frame(w, h, 1 + i % 3, 700 + i) for i in range(1, n)]
    bufs = np.stack([synth.to_yuv420(f, fmt) for f in bgr])
    h3 = h * 3 // 2
    pitch = w + 1 if layout == "device-pitch" else w
    size = h3 * pitch + (1 if layout in ("host", "device-odd") else 0)
    flat = np.zeros(n * size + 8, np.uint8)
    for i in range(n):
        flat[i * size:i * size + h3 * pitch].reshape(h3, pitch)[:, :w] = bufs[i]
    if layout == "host":
        src = np.lib.stride_tricks.as_strided(flat, shape=bufs.shape, strides=(size, pitch, 1))
    else:
        src = torch.as_strided(torch.from_numpy(flat).cuda(), bufs.shape, (size, pitch, 1))
    vectorised = layout in ("host", "device")
    c = nv.Context(0, W, H)
    for mn in (3, 0):
        got, kernels = prep_kernels(lambda: c.face_detect_batch_yuv(ncasc, src, fmt, 160, 1.25, mn, None))
        assert raw_counters(c)[3] == 6
        assert len(kernels) == 1, kernels
        assert ("k_face_prep_yuv4" in kernels.pop()) == vectorised, (layout, kernels)
        for i in range(n):
            exp = O.face_process(ora_bgr(bufs[i], fmt, w, h), ocasc, 160, 1.25, mn, None)[0]
            assert same(got[i], exp), (i, got[i], exp)
    c.close()


def _frame_struct(fmt, w, h, planes, strides, on_device=0):
    f = nv.YuvFrame()
    f.format, f.width, f.height, f.on_device = nv._FMT[fmt], w, h, on_device
    for k, (p, s) in enumerate(zip(planes, strides)):
        f.plane[k], f.stride[k] = p, s
    return f


@pytest.mark.parametrize("fmt", ["I420", "NV12"])
def test_yuv_batch_scattered_planes(ctx, face, fmt):
    """Every plane of every image in an allocation of its own, page-locked and pageable planes mixed within one batch."""
    ncasc, ocasc = face
    n = 6
    keep, pinned, frames = [], [], (nv.YuvFrame * n)()
    for i in range(n):
        buf = yuv_buf(10 + i, fmt)
        planes = synth.yuv420_planes(buf, W, H, fmt)
        ptrs, strides = [], []
        for k, p in enumerate(planes):
            if (i + k) % 2:
                a, ptr = _pinned(p.shape)
                pinned.append(ptr)
            else:
                a = np.empty(p.shape, np.uint8)
            a[:] = p
            keep.append(a)
            ptrs.append(a.ctypes.data); strides.append(a.strides[0])
        frames[i] = _frame_struct(fmt, W, H, ptrs, strides)
    fp = nv.FaceParams(160, 1.25, 3, -1, -1)
    out = (nv.Rect * 4096)(); counts = (C.c_int * n)(); total = C.c_int(0)
    try:
        assert nv._lib.nv_face_detect_batch_yuv(ctx.handle, ncasc.handle, frames, n, C.byref(fp), out, 4096, counts, C.byref(total)) == 0
        assert raw_counters(ctx)[3] == 6
        flat = np.frombuffer(out, np.int32, 4 * total.value).reshape(-1, 4)
        single = nv.Context(0, W, H)
        o = 0
        for i in range(n):
            s = single_yuv(single, ncasc, yuv_buf(10 + i, fmt), fmt)
            assert same(flat[o:o + counts[i]], s) and same(s, oracle_faces(ocasc, 10 + i, 3)), i
            o += counts[i]
        single.close()
    finally:
        for p in pinned:
            nv._lib.nv_host_free(p)


@pytest.mark.parametrize("fmt", ["I420", "NV12"])
@pytest.mark.parametrize("xml,w,h,w2p", [("haarcascade_frontalface_alt.xml", 1280, 720, 640),
                                          ("haarcascade_eye_tree_eyeglasses.xml", 640, 480, 160)],
                         ids=["large-plan", "tree-model"])
def test_yuv_batch_fallback(cascade_dir, fmt, xml, w, h, w2p):
    """Shapes the batched chain does not take run the single 4:2:0 call per image: the same rectangles and launches."""
    path = os.path.join(cascade_dir, xml)
    ncasc = nv.Cascade(path)
    n = 3
    bufs = np.stack([synth.to_yuv420(synth.frame(w, h, 2 + i, 900 + i), fmt) for i in range(n)])
    one = nv.Context(0, w, h)
    exp, per_call = [], 0
    for i in range(n):
        before = one.counters()["launches"]
        exp.append(single_yuv(one, ncasc, bufs[i], fmt, w, h, w2p))
        per_call += one.counters()["launches"] - before
    one.close()
    c = nv.Context(0, w, h)
    got = c.face_detect_batch_yuv(ncasc, bufs, fmt, w2p, 1.25, 3, None)
    assert raw_counters(c)[3] == per_call
    for i in range(n):
        assert same(got[i], exp[i]), i
    c.close()


def permissive_model(path):
    """Two stump stages that every window with some contrast passes (leaves +-0.5, thresholds -5): more than 1024 raw
    candidates on a 160x120 image, with the exactness certificates of the batched route."""
    feats = [[(0, 0, 20, 10, -1.0), (0, 0, 20, 5, 2.0)], [(0, 0, 10, 20, -1.0), (0, 0, 5, 20, 2.0)]]
    write_cascade(path, 20, 20, [(-5.0, [(0, 0.0, 0.5, -0.5), (1, 0.0, -0.5, 0.5)]), (-5.0, [(1, 0.1, 0.5, -0.5)])], feats)


@pytest.mark.parametrize("source", ["pageable", "device"])
@pytest.mark.parametrize("fmt", ["I420", "NV21"])
def test_yuv_batch_overflow_rerun(ctx, tmp_path, fmt, source):
    """An image with more raw candidates than the batched grouping holds is detected again alone in collect, from its
    device planes (for host frames: the uploaded copy, luma row pairs only); the others keep their batched results."""
    import torch
    p = str(tmp_path / "permissive.xml")
    permissive_model(p)
    ncasc, ocasc = nv.Cascade(p), O.Cascade(p)
    rng = np.random.default_rng(9)
    noise = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    patch = np.full((H, W, 3), 128, np.uint8)                     # a few hundred candidates: stays in the batched grouping
    patch[200:212, 300:312] = rng.integers(0, 256, (12, 12, 3), dtype=np.uint8)
    bufs = np.stack([synth.to_yuv420(f, fmt) for f in (np.full((H, W, 3), 128, np.uint8), noise, patch)])
    src = torch.from_numpy(bufs).cuda() if source == "device" else bufs
    for mn in (0, 3):
        one = nv.Context(0, W, H)
        before = one.counters()["launches"]
        s1 = single_yuv(one, ncasc, bufs[1], fmt, mn=mn)
        per_face = one.counters()["launches"] - before
        assert one.counters()["candidates"] > 1024
        s = [single_yuv(one, ncasc, bufs[0], fmt, mn=mn), s1, single_yuv(one, ncasc, bufs[2], fmt, mn=mn)]
        got = ctx.face_detect_batch_yuv(ncasc, src, fmt, 160, 1.25, mn, None)
        assert 6 < raw_counters(ctx)[3] <= 6 + per_face
        for i in range(3):
            exp = O.face_process(ora_bgr(bufs[i], fmt), ocasc, 160, 1.25, mn, None, cap=1 << 16)[0]
            assert same(got[i], exp) and same(got[i], s[i]), i
        one.close()


@pytest.mark.parametrize("fmt", FMTS)
def test_yuv_batch_equals_bgr_batch(ctx, face, fmt):
    ncasc, _ = face
    b = yuv_batch(16, fmt, 20)
    bgr = np.stack([ctx.yuv2bgr(synth.yuv420_planes(b[i], W, H, fmt), fmt) for i in range(16)])
    got = ctx.face_detect_batch_yuv(ncasc, b, fmt, 160, 1.25, 3, None)
    exp = ctx.face_detect_batch(ncasc, bgr, 160, 1.25, 3, None)
    for i in range(16):
        assert same(got[i], exp[i]), i


def test_yuv_batches_interleaved(face):
    """4:2:0 batches of two formats, a BGR batch of the same size and single calls on one context: no call replays a graph
    another shape captured, every result stays exact."""
    ncasc, ocasc = face
    c = nv.Context(0, W, H)
    n = 8
    nv12, i420 = yuv_batch(n, "NV12", 30), yuv_batch(n, "I420", 30)
    bgr = np.stack([ora_bgr(nv12[i], "NV12") for i in range(n)])
    for rep in range(3):
        check(c.face_detect_batch_yuv(ncasc, nv12, "NV12", 160, 1.25, 3, None), ocasc, 3, 30)
        check(c.face_detect_batch(ncasc, bgr, 160, 1.25, 3, None), ocasc, 3, 30)
        check(c.face_detect_batch_yuv(ncasc, i420, "I420", 160, 1.25, 3, None), ocasc, 3, 30)
        assert same(single_yuv(c, ncasc, nv12[rep], "NV12"), oracle_faces(ocasc, 30 + rep, 3))
        assert same(c.face_detect(ncasc, bgr[rep], 160, 1.25, 3, None), oracle_faces(ocasc, 30 + rep, 3))
        check(c.face_detect_batch_yuv(ncasc, nv12[:3], "NV12", 160, 1.25, 0, None), ocasc, 0, 30)
    c.close()


def test_yuv_batch_refusals(ctx, face):
    ncasc, ocasc = face
    L = nv._lib
    n = 4
    bufs = yuv_batch(n, "NV12", 2)
    fp = nv.FaceParams(160, 1.25, 0, -1, -1)

    def table(fmt="NV12"):
        t = (nv.YuvFrame * n)()
        for i in range(n):
            t[i] = _frame_struct(fmt, W, H, [bufs[i].ctypes.data, bufs[i].ctypes.data + W * H], [W, W])
        return t

    def submit(t, c=ctx):
        return L.nv_face_submit_batch_yuv(c.handle, ncasc.handle, t, n, C.byref(fp))

    for bad_n in (0, -1, nv.BATCH_MAX + 1):                       # n out of range, with a real context
        assert L.nv_face_submit_batch_yuv(ctx.handle, ncasc.handle, table(), bad_n, C.byref(fp)) == -1
        assert b"batch of" in L.nv_last_error(), bad_n
    for field, value in (("format", nv.FMT_NV21), ("width", W - 2), ("height", H - 2), ("on_device", 1)):
        t = table()
        setattr(t[2], field, value)
        assert submit(t) == -1, field
        assert b"image 2" in L.nv_last_error(), field
    t = table()
    t[3].stride[1] = W + 4
    assert submit(t) == -1 and b"image 3" in L.nv_last_error()
    t = table()
    for i in range(n):
        t[i].width = W - 1                                        # odd width
    assert submit(t) == -1
    small = nv.Context(0, 320, 240)
    assert submit(table(), small) == -6                           # larger than the context
    small.close()
    ctx.set_scores(True)
    try:
        assert submit(table()) == -8
    finally:
        ctx.set_scores(False)
    # a pending 4:2:0 batch is collected with nv_face_collect_batch only
    full = ctx.face_detect_batch_yuv(ncasc, bufs, "NV12", 160, 1.25, 0, None)
    counts = [len(g) for g in full]
    assert sum(counts) > 1
    assert submit(table()) == 0
    one = (nv.Rect * 16)(); k = C.c_int(0)
    assert L.nv_face_collect(ctx.handle, one, 16, C.byref(k)) == -8
    out = (nv.Rect * 4096)(); cn = (C.c_int * n)(); total = C.c_int(0)
    assert L.nv_face_collect_batch(ctx.handle, out, 4096, cn, C.byref(total)) == 0
    assert list(cn) == counts and (np.frombuffer(out, np.int32, 4 * total.value).reshape(-1, 4) == np.concatenate(full)).all()
    # too small a capacity: true counts, the first cap rectangles
    cap = sum(counts) // 2
    out = (nv.Rect * max(cap, 1))(); cn = (C.c_int * n)(); total = C.c_int(0)
    rc = L.nv_face_detect_batch_yuv(ctx.handle, ncasc.handle, table(), n, C.byref(fp), out, cap, cn, C.byref(total))
    assert rc == -6 and list(cn) == counts and total.value == cap
    assert (np.frombuffer(out, np.int32, 4 * cap).reshape(-1, 4) == np.concatenate(full)[:cap]).all()
