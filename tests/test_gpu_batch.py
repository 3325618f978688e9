"""Batched detection on the GPU: every image of a batch gets exactly the rectangles of the single-image call on it (and
of the CPU oracle), whatever the route (the batched chain or the sequential fallback), the frame source (pageable,
page-locked, device), the row stride and the batch size; the batched route launches the same kernels for any N."""
import ctypes as C
import os

import numpy as np
import pytest

import nubovca as nv
import oracle as O
from cascade_xml_util import write_cascade
from nubovca import synth

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
W, H = 640, 480                                   # BASELINE config 1: processed at 160 x 120


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


_POOL = {}


def frames(n, start=0):
    out = np.empty((n, H, W, 3), np.uint8)
    for i in range(n):
        s = start + i
        if s not in _POOL:
            _POOL[s] = config1_frame(s)
        out[i] = _POOL[s]
    return out


_ORACLE = {}


def oracle_faces(ocasc, seed, mn):
    if (seed, mn) not in _ORACLE:
        _ORACLE[(seed, mn)] = O.face_process(_POOL[seed], ocasc, 160, 1.25, mn, None)[0]
    return _ORACLE[(seed, mn)]


def check(got, batch, ocasc, mn, start=0, single_ctx=None, ncasc=None):
    assert len(got) == len(batch)
    for i, g in enumerate(got):
        exp = oracle_faces(ocasc, start + i, mn)
        assert g.shape == exp.shape and (g == exp).all(), (i, g, exp)
        if single_ctx is not None:
            s = single_ctx.face_detect(ncasc, batch[i], 160, 1.25, mn, None)
            assert s.shape == g.shape and (s == g).all(), (i, s, g)


@pytest.mark.parametrize("mn", [3, 0])
@pytest.mark.parametrize("n", [1, 2, 7, 32, 100, nv.BATCH_MAX])
def test_face_batch_config1(ctx, face, n, mn):
    ncasc, ocasc = face
    b = frames(n)
    single = nv.Context(0, W, H) if n <= 32 else None
    got = ctx.face_detect_batch(ncasc, b, 160, 1.25, mn, None)
    check(got, b, ocasc, mn, 0, single, ncasc)
    if n >= 32:                                       # the batch holds images with and without detections
        assert any(len(g) == 0 for g in got) and any(len(g) > 0 for g in got)
    c = ctx.counters()
    assert c["launches"] == 6                         # the batched route: six launches for the whole batch
    if single:
        single.close()


def test_batch_size_limit(ctx, face):
    ncasc, _ = face
    with pytest.raises(nv.NuboError) as e:
        ctx.face_detect_batch(ncasc, np.zeros((nv.BATCH_MAX + 1, 48, 64, 3), np.uint8))
    assert e.value.code == -1


def _pinned(shape):
    ptr = C.c_void_p()
    size = int(np.prod(shape))
    assert nv._lib.nv_host_alloc(size, C.byref(ptr)) == 0
    arr = np.ctypeslib.as_array((C.c_uint8 * size).from_address(ptr.value)).reshape(shape)
    return arr, ptr


def raw_counters(ctx):
    o = (C.c_longlong * 8)()
    assert nv._lib.nv_debug_get_counters(ctx.handle, o) == 0
    return list(o)


@pytest.mark.parametrize("n", [9, 32, nv.BATCH_MAX])
@pytest.mark.parametrize("source", ["pageable", "pinned", "device"])
@pytest.mark.parametrize("pad", [0, 36])
def test_face_batch_sources_strides_and_replay(face, source, pad, n):
    """New contents in new buffers on every call, the same shape: the graph replays (counter [4]) and every result stays
    exact."""
    import torch
    ncasc, ocasc = face
    rowbytes = W * 3 + pad
    ctx = nv.Context(0, W, H)
    for it in range(3):
        start = 3 + n * it
        b = frames(n, start)
        keep = None
        if source == "pinned":
            wide, keep = _pinned((n, H, rowbytes))
        else:
            wide = np.zeros((n, H, rowbytes), np.uint8)
        wide[:, :, :W * 3] = b.reshape(n, H, W * 3)
        if source == "device":
            t = torch.from_numpy(wide).cuda()
            src = t.as_strided((n, H, W, 3), (t.stride(0), t.stride(1), 3, 1))
        else:
            src = np.lib.stride_tricks.as_strided(wide, shape=(n, H, W, 3), strides=(wide.strides[0], wide.strides[1], 3, 1))
        got = ctx.face_detect_batch(ncasc, src, 160, 1.25, 3, None)
        check(got, b, ocasc, 3, start)
        c = raw_counters(ctx)
        assert c[3] == 6 and c[4] == (it == 2)         # seen, captured, replayed
        if keep is not None:
            del src, wide
            nv._lib.nv_host_free(keep)
    ctx.close()


def test_single_calls_interleaved_with_batches(face):
    ncasc, ocasc = face
    fresh = nv.Context(0, 1920, 1080)
    ctx = nv.Context(0, 1920, 1080)
    b = frames(8, 40)
    big = synth.frame(960, 540, 5, 7)
    gray = synth.frame(160, 120, 2, 77)[..., 1].copy()
    exp_face = [fresh.face_detect(ncasc, f, 160, 1.25, 3, None) for f in b[:2]]
    exp_big = fresh.face_detect(ncasc, big, 960, 1.1, 3, (24, 24))
    exp_gray = fresh.detect_multiscale(ncasc, gray, 1.1, 3)
    for rep in range(3):
        check(ctx.face_detect_batch(ncasc, b, 160, 1.25, 3, None), b, ocasc, 3, 40)
        for f, e in zip(b[:2], exp_face):
            g = ctx.face_detect(ncasc, f, 160, 1.25, 3, None)
            assert (g.shape == e.shape) and (g == e).all()
        g = ctx.face_detect(ncasc, big, 960, 1.1, 3, (24, 24))
        assert g.shape == exp_big.shape and (g == exp_big).all()
        ctx.face_submit_batch(ncasc, b[:3], 160, 1.25, 0, None)
        got = ctx.face_collect_batch()
        check(got, b[:3], ocasc, 0, 40)
        g = ctx.detect_multiscale(ncasc, gray, 1.1, 3)
        assert g.shape == exp_gray.shape and (g == exp_gray).all()
        # taps that describe single calls refuse to describe a batch
        ctx.face_detect_batch(ncasc, b[:2], 160, 1.25, 3, None)
        with pytest.raises(nv.NuboError) as e:
            ctx.gray()
        assert e.value.code == -8
    ctx.close(); fresh.close()


def test_route_visible_in_launch_counts(face, cascade_dir):
    ncasc, _ = face
    ctx = nv.Context(0, 1920, 1080)
    ctx.face_detect_batch(ncasc, frames(1), 160, 1.25, 3, None)
    l1 = ctx.counters()["launches"]
    ctx.face_detect_batch(ncasc, frames(64), 160, 1.25, 3, None)
    assert ctx.counters()["launches"] == l1 == 6
    # fallback (a large plan, a tree model with tilted features): N single calls
    for xml, size in (("haarcascade_frontalface_alt.xml", (640, 360)), ("haarcascade_eye_tree_eyeglasses.xml", (160, 120))):
        c = nv.Cascade(os.path.join(cascade_dir, xml))
        imgs = np.stack([synth.frame(size[0], size[1], 2, 300 + i)[..., 1] for i in range(5)])
        one = nv.Context(0, 1920, 1080)
        before = one.counters()["launches"]
        one.detect_multiscale(c, imgs[0], 1.1, 3)
        per_call = one.counters()["launches"] - before
        one.close()
        ctx.detect_multiscale_batch(c, imgs, 1.1, 3)
        assert ctx.counters()["launches"] == 5 * per_call, xml
    ctx.close()


GRAY_CASES = [
    ("haarcascade_frontalface_alt.xml", 96, 64, 1.1, (0, 0), True),
    ("haarcascade_frontalface_alt.xml", 160, 120, 1.25, (0, 0), True),
    ("haarcascade_frontalface_alt.xml", 160, 120, 1.1, (0, 0), False),     # more than 16 384 windows: a large plan
    ("haarcascade_eye_tree_eyeglasses.xml", 160, 120, 1.1, (0, 0), False),
    ("haarcascade_lefteye_2splits.xml", 160, 120, 1.1, (0, 0), False),
    ("lbp_random_0.xml", 160, 120, 1.1, (0, 0), False),
    ("haarcascade_frontalface_alt.xml", 1920, 1080, 1.2, (40, 40), False),
]


@pytest.mark.parametrize("xml,w,h,sf,ms,routed", GRAY_CASES, ids=[f"{c[0]}-{c[1]}x{c[2]}-{c[3]}" for c in GRAY_CASES])
@pytest.mark.parametrize("mn", [3, 0])
def test_gray_batch(ctx, cascade_dir, xml, w, h, sf, ms, routed, mn):
    path = os.path.join(HERE, "golden", xml) if xml.startswith("lbp") else os.path.join(cascade_dir, xml)
    ncasc, ocasc = nv.Cascade(path), O.Cascade(path)
    n = 2 if w > 1000 else 6
    imgs = np.stack([synth.frame(w, h, 1 + i % 3, 500 + i)[..., 1] for i in range(n)])
    imgs[0] = 120                                       # a flat image
    got = ctx.detect_multiscale_batch(ncasc, imgs, sf, mn, ms)
    single = nv.Context(0, 1920, 1080)
    for i in range(n):
        exp = O.detect_multiscale(imgs[i], ocasc, sf, mn, ms)
        s = single.detect_multiscale(ncasc, imgs[i], sf, mn, ms)
        assert got[i].shape == exp.shape and (got[i] == exp).all(), (i, got[i], exp)
        assert (s == got[i]).all()
    single.close()
    assert (ctx.counters()["launches"] == 5) == routed


def test_batch_capacity_and_refusals(ctx, face):
    ncasc, ocasc = face
    b = frames(6, 2)
    full = ctx.face_detect_batch(ncasc, b, 160, 1.25, 0, None)
    counts = [len(g) for g in full]
    cap = sum(counts) // 2
    ptrs = (C.c_void_p * 6)(*[b.ctypes.data + i * b.strides[0] for i in range(6)])
    out = (nv.Rect * max(cap, 1))(); cn = (C.c_int * 6)(); total = C.c_int(0)
    p = nv.FaceParams(160, 1.25, 0, -1, -1)
    rc = nv._lib.nv_face_detect_batch(ctx.handle, ncasc.handle, ptrs, 6, W, H, b.strides[1], 0, C.byref(p), out, cap, cn, C.byref(total))
    assert rc == -6 and list(cn) == counts and total.value == cap
    flat = np.concatenate(full)[:cap]
    assert (np.frombuffer(out, np.int32, 4 * cap).reshape(-1, 4) == flat).all()
    ctx.set_scores(True)
    try:
        with pytest.raises(nv.NuboError) as e:
            ctx.face_detect_batch(ncasc, b, 160, 1.25, 3, None)
        assert e.value.code == -8
    finally:
        ctx.set_scores(False)


@pytest.mark.parametrize("w,h,pad", [(160, 120, 0), (320, 240, 0), (160, 120, 1), (320, 240, 1)],
                         ids=["copy", "box2", "copy-unaligned", "box2-unaligned"])
def test_face_batch_streaming_modes(ctx, face, w, h, pad):
    """Frames of the processing size (copy) and of twice it (2x box): the vectorised prep kernel when rows are 4-byte
    aligned, the byte-per-lane one when the stride is odd."""
    ncasc, ocasc = face
    n = 12
    imgs = [np.full((h, w, 3), 90, np.uint8)] + [synth.frame(w, h, 1 + i % 3, 700 + i) for i in range(1, n)]
    wide = np.zeros((n, h, 3 * w + pad), np.uint8)
    for i in range(n):
        wide[i, :, :3 * w] = imgs[i].reshape(h, 3 * w)
    src = np.lib.stride_tricks.as_strided(wide, shape=(n, h, w, 3), strides=(wide.strides[0], wide.strides[1], 3, 1))
    single = nv.Context(0, w, h)
    for mn in (3, 0):
        got = ctx.face_detect_batch(ncasc, src, 160, 1.25, mn, None)
        assert raw_counters(ctx)[3] == 6
        for i in range(n):
            exp = O.face_process(imgs[i], ocasc, 160, 1.25, mn, None)[0]
            s = single.face_detect(ncasc, imgs[i], 160, 1.25, mn, None)
            assert got[i].shape == exp.shape and (got[i] == exp).all(), (i, got[i], exp)
            assert s.shape == exp.shape and (s == exp).all()
    single.close()


def permissive_model(path):
    """Two stump stages that every window with some contrast passes (leaves +-0.5, thresholds -5): more than 1024 raw
    candidates on a 160x120 image, with the exactness certificates of the batched route."""
    feats = [[(0, 0, 20, 10, -1.0), (0, 0, 20, 5, 2.0)], [(0, 0, 10, 20, -1.0), (0, 0, 5, 20, 2.0)]]
    write_cascade(path, 20, 20, [(-5.0, [(0, 0.0, 0.5, -0.5), (1, 0.0, -0.5, 0.5)]), (-5.0, [(1, 0.1, 0.5, -0.5)])], feats)


def test_batch_overflow_rerun(ctx, tmp_path):
    """An image with more raw candidates than the batched grouping holds is detected again alone in collect, from its
    device copy (for host face frames: the uploaded row pairs only); the others keep their batched results."""
    p = str(tmp_path / "permissive.xml")
    permissive_model(p)
    ncasc, ocasc = nv.Cascade(p), O.Cascade(p)
    assert ncasc.info.order_free_sums == 1
    rng = np.random.default_rng(9)
    noise = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    patch = np.full((H, W, 3), 128, np.uint8)                     # a few hundred candidates: stays in the batched grouping
    patch[200:212, 300:312] = rng.integers(0, 256, (12, 12, 3), dtype=np.uint8)
    b = np.stack([np.full((H, W, 3), 128, np.uint8), noise, patch])
    gray = np.ascontiguousarray(b[:, ::4, ::4, 1])                                  # 160 x 120
    for mn in (0, 3):
        one = nv.Context(0, W, H)
        before = one.counters()["launches"]
        s_face = one.face_detect(ncasc, noise, 160, 1.25, mn, None)
        per_face = one.counters()["launches"] - before
        assert one.counters()["candidates"] > 1024
        before = one.counters()["launches"]
        s_gray = one.detect_multiscale(ncasc, gray[1], 1.25, mn)
        per_gray = one.counters()["launches"] - before
        got = ctx.face_detect_batch(ncasc, b, 160, 1.25, mn, None)
        # the batched chain, then image 1 alone (per_face: a call whose own candidate buffers overflow first and re-run
        # too; the batch's re-run may find them grown already); the fallback would be three single calls
        assert 6 < raw_counters(ctx)[3] <= 6 + per_face
        for i in range(3):
            exp = O.face_process(b[i], ocasc, 160, 1.25, mn, None, cap=1 << 16)[0]
            assert got[i].shape == exp.shape and (got[i] == exp).all(), i
        assert (got[1] == s_face).all()
        got = ctx.detect_multiscale_batch(ncasc, gray, 1.25, mn)
        assert 5 < raw_counters(ctx)[3] <= 5 + per_gray
        for i in range(3):
            exp = O.detect_multiscale(gray[i], ocasc, 1.25, mn)
            assert got[i].shape == exp.shape and (got[i] == exp).all(), i
        assert (got[1] == s_gray).all()
        one.close()
