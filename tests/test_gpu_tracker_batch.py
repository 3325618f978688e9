"""The batched tracker on the GPU (nv_tracker_process_batch / _yuv / nv_tracker_reset_batch): every slot of a batch gets
exactly the rectangles of the CPU oracle's tracker (O.TrackerState) fed that slot's frames, timestamps and parameters, and
of nv_tracker_process(_yuv) on a separate context, whatever the sources, formats, slot history and interleaved calls."""
import ctypes as C
import os

import numpy as np
import pytest

import nubovca as nv
import oracle as O
from nubovca import synth

pytestmark = pytest.mark.gpu
NV_ERR_ARG, NV_ERR_CAPACITY = -1, -6


def same(a, b):
    a = np.asarray(a, np.int32).reshape(-1, 4); b = np.asarray(b, np.int32).reshape(-1, 4)
    return a.shape == b.shape and bool((a == b).all())


def slot_params(i):
    """Per-slot element properties: thresholds, areas and distances differ from slot to slot."""
    return dict(threshold=12 + 4 * (i % 5), min_area=20 + 15 * (i % 4), max_area=30000 + 20000 * (i % 3), distance=20 + 8 * (i % 4))


def slot_ts(i, f):
    """Slot i's timestamp of frame f: even slots repeat timestamps closer than MHI_DURATION (stale history stays alive, as in
    test_tracker_vs_oracle_with_join_and_stale_history), every third slot jumps by more than 200 ms, the rest run at 30 fps."""
    if i % 2 == 0:
        return 1000.0 + i + (0.1 * f if f < 3 else 33.3 * f)
    if i % 3 == 0:
        return 500.0 + 250.0 * f
    return 100.0 + 33.3 * f


def sequences(n, w, h, nf, seed0=100):
    return [synth.tracker_sequence(w, h, nf, seed=seed0 + i, noise=300) for i in range(n)]


class Oracle:
    """O.TrackerState per slot, driven like the library's slots."""
    def __init__(self, w, h):
        self.w, self.h, self.st = w, h, {}

    def step(self, i, frame, ts, p):
        if i not in self.st:
            self.st[i] = O.TrackerState(self.w, self.h)
        return self.st[i].process(frame, ts, p["threshold"], p["min_area"], p["max_area"], p["distance"])[0]

    def reset(self, i=None):
        for k in ([i] if i is not None else list(self.st)):
            self.st.pop(k, None)


def batch(ctx, frames, ts, params):
    cols = {k: [p[k] for p in params] for k in ("threshold", "min_area", "max_area", "distance")}
    return ctx.tracker_process_batch(frames, ts, **cols)


def run_against_oracle(ctx, seqs, w, h, to_src=lambda b: b, ora=None, slots=None):
    n, nf = len(seqs), len(seqs[0])
    ora = ora or Oracle(w, h)
    slots = slots or list(range(n))
    params = [slot_params(i) for i in slots]
    for f in range(nf):
        frames = np.stack([s[f] for s in seqs])
        ts = [slot_ts(i, f) for i in slots]
        got = batch(ctx, to_src(frames), ts, params)
        assert len(got) == n
        for k, i in enumerate(slots):
            exp = ora.step(i, seqs[k][f], ts[k], params[k])
            assert same(got[k], exp), (f, i, got[k], exp)
            if f == 0:
                assert len(got[k]) == 0                 # a slot's first frame only primes it
    return ora


@pytest.mark.parametrize("n,w,h", [(1, 640, 360), (7, 640, 360), (32, 640, 360), (4, 1280, 720)])
def test_tracker_batch_parity(n, w, h):
    ctx = nv.Context(0, w, h)
    seqs = sequences(n, w, h, 6)
    run_against_oracle(ctx, seqs, w, h)
    single = [nv.Context(0, w, h) for _ in range(min(n, 4))]          # the single call on separate contexts, for a few slots
    ctx.tracker_reset_batch()
    for f in range(6):
        ts = [slot_ts(i, f) for i in range(n)]
        got = batch(ctx, np.stack([s[f] for s in seqs]), ts, [slot_params(i) for i in range(n)])
        for i, s in enumerate(single):
            assert same(got[i], s.tracker_process(seqs[i][f], ts[i], **slot_params(i))), (f, i)
    for s in single:
        s.close()
    ctx.close()


def _pinned(shape):
    ptr = C.c_void_p()
    size = int(np.prod(shape))
    assert nv._lib.nv_host_alloc(size, C.byref(ptr)) == 0
    return np.ctypeslib.as_array((C.c_uint8 * size).from_address(ptr.value)).reshape(shape), ptr


# sources x layouts: packed rows of a width that is a multiple of 4, or pitched rows of a width that is not (scalar path)
@pytest.mark.parametrize("w,pad", [(640, 0), (638, 5)], ids=["packed", "pitched-w638"])
@pytest.mark.parametrize("source", ["pageable", "pinned", "device"])
def test_tracker_batch_sources(source, w, pad):
    import torch
    n, h = 5, 360
    seqs = sequences(n, w, h, 5, 300)
    keep = []

    def to_src(frames):
        if source == "pinned":
            wide, ptr = _pinned((n, h, w + pad, 4))
            keep.append(ptr)
        else:
            wide = np.zeros((n, h, w + pad, 4), np.uint8)
        wide[:, :, :w] = frames
        if source == "device":
            return torch.from_numpy(wide).cuda()[:, :, :w]
        return wide[:, :, :w]

    ctx = nv.Context(0, 1280, 720)
    run_against_oracle(ctx, seqs, w, h, to_src)
    ctx.close()
    for p in keep:
        nv._lib.nv_host_free(p)


def test_tracker_batch_device_odd_spacing():
    """A CUDA tensor whose images are an odd number of bytes apart: image 1's pixels lie at odd addresses (scalar path)."""
    import torch
    n, w, h = 4, 640, 360
    seqs = sequences(n, w, h, 5, 400)
    per = h * w * 4 + 1

    def to_src(frames):
        flat = torch.zeros(n * per, dtype=torch.uint8, device="cuda")
        t = flat.as_strided((n, h, w, 4), (per, w * 4, 4, 1))
        t.copy_(torch.from_numpy(frames).cuda())
        return t

    ctx = nv.Context(0, w, h)
    run_against_oracle(ctx, seqs, w, h, to_src)
    ctx.close()


@pytest.mark.parametrize("fmt", ["I420", "YV12", "NV12", "NV21"])
def test_tracker_batch_yuv(fmt):
    n, w, h, nf = 5, 640, 360, 5
    seqs = sequences(n, w, h, nf, 500)
    bufs = [[synth.to_yuv420(np.ascontiguousarray(f[..., :3]), fmt) for f in s] for s in seqs]
    ctx = nv.Context(0, w, h)
    single = [nv.Context(0, w, h) for _ in range(n)]
    params = [slot_params(i) for i in range(n)]
    cols = {k: [p[k] for p in params] for k in params[0]}
    for f in range(nf):
        ts = [slot_ts(i, f) for i in range(n)]
        got = ctx.tracker_process_batch_yuv(np.stack([b[f] for b in bufs]), fmt, ts, **cols)
        for i in range(n):
            planes = synth.yuv420_planes(bufs[i][f], w, h, fmt)
            exp = single[i].tracker_process_yuv(planes, "I420" if fmt == "YV12" else fmt, ts[i], **params[i])
            assert same(got[i], exp), (f, i)
        assert f == 0 or any(len(g) for g in got)
    for s in single:
        s.close()
    ctx.close()


def test_tracker_batch_slots_reset_grow_shrink_resize():
    w, h = 640, 360
    seqs = sequences(8, w, h, 12, 600)
    ctx = nv.Context(0, 1280, 720)
    ora = Oracle(w, h)
    params = [slot_params(i) for i in range(8)]

    def step(slots, f):
        frames = np.stack([seqs[i][f] for i in slots])
        ts = [slot_ts(i, f) for i in slots]
        got = batch(ctx, frames, ts, [params[i] for i in slots])
        for k, i in enumerate(slots):
            assert same(got[k], ora.step(i, seqs[i][f], ts[k], params[i])), (f, i)
        return got

    step(range(3), 0); step(range(3), 1)
    step(range(6), 2)                         # grows: slots 0..2 continue, 3..5 prime
    step(range(2), 3)                         # shrinks: 2..5 wait
    got = step(range(6), 4)                   # 2..5 resume where they stopped
    assert any(len(g) for g in got[:3])
    ctx.tracker_reset_batch(1); ora.reset(1)
    got = step(range(6), 5)
    assert len(got[1]) == 0                   # slot 1 primes again, the others go on
    step(range(6), 6)
    ctx.tracker_reset_batch(); ora.reset()
    got = step(range(6), 7)
    assert all(len(g) == 0 for g in got)
    step(range(6), 8)
    # another frame size starts every slot afresh
    small = sequences(6, 320, 240, 2, 700)
    got = ctx.tracker_process_batch(np.stack([s[0] for s in small]), [1.0] * 6)
    assert all(len(g) == 0 for g in got)
    ora.reset()
    step(range(6), 9)
    got = step(range(6), 10)
    assert any(len(g) for g in got)
    ctx.close()


def test_tracker_batch_isolation(cascade_dir):
    """Single-tracker calls interleaved on the same context and a pending face batch are left as they are."""
    w, h = 640, 360
    seqs = sequences(3, w, h, 6, 800)
    single_seq = synth.tracker_sequence(w, h, 6, seed=900, noise=300)
    ctx = nv.Context(0, 1280, 720)
    ora, ora_single = Oracle(w, h), O.TrackerState(w, h)
    casc = nv.Cascade(os.path.join(cascade_dir, "haarcascade_frontalface_alt.xml"))
    faces = np.stack([synth.frame(640, 480, 1 + i, 1000 + i) for i in range(4)])
    ref = nv.Context(0, 640, 480).face_detect_batch(casc, faces)
    for f in range(6):
        a = ctx.tracker_process(single_seq[f], 40.0 * f + 7)
        assert same(a, ora_single.process(single_seq[f], 40.0 * f + 7)[0]), f
        if f == 3:
            ctx.face_submit_batch(casc, faces)
        ts = [slot_ts(i, f) for i in range(3)]
        got = batch(ctx, np.stack([s[f] for s in seqs]), ts, [slot_params(i) for i in range(3)])
        for i in range(3):
            assert same(got[i], ora.step(i, seqs[i][f], ts[i], slot_params(i))), (f, i)
        if f == 3:
            got_faces = ctx.face_collect_batch()
            assert len(got_faces) == 4 and all(same(a, b) for a, b in zip(got_faces, ref))
    ctx.tracker_reset()                        # the single tracker's reset leaves the slots alone
    ctx.close()


def _call(ctx, frames, ts, params, cap):
    n, h, w = frames.shape[:3]
    ptrs = (C.c_void_p * n)(*[frames[i].ctypes.data for i in range(n)])
    tsa = (C.c_double * n)(*ts)
    pa = (nv.TrackerParams * n)(*[nv.TrackerParams(p["threshold"], p["min_area"], p["max_area"], p["distance"]) for p in params])
    out = (nv.Rect * max(cap, 1))()
    counts = (C.c_int * n)()
    total = C.c_int(-1)
    rc = nv._lib.nv_tracker_process_batch(ctx.handle, ptrs, n, w, h, frames.strides[1], 0, tsa, pa, out, cap, counts, C.byref(total))
    return rc, nv._rects(out, total.value), list(counts), total.value


def test_tracker_batch_capacity():
    w, h, n = 640, 360, 3
    seqs = sequences(n, w, h, 3, 1100)
    ctx = nv.Context(0, w, h)
    ora = Oracle(w, h)
    params = [dict(threshold=20, min_area=0, max_area=1 << 30, distance=0)] * n      # every component stays
    for f in range(3):
        frames = np.stack([s[f] for s in seqs])
        ts = [33.3 * (f + 1)] * n
        exp = [ora.step(i, seqs[i][f], ts[i], params[i]) for i in range(n)]
        rc, got, counts, total = _call(ctx, frames, ts, params, 5)
        assert counts == [len(e) for e in exp]
        flat = np.concatenate([np.asarray(e, np.int32).reshape(-1, 4) for e in exp])
        assert total == min(5, len(flat)) and same(got, flat[:5])
        assert rc == (NV_ERR_CAPACITY if len(flat) > 5 else 0)
    ctx.close()


def _speckle(w, h, period, seed):
    """Two frames whose difference is a lattice of isolated single pixels (one component each)."""
    rng = np.random.default_rng(seed)
    a = np.full((h, w, 4), 100, np.uint8)
    b = a.copy()
    mask = np.zeros((h, w), bool)
    mask[::period, ::period] = True
    if period == 1:                            # one-pixel checkerboard
        mask = (np.add.outer(np.arange(h), np.arange(w)) % 2) == 0
    b[mask] = 200
    b[..., 3] = rng.integers(0, 256, (h, w))   # alpha is ignored
    return a, b


def test_tracker_batch_many_components():
    """More than 1024 components in one image (the rest read from the device), and a one-pixel checkerboard of motion at
    720p (more than 16384 raw components): the single call's truncated result and NV_ERR_CAPACITY naming that image."""
    w, h = 1280, 720
    params = [dict(threshold=20, min_area=0, max_area=1 << 30, distance=0), dict(threshold=20, min_area=50, max_area=30000, distance=35)]
    a0, b0 = _speckle(w, h, 20, 1)             # 64 x 36 = 2304 isolated pixels
    a1, b1 = _speckle(w, h, 1, 2)              # 460 800 isolated pixels
    ctx = nv.Context(0, w, h)
    singles = [nv.Context(0, w, h) for _ in range(2)]
    rc, _, _, _ = _call(ctx, np.stack([a0, a1]), [10.0, 10.0], params, 1 << 20)
    assert rc == 0
    rc, got, counts, total = _call(ctx, np.stack([b0, b1]), [43.0, 43.0], params, 1 << 20)
    assert rc == NV_ERR_CAPACITY and b"image 1" in nv._lib.nv_last_error()
    exp = []
    for i, (a, b) in enumerate([(a0, b0), (a1, b1)]):
        singles[i].tracker_process(a, 10.0, **params[i])
        try:
            exp.append(singles[i].tracker_process(b, 43.0, **params[i]))
        except nv.NuboError as e:
            assert i == 1 and e.code == NV_ERR_CAPACITY
            exp.append(np.zeros((0, 4), np.int32))      # min_area 50 drops every one-pixel component
    assert counts == [2304, 0] and same(got, np.concatenate(exp))
    st = O.TrackerState(w, h)
    st.process(a0, 10.0, **params[0])
    assert same(exp[0], st.process(b0, 43.0, **params[0])[0])
    for s in singles:
        s.close()
    ctx.close()


def test_tracker_batch_timestamp_capacity():
    """256 distinct timestamps inside 0.2 ms in slot 1: refused naming slot 1, and no slot changes."""
    w, h = 320, 240
    seqs = sequences(2, w, h, 260, 1200)
    ctx = nv.Context(0, w, h)
    ora = Oracle(w, h)
    p = [dict(threshold=20, min_area=50, max_area=30000, distance=35)] * 2
    for f in range(256):                       # slot 1: 255 distinct timestamps after its priming frame, inside 0.2 ms
        ts = [1000.0 + 40.0 * f, 2000.0 + f * 0.0005]
        got = batch(ctx, np.stack([seqs[0][f], seqs[1][f]]), ts, p)
        for i in range(2):
            assert same(got[i], ora.step(i, seqs[i][f], ts[i], p[i])), (f, i)
    with pytest.raises(nv.NuboError) as e:
        batch(ctx, np.stack([seqs[0][256], seqs[1][256]]), [1000.0 + 40.0 * 256, 2000.0 + 256 * 0.0005], p)
    assert e.value.code == NV_ERR_CAPACITY and "slot 1" in str(e.value)
    # slot 0 continues as if the refused call had not happened; slot 1 has no free index until it is reset, as with
    # nv_tracker_process
    f = 257
    got = batch(ctx, seqs[0][f][None], [1000.0 + 40.0 * f], p[:1])
    assert same(got[0], ora.step(0, seqs[0][f], 1000.0 + 40.0 * f, p[0]))
    ctx.tracker_reset_batch(1); ora.reset(1)
    f = 258
    ts = [1000.0 + 40.0 * f, 2001.0]
    got = batch(ctx, np.stack([seqs[0][f], seqs[1][f]]), ts, p)
    for i in range(2):
        assert same(got[i], ora.step(i, seqs[i][f], ts[i], p[i])), i
    assert len(got[1]) == 0
    ctx.close()


def _launches(ctx):
    """nv_debug_get_counters [3]: the kernel launches this context has issued."""
    o = (C.c_longlong * 8)()
    assert nv._lib.nv_debug_get_counters(ctx.handle, o) == 0
    return o[3]


def test_tracker_batch_one_launch_and_profiling():
    """One kernel launch per call, whatever N (the context's launch counter), and it is the batched k_trk_fused
    (torch.profiler: no single-frame instantiation runs).  With profiling on, nv_ctx_get_tracker_kernel_ms reports the
    batched kernel of every call.  torch.profiler names the kernels that ran; it is not used to count them, since in a
    process that has run many profiler sessions it has been seen to miss a kernel record."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    w, h = 640, 360
    seqs = sequences(32, w, h, 4, 1300)
    ctx = nv.Context(0, w, h)
    ctx.set_profile(True)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for f, n in enumerate((8, 32, 1, 32)):
            before = _launches(ctx)
            ctx.tracker_process_batch(np.stack([s[f] for s in seqs[:n]]), [33.3 * (f + 1)] * n)
            assert _launches(ctx) == before + 1, (f, n)
            assert ctx.tracker_kernel_ms() > 0
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "k_trk_fused" in e.name}
    assert names == {"void k_trk_fused<0, true>(TrkParams)"}, names
    ctx.close()


def test_tracker_batch_refusals():
    w, h = 640, 360
    ctx = nv.Context(0, w, h)
    L = nv._lib
    n = 2
    frames = np.zeros((n, h, w, 4), np.uint8)
    ptrs = (C.c_void_p * (nv.BATCH_MAX + 1))(*([frames.ctypes.data] * (nv.BATCH_MAX + 1)))
    ts = (C.c_double * (nv.BATCH_MAX + 1))()
    pa = (nv.TrackerParams * (nv.BATCH_MAX + 1))(*[nv.TrackerParams(20, 50, 30000, 35)] * (nv.BATCH_MAX + 1))
    out = (nv.Rect * 16)()
    counts = (C.c_int * (nv.BATCH_MAX + 1))()
    stride = w * 4
    for bad_n in (0, -1, nv.BATCH_MAX + 1):
        assert L.nv_tracker_process_batch(ctx.handle, ptrs, bad_n, w, h, stride, 0, ts, pa, out, 16, counts, None) == NV_ERR_ARG
    assert L.nv_tracker_process_batch(ctx.handle, None, n, w, h, stride, 0, ts, pa, out, 16, counts, None) == NV_ERR_ARG
    assert L.nv_tracker_process_batch(ctx.handle, ptrs, n, w, h, stride, 0, None, pa, out, 16, counts, None) == NV_ERR_ARG
    assert L.nv_tracker_process_batch(ctx.handle, ptrs, n, w, h, stride, 0, ts, None, out, 16, counts, None) == NV_ERR_ARG
    assert L.nv_tracker_process_batch(ctx.handle, ptrs, n, w, h, stride, 0, ts, pa, out, 16, None, None) == NV_ERR_ARG
    assert L.nv_tracker_process_batch(ctx.handle, ptrs, n, w, h, stride, 0, ts, pa, None, 16, counts, None) == NV_ERR_ARG
    assert L.nv_tracker_process_batch(ctx.handle, ptrs, n, w, h, stride + 2, 0, ts, pa, out, 16, counts, None) == NV_ERR_ARG
    assert L.nv_tracker_process_batch(ctx.handle, ptrs, n, w, h, w * 3, 0, ts, pa, out, 16, counts, None) == NV_ERR_ARG
    nullrow = (C.c_void_p * 2)(frames.ctypes.data, None)
    assert L.nv_tracker_process_batch(ctx.handle, nullrow, n, w, h, stride, 0, ts, pa, out, 16, counts, None) == NV_ERR_ARG
    assert b"image 1" in L.nv_last_error()
    # a frame larger than the context: refused as by nv_tracker_process
    big = L.nv_tracker_process_batch(ctx.handle, ptrs, n, 1280, 720, 1280 * 4, 0, ts, pa, out, 16, counts, None)
    assert big == L.nv_tracker_process(ctx.handle, ptrs[0], 1280, 720, 1280 * 4, 1.0, pa, out, 16, counts) != 0
    # 4:2:0 frames that differ from frame 0
    buf = np.zeros((n, h * 3 // 2, w), np.uint8)
    table, _, _ = nv._batch_yuv_frames(buf, "NV12")
    table[1].stride[0] = w + 2
    assert L.nv_tracker_process_batch_yuv(ctx.handle, table, n, ts, pa, out, 16, counts, None) == NV_ERR_ARG
    assert b"image 1" in L.nv_last_error()
    table[1].stride[0] = w
    table[1].format = nv.FMT_I420
    assert L.nv_tracker_process_batch_yuv(ctx.handle, table, n, ts, pa, out, 16, counts, None) == NV_ERR_ARG
    table[1].format = nv.FMT_NV12
    table[0].width = w + 1; table[1].width = w + 1
    assert L.nv_tracker_process_batch_yuv(ctx.handle, table, n, ts, pa, out, 16, counts, None) == NV_ERR_ARG
    assert L.nv_tracker_reset_batch(ctx.handle, nv.BATCH_MAX) == NV_ERR_ARG
    assert L.nv_tracker_reset_batch(ctx.handle, 5) == 0          # a slot that does not exist yet
    # nothing above touched the slots: the next call primes them
    got = ctx.tracker_process_batch(frames, [1.0, 1.0])
    assert all(len(g) == 0 for g in got)
    ctx.close()
