"""Randomised parity run (not part of the test suite): random frame sizes, strides, processing widths, scale factors,
minNeighbors and input formats through a few long-lived contexts (plan cache, graph replay, format switches) against the
CPU oracle, for a wall-clock budget.  --scores: every context runs with detection scores on, and each call's neighbour
counts and level weights are checked too.  Usage: python tools/fuzz_parity.py [seconds] [seed] [--scores]"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "nubomedia-vca_b200", "python"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import nubovca as nv  # noqa: E402
import oracle as O  # noqa: E402
import scores_ref as S  # noqa: E402
from nubovca import synth  # noqa: E402

scores = "--scores" in sys.argv
args = [a for a in sys.argv[1:] if a != "--scores"]
budget = float(args[0]) if len(args) > 0 else 120.0
seed = int(args[1]) if len(args) > 1 else 0
rng = np.random.default_rng(seed)
xml = os.path.join(ROOT, "nubomedia-vca_b200", "cascades", "haarcascade_frontalface_alt.xml")
ncasc, ocasc = nv.Cascade(xml), O.Cascade(xml)
ctxs = [nv.Context(0, 1920, 1080, debug=False) for _ in range(3)] + [nv.Context(0, 1920, 1080, debug=True)]
for c in ctxs:
    c.set_scores(scores)
t0 = time.time()
n = bad = 0
shapes = []
while time.time() - t0 < budget:
    if shapes and rng.random() < 0.5:
        W, H, w2p, sf, mn = shapes[int(rng.integers(len(shapes)))]          # revisit a shape: plan cache + graph replay
    else:
        W = int(rng.integers(24, 700)) * 2; H = int(rng.integers(24, 400)) * 2
        w2p = int(rng.choice([W, max(1, W // 2), max(1, W // 3), 160, 320, int(rng.integers(40, W + 1))]))
        sf = float(rng.choice([1.1, 1.2, 1.25, 1.5])); mn = int(rng.choice([0, 2, 3]))
        shapes = (shapes + [(W, H, w2p, sf, mn)])[-6:]
    fr = synth.frame(W, H, int(rng.integers(0, 4)), int(rng.integers(1 << 30)), smin=min(0.2, 0.5 * W / H), smax=min(0.7, 0.9 * W / H))
    fmt = str(rng.choice(["BGR", "BGR", "I420", "NV12", "NV21", "YV12"]))
    pad = int(rng.choice([0, 0, 1, 2, 4, 16]))
    c = ctxs[int(rng.integers(len(ctxs)))]
    ms = None if rng.random() < 0.7 else (int(rng.integers(0, 40)), int(rng.integers(0, 40)))
    if fmt == "BGR":
        buf = rng.integers(0, 256, (H, 3 * W + pad), dtype=np.uint8)
        buf[:, :3 * W] = fr.reshape(H, -1)
        view = np.lib.stride_tricks.as_strided(buf, (H, W, 3), (buf.strides[0], 3, 1))
        exp, eq = O.face_process(fr, ocasc, w2p, sf, mn, ms)
        got = c.face_detect(ncasc, view, w2p, sf, mn, ms) if pad == 0 else None
        if got is None:
            import ctypes as C
            k = C.c_int(0)
            a = nv.Context._face_params(w2p, sf, mn, ms)
            rc = nv._lib.nv_face_detect(c.handle, ncasc.handle, buf.ctypes.data_as(C.c_void_p), W, H, buf.strides[0], C.byref(a),
                                        c._out, c._cap, C.byref(k))
            assert rc == 0, nv._lib.nv_last_error()
            got = nv._rects(c._out, k.value)
    else:
        y = synth.to_yuv420(fr, fmt)
        planes = synth.yuv420_planes(y, W, H, fmt)
        if pad:
            planes = tuple(np.ascontiguousarray(np.pad(p, ((0, 0), (0, pad))))[:, :p.shape[1]] for p in planes)
        exp, eq = O.face_process(O.yuv420_to_bgr(*O.yuv420_planes(y, W, H, fmt), fmt=fmt), ocasc, w2p, sf, mn, ms)
        got = c.face_detect_yuv(ncasc, planes, fmt, w2p, sf, mn, ms)
    ok = got.shape == exp.shape and (got == exp).all()
    if c is ctxs[-1]:
        ok = ok and (c.gray() == eq).all()
    if scores:
        rows, cols = eq.shape
        _, enb, ewt = S.detect_multiscale_scores(eq, ocasc, sf, mn, (cols // 20, rows // 20) if ms is None else ms)
        nb, wt = c.scores()
        ok = ok and nb.shape == enb.shape and (nb == enb).all() and (wt == ewt).all()
    n += 1
    if not ok:
        bad += 1
        print("MISMATCH", W, H, w2p, sf, mn, ms, fmt, pad, got.tolist()[:4], exp.tolist()[:4], flush=True)
print(f"fuzz: {n} cases, {bad} mismatches, seed {seed}, {time.time() - t0:.0f} s")
sys.exit(1 if bad else 0)
