"""Detection scores on the GPU (nv_ctx_set_scores / nv_get_scores): per output rectangle, cv2 detectMultiScale2's
numDetections and detectMultiScale3(outputRejectLevels=True)'s levelWeights.  Bit-exact against the CPU oracle on every
route of the pipeline, and the rectangles identical to the same call with scores off."""
import os
import subprocess
import sys

import numpy as np
import pytest

import nubovca as nv
import oracle as O
import scores_ref as S
from cascade_xml_util import random_int_cascade, write_cascade
from nubovca import synth

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FACE_XML = "haarcascade_frontalface_alt.xml"


@pytest.fixture(scope="module")
def ctx():
    c = nv.Context(0, 1920, 1080)
    yield c
    c.close()


@pytest.fixture(scope="module")
def face(cascade_dir):
    p = os.path.join(cascade_dir, FACE_XML)
    return nv.Cascade(p), O.Cascade(p)


def check_detect(ctx, ncasc, ocasc, gray, sf, mn, ms=(0, 0)):
    """detect_multiscale with scores on: rectangles as with scores off, counts and weights as the oracle's."""
    off = ctx.detect_multiscale(ncasc, gray, sf, mn, ms)
    r, nb, wt = ctx._with_scores(lambda: ctx.detect_multiscale(ncasc, gray, sf, mn, ms))
    er, enb, ewt = S.detect_multiscale_scores(gray, ocasc, sf, mn, ms)
    assert r.shape == er.shape and (r == er).all() and (r == off).all(), (mn, len(r), len(er))
    assert (nb == enb).all(), mn
    assert (wt == ewt).all(), (mn, np.abs(wt - ewt).max() if len(wt) else 0)
    return r, nb, wt


def models(cascade_dir, name):
    p = os.path.join(cascade_dir, name)
    return nv.Cascade(p), O.Cascade(p)


def test_small_plans(ctx, face, cascade_dir):
    """Config 1 through the face pipeline and a 96x64 ROI: k_group_fused."""
    ncasc, ocasc = face
    fr = synth.frame(640, 480, 4, 1)
    r, nb, wt = ctx.face_detect(ncasc, fr, 160, 1.25, 3, None, scores=True)
    exp, eq = O.face_process(fr, ocasc, 160, 1.25, 3, None)
    er, enb, ewt = S.detect_multiscale_scores(eq, ocasc, 1.25, 3, (eq.shape[1] // 20, eq.shape[0] // 20))
    assert (r == exp).all() and (r == er).all() and len(r) >= 1
    assert (nb == enb).all() and (wt == ewt).all()
    roi = synth.frame(96, 64, 1, 5, smin=0.5, smax=0.9)[..., 0]
    for mn in (0, 2):
        check_detect(ctx, ncasc, ocasc, roi, 1.1, mn, (20, 20))
    r, nb, wt = check_detect(ctx, ncasc, ocasc, O.equalize_hist(O.bgr2gray(fr)), 1.1, 3, (24, 24))
    assert len(r) >= 1 and (nb > 3).all() and (wt > 105.76).all()       # alt's last stage threshold is 105.76


def test_large_fast_plan_cfg3(ctx, face):
    """Config 3 at 1920x1080 (40 levels): stage 0 on tiles, bulk bank-class kernels, fast tail, k_cand_sort + k_group."""
    ncasc, ocasc = face
    fr = synth.frame(1920, 1080, 6, 3)
    exp, eq = O.face_process(fr, ocasc, 1920, 1.1, 3, (24, 24))
    for mn in (3, 0):
        r, nb, wt = ctx.face_detect(ncasc, fr, 1920, 1.1, mn, (24, 24), scores=True)
        er, enb, ewt = S.detect_multiscale_scores(eq, ocasc, 1.1, mn, (24, 24))
        assert r.shape == er.shape and (r == er).all() and (nb == enb).all() and (wt == ewt).all(), mn
    assert ctx.counters()["windows"] > 16384


def test_bulk_kernels_end_the_cascade(ctx, tmp_path):
    """A short exact-integer stump model over a large plan: the bulk kernels run the last stage themselves (final_stage) and
    keep no stage sums, so the weight is evaluated again in the sort."""
    p = str(tmp_path / "short.xml")
    random_int_cascade(p, np.random.default_rng(5), nstages=3, max_trees=12)
    ncasc, ocasc = nv.Cascade(p), O.Cascade(p)
    g = O.equalize_hist(O.bgr2gray(synth.frame(1280, 720, 4, 2)))
    n = sum(len(check_detect(ctx, ncasc, ocasc, g, 1.2, mn)[0]) for mn in (0, 3))
    assert n > 0 and ctx.counters()["windows"] > 16384


def uncertified_cascade(path, rng):
    """Random stumps whose last stage adds 3e9 and later -3e9 around small leaves: its double sum depends on the order
    of the additions (no order-free certificate), so only a sum in XML order gives the reference's weight."""
    feats = [[(int(rng.integers(0, 10)), int(rng.integers(0, 10)), int(rng.integers(2, 10)), int(rng.integers(2, 10)),
               float(np.float32(rng.uniform(-2, 2)))) for _ in range(2)] for _ in range(8)]

    def stump():
        return (int(rng.integers(0, 8)), float(np.float32(rng.normal(0, 0.05))), float(np.float32(rng.uniform(-1, 1))),
                float(np.float32(rng.uniform(-1, 1))))
    stages = [(-0.7, [stump() for _ in range(3)]), (-0.7, [stump() for _ in range(3)]),
              (-100.0, [(0, 0.0, 3e9, 3e9), stump(), stump(), (1, 0.0, -3e9, -3e9), stump(), stump()])]
    write_cascade(path, 20, 20, stages, feats)


def test_uncertified_stump_models(ctx, cascade_dir, tmp_path):
    """A stump model without the order-free certificate, small and large plans; frontalface_default (24x24 window)."""
    p = str(tmp_path / "uncert.xml")
    uncertified_cascade(p, np.random.default_rng(7))
    nr, orc = nv.Cascade(p), O.Cascade(p)
    assert nr.info.order_free_sums == 0
    n = 0
    for W, H in ((160, 120), (320, 240)):
        g = O.equalize_hist(O.bgr2gray(synth.frame(W, H, 2, 13)))
        for mn in (0, 1):
            r, nb, wt = check_detect(ctx, nr, orc, g, 1.2, mn)
            n += len(r)
    assert n > 0
    nd, od = models(cascade_dir, "haarcascade_frontalface_default.xml")
    g = O.equalize_hist(O.bgr2gray(synth.frame(480, 360, 3, 21)))
    for mn in (0, 2):
        check_detect(ctx, nd, od, g, 1.1, mn)


@pytest.mark.parametrize("name", ["haarcascade_lefteye_2splits.xml", "haarcascade_eye_tree_eyeglasses.xml",
                                  "haarcascade_smile.xml", "haarcascade_profileface.xml"])
def test_general_cascades_small_and_large(ctx, cascade_dir, name):
    """Trees and tilted features: warp-per-window kernels on small plans, staged compaction on large ones."""
    ncasc, ocasc = models(cascade_dir, name)
    n = 0
    for W, H in ((400, 300), (1280, 720)):
        g = O.equalize_hist(O.bgr2gray(synth.frame(W, H, 2, 3, smin=0.5, smax=0.9)))
        for mn in (0, 2):
            n += len(check_detect(ctx, ncasc, ocasc, g, 1.1, mn)[0])
    assert n > 0


@pytest.mark.parametrize("idx", range(3))
def test_lbp_small_and_large(ctx, idx):
    p = os.path.join(HERE, "golden", f"lbp_random_{idx}.xml")
    ncasc, ocasc = nv.Cascade(p), O.Cascade(p)
    for W, H in ((320, 240), (1280, 720)):
        g = O.equalize_hist(O.bgr2gray(synth.frame(W, H, 3, 41 + idx)))
        for mn in (0, 2):
            check_detect(ctx, ncasc, ocasc, g, 1.1, mn)


def test_union_find_tail_and_overflow(cascade_dir):
    """smile at 1080p on a fresh context: the first call overflows the initial candidate capacity and is re-run by collect
    (scores included); more than 2048 raw candidates group by union-find; with min_neighbors 0 more than 1024 rectangles
    come back, so the scores beyond the inline part of the result block are copied too."""
    ncasc, ocasc = models(cascade_dir, "haarcascade_smile.xml")
    g = O.equalize_hist(O.bgr2gray(synth.frame(1920, 1080, 6, 3)))
    c = nv.Context(0, 1920, 1080)
    try:
        c.set_scores(True)
        r = c.detect_multiscale(ncasc, g, 1.1, 0)
        nb, wt = c.scores()
        er, enb, ewt = S.detect_multiscale_scores(g, ocasc, 1.1, 0)
        assert c.counters()["candidates"] > 8192 and len(r) > 1024
        assert r.shape == er.shape and (r == er).all() and (nb == 1).all() and (wt == ewt).all()
        r, nb, wt = check_detect(c, ncasc, ocasc, g, 1.1, 3)
        assert c.counters()["candidates"] > 2048 and len(r) > 0
    finally:
        c.close()


def test_face_pipeline_formats_and_contexts(face):
    """BGR, 4:2:0 and device frames through submit / collect on several contexts at once."""
    torch = pytest.importorskip("torch")
    ncasc, ocasc = face
    ctxs = [nv.Context(0, 1280, 720) for _ in range(3)]
    try:
        for c in ctxs:
            c.set_scores(True)
        frames = [synth.frame(1280, 720, 3, 40 + i) for i in range(3)]
        for rep in range(2):
            y = synth.to_yuv420(frames[1], "NV12")
            d = torch.from_numpy(frames[2]).cuda()
            ctxs[0].face_submit(ncasc, frames[0], 640, 1.25, 3, None)
            ctxs[1].face_submit_yuv(ncasc, synth.yuv420_planes(y, 1280, 720, "NV12"), "NV12", 640, 1.25, 3, None)
            ctxs[2].face_submit_device(ncasc, d.data_ptr(), 1280, 720, 1280 * 3, 640, 1.25, 3, None)
            bgrs = [frames[0], O.yuv420_to_bgr(*O.yuv420_planes(y, 1280, 720, "NV12"), fmt="NV12"), frames[2]]
            for c, bgr in zip(ctxs, bgrs):
                r, nb, wt = c.face_collect(scores=True)
                exp, eq = O.face_process(bgr, ocasc, 640, 1.25, 3, None)
                er, enb, ewt = S.detect_multiscale_scores(eq, ocasc, 1.25, 3, (eq.shape[1] // 20, eq.shape[0] // 20))
                assert (r == exp).all() and (r == er).all() and (nb == enb).all() and (wt == ewt).all(), rep
            torch.cuda.synchronize()
    finally:
        for c in ctxs:
            c.close()


def test_alternating_scores_on_one_context(face):
    """Same shapes, scores on and off in turn: each call replays the graph of its own setting (never the other's)."""
    ncasc, ocasc = face
    c = nv.Context(0, 640, 480)
    try:
        fr = synth.frame(640, 480, 4, 1)
        exp, eq = O.face_process(fr, ocasc, 160, 1.25, 3, None)
        er, enb, ewt = S.detect_multiscale_scores(eq, ocasc, 1.25, 3, (eq.shape[1] // 20, eq.shape[0] // 20))
        gray = O.equalize_hist(O.bgr2gray(fr))
        dr, dnb, dwt = S.detect_multiscale_scores(gray, ocasc, 1.1, 2, (24, 24))
        for i in range(8):
            on = i % 2 == 0
            c.set_scores(on)
            assert (c.face_detect(ncasc, fr, 160, 1.25, 3, None) == exp).all()
            if on:
                nb, wt = c.scores()
                assert (nb == enb).all() and (wt == ewt).all(), i
            else:
                with pytest.raises(nv.NuboError):
                    c.scores()
            assert (c.detect_multiscale(ncasc, gray, 1.1, 2, (24, 24)) == dr).all()
            if on:
                nb, wt = c.scores()
                assert (nb == dnb).all() and (wt == dwt).all(), i
        # a rectangle-only consumer sees nothing new: elements keep their contexts at scores off
        c.set_scores(False)
        assert (c.face_detect(ncasc, fr, 160, 1.25, 3, None) == exp).all()
    finally:
        c.close()


def test_detect_multiscale2_and_3_shapes(ctx, face):
    ncasc, ocasc = face
    g = O.equalize_hist(O.bgr2gray(synth.frame(640, 480, 4, 1)))
    r2, nd = ctx.detect_multiscale2(ncasc, g, 1.1, 3, (24, 24))
    r3, rl, lw = ctx.detect_multiscale3(ncasc, g, 1.1, 3, (24, 24))
    er, enb, ewt = S.detect_multiscale_scores(g, ocasc, 1.1, 3, (24, 24))
    assert (r2 == er).all() and (r3 == er).all() and (nd == enb).all() and (lw == ewt).all()
    assert (rl == ncasc.info.nstages).all() and rl.dtype == np.int32 and lw.dtype == np.float64
    assert (ctx.detect_multiscale(ncasc, g, 1.1, 3, (24, 24)) == er).all()       # the context's own setting is back to off
    with pytest.raises(nv.NuboError):
        ctx.scores()


def test_short_randomised_scores_run():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_parity.py"), "15", "11", "--scores"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "0 mismatches" in r.stdout
