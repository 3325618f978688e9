"""GPU parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the same
seeded inputs and against the committed cv2 golden fixtures.  Bit-exact everywhere: gray/equalised
images, every level's integral and squared integral, every level's stage-exit depth map, raw
candidates (canonical order) and grouped rectangles.  The north-star tolerance (disagreement only for
windows whose stage sum is within 1e-5 relative of a threshold) is therefore never used."""
import json
import os

import numpy as np
import pytest

import nubovca as nv
import oracle as O
from cascade_xml_util import random_cascade, random_general_model, random_int_cascade, random_lbp_cascade, write_old_format
from nubovca import synth

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
FACE_XML = "haarcascade_frontalface_alt.xml"


@pytest.fixture(scope="module")
def ctx():
    c = nv.Context(0, 1920, 1080, debug=True)
    yield c
    c.close()


@pytest.fixture(scope="module")
def face(cascade_dir):
    p = os.path.join(cascade_dir, FACE_XML)
    return nv.Cascade(p), O.Cascade(p)


def rects_equal(a, b):
    a = np.asarray(a, np.int32).reshape(-1, 4); b = np.asarray(b, np.int32).reshape(-1, 4)
    return a.shape == b.shape and bool((a == b).all())


def check_levels(ctx, eq, ocasc, sf, ms):
    """integrals, depth maps and candidates of the last detect call vs the oracle; returns #windows checked."""
    levels = O.eval_pyramid(eq, ocasc, sf, ms, keep_integrals=True)
    got = ctx.levels()
    assert len(got) == len(levels)
    nwin = 0
    cands = []
    for i, (g, o) in enumerate(zip(got, levels)):
        assert (g["lw"], g["lh"], g["ystep"]) == (o["lw"], o["lh"], o["ystep"]), i
        assert g["scale"] == np.float32(o["scale"])
        assert (g["ny"], g["nx"]) == o["depth"].shape, i
        s, q = ctx.integral(i)
        assert (s == o["sum"]).all(), f"level {i} integral"
        assert (q == o["sqsum"]).all(), f"level {i} squared integral"
        if ocasc.has_tilted:
            assert (ctx.tilted(i) == o["tilted"]).all(), f"level {i} tilted integral"
        d = ctx.depth_map(i)
        bad = np.argwhere(d != o["depth"])
        assert len(bad) == 0, f"level {i}: {len(bad)} depth mismatches, first {bad[:3]} gpu {d[tuple(bad[0])]} ora {o['depth'][tuple(bad[0])]}"
        nwin += d.size
        cands.append(o["cand"])
    cand = np.concatenate(cands) if cands else np.zeros((0, 4), np.int32)
    assert rects_equal(ctx.candidates(), cand)
    return nwin, levels


# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("idx", range(6))
def test_face_golden_cases(ctx, face, idx):
    """cfg1 / cfg5 / cfg2-face-stage / cfg3-parameter cases of tests/golden (cv2 4.13 outputs)."""
    c = json.load(open(os.path.join(HERE, "golden", "face_golden.json")))["cases"][idx]
    ncasc, ocasc = face
    fr = synth.frame(c["W"], c["H"], c["k"], c["seed"])
    ms = tuple(c["min_size"])
    got = ctx.face_detect(ncasc, fr, c["width_to_process"], c["scale_factor"], c["min_neighbors"], ms)
    assert rects_equal(got, c["grouped"])
    exp, eq = O.face_process(fr, ocasc, c["width_to_process"], c["scale_factor"], c["min_neighbors"], ms)
    assert rects_equal(got, exp)
    assert (ctx.gray() == eq).all()
    nwin, _ = check_levels(ctx, eq, ocasc, c["scale_factor"], ms)
    assert nwin > 1000
    raw = ctx.face_detect(ncasc, fr, c["width_to_process"], c["scale_factor"], 0, ms)
    assert rects_equal(raw, c["raw"])


@pytest.mark.parametrize("idx", range(2))
def test_cfg3_full_size_golden(face, idx):
    """BASELINE config 3 at FULL size (the bench.py frames of rank 0) against the committed cv2 output: raw candidates and
    grouped rectangles of 3.66 M windows."""
    c = json.load(open(os.path.join(HERE, "golden", "cfg3_golden.json")))["cases"][idx]
    ncasc, _ = face
    fr = synth.frame(c["W"], c["H"], c["k"], c["seed"])
    big = nv.Context(0, 1920, 1080)
    try:
        ms = tuple(c["min_size"])
        assert rects_equal(big.face_detect(ncasc, fr, c["width_to_process"], c["scale_factor"], c["min_neighbors"], ms), c["grouped"])
        assert rects_equal(big.face_detect(ncasc, fr, c["width_to_process"], c["scale_factor"], 0, ms), c["raw"])
        assert big.counters()["windows"] > 3_000_000
    finally:
        big.close()


def test_grouping_with_thousands_of_candidates(cascade_dir):
    """A permissive model over a large image leaves thousands of raw candidates: groupRectangles then builds its classes by
    neighbour search + union-find (uf_link, kernels_group.cu) instead of the similarity bit-matrix; same classes, same order."""
    nc = nv.Cascade(os.path.join(cascade_dir, "haarcascade_smile.xml"))
    oc = O.Cascade(os.path.join(cascade_dir, "haarcascade_smile.xml"))
    g = O.equalize_hist(O.bgr2gray(synth.frame(1280, 720, 4, 9, smin=0.2, smax=0.5)))
    big = nv.Context(0, 1280, 720)
    try:
        for mn in (3, 1):
            got = big.detect_multiscale(nc, g, 1.1, mn)
            assert big.counters()["candidates"] > 2048
            assert rects_equal(got, O.detect_multiscale(g, oc, 1.1, mn)), mn
    finally:
        big.close()


def test_face_element_min_size_rule(ctx, face):
    # min_size=None -> Size(cols/20, rows/20), kmsfacedetect.cpp:811
    ncasc, ocasc = face
    fr = synth.frame(640, 480, 4, 1)
    got = ctx.face_detect(ncasc, fr, 160, 1.25, 3, None)
    exp, _ = O.face_process(fr, ocasc, 160, 1.25, 3, None)
    assert rects_equal(got, exp) and len(got) >= 1


def test_depth_maps_reach_every_stage(ctx, face):
    """The procedurally composited patches drive windows through all 22 stages (SURVEY.md §8d)."""
    ncasc, ocasc = face
    fr = synth.frame(480, 360, 10, 5)
    ctx.face_detect(ncasc, fr, 480, 1.1, 3, (0, 0))
    _, eq = O.face_process(fr, ocasc, 480, 1.1, 3, (0, 0))
    nwin, levels = check_levels(ctx, eq, ocasc, 1.1, (0, 0))
    codes = np.concatenate([l["depth"].ravel() for l in levels])
    for st in range(1, 22):
        assert (codes == -st).any(), f"no window exits at stage {st}"
    assert (codes == 0).any() and (codes == 1).any() and (codes == O.DEPTH_SKIPPED).any() and (codes == O.DEPTH_VARREJ).any()
    assert ctx.counters()["windows"] == nwin


@pytest.mark.parametrize("name,sf,ms", [("haarcascade_profileface.xml", 1.25, (3, 3)),
                                        ("haarcascade_eye.xml", 1.1, (20, 20)),
                                        ("haarcascade_frontalface_default.xml", 1.2, (0, 0))])
def test_other_cascades(ctx, cascade_dir, name, sf, ms):
    """profileface = the ear element's face stage (kmseardetect.cpp:656-659); eye = stand-in for the absent
    mcs_* feature cascades; frontalface_default = a 24x24 window."""
    p = os.path.join(cascade_dir, name)
    ncasc, ocasc = nv.Cascade(p), O.Cascade(p)
    g = O.equalize_hist(O.bgr2gray(synth.frame(320, 240, 4, 9)))
    for mn in (0, 2):
        assert rects_equal(ctx.detect_multiscale(ncasc, g, sf, mn, ms), O.detect_multiscale(g, ocasc, sf, mn, ms))
    check_levels(ctx, g, ocasc, sf, ms)


@pytest.mark.parametrize("name,sf,ms", [("haarcascade_lefteye_2splits.xml", 1.1, (20, 20)),
                                        ("haarcascade_righteye_2splits.xml", 1.1, (0, 0)),
                                        ("haarcascade_smile.xml", 1.1, (1, 1)),
                                        ("haarcascade_eye_tree_eyeglasses.xml", 1.25, (0, 0)),
                                        ("haarcascade_frontalface_alt2.xml", 1.2, (0, 0))])
def test_general_cascades(ctx, cascade_dir, tmp_path, name, sf, ms):
    """Tree weak classifiers and tilted features (OpenCV's predictOrdered path): tilted integrals, depth maps,
    candidates and grouped rectangles against the oracle, in the new and the OpenCV-2.x XML layout; then a plain stump
    cascade on the same context (the tilted buffers come and go with the cascade)."""
    from cascade_xml_util import write_old_format
    p = os.path.join(cascade_dir, name)
    ncasc, ocasc = nv.Cascade(p), O.Cascade(p)
    assert ncasc.info.general == 1 and ocasc.general
    g = O.equalize_hist(O.bgr2gray(synth.frame(400, 300, 2, 3, smin=0.5, smax=0.9)))      # faces big enough for their eyes to fire
    n = 0
    for mn in (0, 2):
        got = ctx.detect_multiscale(ncasc, g, sf, mn, ms)
        assert rects_equal(got, O.detect_multiscale(g, ocasc, sf, mn, ms)), mn
        n += len(got)
    assert n > 0
    nwin, levels = check_levels(ctx, g, ocasc, sf, ms)
    assert nwin > 1000
    old = str(tmp_path / "old.xml")
    write_old_format(old, O.parse_cascade_xml(p))
    assert rects_equal(ctx.detect_multiscale(nv.Cascade(old), g, sf, 0, ms), O.detect_multiscale(g, ocasc, sf, 0, ms))
    fp = os.path.join(cascade_dir, FACE_XML)
    assert rects_equal(ctx.detect_multiscale(nv.Cascade(fp), g, 1.2, 2), O.detect_multiscale(g, O.Cascade(fp), 1.2, 2))


@pytest.mark.parametrize("seed", range(6))
def test_random_cascades_and_ragged_sizes(ctx, tmp_path, seed):
    """Random stump cascades (stage-0 skip rule, 3-rect features, odd window sizes) on odd image sizes."""
    rng = np.random.default_rng(300 + seed)
    p = str(tmp_path / "rand.xml")
    w, h = [(20, 20), (24, 24), (25, 15), (18, 15), (12, 30), (33, 9)][seed]
    random_cascade(p, rng, w=w, h=h, nstages=int(rng.integers(1, 7)), max_trees=8)
    W, H = int(rng.integers(w + 1, 500)), int(rng.integers(h + 1, 400))
    g = synth.frame(W, H, 2, seed)[..., 1] if seed % 2 else rng.integers(0, 256, (H, W), dtype=np.uint8)
    sf = float(rng.choice([1.1, 1.25, 1.4]))
    ncasc, ocasc = nv.Cascade(p), O.Cascade(p)
    for mn in (0, 2):
        assert rects_equal(ctx.detect_multiscale(ncasc, g, sf, mn), O.detect_multiscale(g, ocasc, sf, mn)), (seed, mn)
    check_levels(ctx, g, ocasc, sf, (0, 0))


@pytest.mark.parametrize("idx", range(5))
def test_general_golden_cases(ctx, cascade_dir, idx):
    """Tree / tilted models against the committed cv2 outputs (tests/golden/general_golden.json)."""
    import hashlib
    c = json.load(open(os.path.join(HERE, "golden", "general_golden.json")))["cases"][idx]
    eq = O.equalize_hist(O.bgr2gray(synth.frame(c["W"], c["H"], c["k"], c["seed"], smin=c["smin"], smax=c["smax"])))
    ncasc = nv.Cascade(os.path.join(cascade_dir, c["cascade"]))
    ms = tuple(c["min_size"])
    assert rects_equal(ctx.detect_multiscale(ncasc, eq, c["scale_factor"], c["min_neighbors"], ms), c["grouped"])
    assert rects_equal(ctx.detect_multiscale(ncasc, eq, c["scale_factor"], 0, ms), c["raw"])
    if ncasc.info.has_tilted:
        lv0 = ctx.levels()[0]
        if (lv0["lw"], lv0["lh"]) == (c["W"], c["H"]):          # the first level is the frame itself when min_size allows scale 1
            assert hashlib.sha256(ctx.tilted(0).tobytes()).hexdigest() == c["tilted_sha"]


@pytest.mark.parametrize("seed", range(6))
def test_random_trainer_shaped_and_general_cascades(ctx, tmp_path, seed):
    """The exact-integer fast kernels (bulk bank-class kernel, six-load features, fast tail) on random cascades shaped
    like the trainer's output — 12 stages of up to 40 classifiers, so the bulk stages AND the tail run — and the
    predictOrdered kernels on random tree / tilted cascades: integrals, tilted integrals, every depth map, candidates
    and grouped rectangles against the oracle, on odd image and window sizes."""
    rng = np.random.default_rng(500 + seed)
    p = str(tmp_path / "int.xml")
    random_int_cascade(p, rng, w=[20, 24, 18, 32, 20, 25][seed], h=[20, 24, 15, 20, 30, 15][seed])
    ncasc, ocasc = nv.Cascade(p), O.Cascade(p)
    assert ncasc.info.order_free_sums == 1 and ncasc.info.general == 0
    W, H = int(rng.integers(150, 700)), int(rng.integers(120, 500))
    g = synth.frame(W, H, 3, seed)[..., 1]
    sf = float(rng.choice([1.1, 1.2, 1.3]))
    for mn in (0, 2):
        assert rects_equal(ctx.detect_multiscale(ncasc, g, sf, mn), O.detect_multiscale(g, ocasc, sf, mn)), (seed, mn)
    nwin, levels = check_levels(ctx, g, ocasc, sf, (0, 0))
    codes = np.concatenate([l["depth"].ravel() for l in levels])
    assert (codes <= -10).any() or (codes == 1).any(), "no window reached the tail stages"
    q = str(tmp_path / "gen.xml")
    write_old_format(q, random_general_model(rng))
    ngen, ogen = nv.Cascade(q), O.Cascade(q)
    assert ngen.info.general == 1
    for mn in (0, 2):
        assert rects_equal(ctx.detect_multiscale(ngen, g, sf, mn), O.detect_multiscale(g, ogen, sf, mn)), (seed, mn)
    check_levels(ctx, g, ogen, sf, (0, 0))


@pytest.mark.parametrize("idx", range(3))
def test_lbp_golden_cases(ctx, idx):
    """BOOST/LBP cascades against the committed cv2 outputs (tests/golden/lbp_golden.json)."""
    import hashlib
    c = json.load(open(os.path.join(HERE, "golden", "lbp_golden.json")))["cases"][idx]
    eq = O.equalize_hist(O.bgr2gray(synth.frame(c["W"], c["H"], c["k"], c["seed"])))
    ncasc = nv.Cascade(os.path.join(HERE, "golden", c["cascade"]))
    assert ncasc.info.lbp == 1
    raw = ctx.detect_multiscale(ncasc, eq, c["scale_factor"], 0)
    assert len(raw) == c["n_raw"] and hashlib.sha256(np.ascontiguousarray(raw, np.int32).tobytes()).hexdigest() == c["raw_sha"]
    assert rects_equal(ctx.detect_multiscale(ncasc, eq, c["scale_factor"], c["min_neighbors"]), c["grouped"])


@pytest.mark.parametrize("seed", range(8))
def test_random_lbp_cascades(ctx, tmp_path, seed):
    """Random LBP cascades (OpenCV's predictCategorical path; categorical stumps for even seeds, trees of up to three nodes
    for odd ones), on small plans (warp per window / thread per window) and on plans above 16 384 windows (stage-range
    passes with compaction): every depth map, candidates and grouped rectangles against the oracle.  A Haar cascade on
    the same context afterwards (the model kind switches with the cascade)."""
    rng = np.random.default_rng(700 + seed)
    p = str(tmp_path / "lbp.xml")
    w, h = [(24, 24), (20, 20), (32, 18), (18, 30)][seed % 4]
    random_lbp_cascade(p, rng, w=w, h=h, nstages=int(rng.integers(2, 8)), max_trees=8, max_nodes=1 if seed % 2 == 0 else 3)
    big = seed >= 4
    W, H = (int(rng.integers(500, 900)), int(rng.integers(400, 600))) if big else (int(rng.integers(60, 100)), int(rng.integers(60, 100)))
    g = synth.frame(W, H, 2, seed)[..., 1] if seed % 3 else rng.integers(0, 256, (H, W), dtype=np.uint8)
    sf = float(rng.choice([1.1, 1.25, 1.4]))
    ncasc, ocasc = nv.Cascade(p), O.Cascade(p)
    assert ncasc.info.lbp == 1 and ocasc.lbp
    n = 0
    for mn in (0, 2):
        got = ctx.detect_multiscale(ncasc, g, sf, mn)
        assert rects_equal(got, O.detect_multiscale(g, ocasc, sf, mn)), (seed, mn)
        n += len(got)
    assert n > 0
    nwin, levels = check_levels(ctx, g, ocasc, sf, (0, 0))
    assert (nwin > 16384) == big                                                # both routes: small plan / staged large plan
    assert not any((l["depth"] == O.DEPTH_VARREJ).any() for l in levels)         # LBP has no variance test
    fp = os.path.join(os.path.dirname(HERE), "nubomedia-vca_b200", "cascades", FACE_XML)
    assert rects_equal(ctx.detect_multiscale(nv.Cascade(fp), g, 1.2, 2), O.detect_multiscale(g, O.Cascade(fp), 1.2, 2))


def test_old_format_and_wide_window_cascade(ctx, tmp_path, cascade_dir):
    """(1) frontalface_alt rewritten in the OpenCV-2.x layout detects exactly like the new layout;
    (2) cv2's genuine old-layout 64x16 plate cascade: wider than the tile kernel's 32x32 limit, so this also
    covers the generic queue path (k_alive_to_queue + k_queue_stages)."""
    from cascade_xml_util import write_old_format
    src = os.path.join(cascade_dir, FACE_XML)
    p = str(tmp_path / "old.xml")
    write_old_format(p, O.parse_cascade_xml(src))
    g = O.equalize_hist(O.bgr2gray(synth.frame(480, 360, 10, 5)))
    a = ctx.detect_multiscale(nv.Cascade(p), g, 1.25, 3)
    assert len(a) >= 3 and rects_equal(a, ctx.detect_multiscale(nv.Cascade(src), g, 1.25, 3))
    assert rects_equal(a, O.detect_multiscale(g, O.Cascade(p), 1.25, 3))
    cv2 = pytest.importorskip("cv2")
    plate = os.path.join(cv2.data.haarcascades, "haarcascade_license_plate_rus_16stages.xml")
    rng = np.random.default_rng(21)
    g2 = O.equalize_hist(cv2.GaussianBlur(rng.integers(0, 256, (240, 400), dtype=np.uint8), (0, 0), 1.2))
    ncasc, ocasc = nv.Cascade(plate), O.Cascade(plate)
    for mn in (0, 2):
        assert rects_equal(ctx.detect_multiscale(ncasc, g2, 1.1, mn), O.detect_multiscale(g2, ocasc, 1.1, mn))
    check_levels(ctx, g2, ocasc, 1.1, (0, 0))


def test_plan_cache_eviction_and_graph_replay(cascade_dir):
    """A context keeps 12 plans (size, cascade, parameters) with their parameter banks, tensor maps and a CUDA graph of
    the launches.  20 image sizes x 2 cascades through ONE non-debug context, three passes: the first pass plans, the
    second captures graphs where a plan survived, the third replays or re-plans after eviction; plus a device-resident
    ROI whose pointer and size repeat (the nested elements' pattern).  Every result against the oracle."""
    c = nv.Context(0, 640, 480)
    cascs = [(nv.Cascade(os.path.join(cascade_dir, n)), O.Cascade(os.path.join(cascade_dir, n)))
             for n in (FACE_XML, "haarcascade_eye.xml")]
    base = O.equalize_hist(O.bgr2gray(synth.frame(640, 480, 6, 21, smin=0.15, smax=0.5)))
    sizes = [(60 + 23 * i, 50 + 17 * i) for i in range(20)]
    exp = {}
    hits = 0
    for rep in range(3):
        for k, (w, h) in enumerate(sizes):
            g = np.ascontiguousarray(base[k:k + h, 2 * k:2 * k + w])
            for ci, (ncasc, ocasc) in enumerate(cascs):
                if (k, ci) not in exp:
                    exp[(k, ci)] = O.detect_multiscale(g, ocasc, 1.1, 2, (20, 20))
                got = c.detect_multiscale(ncasc, g, 1.1, 2, (20, 20))
                assert rects_equal(got, exp[(k, ci)]), (rep, k, ci)
                hits += len(got)
    assert hits > 0
    # cascades that are freed and re-created in turn (a new one may land on the old one's ADDRESS: plans are keyed by a
    # never-reused id, not by the pointer), same image and parameters every time
    g = np.ascontiguousarray(base[:300, :400])
    names = [FACE_XML, "haarcascade_frontalface_alt2.xml", "haarcascade_eye.xml", "haarcascade_lefteye_2splits.xml"]
    want = [O.detect_multiscale(g, O.Cascade(os.path.join(cascade_dir, n)), 1.2, 2) for n in names]
    for rep in range(3):
        for n, w_ in zip(names, want):
            tmp = nv.Cascade(os.path.join(cascade_dir, n))
            assert rects_equal(c.detect_multiscale(tmp, g, 1.2, 2), w_), (rep, n)
            del tmp
    # the same two sizes alternating many times: both plans stay cached and their graphs are replayed
    for rep in range(6):
        for k in (3, 11):
            w, h = sizes[k]
            g = np.ascontiguousarray(base[k:k + h, 2 * k:2 * k + w])
            assert rects_equal(c.detect_multiscale(cascs[0][0], g, 1.1, 2, (20, 20)), exp[(k, 0)])
    c.close()


def test_edge_cases(ctx, face):
    ncasc, ocasc = face
    rng = np.random.default_rng(1)
    # image smaller than the window: empty result, no error (A.9)
    assert len(ctx.detect_multiscale(ncasc, rng.integers(0, 256, (15, 19), dtype=np.uint8), 1.1, 3)) == 0
    # exactly one window
    g = rng.integers(0, 256, (20, 20), dtype=np.uint8)
    assert rects_equal(ctx.detect_multiscale(ncasc, g, 1.1, 0), O.detect_multiscale(g, ocasc, 1.1, 0))
    # flat image: every window variance-rejected
    assert len(ctx.detect_multiscale(ncasc, np.full((100, 100), 128, np.uint8), 1.1, 0)) == 0
    # padded stride (GStreamer rows are 4-byte aligned: stride != 3*width)
    fr = synth.frame(322, 241, 3, 11)
    pad = np.zeros((241, 322 * 3 + 2), np.uint8); pad[:, :966] = fr.reshape(241, -1)
    view = pad[:, :966].reshape(241, 322, 3)
    a = nv.Context._face_params(161, 1.25, 3, None)
    import ctypes as C
    n = C.c_int(0)
    rc = nv._lib.nv_face_detect(ctx.handle, ncasc.handle, pad.ctypes.data_as(C.c_void_p), 322, 241, pad.strides[0],
                                C.byref(a), ctx._out, ctx._cap, C.byref(n))
    assert rc == 0
    exp, _ = O.face_process(np.ascontiguousarray(view), ocasc, 161, 1.25, 3, None)
    assert rects_equal(nv._rects(ctx._out, n.value), exp)
    # bad parameters are reported, not crashed on
    with pytest.raises(nv.NuboError):
        ctx.detect_multiscale(ncasc, g, 1.0, 3)
    with pytest.raises(nv.NuboError):
        ctx.face_detect(ncasc, fr, 0)
    with pytest.raises(nv.NuboError):
        ctx.face_detect(ncasc, np.zeros((2000, 3000, 3), np.uint8), 160)


@pytest.mark.parametrize("case", [(648, 480, 648, 0), (642, 480, 642, 0), (1288, 720, 644, 0), (1284, 720, 642, 0),
                                  (648, 480, 648, 4), (648, 480, 648, 3), (1288, 720, 644, 8), (1288, 720, 644, 2),
                                  (648, 480, 216, 0)])
def test_prep_modes_and_alignment(ctx, face, case):
    """k_face_prep: same-size and exact-2x frames go through the vectorised kernels when output width, pointer and row
    stride are multiples of 4, else (and for every other ratio) through the byte-per-lane kernel; all against the oracle."""
    import ctypes as C
    ncasc, ocasc = face
    W, H, w2p, pad = case
    fr = synth.frame(W, H, 3, 30 + W + pad)
    buf = np.random.default_rng(pad).integers(0, 256, (H, 3 * W + pad), dtype=np.uint8)
    buf[:, :3 * W] = fr.reshape(H, -1)
    n = C.c_int(0)
    a = nv.Context._face_params(w2p, 1.2, 2, None)
    assert nv._lib.nv_face_detect(ctx.handle, ncasc.handle, buf.ctypes.data_as(C.c_void_p), W, H, buf.strides[0], C.byref(a),
                                  ctx._out, ctx._cap, C.byref(n)) == 0
    exp, eq = O.face_process(fr, ocasc, w2p, 1.2, 2, None)
    assert (ctx.gray() == eq).all()
    assert rects_equal(nv._rects(ctx._out, n.value), exp)


@pytest.mark.parametrize("case", [(640, 480, 160, 0), (640, 480, 160, 16), (480, 360, 160, 0), (800, 600, 160, 4),
                                  (960, 540, 160, 0), (646, 486, 160, 0), (1920, 1080, 320, 0)])
@pytest.mark.parametrize("pinned", [False, True])
def test_integer_downscale_uploads_row_pairs(face, case, pinned):
    """An integer down-scale by 3 or more (the element's default 640 -> 160) reads two of every `scale` source rows; only
    those row pairs are uploaded (context.cu: upload_rows; page-locked frames in place, others through the staging
    buffer).  The rows that stay on the host are POISONED on the device side here by a first, full-size call with a frame of 0xFF, so a
    kernel that read one of them would not reproduce the oracle's gray image.  646x486 is the irregular case (646 / 160 = 4
    but 486 rows do not divide: the whole frame travels).  Non-debug context: graph replay on the third call."""
    import ctypes as C
    import torch
    ncasc, ocasc = face
    W, H, w2p, pad = case
    c = nv.Context(0, 1920, 1080)
    try:
        fr = synth.frame(W, H, 3, 77 + W + pad)
        stride = 3 * W + pad
        host = torch.empty((H, stride), dtype=torch.uint8)
        if pinned:
            host = host.pin_memory()
        buf = host.numpy()
        n = C.c_int(0)
        a = nv.Context._face_params(w2p, 1.2, 2, None)
        exp, eq = O.face_process(fr, ocasc, w2p, 1.2, 2, None)
        for it in range(4):
            buf[:] = 255 if it == 0 else np.random.default_rng(it).integers(0, 256, buf.shape, dtype=np.uint8)
            if it > 0:
                buf[:, :3 * W] = fr.reshape(H, -1)
            # the poison frame goes up whole (processing width = frame width: same-size mode, every row is read)
            prm = nv.Context._face_params(W, 1.2, 2, None) if it == 0 else a
            assert nv._lib.nv_face_detect(c.handle, ncasc.handle, buf.ctypes.data_as(C.c_void_p), W, H, stride, C.byref(prm),
                                          c._out, c._cap, C.byref(n)) == 0
            if it > 0:
                assert rects_equal(nv._rects(c._out, n.value), exp), it
        c.set_debug(True)
        assert nv._lib.nv_face_detect(c.handle, ncasc.handle, buf.ctypes.data_as(C.c_void_p), W, H, stride, C.byref(a),
                                      c._out, c._cap, C.byref(n)) == 0
        assert (c.gray() == eq).all()
    finally:
        c.close()


def test_cfg3_full_size_1080p(ctx, face):
    """BASELINE config 3 at full size: 1920x1080, processing width 1920, sf 1.1, min 24x24.
    Full oracle comparison (a few seconds of CPU) including every depth map."""
    ncasc, ocasc = face
    fr = synth.frame(1920, 1080, 6, 3)
    got = ctx.face_detect(ncasc, fr, 1920, 1.1, 3, (24, 24))
    exp, eq = O.face_process(fr, ocasc, 1920, 1.1, 3, (24, 24))
    assert rects_equal(got, exp) and len(got) >= 4
    assert (ctx.gray() == eq).all()
    nwin, _ = check_levels(ctx, eq, ocasc, 1.1, (24, 24))
    assert nwin > 3_000_000
    assert len(ctx.levels()) == 40


def test_beyond_1080p_4k_frame(face):
    """Maximum sizes: a 3840x2160 frame at full processing width (the packed candidate key keeps 13 bits per coordinate),
    BGR and NV12, with every level's integrals and depth maps against the oracle."""
    ncasc, ocasc = face
    c = nv.Context(0, 3840, 2160, debug=True)
    try:
        fr = synth.frame(3840, 2160, 5, 21)
        exp, eq = O.face_process(fr, ocasc, 3840, 1.2, 3, (40, 40))
        got = c.face_detect(ncasc, fr, 3840, 1.2, 3, (40, 40))
        assert rects_equal(got, exp) and len(got) >= 4
        assert (c.gray() == eq).all()
        nwin, _ = check_levels(c, eq, ocasc, 1.2, (40, 40))
        assert nwin > 5_000_000
        buf = synth.to_yuv420(fr, "NV12")
        exp, eq = O.face_process(O.yuv420_to_bgr(*O.yuv420_planes(buf, 3840, 2160, "NV12"), fmt="NV12"), ocasc, 1920, 1.2, 3, None)
        got = c.face_detect_yuv(ncasc, synth.yuv420_planes(buf, 3840, 2160, "NV12"), "NV12", 1920, 1.2, 3, None)
        assert rects_equal(got, exp) and (c.gray() == eq).all()
    finally:
        c.close()


def test_full_size_properties_without_the_oracle(face):
    """Size-independent properties at BASELINE's full sizes, where a second oracle run would only repeat
    test_cfg3_full_size_1080p: (1) a frame padded to a wider stride gives the same rectangles; (2) the device-resident
    input path equals the host path; (3) ten replays of the captured graph are identical; (4) raw candidates
    (minNeighbors 0) contain every grouped rectangle's neighbourhood: each grouped rect has >= 3 raw candidates within
    the 0.2 similarity bound; (5) 32 contexts on different frames (config 5's shape) agree with one context run alone."""
    torch = pytest.importorskip("torch")
    ncasc, _ = face
    fr = synth.frame(1920, 1080, 6, 3)
    c = nv.Context(0, 1920, 1080)
    base = c.face_detect(ncasc, fr, 1920, 1.1, 3, (24, 24))
    assert len(base) >= 4
    import ctypes as C
    pad = np.zeros((1080, 1920 * 3 + 64), np.uint8); pad[:, :5760] = fr.reshape(1080, -1)
    n = C.c_int(0)
    a = nv.Context._face_params(1920, 1.1, 3, (24, 24))
    assert nv._lib.nv_face_detect(c.handle, ncasc.handle, pad.ctypes.data_as(C.c_void_p), 1920, 1080, pad.strides[0], C.byref(a),
                                  c._out, c._cap, C.byref(n)) == 0
    assert rects_equal(nv._rects(c._out, n.value), base)
    d = torch.from_numpy(fr).cuda()
    for _ in range(10):
        c.face_submit_device(ncasc, d.data_ptr(), 1920, 1080, 5760, 1920, 1.1, 3, (24, 24))
        assert rects_equal(c.face_collect(), base)
    raw = c.face_detect(ncasc, fr, 1920, 1.1, 0, (24, 24)).astype(np.int64)
    for (x, y, w, h) in base.astype(np.int64):
        delta = 0.2 * (np.minimum(w, raw[:, 2]) + np.minimum(h, raw[:, 3])) * 0.5
        near = (np.abs(raw[:, 0] - x) <= delta) & (np.abs(raw[:, 1] - y) <= delta) & \
               (np.abs(raw[:, 0] + raw[:, 2] - x - w) <= delta) & (np.abs(raw[:, 1] + raw[:, 3] - y - h) <= delta)
        assert near.sum() >= 3, (x, y, w, h)
    c.close()
    frames = [synth.frame(1280, 720, 3, 1000 + i) for i in range(32)]
    ctxs = [nv.Context(0, 1280, 720) for _ in frames]
    for rep in range(2):                                        # second round: every context replays its graph
        for cx, f in zip(ctxs, frames):
            cx.face_submit(ncasc, f, 640, 1.25, 3, None)
        outs = [cx.face_collect() for cx in ctxs]
    solo = nv.Context(0, 1280, 720)
    for f, o in zip(frames, outs):
        assert rects_equal(solo.face_detect(ncasc, f, 640, 1.25, 3, None), o)
    for cx in ctxs + [solo]:
        cx.close()


def test_async_streams_are_independent(face):
    """cfg5 mechanics: many contexts in flight give the same per-stream results as one at a time."""
    ncasc, ocasc = face
    ctxs = [nv.Context(0, 1280, 720) for _ in range(4)]
    frames = [synth.frame(1280, 720, 3, 1000 + i) for i in range(4)]
    for c, f in zip(ctxs, frames):
        c.face_submit(ncasc, f, 640, 1.25, 3, None)
    outs = [c.face_collect() for c in ctxs]
    for f, o in zip(frames, outs):
        exp, _ = O.face_process(f, ocasc, 640, 1.25, 3, None)
        assert rects_equal(o, exp)
    for c in ctxs:
        c.close()


# ------------------------------------------------------------------------------------------
def test_image_ops(ctx):
    rng = np.random.default_rng(2)
    img = rng.integers(0, 256, (217, 333, 3), dtype=np.uint8)
    assert (ctx.bgr2gray(img) == O.bgr2gray(img)).all()
    img4 = rng.integers(0, 256, (45, 67, 4), dtype=np.uint8)
    assert (ctx.bgr2gray(img4) == O.bgr2gray(img4)).all()
    g = img[..., 0].copy()
    assert (ctx.equalize_hist(g) == O.equalize_hist(g)).all()
    assert (ctx.equalize_hist(np.full((10, 10), 7, np.uint8)) == 7).all()
    for (dw, dh) in [(160, 104), (166, 108), (333, 217), (400, 300), (100, 300), (666, 434)]:
        assert (ctx.resize_linear(img, dw, dh) == O.resize_linear(img, dw, dh)).all(), (dw, dh)
        assert (ctx.resize_linear(g, dw, dh) == O.resize_linear(g, dw, dh)).all(), (dw, dh)
    big = rng.integers(0, 256, (720, 1280), dtype=np.uint8)
    assert (ctx.resize_linear(big, 640, 360) == O.resize_linear(big, 640, 360)).all()      # 2x fast path
    assert (ctx.flip_horizontal(g) == g[:, ::-1]).all()


# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("idx", range(2))
def test_tracker_golden(idx):
    c = json.load(open(os.path.join(HERE, "golden", "tracker_golden.json")))["cases"][idx]
    frames = synth.tracker_sequence(c["W"], c["H"], c["nframes"], c["seed"], noise=c["noise"])
    t = nv.Context(0, c["W"], c["H"])
    for i, (f, g) in enumerate(zip(frames, c["frames"])):
        r = t.tracker_process(f, 33.3 * (i + 1), c["threshold"], -1, 1 << 40, 0)
        assert rects_equal(r, g["rects"]), i
    t.close()


def test_tracker_vs_oracle_with_join_and_stale_history():
    """cfg4 parameters at 720p; timestamps closer than MHI_DURATION keep stale history alive, which
    exercises the floating-range connectivity beyond plain connected components."""
    W, H = 1280, 720
    frames = synth.tracker_sequence(W, H, 6, seed=4, noise=300)
    t = nv.Context(0, W, H)
    st = O.TrackerState(W, H)
    for i, f in enumerate(frames):
        ts = 1000.0 + (0.1 * i if i < 3 else 33.3 * i)
        got = t.tracker_process(f, ts, 20, 50, 30000, 35)
        exp, nraw, _ = st.process(f, ts, 20, 50, 30000, 35)
        assert rects_equal(got, exp), i
    t.tracker_reset()
    assert len(t.tracker_process(frames[0], 5000.0)) == 0       # first frame after reset only primes
    t.close()
