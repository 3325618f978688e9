"""Detection scores of the CPU reference (tests/scores_ref.py, built on the oracle's artefacts): cv2 detectMultiScale2's
numDetections and detectMultiScale3(outputRejectLevels=True)'s levelWeights, compared with `==` (no tolerance) against the
committed cv2 4.13 answers of tests/golden/make_scores_golden.py everywhere, and against cv2 itself where it imports."""
import json
import os

import numpy as np
import pytest

import oracle as O
import scores_ref as S
from cascade_xml_util import random_cascade
from nubovca import synth

try:
    import cv2
    cv2.setNumThreads(1)
except Exception:  # pragma: no cover
    cv2 = None

needs_cv2 = pytest.mark.skipif(cv2 is None, reason="cv2 not importable")
HERE = os.path.dirname(os.path.abspath(__file__))
CASC = os.path.join(os.path.dirname(HERE), "nubomedia-vca_b200", "cascades")
with open(os.path.join(HERE, "golden", "scores_golden.json")) as _f:
    GOLDEN = json.load(_f)["cases"]


def model_path(name, tmp):
    """As make_scores_golden.model_path: a shipped cascade, a committed LBP model, or a seeded random stump model."""
    if name.startswith("random_stump:"):
        path = os.path.join(str(tmp), name.replace(":", "_") + ".xml")
        random_cascade(path, np.random.default_rng(int(name.split(":")[1]) + 100), nstages=4, max_trees=6)
        return path
    if name.startswith("lbp_random"):
        return os.path.join(HERE, "golden", name)
    return os.path.join(CASC, name)


def case_gray(c):
    fr = np.full((c["H"], c["W"], 3), 128, np.uint8) if c["k"] == 0 else synth.frame(c["W"], c["H"], c["k"], c["seed"])
    return O.equalize_hist(O.bgr2gray(fr))


def golden_scores(c):
    return (np.asarray(c["rects"], np.int32).reshape(-1, 4), np.asarray(c["num_detections"], np.int32),
            np.array([float.fromhex(v) for v in c["level_weights"]], np.float64))


@pytest.mark.parametrize("idx", range(len(GOLDEN)), ids=[f"{c['cascade']}-mn{c['min_neighbors']}-{i}" for i, c in enumerate(GOLDEN)])
def test_oracle_scores_golden(idx, tmp_path):
    c = GOLDEN[idx]
    casc = O.Cascade(model_path(c["cascade"], tmp_path))
    r, nb, wt = S.detect_multiscale_scores(case_gray(c), casc, c["scale_factor"], c["min_neighbors"], tuple(c["min_size"]))
    er, enb, ewt = golden_scores(c)
    assert r.shape == er.shape and (r == er).all()
    assert (nb == enb).all() and (wt == ewt).all()
    # the rectangles are those of the scores-off call; rejectLevels is the stage count
    assert (O.detect_multiscale(case_gray(c), casc, c["scale_factor"], c["min_neighbors"], tuple(c["min_size"])) == r).all()
    assert c["reject_levels"] in ([], [casc.nstages])
    if c["min_neighbors"] <= 0:
        assert (nb == 1).all()
    else:
        assert (nb > c["min_neighbors"]).all()


def test_golden_covers_the_cases():
    """Raw and grouped calls, an empty result, a rectangle on the image border, thousands of raw candidates."""
    assert any(c["min_neighbors"] == 0 and len(c["rects"]) > 1000 for c in GOLDEN)
    assert any(c["min_neighbors"] > 0 and len(c["rects"]) > 0 for c in GOLDEN)
    assert any(len(c["rects"]) == 0 for c in GOLDEN)
    assert any(x == 0 or y == 0 or x + w == c["W"] or y + h == c["H"] for c in GOLDEN for x, y, w, h in c["rects"])


def test_weight_is_last_stage_sum(cascade_dir):
    """A raw window's weight is its last stage's sum: at or above that stage's threshold, and a grouped rectangle carries the
    largest weight of its class."""
    casc = O.Cascade(os.path.join(cascade_dir, "haarcascade_frontalface_alt.xml"))
    d = O.parse_cascade_xml(os.path.join(cascade_dir, "haarcascade_frontalface_alt.xml"))
    thr = float(np.float32(d["stage_thr"][-1]) - np.float32(1e-5))
    gray = O.equalize_hist(O.bgr2gray(synth.frame(640, 480, 4, 1)))
    raw, nb, wt = S.detect_multiscale_scores(gray, casc, 1.1, 0, (24, 24))
    assert len(raw) > 50 and (nb == 1).all() and (wt >= thr).all()
    g, gn, gw = S.group_weighted(raw, wt, 3)
    r, n3, w3 = S.detect_multiscale_scores(gray, casc, 1.1, 3, (24, 24))
    assert (g == r).all() and (gn == n3).all() and (gw == w3).all()
    assert gn.sum() <= len(raw) and set(gw.tolist()) <= set(wt.tolist())


def test_group_rectangles_weighted_unit():
    rects = [(10, 10, 20, 20), (11, 10, 20, 20), (10, 11, 20, 20), (100, 100, 20, 20)]
    w = [1.5, 3.25, -2.0, 7.0]
    r, n, lw = S.group_weighted(rects, w, 2)
    assert r.tolist() == [[10, 10, 20, 20]] and n.tolist() == [3] and lw.tolist() == [3.25]
    r, n, lw = S.group_weighted(rects, w, 0)
    assert r.tolist() == [list(x) for x in rects] and n.tolist() == [1, 1, 1, 1] and lw.tolist() == w
    r, n, lw = S.group_weighted(rects[:3], [-4.0, -1.0, -3.0], 1)       # all-negative weights: still the maximum
    assert n.tolist() == [3] and lw.tolist() == [-1.0]


@needs_cv2
@pytest.mark.parametrize("name,W,H,k,seed,mn", [
    ("haarcascade_frontalface_alt.xml", 640, 480, 4, 1, 3),
    ("haarcascade_frontalface_default.xml", 480, 360, 3, 21, 2),
    ("haarcascade_smile.xml", 640, 480, 4, 2, 0),
    ("haarcascade_smile.xml", 640, 480, 4, 2, 3),
    ("haarcascade_eye.xml", 640, 480, 2, 8, 0),
    ("lbp_random_1.xml", 480, 360, 4, 23, 3),
])
def test_oracle_scores_vs_cv2(name, W, H, k, seed, mn, tmp_path):
    gray = O.equalize_hist(O.bgr2gray(synth.frame(W, H, k, seed)))
    path = model_path(name, tmp_path)
    cc = cv2.CascadeClassifier(path)
    r2, nd = cc.detectMultiScale2(gray, 1.1, mn, 0, (0, 0))
    r3, rl, lw = cc.detectMultiScale3(gray, 1.1, mn, 0, (0, 0), outputRejectLevels=True)
    casc = O.Cascade(path)
    r, nb, wt = S.detect_multiscale_scores(gray, casc, 1.1, mn)
    assert (np.asarray(r2, np.int32).reshape(-1, 4) == r).all() and (np.asarray(r3, np.int32).reshape(-1, 4) == r).all()
    assert (np.asarray(nd).ravel() == nb).all()
    assert (np.asarray(lw, np.float64).ravel() == wt).all()
    assert set(np.asarray(rl).ravel().tolist()) <= {casc.nstages}
