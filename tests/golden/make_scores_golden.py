"""Generates tests/golden/scores_golden.json from cv2 4.13 with one thread:

    python tests/golden/make_scores_golden.py

For each case (a cascade, a seeded synthetic frame, detectMultiScale parameters) it stores cv2's
detectMultiScale2 rectangles and numDetections and detectMultiScale3(outputRejectLevels=True) rectangles,
rejectLevels and levelWeights.  Weights are stored as float.hex() strings so that the tests compare them
exactly.  Tests check the oracle (and on the GPU the CUDA path) against this file without cv2.
"""
import hashlib
import json
import os
import sys
import tempfile

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "nubomedia-vca_b200", "python"))
sys.path.insert(0, os.path.dirname(HERE))
from cascade_xml_util import random_cascade  # noqa: E402
from nubovca import synth  # noqa: E402

CASC = os.path.join(ROOT, "nubomedia-vca_b200", "cascades")

# (model, W, H, k, seed, scale_factor, min_neighbors list, min_size)
CASES = [
    ("haarcascade_frontalface_alt.xml", 640, 480, 4, 1, 1.1, [0, 3], (24, 24)),
    ("haarcascade_frontalface_alt2.xml", 320, 240, 3, 5, 1.1, [0, 3], (0, 0)),
    ("haarcascade_frontalface_default.xml", 320, 240, 3, 5, 1.1, [0, 3], (0, 0)),
    ("haarcascade_profileface.xml", 640, 480, 2, 3, 1.1, [0, 1], (0, 0)),
    ("haarcascade_lefteye_2splits.xml", 640, 480, 1, 9, 1.1, [0, 1], (0, 0)),
    ("haarcascade_eye_tree_eyeglasses.xml", 640, 480, 1, 9, 1.1, [0, 1], (0, 0)),
    ("haarcascade_smile.xml", 320, 240, 3, 11, 1.1, [0, 3], (0, 0)),
    ("lbp_random_0.xml", 320, 240, 3, 41, 1.1, [0, 2], (0, 0)),
    ("lbp_random_1.xml", 320, 240, 3, 42, 1.1, [0, 2], (0, 0)),
    ("lbp_random_2.xml", 320, 240, 3, 43, 1.1, [0, 2], (0, 0)),
    ("random_stump:3", 160, 120, 2, 13, 1.2, [0, 1, 4], (0, 0)),
    ("random_stump:3", 160, 120, 3, 17, 1.2, [0, 2], (0, 0)),
    ("haarcascade_frontalface_alt.xml", 320, 240, 0, 3, 1.1, [0, 3], (0, 0)),      # blank frame: no detections
]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def model_path(name, tmp):
    """Cascade file of a case: a shipped cascade, a committed LBP model, or a seeded random stump model."""
    if name.startswith("random_stump:"):
        path = os.path.join(tmp, name.replace(":", "_") + ".xml")
        random_cascade(path, np.random.default_rng(int(name.split(":")[1]) + 100), nstages=4, max_trees=6)
        return path
    if name.startswith("lbp_random"):
        return os.path.join(HERE, name)
    return os.path.join(CASC, name)


def frame(W, H, k, seed):
    if k == 0:
        return np.full((H, W, 3), 128, np.uint8)
    return synth.frame(W, H, k, seed)


def main():
    cv2.setNumThreads(1)
    out = []
    with tempfile.TemporaryDirectory() as tmp:
        for name, W, H, k, seed, sf, mns, ms in CASES:
            cc = cv2.CascadeClassifier(model_path(name, tmp))
            assert not cc.empty(), name
            eq = cv2.equalizeHist(cv2.cvtColor(frame(W, H, k, seed), cv2.COLOR_BGR2GRAY))
            for mn in mns:
                r2, nd = cc.detectMultiScale2(eq, sf, mn, 0, ms)
                r3, rl, lw = cc.detectMultiScale3(eq, sf, mn, 0, ms, outputRejectLevels=True)
                r2 = np.asarray(r2, np.int32).reshape(-1, 4); r3 = np.asarray(r3, np.int32).reshape(-1, 4)
                assert (r2 == r3).all(), name
                out.append(dict(cascade=name, W=W, H=H, k=k, seed=seed, scale_factor=sf, min_neighbors=mn, min_size=list(ms),
                                eq_sha=sha(eq), rects=r2.tolist(), num_detections=np.asarray(nd).ravel().tolist(),
                                reject_levels=sorted(set(np.asarray(rl).ravel().tolist())),
                                level_weights=[float(v).hex() for v in np.asarray(lw, np.float64).ravel()]))
                print(f"{name:38s} mn={mn} rects={len(r2)}", flush=True)
    with open(os.path.join(HERE, "scores_golden.json"), "w") as f:
        json.dump({"generator": "cv2 " + cv2.__version__ + ", setNumThreads(1)", "cases": out}, f)


if __name__ == "__main__":
    main()
