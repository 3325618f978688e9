"""What the reference's six elements, compiled from their own sources (oracle/build_ref.py) and run on the CPU, answered
(tests/golden/ref_elements.json), against this repository:

  * what their class_init declares (factory names, pad caps, properties with ranges, signals) equals SURVEY.md §2.2 and
    the property table of the nv_element mirrors;
  * tests/element_ref.py — the Python restatement the GPU element tests were written against in round 1 — emits the same
    messages as the compiled reference on the same frames, so both restatements are pinned to the reference itself;
  * __receive_event semantics (any queued message uses up the frame's pop; a message without timestamp is dropped), on the
    GStreamer shell.

No GPU needed except for the last: the restatements compute through the CPU oracle."""
import os
import shutil

import numpy as np
import pytest

import nubovca as nv
import oracle as O
import refgst
from cascade_xml_util import permissive_cascade
from element_ref import EarRef, FaceRef, FeatureRef
from nubovca import synth
from refgst import GOLDEN

STANDINS = {"haarcascade_mcs_righteye.xml": (18, 12, 0), "haarcascade_mcs_lefteye.xml": (18, 12, 1),
            "haarcascade_mcs_mouth.xml": (25, 15, 4), "haarcascade_mcs_nose.xml": (18, 15, 5),
            "haarcascade_mcs_rightear.xml": (12, 20, 0), "haarcascade_mcs_leftear.xml": (12, 20, 1)}


def make_cascade_dir(d, cascade_dir):
    shutil.copy(os.path.join(cascade_dir, "haarcascade_frontalface_alt.xml"), os.path.join(d, "haarcascade_frontalface_alt.xml"))
    shutil.copy(os.path.join(cascade_dir, "haarcascade_frontalface_alt.xml"), os.path.join(d, "haarcascade_profileface.xml"))
    for name, (w, h, seed) in STANDINS.items():
        permissive_cascade(os.path.join(d, name), np.random.default_rng(seed), w, h)
    return str(d)


@pytest.fixture(scope="module")
def cdir(tmp_path_factory, cascade_dir):
    return make_cascade_dir(str(tmp_path_factory.mktemp("cascades_ref")), cascade_dir)


def oc(cdir, name):
    return O.Cascade(os.path.join(cdir, name))


def sequence(W, H, k, seed, n, **kw):
    base = synth.frame(W, H, k, seed, **kw)
    rng = np.random.default_rng(seed + 77)
    out = []
    for _ in range(n):
        f = base.astype(np.int16) + rng.integers(-3, 4, base.shape, dtype=np.int16)
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return out


# ---- class_init: what the elements declare ------------------------------------------------------------------------------
EXPECTED_PROPS = {
    "nubofacedetector": [("view-faces", 0, 1), ("detect-event", 0, 1), ("send-meta-data", 0, 1), ("width-to-process", 0, 640),
                         ("process-x-every-4-frames", 0, 4), ("euclidean-distance", 0, 20), ("track-threshold", 0, 100),
                         ("area-threshold", 0, 1000), ("multi-scale-factor", 0, 51), ("activate-events", 0, 1), ("events-ms", 0, 30000)],
    "nubotracker": [("set_threshold", 0, 255), ("set_min_area", 0, 10000), ("set_max_area", 0, 300000), ("set_distance", 0, 2000),
                    ("set_visual_mode", 0, 4), ("activate-events", 0, 1), ("events-ms", 0, 30000)],
}
INIT_VALUES = {       # *_init(): the values a fresh element reports (the pspec default is 0 for every property)
    "nubofacedetector": {"width-to-process": 160, "process-x-every-4-frames": 4, "multi-scale-factor": 25, "euclidean-distance": 8,
                         "track-threshold": 40, "area-threshold": 500, "events-ms": 30001, "view-faces": 0, "detect-event": 0},
    "nuboeyedetector": {"width-to-process": 320, "process-x-every-4-frames": 4, "multi-scale-factor": 25, "events-ms": 30001},
    "nubomouthdetector": {"width-to-process": 320, "process-x-every-4-frames": 4, "multi-scale-factor": 25, "events-ms": 30001},
    "nubonosedetector": {"width-to-process": 320, "process-x-every-4-frames": 4, "multi-scale-factor": 25, "events-ms": 30001},
    "nuboeardetector": {"width-to-process": 320, "process-x-every-4-frames": 4, "multi-scale-factor": 25, "events-ms": 0, "view-ears": -1},
    "nubotracker": {"set_threshold": 20, "set_min_area": 50, "set_max_area": 30000, "set_distance": 35, "events-ms": 30001},
}


def parse_description(text):
    d = {"property": [], "pad": [], "signal": []}
    for line in text.strip().split("\n"):
        k, *rest = line.split("|")
        if k in d:
            d[k].append(rest)
        else:
            d[k] = rest
    return d


@pytest.mark.parametrize("factory", refgst.FACTORIES)
def test_reference_class_init_matches_the_mirror(cdir, factory):
    d = parse_description(GOLDEN["describe"][factory])
    assert d["factory"] == [factory, "rank=0"]                                  # GST_RANK_NONE
    fmt = "BGRA" if factory == "nubotracker" else "BGR"
    assert [(p[0], p[1]) for p in d["pad"]] == [("src", "src"), ("sink", "sink")] and all(f"{{ {fmt} }}" in p[3] for p in d["pad"])
    sig = {"nubofacedetector": "face-event", "nuboeyedetector": "eye-event", "nubomouthdetector": "mouth-event",
           "nubonosedetector": "nose-event", "nuboeardetector": "ear-event", "nubotracker": "tracker-event"}[factory]
    assert [s[0] for s in d["signal"]] == [sig]
    ref_props = {p[0]: (p[1], int(p[2][4:]), int(p[3][4:]), int(p[4][8:])) for p in d["property"]}
    if factory in EXPECTED_PROPS:
        assert [(n, ref_props[n][1], ref_props[n][2]) for n, _, _ in EXPECTED_PROPS[factory]] == EXPECTED_PROPS[factory]
    assert all(v[3] == 0 for v in ref_props.values())                          # g_param_spec_int(.., FALSE, ..) everywhere
    if factory != "nubotracker":
        assert ref_props["image-to-overlay"][0] == "GstStructure"
    # the mirror's table: same names, same ranges (its "default" column is the *_init() value a fresh element reports)
    m = nv.Element(factory, 0, cdir)
    fresh = {n: v for step, n, _, v in GOLDEN["round_trip"][factory] if step == "init"}
    mirror = {n: (lo, hi, de) for n, lo, hi, de in m.properties()}
    ints = {n: v for n, v in ref_props.items() if v[0] in ("int", "long")}
    assert set(mirror) == set(ints) == set(fresh), (sorted(mirror), sorted(ints))
    for n, (typ, lo, hi, _) in ints.items():
        assert mirror[n][:2] == (lo, hi), n
        assert fresh[n] == m.get(n), (n, fresh[n], m.get(n))                    # fresh-instance values
    for n, v in INIT_VALUES[factory].items():
        assert fresh[n] == v, (n, fresh[n])
    # out-of-range values are rejected by both (the reference through a GLib warning)
    some = "set_threshold" if factory == "nubotracker" else "multi-scale-factor"
    assert GOLDEN["out_of_range"][factory] == {"property": some, "value": 10 ** 6, "accepted": False, "warnings": 1}
    with pytest.raises(nv.NuboError):
        m.set(some, 10 ** 6)
    m.close()


def test_face_track_threshold_setter_quirk(cdir, monkeypatch):
    """kmsfacedetect.cpp:548-550: the track-threshold setter writes euclidean_threshold; the getter reads track_threshold."""
    monkeypatch.setenv("NUBOVCA_CASCADE_DIR", cdir)
    s, m = refgst.shell().element("nubofacedetector"), nv.Element("nubofacedetector", 0, cdir)
    for e in (s, m):
        e.set("track-threshold", 17)
    assert (s.get("track-threshold"), s.get("euclidean-distance")) == (40, 17) == (m.get("track-threshold"), m.get("euclidean-distance"))
    s.close(); m.close()


# ---- element_ref.py against the compiled reference ----------------------------------------------------------------------
def face_restatement(cdir):
    """FaceRef's message rows per frame, for each process-x-every-4-frames value."""
    frames = sequence(640, 480, 4, 1, 6) + [np.full((480, 640, 3), 90, np.uint8)] * 3
    out = {}
    for x4 in (4, 3, 2, 1):
        py = FaceRef(oc(cdir, "haarcascade_frontalface_alt.xml"))
        py.p["x4"] = x4
        out[str(x4)] = [[list(m) for m in py.process(f)] for f in frames]
    return out


def test_face_restatement_equals_reference(cdir):
    got, exp = face_restatement(cdir), GOLDEN["face_restatement"]
    assert sorted(got) == sorted(exp)
    for x4 in exp:
        assert len(got[x4]) == len(exp[x4])
        for i, (g, x) in enumerate(zip(got[x4], exp[x4])):
            assert g == x, (x4, i, g, x)
        assert sum(len(x) for x in exp[x4]) > 0


FEATURES = {"eye": ("nuboeyedetector", ("haarcascade_mcs_righteye.xml", "haarcascade_mcs_lefteye.xml")),
            "mouth": ("nubomouthdetector", ("haarcascade_mcs_mouth.xml",)),
            "nose": ("nubonosedetector", ("haarcascade_mcs_nose.xml",))}


def feature_restatement(cdir, kind):
    frames = sequence(640, 360, 3, 2, 4, smin=0.4, smax=0.6)
    py = FeatureRef(kind, oc(cdir, "haarcascade_frontalface_alt.xml"), *[oc(cdir, f) for f in FEATURES[kind][1]])
    return [[list(m) for m in py.process(f)] for f in frames]


@pytest.mark.parametrize("kind,factory,files", [(k, f, fs) for k, (f, fs) in FEATURES.items()])
def test_feature_restatement_equals_reference(cdir, kind, factory, files):
    got, exp = feature_restatement(cdir, kind), GOLDEN["feature_restatement"][kind]
    assert len(got) == len(exp)
    for i, (g, x) in enumerate(zip(got, exp)):
        assert g == x, (kind, i, g, x)
    assert sum(1 for x in exp for m in x if m[1] != "face") > 0


def ear_restatement(cdir):
    """The ear-event signals EarRef implies per frame with activate-events 1, events-ms 0 (kmseardetect.cpp:210-290 builds
    the message, never pushes it: the signal is all that leaves the element)."""
    frames = sequence(640, 360, 3, 2, 4, smin=0.4, smax=0.6)
    py = EarRef(oc(cdir, "haarcascade_profileface.xml"), oc(cdir, "haarcascade_mcs_rightear.xml"), oc(cdir, "haarcascade_mcs_leftear.xml"))
    out = []
    for f in frames:
        exp = [m for m in py.process(f) if m[0] == "ear"]
        payload = "".join(f"x:{m[2]},y:{m[3]},width:{m[4]},height:{m[5]};" for m in exp)
        out.append([["ear-event", payload]] if exp else [])
    return out


def test_ear_restatement_equals_reference(cdir):
    got, exp = ear_restatement(cdir), GOLDEN["ear_restatement"]
    assert len(got) == len(exp)
    for i, (g, x) in enumerate(zip(got, exp)):
        assert g == x, (i, g, x)


# ---- __receive_event ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_reference_receive_event_semantics(cdir, monkeypatch):
    """The reference's semantics, on the GStreamer shell."""
    monkeypatch.setenv("NUBOVCA_CASCADE_DIR", cdir)
    S = refgst.shell()
    f = synth.frame(640, 480, 4, 1)
    r = S.element("nubofacedetector")
    assert r.set("detect-event", 1)
    n = lambda: len(r.process(f.copy())[1][0][2])
    assert n() == 0                                                            # nothing queued: no detection
    r.send_event(S.faces_message([(1, 2, 3, 4)]))                              # a non-motion message ...
    r.send_event(S.motion_message())
    assert n() == 0                                                            # ... uses up this frame's pop
    assert n() >= 1                                                            # the motion message arms 10 frames
    r.close()
    r = S.element("nubofacedetector")
    assert r.set("detect-event", 1)
    r.send_event(S.motion_message(timestamp=False))                            # no timestamp: dropped unread
    assert len(r.process(f.copy())[1][0][2]) == 0
    r.close()
