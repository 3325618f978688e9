"""The GStreamer shells (nubomedia-vca_b200/gst/gstnubovca.cpp) built against the mock GStreamer, next to what the
reference's own elements, built against the same mock (oracle/build_ref.py), answered to the same calls
(tests/golden/ref_elements.json): what class_init declares must agree — factory names, rank, pad templates and caps, every
property (name, type, range, pspec default, flags, the boxed image-to-overlay), the signal and its signature, the
overridden virtual functions.  Compute paths need a GPU and live in tests/test_gst_shells_gpu.py."""
import ctypes as C

import pytest

import refgst
from refgst import GOLDEN


def parse(text):
    d = {"property": {}, "pad": [], "signal": [], "vfuncs": None, "factory": None}
    for line in text.strip().split("\n"):
        k, *rest = line.split("|")
        if k == "property":
            # name | type | min | max | default | flags   (ids and nicks are private to a class)
            d["property"][rest[0]] = tuple(rest[1:6])
        elif k in ("pad", "signal"):
            d[k].append(tuple(rest))
        elif k in ("vfuncs", "factory"):
            d[k] = tuple(rest)
    return d


@pytest.mark.parametrize("factory", refgst.FACTORIES)
def test_shell_declares_what_the_reference_declares(factory):
    ref, sh = parse(GOLDEN["describe"][factory]), parse(refgst.shell().describe(factory))
    assert sh["factory"] == ref["factory"]                     # name and GST_RANK_NONE
    assert sh["pad"] == ref["pad"]                             # src / sink, always, identical caps strings
    assert sh["property"] == ref["property"], (set(sh["property"]) ^ set(ref["property"]))
    assert sh["signal"] == ref["signal"]
    assert sh["vfuncs"] == ref["vfuncs"]


def property_round_trip(h, factory):
    """*_init() values, then g_object_set / g_object_get of every int property over in- and out-of-range values, then the
    boxed image-to-overlay: [(step, name, value, answer), ..] in call order."""
    e = h.element(factory)
    names = [ln.split("|")[1] for ln in h.describe(factory).split("\n") if ln.startswith("property|") and "GstStructure" not in ln]
    out = [("init", n, None, e.get(n)) for n in names]
    for n in names:
        for v in (0, 1, 3, 160, 640, 30000, 300000, -1, 10 ** 7):
            out.append(("set", n, v, e.set(n, v)))             # GLib range validation
            out.append(("get", n, v, e.get(n)))
    if factory != "nubotracker":                                # image-to-overlay: boxed GstStructure, get on a fresh element gives an empty one
        buf = C.create_string_buffer(4096)
        st = h.L.mh_get_structure(e.e, b"image-to-overlay")
        h.L.mh_st_to_string(st, buf, 4096)
        h.L.mh_st_free(st)
        out.append(("overlay", "fresh", None, buf.value.decode()))
        st = h.structure("image_to_overlay", [("offsetXPercent", "double", 0.1), ("offsetYPercent", "double", 0.2), ("widthPercent", "double", 1.0),
                                              ("heightPercent", "double", 1.0), ("url", "string", "/nonexistent.png")])
        out.append(("overlay", "set", None, h.L.mh_set_structure(e.e, b"image-to-overlay", st)))
        h.L.mh_st_free(st)
        st = h.L.mh_get_structure(e.e, b"image-to-overlay")
        h.L.mh_st_to_string(st, buf, 4096)
        h.L.mh_st_free(st)
        out.append(("overlay", "get", None, buf.value.decode()))
    e.close()
    return [list(step) for step in out]


@pytest.mark.parametrize("factory", refgst.FACTORIES)
def test_shell_property_round_trip_like_the_reference(factory):
    got, exp = property_round_trip(refgst.shell(), factory), GOLDEN["round_trip"][factory]
    assert len(got) == len(exp)
    for g, x in zip(got, exp):
        assert g == x, (g, x)
    if factory != "nubotracker":
        assert got[-3][3] == "image_to_overlay;" and "url=(string)/nonexistent.png" in got[-1][3]


def forwarded_event_counts(h):
    """Downstream events an element pushes after one custom face message and one non-custom event, per factory."""
    counts = {}
    for factory in refgst.FACTORIES:
        e = h.element(factory)
        e.send_event(h.faces_message([(1, 2, 3, 4)]))
        e.send_event(h.structure("eos-like"), downstream_custom=False)
        counts[factory] = h.L.mh_pushed_count(e.e)
        e.close()
    return counts


def test_custom_events_are_forwarded_like_the_reference():
    """kmseyedetect.cpp:192-218 hands every sink event on through gst_pad_event_default; the face element keeps custom
    downstream events to itself (kmsfacedetect.cpp:251-280); ear and tracker do not override sink_event."""
    assert forwarded_event_counts(refgst.shell()) == GOLDEN["custom_events"]
