#!/usr/bin/env python3
"""Records what the reference NUBOMEDIA-VCA elements answered in the tests that compare this repository with them, so
that those tests run from this repository alone:

  ref_elements.json      tests/test_gst_shells_cpu.py, tests/test_ref_elements_cpu.py, tests/test_ref_glue.py (no GPU)
  ref_elements_gpu.json  tests/test_gst_shells_gpu.py and tools/fuzz_ref_elements.py (needs a CUDA device)

The reference's element sources are not part of this repository (oracle/build_ref.py compiles them where they are
present).  The answers were therefore taken from this repository's GStreamer shells, host functions and
tests/element_ref.py at commit 00d7895, whose tests compared each of them, call for call, with the reference's own
elements and helper functions compiled by oracle/build_ref.py.  One exception: after a reference element threw (an ROI
outside the image, which the shells clamp instead), the old fuzz run compared nothing more of that sequence; the recorded
sequences hold the shell's answers there.  Re-recording from a later tree would pin that tree
instead of the reference: only re-record when a test's inputs change, and from a tree that still answers as the
reference did.

  python tests/golden/make_ref_golden.py            # -> tests/golden/ref_elements.json
  python tests/golden/make_ref_golden.py --gpu      # -> tests/golden/ref_elements_gpu.json
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "nubomedia-vca_b200", "python"),
                os.path.join(ROOT, "tools")]
CASCADE_DIR = os.path.join(ROOT, "nubomedia-vca_b200", "cascades")
FUZZ_SEED, FUZZ_SEQUENCES = 3, 40


def describe_as_compared(text):
    """The lines of mh_describe the tests compare, property lines cut to name|type|min|max|default|flags."""
    out = []
    for line in text.strip().split("\n"):
        k = line.split("|", 1)[0]
        if k == "property":
            out.append("|".join(line.split("|")[:7]))
        elif k in ("factory", "pad", "signal", "vfuncs"):
            out.append(line)
    return "\n".join(out) + "\n"


def record_cpu():
    import refgst
    import test_gst_shells_cpu as shells
    import test_ref_elements_cpu as elements
    import test_ref_glue as glue

    S = refgst.shell()
    g = {"describe": {f: describe_as_compared(S.describe(f)) for f in refgst.FACTORIES},
         "round_trip": {f: shells.property_round_trip(S, f) for f in refgst.FACTORIES},
         "custom_events": shells.forwarded_event_counts(S), "out_of_range": {}}
    for f in refgst.FACTORIES:
        some = "set_threshold" if f == "nubotracker" else "multi-scale-factor"
        e, w = S.element(f), S.warnings()
        g["out_of_range"][f] = {"property": some, "value": 10 ** 6, "accepted": e.set(some, 10 ** 6), "warnings": S.warnings() - w}
        e.close()
    with tempfile.TemporaryDirectory() as d:
        cdir = elements.make_cascade_dir(d, CASCADE_DIR)
        g["face_restatement"] = elements.face_restatement(cdir)
        g["feature_restatement"] = {k: elements.feature_restatement(cdir, k) for k in elements.FEATURES}
        g["ear_restatement"] = elements.ear_restatement(cdir)
    zero = {"shrunk": 0, "kept": 0, "merged": 0}
    g["glue"] = {"track_faces": glue.digests(glue.track_faces_answers()),
                 "merge_eyes_current_frame": glue.digests(glue.merge_eyes_current_frame_answers(dict(zero))),
                 **{name: glue.digests(glue.merge_consecutive_answers(k, dict(zero))) for k, name in glue.KINDS.items()},
                 "eye_to_global": glue.digests(glue.eye_to_global_answers()),
                 "join_objects": glue.digests(glue.join_objects_answers(dict(zero)))}
    return g


def record_gpu():
    import fuzz_ref_elements as fuzz
    import nubovca as nv
    import test_gst_shells_gpu as shells_gpu

    if nv.device_count() < 1:                # without a device the shells pass buffers through untouched
        raise SystemExit("--gpu needs a CUDA device")
    g = {"config1": shells_gpu.config1_run(CASCADE_DIR)}
    assert all(len(x["events"]) == 1 for x in g["config1"]) and sum(len(x["events"][0][2]) for x in g["config1"]) >= 8
    _, _, seqs = fuzz.run(FUZZ_SEQUENCES, FUZZ_SEED, [fuzz.ShellTarget])
    g["fuzz"] = {"seed": FUZZ_SEED, "sequences": seqs}
    return g


def main():
    gpu = "--gpu" in sys.argv[1:]
    g = record_gpu() if gpu else record_cpu()
    path = os.path.join(HERE, "ref_elements_gpu.json" if gpu else "ref_elements.json")
    with open(path, "w") as f:
        json.dump(g, f, separators=(",", ":"))
        f.write("\n")
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
