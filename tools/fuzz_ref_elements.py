"""Randomised element-level parity run against what the REFERENCE'S OWN ELEMENTS (the six kms*detect.cpp /
gstnubotracker.cpp sources compiled unmodified by oracle/build_ref.py, computing through the CPU oracle) answered on the
same sequences, recorded in tests/golden/ref_elements_gpu.json:

  target "mirror": the nv_element C ABI of libnubovca.so (CUDA),
  target "shell":  this repo's GStreamer shells (nubomedia-vca_b200/gst/) built against the mock GStreamer, driven through
                   the same harness calls as the reference elements.

Random frame sizes, face layouts, stand-in feature models, property values (including out-of-range ones, view-*,
detect-event with random upstream event streams — face messages, motion messages, foreign messages, messages without a
timestamp —, activate-events / events-ms under an injected wall clock), frame sequences with noise and empty frames, all
drawn from the recorded seed.  Compared per frame: the pushed downstream event (structure name, timestamp, every
sub-structure field by field), the emitted signal payload, and a digest of the frame's pixels after the element drew into
it.  Needs a CUDA device.
Usage: python tools/fuzz_ref_elements.py [mirror|shell|both]"""
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "nubomedia-vca_b200", "python"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import nubovca as nv  # noqa: E402
import refgst  # noqa: E402
from cascade_xml_util import permissive_cascade  # noqa: E402
from nubovca import synth  # noqa: E402

SRC = os.path.join(ROOT, "nubomedia-vca_b200", "cascades")
STANDINS = {"haarcascade_mcs_righteye.xml": (18, 12), "haarcascade_mcs_lefteye.xml": (18, 12), "haarcascade_mcs_mouth.xml": (25, 15),
            "haarcascade_mcs_nose.xml": (18, 15), "haarcascade_mcs_rightear.xml": (12, 20), "haarcascade_mcs_leftear.xml": (12, 20)}
VIEW = {"nubofacedetector": "view-faces", "nuboeyedetector": "view-eyes", "nubomouthdetector": "view-mouths",
        "nubonosedetector": "view-noses", "nuboeardetector": "view-ears", "nubotracker": "set_visual_mode"}


class MirrorTarget:
    name = "mirror"

    def __init__(self, factory, cdir):
        self.e = nv.Element(factory, 0, cdir)

    def set(self, prop, v):
        try:
            self.e.set(prop, v)
            return True
        except nv.NuboError:
            return False

    def get(self, prop):
        return self.e.get(prop)

    def event(self, kind, faces, ts):
        f = [("timestamp", True, None, (0, 0, 0, 0))] if ts else []
        if kind == "faces":
            f += [(str(i), True, "face", r) for i, r in enumerate(faces)]
        elif kind == "motion":
            f.append(("motion", True, "motion", (0, 0, 0, 0)))
        else:
            f.append(("x", True, "thing", (0, 0, 0, 0)))
        self.e.push_message(f)

    def process(self, frame, pts_ns, wall_ms):
        nv._lib.nv_debug_set_wall_clock_ms(float(wall_ms))
        msg, pushed, sig = self.e.process(frame, pts_ns=pts_ns)
        return (msg if pushed else None), sig

    def close(self):
        self.e.close()


class ShellTarget:
    name = "shell"

    def __init__(self, factory, cdir):
        self.S = refgst.shell()
        os.environ["NUBOVCA_CASCADE_DIR"] = cdir
        self.factory = factory
        self.e = self.S.element(factory)

    def set(self, prop, v):
        return self.e.set(prop, v)

    def get(self, prop):
        return self.e.get(prop)

    def event(self, kind, faces, ts):
        S = self.S
        if kind == "faces":
            st = S.faces_message([tuple(int(v) for v in f) for f in faces], timestamp=ts)
        elif kind == "motion":
            st = S.motion_message(timestamp=ts)
        else:
            st = S.structure("message", ([("timestamp", "struct", S.structure("time", [("pts", "uint64", 0)]))] if ts else []) +
                             [("x", "struct", S.structure("thing", [("type", "string", "thing")]))])
        self.e.send_event(st)

    def process(self, frame, pts_ns, wall_ms):
        self.S.set_time(pts_ns / 1e6, wall_ms)
        nv._lib.nv_debug_set_wall_clock_ms(float(wall_ms))
        threw, events, sig = self.e.process(frame, pts_ns=pts_ns, fmt="BGRA" if self.factory == "nubotracker" else "BGR")
        assert not threw
        assert len(events) <= 1
        msg = None
        if events:
            msg = events[0]                           # (structure name, timestamp.pts or ~0, rows with their field names)
        return msg, (sig[0][1] if sig else None)

    def close(self):
        self.e.close()


def run(nseq, seed, targets, expected=None):
    """nseq random sequences from `seed` through `targets`.  With `expected` (the recorded sequences) every target is compared
    with it; without, the first target's answers are returned as the record."""
    rng = np.random.default_rng(seed)
    t0 = time.time()
    stats = dict(sequences=0, frames=0, rects=0, signals=0, drawn_frames=0, events_sent=0, rejected_sets=0, mismatches=0)
    record = []
    # ONE set of stand-in models per process: the reference's nose element keeps its cascades in file-static objects that
    # only the first instance loads (kmsnosedetect.cpp:151-152,1049-1051), so the models cannot change between sequences
    d = tempfile.mkdtemp(prefix="nubovca_fzr_")
    shutil.copy(os.path.join(SRC, "haarcascade_frontalface_alt.xml"), d)
    shutil.copy(os.path.join(SRC, "haarcascade_frontalface_alt.xml"), os.path.join(d, "haarcascade_profileface.xml"))
    for name, (w, h) in STANDINS.items():
        permissive_cascade(os.path.join(d, name), np.random.default_rng(int(rng.integers(1 << 30))), w, h,
                           bias=float(rng.choice([0.2, 0.35, 0.5])))
    for q in range(nseq):
        els = []
        exp = expected[q] if expected is not None else None
        rec = {"sets": [], "gets": [], "frames": []}
        record.append(rec)
        try:
            factory = refgst.FACTORIES[int(rng.integers(6))]
            trk = factory == "nubotracker"
            W, H = [(640, 480), (1280, 720), (960, 540), (800, 600), (320, 240)][int(rng.integers(5))]
            if trk:
                frames = synth.tracker_sequence(W, H, int(rng.integers(3, 8)), seed=int(rng.integers(1 << 30)), noise=int(rng.choice([0, 0, 12, 25])))
            else:
                base = synth.frame(W, H, int(rng.integers(1, 4)), int(rng.integers(1 << 30)), smin=0.3, smax=0.7)
                frames = []
                for i in range(int(rng.integers(3, 9))):
                    if rng.random() < 0.2:
                        frames.append(np.full((H, W, 3), 90, np.uint8))
                    else:
                        frames.append(np.clip(base.astype(np.int16) + rng.integers(-3, 4, base.shape, dtype=np.int16), 0, 255).astype(np.uint8))
            els = [t(factory, d) for t in targets]
            props = {}
            if trk:
                props = {"set_threshold": int(rng.choice([5, 20, 60, 300])), "set_min_area": int(rng.choice([0, 50, 500])),
                         "set_max_area": int(rng.choice([2000, 30000, 300000])), "set_distance": int(rng.choice([0, 35, 200, 5000])),
                         "set_visual_mode": int(rng.choice([0, 1, 3]))}
            else:
                props = {"process-x-every-4-frames": int(rng.choice([0, 1, 2, 3, 4, 7])), "multi-scale-factor": int(rng.choice([10, 25, 40, 60])),
                         "width-to-process": int(rng.choice([160, 320, 640, 800] if factory == "nubofacedetector" else [320, 640, 480, 200])),
                         VIEW[factory]: int(rng.choice([0, 1, 1, 2])), "detect-event": int(rng.choice([0, 0, 1]))}
                if factory == "nubofacedetector":
                    props["track-threshold"] = int(rng.choice([5, 40, 100]))
            props["activate-events"] = int(rng.choice([0, 1, 1]))
            props["events-ms"] = int(rng.choice([0, 50, 1000]))
            wall = 1e12
            nv._lib.nv_debug_set_wall_clock_ms(wall)
            for k, v in props.items():
                oks = [e.set(k, v) for e in els]
                assert len(set(oks)) == 1, (factory, k, v, oks)
                rec["sets"].append(oks[0])
                stats["rejected_sets"] += not oks[0]
            for k in props:
                vals = [e.get(k) for e in els]
                assert len(set(vals)) == 1, (factory, k, vals)
                rec["gets"].append(vals[0])
            if exp is not None:
                assert (rec["sets"], rec["gets"]) == (exp["sets"], exp["gets"]), (factory, props, rec, exp)
            for i, f in enumerate(frames):
                pts = i * 33_333_000
                wall += float(rng.choice([5, 40, 700]))
                if not trk and props.get("detect-event") == 1:
                    for _ in range(int(rng.choice([0, 1, 1, 2]))):
                        kind = str(rng.choice(["faces", "faces", "motion", "other"]))
                        ts = bool(rng.random() < 0.85)
                        faces = [(int(rng.integers(0, W - 80)), int(rng.integers(0, H - 80)), int(s), int(s)) for s in rng.integers(40, min(H, 260), int(rng.integers(0, 3)))]
                        for e in els:
                            e.event(kind, faces, ts)
                        stats["events_sent"] += 1
                outs = []
                for e in els:
                    g = f.copy()
                    msg, s = e.process(g, pts, wall)
                    outs.append((e, refgst.plain(msg), s, refgst.frame_digest(g), int((g != f).any(axis=-1).sum())))
                if exp is None:
                    _, event, sig, pixels, drawn = outs[0]
                    rec["frames"].append({"event": event, "signal": sig, "pixels": pixels, "drawn": drawn})
                    continue
                x = exp["frames"][i]
                exp_event, exp_sig = x["event"], x["signal"]
                exp_msg = None
                if exp_event is not None:
                    name, epts, rows = exp_event
                    assert [r[0] for r in rows] == [str(j) for j in range(len(rows))]
                    assert (name, epts) == (("noses", 2 ** 64 - 1) if factory == "nubonosedetector" else ("message", pts))
                    exp_msg = [r[1:] for r in rows]
                stats["frames"] += 1
                stats["rects"] += len(exp_msg or [])
                stats["signals"] += exp_sig is not None
                stats["drawn_frames"] += bool(x["drawn"])
                for e, msg, s, pixels, drawn in outs:
                    if e.name == "mirror" and (trk or factory == "nuboeardetector"):
                        msg = None                   # the mirror reports the message it built; neither element pushes one
                    if msg != (exp_event if e.name == "shell" else exp_msg) or s != exp_sig or pixels != x["pixels"]:
                        stats["mismatches"] += 1
                        print("MISMATCH", e.name, factory, (W, H), props, "sequence", q, "frame", i, "\n  msg", msg, "\n  exp", exp_msg,
                              "\n  sig", s, "\n  exp", exp_sig, "\n  drawn pixels", drawn, "expected", x["drawn"], flush=True)
                        raise StopIteration
            stats["sequences"] += 1
        except StopIteration:
            pass
        finally:
            for e in els:
                e.close()
    shutil.rmtree(d, ignore_errors=True)
    nv._lib.nv_debug_set_wall_clock_ms(-1.0)
    return stats, time.time() - t0, record


if __name__ == "__main__":
    which = sys.argv[1] if len(sys.argv) > 1 else "both"
    targets = {"mirror": [MirrorTarget], "shell": [ShellTarget], "both": [MirrorTarget, ShellTarget]}[which]
    golden = refgst.load_golden("ref_elements_gpu.json")["fuzz"]
    stats, dt, _ = run(len(golden["sequences"]), golden["seed"], targets, golden["sequences"])
    print(f"fuzz_ref_elements[{which}]: " + ", ".join(f"{v} {k}" for k, v in stats.items()) + f", seed {golden['seed']}, {dt:.0f} s")
    sys.exit(1 if stats["mismatches"] or stats["sequences"] < len(golden["sequences"]) else 0)
