"""GPU: the GStreamer shells (mock build) and the nv_element mirrors against what the REFERENCE'S OWN ELEMENTS (compiled by
oracle/build_ref.py) answered on the same buffers, properties and upstream events (tests/golden/ref_elements_gpu.json):
pushed downstream events (field by field), signal payloads and drawn pixels.  BASELINE config 1 literally (640x480 BGR,
element defaults, haarcascade_frontalface_alt) plus the randomised sequences of tools/fuzz_ref_elements.py over all six
elements."""
import os
import subprocess
import sys

import numpy as np
import pytest

import refgst
from nubovca import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def config1_run(cascade_dir):
    """videotestsrc-like stream ! nubofacedetector ! fakesink with the element's defaults and view-faces 1, on the shell:
    per frame the pushed events, the signals and a digest of the drawn frame."""
    os.environ["NUBOVCA_CASCADE_DIR"] = cascade_dir
    s = refgst.shell().element("nubofacedetector")
    assert s.set("view-faces", 1)
    base = synth.frame(640, 480, 4, 1)
    rng = np.random.default_rng(5)
    out = []
    for i in range(12):
        f = np.clip(base.astype(np.int16) + rng.integers(-3, 4, base.shape, dtype=np.int16), 0, 255).astype(np.uint8)
        if i in (6, 7, 8):
            f[:] = 90                                                         # faces leave: the two-empty-frames rule
        b = f.copy()
        threw, ev, sig = s.process(b, pts_ns=i * 33_333_333)
        out.append({"threw": threw, "events": ev, "signals": sig, "pixels": refgst.frame_digest(b),
                    "drawn": int((b != f).any(axis=-1).sum())})
    s.close()
    return refgst.plain(out)


def test_config1_shell_equals_reference_element(cascade_dir, monkeypatch):
    monkeypatch.setenv("NUBOVCA_CASCADE_DIR", cascade_dir)
    exp = refgst.load_golden("ref_elements_gpu.json")["config1"]
    got = config1_run(cascade_dir)
    assert len(got) == len(exp)
    for i, (g, x) in enumerate(zip(got, exp)):
        assert not g["threw"] and g == x, (i, g, x)
    assert sum(len(x["events"][0][2]) for x in exp) >= 8


def test_randomised_elements_against_the_reference_elements():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_ref_elements.py"), "both"], capture_output=True,
                       text=True, timeout=600)
    tail = r.stdout[-3000:] + r.stderr[-3000:]
    assert r.returncode == 0, tail
    assert " 0 mismatches" in r.stdout, tail
