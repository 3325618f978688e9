"""ctypes driver of tests/mock_gst/harness.cpp.  The same harness is linked into two libraries:

  * oracle/_ref/libnubo_ref_elements.so — the REFERENCE's own element sources compiled unmodified against the mock
    GStreamer and the oracle-backed OpenCV stand-in (oracle/build_ref.py) — `ref()`;
  * nubomedia-vca_b200/lib/libnubovca_gst_mock.so — this repo's GStreamer shells compiled against the same mock
    (nubomedia-vca_b200/gst/, built by the Makefile) — `shell()`.

Test infrastructure only."""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

FACTORIES = ["nubofacedetector", "nuboeyedetector", "nubomouthdetector", "nubonosedetector", "nuboeardetector", "nubotracker"]
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def load_golden(name):
    """What the reference elements answered in a test, as tests/golden/make_ref_golden.py recorded it."""
    with open(os.path.join(GOLDEN_DIR, name)) as f:
        return json.load(f)


GOLDEN = load_golden("ref_elements.json") if os.path.exists(os.path.join(GOLDEN_DIR, "ref_elements.json")) else {}


def plain(x):
    """x as it reads back from JSON (tuples become lists)."""
    return json.loads(json.dumps(x))


def frame_digest(frame):
    """First 16 hex digits of the SHA-256 of a frame's pixels: how the recorded answers hold the frames an element drew into."""
    return hashlib.sha256(np.ascontiguousarray(frame).tobytes()).hexdigest()[:16]
FMT = {"BGR": 0, "BGRA": 1, "I420": 2, "NV12": 3}


class MhRect(C.Structure):
    _fields_ = [("field", C.c_char * 16), ("name", C.c_char * 16), ("type", C.c_char * 16),
                ("x", C.c_uint), ("y", C.c_uint), ("width", C.c_uint), ("height", C.c_uint)]


class MhDraw(C.Structure):
    _fields_ = [("kind", C.c_int), ("x0", C.c_int), ("y0", C.c_int), ("x1", C.c_int), ("y1", C.c_int), ("color", C.c_double * 4),
                ("thickness", C.c_int), ("line_type", C.c_int), ("shift", C.c_int), ("offset", C.c_longlong)]


class Harness:
    def __init__(self, path, is_ref):
        self.path, self.is_ref = path, is_ref
        L = self.L = C.CDLL(path)
        L.mh_element_new.restype = C.c_void_p
        L.mh_element_new.argtypes = [C.c_char_p]
        L.mh_element_free.argtypes = [C.c_void_p]
        L.mh_set_long.argtypes = [C.c_void_p, C.c_char_p, C.c_long]
        L.mh_get_long.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_long)]
        L.mh_set_structure.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p]
        L.mh_get_structure.restype = C.c_void_p
        L.mh_get_structure.argtypes = [C.c_void_p, C.c_char_p]
        L.mh_describe.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        L.mh_st_new.restype = C.c_void_p
        L.mh_st_new.argtypes = [C.c_char_p]
        L.mh_st_free.argtypes = [C.c_void_p]
        L.mh_st_set_uint.argtypes = [C.c_void_p, C.c_char_p, C.c_uint]
        L.mh_st_set_int.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.mh_st_set_uint64.argtypes = [C.c_void_p, C.c_char_p, C.c_ulonglong]
        L.mh_st_set_double.argtypes = [C.c_void_p, C.c_char_p, C.c_double]
        L.mh_st_set_string.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
        L.mh_st_set_struct.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p]
        L.mh_st_to_string.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.mh_send_event.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.mh_transform_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_ulonglong, C.c_int]
        L.mh_pushed_count.argtypes = [C.c_void_p]
        L.mh_clear_pushed.argtypes = [C.c_void_p]
        L.mh_pushed_to_string.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_int]
        L.mh_pushed_rects.argtypes = [C.c_void_p, C.c_int, C.POINTER(MhRect), C.c_int, C.POINTER(C.c_ulonglong), C.c_char_p]
        L.mh_emissions.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.mh_clear_emissions.argtypes = [C.c_void_p]
        L.mh_set_time.argtypes = [C.c_double, C.c_double]
        if is_ref:
            L.mh_register_cascade.argtypes = [C.c_char_p, C.c_void_p]
            L.mh_get_draws.argtypes = [C.c_void_p, C.POINTER(MhDraw), C.c_int]
            self._cascades = {}

    def describe(self, factory):
        buf = C.create_string_buffer(1 << 16)
        n = self.L.mh_describe(factory.encode(), buf, len(buf))
        if n < 0:
            raise KeyError(factory)
        return buf.value.decode()

    def set_time(self, clock_ms, wall_ms):
        self.L.mh_set_time(float(clock_ms), float(wall_ms))

    def warnings(self):
        return self.L.mh_warning_count()

    # reference build only: CascadeClassifier::load("/usr/share/opencv/haarcascades/<basename>") resolves to this model
    def register_cascade(self, basename, ocascade):
        assert self.is_ref
        # Keeps the arrays behind the C struct alive FOR THE LIFE OF THE PROCESS: the reference's nose element holds its
        # cascades in file-static objects loaded by the first instance only (kmsnosedetect.cpp:151-152,1049-1051), so a
        # model registered once may be referenced for ever.  For the same reason a test process must not re-register
        # haarcascade_frontalface_alt.xml / haarcascade_mcs_nose.xml with other content and expect the nose element to follow.
        self._keep = getattr(self, "_keep", [])
        self._keep.append(ocascade)
        self._cascades[basename] = ocascade
        self.L.mh_register_cascade(basename.encode(), C.addressof(ocascade.c) if ocascade is not None else None)

    def register_cascade_dir(self, cdir):
        import oracle as O
        for f in sorted(os.listdir(cdir)):
            if f.endswith(".xml"):
                self.register_cascade(f, O.Cascade(os.path.join(cdir, f)))

    def structure(self, name, fields=()):
        """fields: (name, kind, value) with kind in uint / int / uint64 / double / string / struct (value: a handle, copied)"""
        s = self.L.mh_st_new(name.encode())
        for fn, kind, v in fields:
            if kind == "string":
                self.L.mh_st_set_string(s, fn.encode(), v.encode())
            elif kind == "struct":
                self.L.mh_st_set_struct(s, fn.encode(), v)
                self.L.mh_st_free(v)
            else:
                getattr(self.L, "mh_st_set_" + kind)(s, fn.encode(), v)
        return s

    def faces_message(self, rects, pts=0, timestamp=True, type_="face", name="face"):
        """The downstream custom event of the face element (kmsfacedetect.cpp:196-226): message{timestamp{pts}, "0"{face..}, ..}"""
        f = []
        if timestamp:
            f.append(("timestamp", "struct", self.structure("time", [("pts", "uint64", pts)])))
        for i, (x, y, w, h) in enumerate(rects):
            f.append((str(i), "struct", self.structure(name, [("type", "string", type_), ("x", "uint", x), ("y", "uint", y),
                                                             ("width", "uint", w), ("height", "uint", h)])))
        return self.structure("message", f)

    def motion_message(self, pts=0, timestamp=True, grid="1"):
        f = []
        if timestamp:
            f.append(("timestamp", "struct", self.structure("time", [("pts", "uint64", pts)])))
        # "type" is given so that the eye / nose elements, which read it from every sub-structure into an uninitialised
        # pointer (kmseyedetect.cpp:703-705), stay defined when a test hands them a motion message
        f.append(("motion", "struct", self.structure("motion", [("type", "string", "motion"), ("grid", "string", grid)])))
        return self.structure("message", f)

    def element(self, factory):
        return Element(self, factory)


class Element:
    def __init__(self, h, factory):
        self.h, self.factory = h, factory
        self.e = h.L.mh_element_new(factory.encode())
        if not self.e:
            raise KeyError(f"no element factory {factory!r} in {h.path}")

    def close(self):
        if self.e:
            self.h.L.mh_element_free(self.e)
            self.e = None

    def set(self, prop, value):
        """g_object_set; returns False when GLib would have rejected the value (out of range) or the name"""
        return self.h.L.mh_set_long(self.e, prop.encode(), int(value)) == 0

    def get(self, prop):
        v = C.c_long()
        rc = self.h.L.mh_get_long(self.e, prop.encode(), C.byref(v))
        if rc != 0:
            raise KeyError(prop)
        return v.value

    def send_event(self, st, downstream_custom=True):
        return self.h.L.mh_send_event(self.e, st, 1 if downstream_custom else 0)

    def process(self, frame, pts_ns=0, fmt="BGR"):
        """transform_frame_ip on `frame` (numpy, modified in place when the element draws).  Returns
        (threw, [pushed events as (structure name, pts, [(field, name, type, x, y, w, h), ..])], [(signal, payload), ..])."""
        L = self.h.L
        L.mh_clear_pushed(self.e)
        L.mh_clear_emissions(self.e)
        if self.h.is_ref:
            L.mh_clear_draws()
        if fmt in ("BGR", "BGRA"):
            H, W = frame.shape[:2]
            stride = frame.strides[0]
        else:
            W = frame.shape[1]
            H = frame.shape[0] * 2 // 3
            stride = W
        assert frame.flags["C_CONTIGUOUS"] or frame.strides[1] == frame.shape[2]
        threw = L.mh_transform_frame(self.e, frame.ctypes.data_as(C.c_void_p), W, H, stride, int(pts_ns), FMT[fmt])
        if threw < 0:
            raise RuntimeError("element has no transform_frame_ip")
        events = []
        arr = (MhRect * 4096)()
        for i in range(L.mh_pushed_count(self.e)):
            pts = C.c_ulonglong()
            name = C.create_string_buffer(16)
            n = L.mh_pushed_rects(self.e, i, arr, 4096, C.byref(pts), name)
            events.append((name.value.decode(), pts.value,
                           [(r.field.decode(), r.name.decode(), r.type.decode(), r.x, r.y, r.width, r.height) for r in arr[:n]]))
        buf = C.create_string_buffer(1 << 18)
        L.mh_emissions(self.e, buf, len(buf))
        sig = [tuple(line.split("\t", 1)) for line in buf.value.decode().split("\n") if line]
        return bool(threw), events, sig

    def pushed_strings(self):
        out = []
        buf = C.create_string_buffer(1 << 18)
        for i in range(self.h.L.mh_pushed_count(self.e)):
            self.h.L.mh_pushed_to_string(self.e, i, buf, len(buf))
            out.append(buf.value.decode())
        return out

    def draws(self, frame):
        """Reference build: the cvRectangle / cv::circle calls of the last process(), for replay with cv2."""
        arr = (MhDraw * 1024)()
        n = self.h.L.mh_get_draws(frame.ctypes.data_as(C.c_void_p), arr, 1024)
        return [dict(kind="rectangle" if d.kind == 0 else "circle", p0=(d.x0, d.y0), p1=(d.x1, d.y1), color=tuple(d.color),
                     thickness=d.thickness, line_type=d.line_type, shift=d.shift, offset=d.offset) for d in arr[:n]]


def replay_draws(frame, draws):
    """Apply recorded drawing calls with the real OpenCV (cv2 4.13), as the reference's cvRectangle / cv::circle would."""
    import cv2
    for d in draws:
        assert d["offset"] == 0, "drawing into something else than the frame"
        col = tuple(d["color"][:frame.shape[2]]) if frame.ndim == 3 else d["color"][0]
        if d["kind"] == "rectangle":
            cv2.rectangle(frame, d["p0"], d["p1"], col, d["thickness"], d["line_type"], d["shift"])
        else:
            cv2.circle(frame, d["p0"], d["p1"][0], col, d["thickness"], d["line_type"], d["shift"])
    return frame


_ref = None
_shell = None


def ref():
    """The reference elements library (built on demand where /root/reference exists; prebuilt elsewhere)."""
    global _ref
    if _ref is None:
        import build_ref
        _ref = Harness(build_ref.build(), True)
    return _ref


def shell():
    global _shell
    if _shell is None:
        p = os.path.join(ROOT, "nubomedia-vca_b200", "lib", "libnubovca_gst_mock.so")
        if not os.path.exists(p):
            raise FileNotFoundError(p + " (run __graft_entry__.build())")
        _shell = Harness(p, False)
    return _shell


def ref_glue():
    """ctypes handle on the static-helper exports of the reference library (oracle/refbuild/wrap_*.cpp)."""
    L = ref().L
    ip = C.POINTER(C.c_int)
    L.ref_faces_new.restype = C.c_void_p
    L.ref_faces_free.argtypes = [C.c_void_p]
    L.ref_faces_clear.argtypes = [C.c_void_p]
    L.ref_faces_track.argtypes = [C.c_void_p, ip, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.ref_faces_get.argtypes = [C.c_void_p, ip, ip, C.c_int]
    L.ref_eye_contain_bb.argtypes = [C.c_int, C.c_int, ip]
    L.ref_eye_merge_current_frame.argtypes = [ip, ip, C.c_int, C.c_int, ip, C.c_int, C.c_int, C.c_int, C.c_int]
    L.ref_eye_merge_consecutive.argtypes = [ip, C.c_int, ip, C.c_int, ip, C.c_int, C.c_int, ip, C.c_int]
    L.ref_eye_to_global.argtypes = [ip, C.c_int, ip, C.c_int]
    L.ref_mouth_merge_consecutive.argtypes = [ip, C.c_int, ip, C.c_int, ip, C.c_int, ip, C.c_int]
    L.ref_nose_merge_consecutive.argtypes = [ip, C.c_int, ip, C.c_int, ip, C.c_int, ip, C.c_int]
    L.ref_trk_calc_dist.restype = C.c_float
    L.ref_trk_calc_dist.argtypes = [ip, ip]
    L.ref_trk_merge.argtypes = [ip, ip, ip]
    L.ref_trk_join_objects.argtypes = [C.c_void_p, ip, C.c_int, C.c_int]
    return L
