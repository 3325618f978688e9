"""ctypes binding of libnubovca.so (include/nubovca.h) for tests and bench.py.

The product is the C-ABI library; this module only marshals numpy arrays across it.  There is no
CPU implementation behind it: if the shared library is missing the import fails, and without a
CUDA device every compute call raises NuboError(NV_ERR_NO_DEVICE).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
LIB_PATH = os.environ.get("NUBOVCA_LIB") or os.path.join(_PKG, "lib", "libnubovca.so")   # override: kernel A/B experiments
CASCADE_DIR = os.path.join(_PKG, "cascades")

NV_OK = 0
NV_ERR_NO_DEVICE = -7
DEPTH_PASS, DEPTH_VARREJ, DEPTH_SKIPPED = 1, -100, -32768

if not os.path.exists(LIB_PATH):
    raise ImportError(f"{LIB_PATH} is missing: build it with `make -C {_PKG}` (or __graft_entry__.build()); "
                      "nubovca has no CPU fallback")

_lib = C.CDLL(LIB_PATH)


class Rect(C.Structure):
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("width", C.c_int), ("height", C.c_int)]


class CascadeInfo(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("win_w", "win_h", "nstages", "nstumps", "nfeatures", "n3rect", "order_free_sums",
                                         "general", "has_tilted", "nnodes", "lbp")]


class DetectParams(C.Structure):
    _fields_ = [("scale_factor", C.c_double), ("min_neighbors", C.c_int), ("flags", C.c_int), ("min_w", C.c_int),
                ("min_h", C.c_int), ("max_w", C.c_int), ("max_h", C.c_int)]


class FaceParams(C.Structure):
    _fields_ = [("width_to_process", C.c_int), ("scale_factor", C.c_double), ("min_neighbors", C.c_int),
                ("min_w", C.c_int), ("min_h", C.c_int)]


class YuvFrame(C.Structure):
    _fields_ = [("format", C.c_int), ("width", C.c_int), ("height", C.c_int), ("plane", C.c_void_p * 3),
                ("stride", C.c_int * 3), ("on_device", C.c_int)]


FMT_BGR, FMT_I420, FMT_NV12, FMT_NV21 = 0, 1, 2, 3
_FMT = {"I420": FMT_I420, "YV12": FMT_I420, "NV12": FMT_NV12, "NV21": FMT_NV21}


class TrackerParams(C.Structure):
    _fields_ = [("threshold", C.c_int), ("min_area", C.c_int), ("max_area", C.c_long), ("distance", C.c_int)]


class EventField(C.Structure):
    _fields_ = [("name", C.c_char_p), ("is_structure", C.c_int), ("type", C.c_char_p), ("rect", Rect)]


class Shape(C.Structure):
    _fields_ = [("kind", C.c_int), ("a", C.c_int), ("b", C.c_int), ("c", C.c_int), ("d", C.c_int),
                ("blue", C.c_ubyte), ("green", C.c_ubyte), ("red", C.c_ubyte), ("pad", C.c_ubyte)]


class LevelInfo(C.Structure):
    _fields_ = [("scale", C.c_float), ("width", C.c_int), ("height", C.c_int), ("ystep", C.c_int), ("nx", C.c_int),
                ("ny", C.c_int)]


_vp, _i, _ip = C.c_void_p, C.c_int, C.POINTER(C.c_int)
_SIGS = {
    "nv_version": (C.c_char_p, []),
    "nv_last_error": (C.c_char_p, []),
    "nv_device_count": (_i, []),
    "nv_cascade_load": (_i, [C.c_char_p, C.POINTER(_vp)]),
    "nv_cascade_get_info": (_i, [_vp, C.POINTER(CascadeInfo)]),
    "nv_cascade_free": (None, [_vp]),
    "nv_ctx_create": (_i, [_i, _i, _i, C.POINTER(_vp)]),
    "nv_ctx_destroy": (None, [_vp]),
    "nv_ctx_set_debug": (_i, [_vp, _i]),
    "nv_ctx_set_scores": (_i, [_vp, _i]),
    "nv_get_scores": (_i, [_vp, _ip, C.POINTER(C.c_double), _i, _ip]),
    "nv_detect_multiscale": (_i, [_vp, _vp, _vp, _i, _i, _i, C.POINTER(DetectParams), _vp, _i, _ip]),
    "nv_face_detect": (_i, [_vp, _vp, _vp, _i, _i, _i, C.POINTER(FaceParams), _vp, _i, _ip]),
    "nv_face_submit": (_i, [_vp, _vp, _vp, _i, _i, _i, C.POINTER(FaceParams)]),
    "nv_face_submit_device": (_i, [_vp, _vp, _vp, _i, _i, _i, C.POINTER(FaceParams)]),
    "nv_face_collect": (_i, [_vp, _vp, _i, _ip]),
    "nv_face_detect_yuv": (_i, [_vp, _vp, C.POINTER(YuvFrame), C.POINTER(FaceParams), _vp, _i, _ip]),
    "nv_face_submit_yuv": (_i, [_vp, _vp, C.POINTER(YuvFrame), C.POINTER(FaceParams)]),
    "nv_yuv2bgr": (_i, [_vp, C.POINTER(YuvFrame), _vp, _i]),
    "nv_host_alloc": (_i, [C.c_size_t, C.POINTER(_vp)]),
    "nv_host_free": (None, [_vp]),
    "nv_host_register": (_i, [_vp, C.c_size_t]),
    "nv_host_unregister": (_i, [_vp]),
    "nv_tracker_process": (_i, [_vp, _vp, _i, _i, _i, C.c_double, C.POINTER(TrackerParams), _vp, _i, _ip]),
    "nv_tracker_reset": (_i, [_vp]),
    "nv_tracker_process_yuv": (_i, [_vp, C.POINTER(YuvFrame), C.c_double, C.POINTER(TrackerParams), _vp, _i, _ip]),
    "nv_bgr2gray": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i]),
    "nv_equalize_hist": (_i, [_vp, _vp, _i, _i, _i, _vp, _i]),
    "nv_resize_linear": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i]),
    "nv_flip_horizontal": (_i, [_vp, _vp, _i, _i, _i, _vp, _i]),
    "nv_element_create": (_i, [C.c_char_p, _i, C.c_char_p, C.POINTER(_vp)]),
    "nv_element_destroy": (None, [_vp]),
    "nv_element_set_property": (_i, [_vp, C.c_char_p, C.c_long]),
    "nv_element_get_property": (_i, [_vp, C.c_char_p, C.POINTER(C.c_long)]),
    "nv_element_property_info": (_i, [_vp, _i, C.POINTER(C.c_char_p), C.POINTER(C.c_long), C.POINTER(C.c_long), C.POINTER(C.c_long)]),
    "nv_element_push_faces_event": (_i, [_vp, _vp, _i]),
    "nv_element_push_motion_event": (_i, [_vp]),
    "nv_element_push_message": (_i, [_vp, _vp, _i]),
    "nv_debug_set_wall_clock_ms": (None, [C.c_double]),
    "nv_debug_merge_eyes_current_frame": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _i, _i, _ip]),
    "nv_debug_merge_consecutive": (_i, [_i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _ip]),
    "nv_debug_eye_to_global": (_i, [_vp, _i, _vp, _i]),
    "nv_debug_join_objects": (_i, [_vp, _i, _i, C.c_long, _i, _ip]),
    "nv_element_transform_frame_ip": (_i, [_vp, _vp, _i, _i, _i, C.c_uint64, C.c_double]),
    "nv_element_transform_frame_yuv": (_i, [_vp, C.POINTER(YuvFrame), C.c_uint64, C.c_double]),
    "nv_element_get_message": (_i, [_vp, _vp, _i, _ip, _ip]),
    "nv_element_get_signal": (_i, [_vp, C.c_char_p, _i, _ip]),
    "nv_element_get_message_info": (_i, [_vp, C.c_char_p, _ip]),
    "nv_debug_track_faces": (_i, [_vp, _vp, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _ip, _ip]),
    "nv_stage_name": (C.c_char_p, [_i]),
    "nv_ctx_set_profile": (_i, [_vp, _i]),
    "nv_ctx_get_stage_times": (_i, [_vp, C.POINTER(C.c_float), _i, _ip]),
    "nv_ctx_get_tracker_kernel_ms": (_i, [_vp, C.POINTER(C.c_float)]),
    "nv_event_create": (_i, [C.POINTER(_vp)]),
    "nv_event_record": (_i, [_vp, _vp]),
    "nv_event_elapsed_ms": (_i, [_vp, _vp, C.POINTER(C.c_float)]),
    "nv_event_destroy": (None, [_vp]),
    "nv_debug_cascade_stage": (_i, [_vp, _i, _ip, C.POINTER(C.c_float)]),
    "nv_debug_cascade_stump": (_i, [_vp, _i, _ip, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "nv_debug_draw_rectangle": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "nv_debug_draw_circle": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "nv_debug_cascade_tree": (_i, [_vp, _i, _i, _ip, _ip, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "nv_debug_cascade_feature": (_i, [_vp, _i, _ip, C.POINTER(C.c_float), _ip]),
    "nv_debug_cascade_subset": (_i, [_vp, _i, _ip]),
    "nv_element_transform_frame_device": (_i, [_vp, _vp, _i, _i, _i, C.c_uint64, C.c_double]),
    "nv_draw_shapes_device": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i]),
    "nv_debug_draw_shapes_spans": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _ip]),
    "nv_debug_num_levels": (_i, [_vp]),
    "nv_debug_level_info": (_i, [_vp, _i, C.POINTER(LevelInfo)]),
    "nv_debug_get_gray": (_i, [_vp, _vp, _i, _ip, _ip]),
    "nv_debug_get_integral": (_i, [_vp, _i, _vp, _vp]),
    "nv_debug_get_tilted": (_i, [_vp, _i, _vp]),
    "nv_debug_get_depth_map": (_i, [_vp, _i, _vp]),
    "nv_debug_get_candidates": (_i, [_vp, _vp, _i, _ip]),
    "nv_debug_get_counters": (_i, [_vp, C.POINTER(C.c_longlong)]),
    "nv_detect_multiscale_batch": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, C.POINTER(DetectParams), _vp, _i, _ip]),
    "nv_face_submit_batch": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, C.POINTER(FaceParams)]),
    "nv_face_collect_batch": (_i, [_vp, _vp, _i, _ip, _ip]),
    "nv_face_detect_batch": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, C.POINTER(FaceParams), _vp, _i, _ip, _ip]),
}
BATCH_MAX = 256           # NV_BATCH_MAX
EXPORTS = sorted(_SIGS)
for _name, (_res, _args) in _SIGS.items():
    _f = getattr(_lib, _name)          # AttributeError here = a declared symbol is not exported
    _f.restype, _f.argtypes = _res, _args


class NuboError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        super().__init__(f"{where}: nv_status {code}: {_lib.nv_last_error().decode(errors='replace')}")


def _check(rc, where):
    if rc != NV_OK:
        raise NuboError(rc, where)


def version() -> str:
    return _lib.nv_version().decode()


def device_count() -> int:
    return _lib.nv_device_count()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


def _rects(buf, n):
    return np.frombuffer(buf, dtype=np.int32, count=4 * n).reshape(n, 4).copy()


def _batch_frames(images, cn):
    """(pointer table, n, w, h, row stride, on_device, keep-alive) of a batch: a uint8 numpy array or CUDA torch tensor
    [N, H, W] (cn == 1) / [N, H, W, 3] (cn == 3) whose pixels are packed within a row; rows and images may be further
    apart than packed.  A torch tensor's stream is synchronised here, so the library reads finished frames."""
    ndim = 3 if cn == 1 else 4
    if type(images).__module__.startswith("torch"):
        import torch
        if images.dtype != torch.uint8:
            raise TypeError(f"batch must be a uint8 tensor, got {images.dtype}")
        if images.dim() != ndim or (cn == 3 and images.shape[3] != 3):
            raise ValueError(f"batch tensor must be [N, H, W{', 3' if cn == 3 else ''}], got {tuple(images.shape)}")
        if not images.is_cuda:
            images = images.numpy()
        else:
            if images.stride(2) != cn or (cn == 3 and images.stride(3) != 1):
                raise ValueError("the pixels of a row must be packed (stride(2) == channels)")
            n, h, w = images.shape[:3]
            torch.cuda.current_stream(images.device).synchronize()
            base = images.data_ptr()
            ptrs = (C.c_void_p * max(n, 1))(*[base + i * images.stride(0) for i in range(n)])
            return ptrs, n, w, h, images.stride(1), 1, images
    if not isinstance(images, np.ndarray) or images.dtype != np.uint8:
        raise TypeError("batch must be a uint8 numpy array or a CUDA torch tensor")
    shape, strides = images.shape, images.strides
    if len(shape) != ndim or (cn == 3 and shape[3] != 3):
        raise ValueError(f"batch array must be [N, H, W{', 3' if cn == 3 else ''}], got {shape}")
    if strides[2] != cn or (cn == 3 and strides[3] != 1) or min(strides) < 0:
        images = np.ascontiguousarray(images)
        strides = images.strides
    n, h, w = shape[:3]
    base, s0 = images.ctypes.data, strides[0]
    ptrs = (C.c_void_p * max(n, 1))(*range(base, base + n * s0, s0)) if s0 else (C.c_void_p * max(n, 1))(*([base] * n))
    return ptrs, n, w, h, strides[1], 0, images


NUM_STAGES = 8
STAGE_NAMES = [_lib.nv_stage_name(i).decode() for i in range(NUM_STAGES)]


class Event:
    """A CUDA event recorded on a context's own stream (torch.cuda.Event only sees torch's stream)."""

    def __init__(self):
        self.handle = _vp()
        _check(_lib.nv_event_create(C.byref(self.handle)), "nv_event_create")

    def elapsed_ms(self, end: "Event") -> float:
        ms = C.c_float(0)
        _check(_lib.nv_event_elapsed_ms(self.handle, end.handle, C.byref(ms)), "nv_event_elapsed_ms")
        return ms.value

    def __del__(self):
        if getattr(self, "handle", None):
            _lib.nv_event_destroy(self.handle)
            self.handle = None


class Cascade:
    """cv::CascadeClassifier::load replacement (kmsfacedetect.cpp:163-177)."""

    def __init__(self, path: str):
        if not os.path.isabs(path) and not os.path.exists(path):
            path = os.path.join(CASCADE_DIR, path)
        self.handle = _vp()
        _check(_lib.nv_cascade_load(path.encode(), C.byref(self.handle)), f"nv_cascade_load({path})")
        self.info = CascadeInfo()
        _check(_lib.nv_cascade_get_info(self.handle, C.byref(self.info)), "nv_cascade_get_info")

    def __del__(self):
        if getattr(self, "handle", None):
            _lib.nv_cascade_free(self.handle)
            self.handle = None

    def stage(self, s):
        nt, thr = C.c_int(0), C.c_float(0)
        _check(_lib.nv_debug_cascade_stage(self.handle, s, C.byref(nt), C.byref(thr)), "nv_debug_cascade_stage")
        return nt.value, np.float32(thr.value)

    def tree(self, t, cap=64):
        """(nodes [n,3] int: feature, left, right), thresholds [n] f32, leaves [n+1] f32 of weak classifier t"""
        nn = C.c_int(0)
        flr, thr, lv = (C.c_int * (3 * cap))(), (C.c_float * cap)(), (C.c_float * (cap + 1))()
        _check(_lib.nv_debug_cascade_tree(self.handle, t, cap, C.byref(nn), flr, thr, lv), "nv_debug_cascade_tree")
        n = nn.value
        return (np.array(flr[:3 * n], np.int32).reshape(n, 3), np.array(thr[:n], np.float32), np.array(lv[:n + 1], np.float32))

    def feature(self, f):
        r, w, t = (C.c_int * 12)(), (C.c_float * 3)(), C.c_int(0)
        _check(_lib.nv_debug_cascade_feature(self.handle, f, r, w, C.byref(t)), "nv_debug_cascade_feature")
        return np.array(r[:], np.int32).reshape(3, 4), np.array(w[:], np.float32), t.value

    def subset(self, node):
        s = (C.c_int * 8)()
        _check(_lib.nv_debug_cascade_subset(self.handle, node, s), "nv_debug_cascade_subset")
        return np.array(s[:], np.int32)

    def stump(self, i):
        r, w, t = (C.c_int * 12)(), (C.c_float * 3)(), (C.c_float * 3)()
        _check(_lib.nv_debug_cascade_stump(self.handle, i, r, w, t), "nv_debug_cascade_stump")
        return np.array(r[:], np.int32).reshape(3, 4), np.array(w[:], np.float32), np.array(t[:], np.float32)


class MetaRect(C.Structure):
    _fields_ = [("name", C.c_char * 16), ("type", C.c_char * 16), ("x", C.c_uint), ("y", C.c_uint), ("width", C.c_uint),
                ("height", C.c_uint)]


class Element:
    """Mirror of one reference GStreamer element (same factory name, properties, per-frame behaviour)."""

    def __init__(self, factory: str, gpu: int = 0, cascade_dir: str | None = None):
        self.handle = _vp()
        _check(_lib.nv_element_create(factory.encode(), gpu, cascade_dir.encode() if cascade_dir else None,
                                      C.byref(self.handle)), f"nv_element_create({factory})")

    def close(self):
        if getattr(self, "handle", None):
            _lib.nv_element_destroy(self.handle)
            self.handle = None

    __del__ = close

    def set(self, name: str, value: int):
        _check(_lib.nv_element_set_property(self.handle, name.encode(), value), f"set {name}")

    def get(self, name: str) -> int:
        v = C.c_long(0)
        _check(_lib.nv_element_get_property(self.handle, name.encode(), C.byref(v)), f"get {name}")
        return v.value

    def properties(self):
        """[(name, minimum, maximum, default)] — the table a GStreamer shell installs its GObject properties from."""
        out = []
        i = 0
        while True:
            name = C.c_char_p(); lo, hi, de = C.c_long(0), C.c_long(0), C.c_long(0)
            if _lib.nv_element_property_info(self.handle, i, C.byref(name), C.byref(lo), C.byref(hi), C.byref(de)) != 0:
                break
            out.append((name.value.decode(), lo.value, hi.value, de.value))
            i += 1
        return out

    def push_faces(self, rects):
        r = np.ascontiguousarray(np.asarray(rects, np.int32).reshape(-1, 4))
        _check(_lib.nv_element_push_faces_event(self.handle, _p(r), len(r)), "nv_element_push_faces_event")

    def push_motion(self):
        _check(_lib.nv_element_push_motion_event(self.handle), "nv_element_push_motion_event")

    def push_message(self, fields):
        """One custom downstream event as the sink pad saw it: fields = [(name, is_structure, type or None, (x, y, w, h))]."""
        arr = (EventField * max(len(fields), 1))()
        for i, (name, is_st, typ, r) in enumerate(fields):
            arr[i] = EventField(name.encode(), int(is_st), typ.encode() if typ is not None else None, Rect(*[int(v) for v in r]))
        _check(_lib.nv_element_push_message(self.handle, arr, len(fields)), "nv_element_push_message")

    def process(self, frame, pts_ns: int = 0, now_ms: float = -1.0):
        """One buffer through transform_frame_ip.  Returns (message [(name, type, x, y, w, h)], pushed, signal or None)."""
        frame = _u8(frame); h, w = frame.shape[:2]
        _check(_lib.nv_element_transform_frame_ip(self.handle, _p(frame), w, h, frame.strides[0], pts_ns, now_ms),
               "nv_element_transform_frame_ip")
        return self._outputs()

    def process_device(self, d_ptr: int, w: int, h: int, stride: int, pts_ns: int = 0, now_ms: float = -1.0):
        """One BGR(A) buffer that lives in device memory (d_ptr: a CUDA device address, e.g. torch.Tensor.data_ptr()) through
        nv_element_transform_frame_device; the overlays are written into it on the device.  Same outputs as process()."""
        _check(_lib.nv_element_transform_frame_device(self.handle, C.c_void_p(d_ptr), w, h, stride, pts_ns, now_ms),
               "nv_element_transform_frame_device")
        return self._outputs()

    def process_yuv(self, planes, fmt="I420", pts_ns: int = 0, now_ms: float = -1.0):
        """One 4:2:0 buffer (nubofacedetector only) through nv_element_transform_frame_yuv; same outputs as process()."""
        f = Context._yuv_frame(planes, fmt)
        _check(_lib.nv_element_transform_frame_yuv(self.handle, C.byref(f), pts_ns, now_ms), "nv_element_transform_frame_yuv")
        return self._outputs()

    def _outputs(self):
        buf = (MetaRect * 4096)(); n = C.c_int(0); pushed = C.c_int(0)
        _check(_lib.nv_element_get_message(self.handle, buf, 4096, C.byref(n), C.byref(pushed)), "nv_element_get_message")
        msg = [(buf[i].name.decode(), buf[i].type.decode(), buf[i].x, buf[i].y, buf[i].width, buf[i].height)
               for i in range(n.value)]
        sbuf = C.create_string_buffer(1 << 16); em = C.c_int(0)
        _check(_lib.nv_element_get_signal(self.handle, sbuf, len(sbuf), C.byref(em)), "nv_element_get_signal")
        return msg, bool(pushed.value), (sbuf.value.decode() if em.value else None)


def draw_rectangle(frame, x0, y0, x1, y1, bgr):
    """cvRectangle(frame, (x0, y0), (x1, y1), Scalar(b, g, r, 0), 3, 8, 0) in place on an HxWx3 / HxWx4 uint8 array."""
    assert frame.dtype == np.uint8 and frame.ndim == 3 and frame.flags["C_CONTIGUOUS"]
    h, w, cn = frame.shape
    _check(_lib.nv_debug_draw_rectangle(_p(frame), w, h, frame.strides[0], cn, int(x0), int(y0), int(x1), int(y1),
                                        int(bgr[0]), int(bgr[1]), int(bgr[2])), "nv_debug_draw_rectangle")
    return frame


def _shape_array(shapes):
    arr = (Shape * max(len(shapes), 1))()
    for i, (kind, a, b, c, d, col) in enumerate(shapes):
        arr[i] = Shape(0 if kind == "rect" else 1, int(a), int(b), int(c), int(d), int(col[0]), int(col[1]), int(col[2]), 0)
    return arr


def draw_shapes_spans(frame, shapes):
    """The host half of the device overlay on a host frame (nv_debug_draw_shapes_spans); returns the number of disjoint spans."""
    assert frame.dtype == np.uint8 and frame.ndim == 3 and frame.flags["C_CONTIGUOUS"]
    h, w, cn = frame.shape
    n = C.c_int(0)
    _check(_lib.nv_debug_draw_shapes_spans(_p(frame), w, h, frame.strides[0], cn, _shape_array(shapes), len(shapes), C.byref(n)),
           "nv_debug_draw_shapes_spans")
    return n.value


def draw_circle(frame, cx, cy, radius, bgr, thickness=4):
    """cv::circle(frame, (cx, cy), radius, Scalar(b, g, r, 0), thickness, 8, 0) in place."""
    assert frame.dtype == np.uint8 and frame.ndim == 3 and frame.flags["C_CONTIGUOUS"]
    h, w, cn = frame.shape
    _check(_lib.nv_debug_draw_circle(_p(frame), w, h, frame.strides[0], cn, int(cx), int(cy), int(radius), int(thickness),
                                     int(bgr[0]), int(bgr[1]), int(bgr[2])), "nv_debug_draw_circle")
    return frame


def track_faces(prev, prev_ids, next_id, cur, track_threshold=40, pos_threshold=8, area_threshold=500):
    """Faces::track_faces (Faces.cpp:78-153) on explicit lists; returns (rects, ids, next_id)."""
    prev = np.ascontiguousarray(np.asarray(prev, np.int32).reshape(-1, 4))
    ids = np.ascontiguousarray(np.asarray(prev_ids, np.int32).reshape(-1))
    cur = np.ascontiguousarray(np.asarray(cur, np.int32).reshape(-1, 4))
    out = np.zeros((len(prev) + len(cur) + 1, 4), np.int32); oid = np.zeros(len(out), np.int32)
    n = C.c_int(0); nid = C.c_int(0)
    _check(_lib.nv_debug_track_faces(_p(prev), _p(ids), len(prev), next_id, _p(cur), len(cur), track_threshold,
                                     pos_threshold, area_threshold, _p(out), _p(oid), len(out), C.byref(n), C.byref(nid)),
           "nv_debug_track_faces")
    return out[:n.value].copy(), oid[:n.value].copy(), nid.value


class Context:
    """One per element instance / video stream."""

    def __init__(self, gpu: int = 0, max_width: int = 1920, max_height: int = 1080, debug: bool = False):
        self.handle = _vp()
        _check(_lib.nv_ctx_create(gpu, max_width, max_height, C.byref(self.handle)), "nv_ctx_create")
        self._cap = 131072
        self._out = (Rect * self._cap)()
        self._scores_on = False
        if debug:
            self.set_debug(True)

    def close(self):
        if getattr(self, "handle", None):
            _lib.nv_ctx_destroy(self.handle)
            self.handle = None

    __del__ = close

    def set_debug(self, on: bool):
        _check(_lib.nv_ctx_set_debug(self.handle, int(on)), "nv_ctx_set_debug")

    # ---- device-side timing ------------------------------------------------------------------
    def set_profile(self, on: bool):
        _check(_lib.nv_ctx_set_profile(self.handle, int(on)), "nv_ctx_set_profile")

    def stage_times(self):
        """{stage name: ms} of the last collected detect call (CUDA events on this ctx's stream)."""
        ms = (C.c_float * NUM_STAGES)(); n = C.c_int(0)
        _check(_lib.nv_ctx_get_stage_times(self.handle, ms, NUM_STAGES, C.byref(n)), "nv_ctx_get_stage_times")
        return {STAGE_NAMES[i]: ms[i] for i in range(n.value)}

    def record(self, ev: "Event"):
        _check(_lib.nv_event_record(self.handle, ev.handle), "nv_event_record")

    # ---- detection scores (cv::CascadeClassifier::detectMultiScale2 / 3) ---------------------------
    def set_scores(self, on: bool):
        """Every later detect call on this context also yields per-rectangle neighbour counts and level weights."""
        _check(_lib.nv_ctx_set_scores(self.handle, int(on)), "nv_ctx_set_scores")
        self._scores_on = bool(on)

    def scores(self):
        """(num_detections int32 [n], level_weights float64 [n]) of the last collected call, parallel to its rectangles."""
        nb = np.empty(self._cap, np.int32); wt = np.empty(self._cap, np.float64); n = C.c_int(0)
        _check(_lib.nv_get_scores(self.handle, nb.ctypes.data_as(_ip), wt.ctypes.data_as(C.POINTER(C.c_double)), self._cap,
                                  C.byref(n)), "nv_get_scores")
        return nb[:n.value].copy(), wt[:n.value].copy()

    def _with_scores(self, fn):
        """fn() run with scores on; the context's own setting is restored afterwards."""
        was = self._scores_on
        self.set_scores(True)
        try:
            rects = fn()
            return (rects,) + self.scores()
        finally:
            self.set_scores(was)

    # ---- detection -------------------------------------------------------------------------
    def detect_multiscale(self, casc: Cascade, gray, scale_factor=1.1, min_neighbors=3, min_size=(0, 0), max_size=(0, 0)):
        gray = _u8(gray); h, w = gray.shape
        p = DetectParams(scale_factor, min_neighbors, 0, min_size[0], min_size[1], max_size[0], max_size[1])
        n = C.c_int(0)
        _check(_lib.nv_detect_multiscale(self.handle, casc.handle, _p(gray), w, h, gray.strides[0], C.byref(p),
                                         self._out, self._cap, C.byref(n)), "nv_detect_multiscale")
        return _rects(self._out, n.value)

    def detect_multiscale2(self, casc: Cascade, gray, scale_factor=1.1, min_neighbors=3, min_size=(0, 0), max_size=(0, 0)):
        """cv2.CascadeClassifier.detectMultiScale2: (rects, num_detections)."""
        r, nb, _ = self._with_scores(lambda: self.detect_multiscale(casc, gray, scale_factor, min_neighbors, min_size, max_size))
        return r, nb

    def detect_multiscale3(self, casc: Cascade, gray, scale_factor=1.1, min_neighbors=3, min_size=(0, 0), max_size=(0, 0)):
        """cv2.CascadeClassifier.detectMultiScale3(..., outputRejectLevels=True): (rects, reject_levels, level_weights).
        reject_levels is always the cascade's stage count, as in OpenCV 4.13."""
        r, _, wt = self._with_scores(lambda: self.detect_multiscale(casc, gray, scale_factor, min_neighbors, min_size, max_size))
        return r, np.full(len(r), casc.info.nstages, np.int32), wt

    @staticmethod
    def _face_params(width_to_process, scale_factor, min_neighbors, min_size):
        mw, mh = (-1, -1) if min_size is None else min_size
        return FaceParams(width_to_process, scale_factor, min_neighbors, mw, mh)

    def face_detect(self, casc: Cascade, bgr, width_to_process=160, scale_factor=1.25, min_neighbors=3, min_size=None,
                    scores=False):
        """scores=True: (rects, num_detections, level_weights), see set_scores."""
        if scores:
            return self._with_scores(lambda: self.face_detect(casc, bgr, width_to_process, scale_factor, min_neighbors, min_size))
        bgr = _u8(bgr); h, w, _ = bgr.shape
        p = self._face_params(width_to_process, scale_factor, min_neighbors, min_size)
        n = C.c_int(0)
        _check(_lib.nv_face_detect(self.handle, casc.handle, _p(bgr), w, h, bgr.strides[0], C.byref(p), self._out,
                                   self._cap, C.byref(n)), "nv_face_detect")
        return _rects(self._out, n.value)

    def face_submit(self, casc: Cascade, bgr, width_to_process=160, scale_factor=1.25, min_neighbors=3, min_size=None):
        h, w, _ = bgr.shape
        p = self._face_params(width_to_process, scale_factor, min_neighbors, min_size)
        _check(_lib.nv_face_submit(self.handle, casc.handle, _p(bgr), w, h, bgr.strides[0], C.byref(p)), "nv_face_submit")

    def face_submit_device(self, casc: Cascade, dev_ptr: int, w: int, h: int, stride: int, width_to_process=160,
                           scale_factor=1.25, min_neighbors=3, min_size=None):
        p = self._face_params(width_to_process, scale_factor, min_neighbors, min_size)
        _check(_lib.nv_face_submit_device(self.handle, casc.handle, _vp(dev_ptr), w, h, stride, C.byref(p)),
               "nv_face_submit_device")

    # ---- batches: N same-size images per call (see nubovca.h).  images: a uint8 numpy array or CUDA torch tensor
    #      [N, H, W] (gray) / [N, H, W, 3] (BGR); a torch tensor's current stream is synchronised before the submit.
    #      Returns a list of N int32 arrays [k, 4], image by image.
    def _batch_out(self, counts):
        flat = np.frombuffer(self._bout, dtype=np.int32, count=4 * sum(counts)).reshape(-1, 4)
        out, o = [], 0
        for k in counts:
            out.append(flat[o:o + k].copy())
            o += k
        return out

    def _batch_buffers(self, n):
        self._bcounts = (C.c_int * max(n, 1))()
        if not hasattr(self, "_bout"):
            self._bout = (Rect * (1 << 20))()

    def detect_multiscale_batch(self, casc: Cascade, images, scale_factor=1.1, min_neighbors=3, min_size=(0, 0), max_size=(0, 0)):
        ptrs, n, w, h, stride, dev, keep = _batch_frames(images, 1)
        p = DetectParams(scale_factor, min_neighbors, 0, min_size[0], min_size[1], max_size[0], max_size[1])
        self._batch_buffers(n)
        _check(_lib.nv_detect_multiscale_batch(self.handle, casc.handle, ptrs, n, w, h, stride, dev, C.byref(p), self._bout,
                                               len(self._bout), self._bcounts), "nv_detect_multiscale_batch")
        return self._batch_out(self._bcounts[:n])

    def face_submit_batch(self, casc: Cascade, frames, width_to_process=160, scale_factor=1.25, min_neighbors=3, min_size=None):
        ptrs, n, w, h, stride, dev, keep = _batch_frames(frames, 3)
        p = self._face_params(width_to_process, scale_factor, min_neighbors, min_size)
        self._batch_buffers(n)
        _check(_lib.nv_face_submit_batch(self.handle, casc.handle, ptrs, n, w, h, stride, dev, C.byref(p)), "nv_face_submit_batch")
        self._batch_keep, self._batch_n = keep, n          # page-locked / device frames are read until collect

    def face_collect_batch(self):
        total = C.c_int(0)
        try:
            _check(_lib.nv_face_collect_batch(self.handle, self._bout, len(self._bout), self._bcounts, C.byref(total)),
                   "nv_face_collect_batch")
        finally:
            self._batch_keep = None
        return self._batch_out(self._bcounts[:self._batch_n])

    def face_detect_batch(self, casc: Cascade, frames, width_to_process=160, scale_factor=1.25, min_neighbors=3, min_size=None):
        self.face_submit_batch(casc, frames, width_to_process, scale_factor, min_neighbors, min_size)
        return self.face_collect_batch()

    # ---- 4:2:0 ingest: planes = (y, u, v) for I420 (YV12: pass the planes in I420 meaning), (y, uv) for NV12 / NV21;
    #      each a 2-D uint8 array with unit column stride (row strides are honoured)
    @staticmethod
    def _yuv_frame(planes, fmt):
        y, c1 = planes[0], planes[1]
        c2 = planes[2] if len(planes) > 2 and planes[2] is not None else None
        for a in (y, c1) + ((c2,) if c2 is not None else ()):
            if a.dtype != np.uint8 or a.ndim != 2 or a.strides[1] != 1:
                raise ValueError("planes must be 2-D uint8 arrays with contiguous rows")
        h, w = y.shape
        f = YuvFrame()
        f.format, f.width, f.height, f.on_device = _FMT[fmt], w, h, 0
        f.plane[0], f.plane[1] = y.ctypes.data, c1.ctypes.data
        f.stride[0], f.stride[1] = y.strides[0], c1.strides[0]
        if c2 is not None:
            f.plane[2], f.stride[2] = c2.ctypes.data, c2.strides[0]
        return f

    def face_detect_yuv(self, casc: Cascade, planes, fmt="I420", width_to_process=160, scale_factor=1.25, min_neighbors=3,
                        min_size=None):
        f = self._yuv_frame(planes, fmt)
        p = self._face_params(width_to_process, scale_factor, min_neighbors, min_size)
        n = C.c_int(0)
        _check(_lib.nv_face_detect_yuv(self.handle, casc.handle, C.byref(f), C.byref(p), self._out, self._cap, C.byref(n)),
               "nv_face_detect_yuv")
        return _rects(self._out, n.value)

    def face_submit_yuv(self, casc: Cascade, planes, fmt="I420", width_to_process=160, scale_factor=1.25, min_neighbors=3,
                        min_size=None):
        f = self._yuv_frame(planes, fmt)
        p = self._face_params(width_to_process, scale_factor, min_neighbors, min_size)
        _check(_lib.nv_face_submit_yuv(self.handle, casc.handle, C.byref(f), C.byref(p)), "nv_face_submit_yuv")

    def yuv2bgr(self, planes, fmt="I420"):
        f = self._yuv_frame(planes, fmt)
        out = np.empty((f.height, f.width, 3), np.uint8)
        _check(_lib.nv_yuv2bgr(self.handle, C.byref(f), _p(out), 3 * f.width), "nv_yuv2bgr")
        return out

    def face_collect(self, scores=False):
        """scores=True: (rects, num_detections, level_weights) of a call submitted with set_scores(True)."""
        n = C.c_int(0)
        _check(_lib.nv_face_collect(self.handle, self._out, self._cap, C.byref(n)), "nv_face_collect")
        rects = _rects(self._out, n.value)
        return (rects,) + self.scores() if scores else rects

    # ---- tracker ---------------------------------------------------------------------------
    def tracker_process(self, bgra, ts_ms, threshold=20, min_area=50, max_area=30000, distance=35):
        bgra = _u8(bgra); h, w, _ = bgra.shape
        p = TrackerParams(threshold, min_area, max_area, distance)
        n = C.c_int(0)
        _check(_lib.nv_tracker_process(self.handle, _p(bgra), w, h, bgra.strides[0], float(ts_ms), C.byref(p),
                                       self._out, self._cap, C.byref(n)), "nv_tracker_process")
        return _rects(self._out, n.value)

    def tracker_process_yuv(self, planes, fmt, ts_ms, threshold=20, min_area=50, max_area=30000, distance=35):
        f = self._yuv_frame(planes, fmt)
        p = TrackerParams(threshold, min_area, max_area, distance)
        n = C.c_int(0)
        _check(_lib.nv_tracker_process_yuv(self.handle, C.byref(f), float(ts_ms), C.byref(p), self._out, self._cap, C.byref(n)),
               "nv_tracker_process_yuv")
        return _rects(self._out, n.value)

    def draw_shapes_device(self, d_ptr: int, w: int, h: int, stride: int, channels: int, shapes):
        """shapes: [("rect", x0, y0, x1, y1, (b, g, r))] / [("circle", cx, cy, radius, thickness, (b, g, r))], drawn in order into
        the BGR(A) frame at device address d_ptr (nv_draw_shapes_device)."""
        _check(_lib.nv_draw_shapes_device(self.handle, C.c_void_p(d_ptr), w, h, stride, channels, _shape_array(shapes), len(shapes)),
               "nv_draw_shapes_device")

    def tracker_kernel_ms(self):
        ms = C.c_float(0)
        _check(_lib.nv_ctx_get_tracker_kernel_ms(self.handle, C.byref(ms)), "nv_ctx_get_tracker_kernel_ms")
        return ms.value

    def tracker_reset(self):
        _check(_lib.nv_tracker_reset(self.handle), "nv_tracker_reset")

    # ---- image ops -------------------------------------------------------------------------
    def bgr2gray(self, img):
        img = _u8(img); h, w, cn = img.shape
        out = np.empty((h, w), np.uint8)
        _check(_lib.nv_bgr2gray(self.handle, _p(img), w, h, img.strides[0], cn, _p(out), w), "nv_bgr2gray")
        return out

    def equalize_hist(self, img):
        img = _u8(img); h, w = img.shape
        out = np.empty((h, w), np.uint8)
        _check(_lib.nv_equalize_hist(self.handle, _p(img), w, h, img.strides[0], _p(out), w), "nv_equalize_hist")
        return out

    def resize_linear(self, img, dw, dh):
        img = _u8(img); h, w = img.shape[:2]; cn = 1 if img.ndim == 2 else img.shape[2]
        out = np.empty((dh, dw) if img.ndim == 2 else (dh, dw, cn), np.uint8)
        _check(_lib.nv_resize_linear(self.handle, _p(img), w, h, img.strides[0], cn, _p(out), dw, dh, dw * cn),
               "nv_resize_linear")
        return out

    def flip_horizontal(self, img):
        img = _u8(img); h, w = img.shape
        out = np.empty((h, w), np.uint8)
        _check(_lib.nv_flip_horizontal(self.handle, _p(img), w, h, img.strides[0], _p(out), w), "nv_flip_horizontal")
        return out

    # ---- parity taps -----------------------------------------------------------------------
    def levels(self):
        out = []
        for i in range(_lib.nv_debug_num_levels(self.handle)):
            li = LevelInfo()
            _check(_lib.nv_debug_level_info(self.handle, i, C.byref(li)), "nv_debug_level_info")
            out.append(dict(scale=li.scale, lw=li.width, lh=li.height, ystep=li.ystep, nx=li.nx, ny=li.ny))
        return out

    def gray(self):
        w, h = C.c_int(0), C.c_int(0)
        _lib.nv_debug_get_gray(self.handle, None, 0, C.byref(w), C.byref(h))       # size query (reports "too small")
        buf = np.empty(max(1, w.value * h.value), np.uint8)
        _check(_lib.nv_debug_get_gray(self.handle, _p(buf), buf.size, C.byref(w), C.byref(h)), "nv_debug_get_gray")
        return buf[:w.value * h.value].reshape(h.value, w.value).copy()

    def integral(self, level):
        lv = self.levels()[level]
        s = np.empty((lv["lh"] + 1, lv["lw"] + 1), np.int32); q = np.empty((lv["lh"] + 1, lv["lw"] + 1), np.uint32)
        _check(_lib.nv_debug_get_integral(self.handle, level, _p(s), _p(q)), "nv_debug_get_integral")
        return s, q

    def tilted(self, level):
        lv = self.levels()[level]
        t = np.empty((lv["lh"] + 1, lv["lw"] + 1), np.int32)
        _check(_lib.nv_debug_get_tilted(self.handle, level, _p(t)), "nv_debug_get_tilted")
        return t

    def depth_map(self, level):
        lv = self.levels()[level]
        d = np.empty((lv["ny"], lv["nx"]), np.int16)
        _check(_lib.nv_debug_get_depth_map(self.handle, level, _p(d)), "nv_debug_get_depth_map")
        return d

    def candidates(self):
        n = C.c_int(0)
        buf = (Rect * 131072)()
        _check(_lib.nv_debug_get_candidates(self.handle, buf, 131072, C.byref(n)), "nv_debug_get_candidates")
        return _rects(buf, n.value)

    def counters(self):
        o = (C.c_longlong * 8)()
        _check(_lib.nv_debug_get_counters(self.handle, o), "nv_debug_get_counters")
        return dict(windows=o[0], alive_after_stage0=o[1], candidates=o[2], launches=o[3])
