"""The host glue of libnubovca.so (csrc/elements.cu, csrc/context.cu) fuzzed against what the REFERENCE'S OWN functions
returned on the same random cases: Faces::track_faces (Faces.cpp:78-153, compiled unmodified), __merge_eyes_current_frame /
__merge_eyes_consecutives_frames / transform_2_global_coordinates / __contain_bb (kmseyedetect.cpp:766-913),
__merge_mouths_consecutives_frames (kmsmouthdetect.cpp:750-796), __merge_noses_consecutives_frames
(kmsnosedetect.cpp:745-790) and calc_dist / __merge / __join_objects (gstnubotracker.cpp:119-200), as compiled by
oracle/build_ref.py.  >= 10 000 random cases per function; the cases come from fixed seeds, and
tests/golden/ref_elements.json holds a SHA-256 digest of the reference's answers for every CHUNK consecutive cases.
Runs without a GPU: the taps are host code."""
import ctypes as C
import hashlib

import numpy as np
import pytest

import nubovca as nv
from refgst import GOLDEN

N_CASES = 10_000
CHUNK = 500


def digests(answers):
    """First 16 hex digits of the SHA-256 of every CHUNK consecutive answers (each a sequence of ints)."""
    out = []
    for i, a in enumerate(answers):
        if i % CHUNK == 0:
            out.append(hashlib.sha256())
        a = np.asarray(a, np.int64).ravel()
        out[-1].update(np.int64(len(a)).tobytes() + a.tobytes())
    return [h.hexdigest()[:16] for h in out]


def check(name, answers):
    got, exp = digests(answers), GOLDEN["glue"][name]
    assert len(got) == len(exp), (name, len(got), len(exp))
    bad = [i for i, (g, x) in enumerate(zip(got, exp)) if g != x]
    assert not bad, f"{name}: cases {bad[0] * CHUNK}..{(bad[0] + 1) * CHUNK - 1} differ from the reference ({len(bad)} chunks)"


def rand_rects(rng, n, span=400, smin=1, smax=140):
    if n == 0:
        return np.zeros((0, 4), np.int32)
    r = np.empty((n, 4), np.int32)
    r[:, 0] = rng.integers(0, span, n)
    r[:, 1] = rng.integers(0, span, n)
    r[:, 2] = rng.integers(smin, smax, n)
    r[:, 3] = rng.integers(smin, smax, n)
    return r


def clustered_rects(rng, n, span=300):
    """Rectangles that overlap and nest often (what a cascade returns around one object)."""
    if n == 0:
        return np.zeros((0, 4), np.int32)
    cx, cy = rng.integers(40, span), rng.integers(40, span)
    r = np.empty((n, 4), np.int32)
    r[:, 2] = rng.integers(4, 90, n)
    r[:, 3] = rng.integers(4, 90, n)
    r[:, 0] = cx + rng.integers(-30, 31, n) - r[:, 2] // 2
    r[:, 1] = cy + rng.integers(-30, 31, n) - r[:, 3] // 2
    return r


def track_faces_answers():
    """Random sequences of detection lists through nv_debug_track_faces carrying (rects, ids, next id) from call to call;
    the tracked faces (rectangles and ids) after every call."""
    rng = np.random.default_rng(11)
    calls = 0
    while calls < N_CASES:
        rects, ids, next_id = np.zeros((0, 4), np.int32), np.zeros(0, np.int32), 0
        track = int(rng.choice([0, 5, 20, 40, 100]))
        anchors = rand_rects(rng, int(rng.integers(1, 6)), span=300, smin=10, smax=120)
        for _ in range(int(rng.integers(2, 9))):
            k = int(rng.integers(0, len(anchors) + 2))
            if k:
                cur = anchors[rng.integers(0, len(anchors), k)].copy()
                cur[:, :2] += rng.integers(-12, 13, (k, 2))                     # jitter: below / around / above the 3-5-8 px limits
                cur[:, 2:] = np.maximum(cur[:, 2:] + rng.integers(-25, 26, (k, 2)), 1)      # the 15 % area rule
            else:
                cur = np.zeros((0, 4), np.int32)
            if k:                                                              # kmsfacedetect.cpp:813: only when something was found
                rects, ids, next_id = nv.track_faces(rects, ids, next_id, cur, track, 8, 500)
            elif rng.random() < 0.3:                                           # :824 after two empty frames
                rects, ids = np.zeros((0, 4), np.int32), np.zeros(0, np.int32)
            yield np.concatenate([np.ravel(rects), np.ravel(ids)])
            calls += 1


def test_track_faces_sequences():
    """The same sequences through one reference Faces object (Faces::track_faces, Faces::clear)."""
    check("track_faces", track_faces_answers())


def _nv_merge_current(face, eye_r, same, eyes, scale, left):
    buf = np.zeros((max(len(eyes), 1), 4), np.int32)
    buf[:len(eyes)] = eyes
    n = C.c_int(0)
    face = np.ascontiguousarray(face, np.int32)
    eye_r = np.ascontiguousarray(eye_r, np.int32)
    rc = nv._lib.nv_debug_merge_eyes_current_frame(face.ctypes.data, eye_r.ctypes.data if len(eye_r) else None, len(eye_r), int(same),
                                                   buf.ctypes.data, len(eyes), scale, int(left), len(buf), C.byref(n))
    assert rc == 0
    return buf[:n.value].copy()


def merge_eyes_current_frame_answers(stats):
    rng = np.random.default_rng(12)
    for case in range(N_CASES):
        scale = int(rng.integers(1, 5))
        face = np.array([rng.integers(0, 200), rng.integers(0, 200), rng.integers(10, 160), rng.integers(10, 120)], np.int32)
        n = int(rng.integers(1, 7))                                            # the caller only merges non-empty lists (:1014,1023)
        eyes = clustered_rects(rng, n) if rng.random() < 0.7 else rand_rects(rng, n)
        eyes[:, 1] += int(face[1] * scale * rng.integers(0, 2))                # both sides of the 60 % eyebrow line
        left = bool(rng.integers(0, 2))
        same = not left                                                        # right eye: eye_r is the list itself
        eye_r = rand_rects(rng, int(rng.integers(0, 3)))
        got = _nv_merge_current(face, eye_r, same, eyes, scale, left)
        stats["shrunk"] += len(got) < n
        yield got


def test_merge_eyes_current_frame():
    stats = {"shrunk": 0}
    check("merge_eyes_current_frame", merge_eyes_current_frame_answers(stats))
    assert stats["shrunk"] > N_CASES // 4                                      # the merging paths were exercised


def _nv_merge_consecutive(kind, cur, prev, face, scale):
    out = np.zeros((len(cur) + len(prev) + 1, 4), np.int32)
    n = C.c_int(0)
    cur = np.ascontiguousarray(cur, np.int32); prev = np.ascontiguousarray(prev, np.int32); face = np.ascontiguousarray(face, np.int32)
    rc = nv._lib.nv_debug_merge_consecutive(kind, cur.ctypes.data if len(cur) else None, len(cur), prev.ctypes.data if len(prev) else None,
                                            len(prev), face.ctypes.data, scale, out.ctypes.data, len(out), C.byref(n))
    assert rc == 0
    return out[:n.value].copy()


KINDS = {0: "eye_merge_consecutive", 1: "mouth_merge_consecutive", 2: "nose_merge_consecutive"}


def merge_consecutive_answers(kind, stats):
    rng = np.random.default_rng(20 + kind)
    for case in range(N_CASES):
        scale = int(rng.integers(1, 5))
        face = np.array([rng.integers(0, 100), rng.integers(0, 100), rng.integers(10, 100), rng.integers(10, 100)], np.int32)
        prev = rand_rects(rng, int(rng.integers(0, 4)), span=300, smin=4, smax=60)
        ncur = int(rng.integers(1, 5))
        cur = rand_rects(rng, ncur, span=300 if kind == 0 else 100, smin=4, smax=60)
        for j in range(ncur):                                                  # put some current rects within a few px of a previous one
            if len(prev) and rng.random() < 0.6:
                o = prev[rng.integers(0, len(prev))]
                d = rng.integers(-6, 7, 2)
                if kind == 0:
                    cur[j] = [o[0] + d[0], o[1] + d[1], o[2], o[3]]
                else:                                                          # mouth / nose compare in original-image coordinates
                    w, h = max(o[2] // scale, 1), max(o[3] // scale, 1)
                    cur[j] = [(o[0] + d[0]) // scale - face[0], (o[1] + d[1]) // scale - face[1], w, h]
        if kind == 0:
            rng.integers(0, 2)                                                 # the reference's eye variant takes a left / right flag
        got = _nv_merge_consecutive(kind, cur, prev, face, scale)
        stats["kept"] += any((got == p).all(axis=1).any() for p in prev) if len(prev) else 0
        yield got


@pytest.mark.parametrize("kind,fn", [(0, "ref_eye_merge_consecutive"), (1, "ref_mouth_merge_consecutive"), (2, "ref_nose_merge_consecutive")])
def test_merge_consecutive_frames(kind, fn):
    stats = {"kept": 0}
    check(KINDS[kind], merge_consecutive_answers(kind, stats))
    assert stats["kept"] > N_CASES // 10                                       # the "keep the previous rectangle" path was exercised


def eye_to_global_answers():
    rng = np.random.default_rng(30)
    for case in range(N_CASES):
        n = int(rng.integers(1, 5))
        eyes = rand_rects(rng, n)
        face = rand_rects(rng, 1)[0]
        scale = int(rng.integers(1, 5))
        b = eyes.copy()
        assert nv._lib.nv_debug_eye_to_global(b.ctypes.data, n, np.ascontiguousarray(face).ctypes.data, scale) == 0
        yield b


def test_eye_to_global_and_contain_bb():
    check("eye_to_global", eye_to_global_answers())


def join_objects_answers(stats):
    rng = np.random.default_rng(40)
    for case in range(N_CASES):
        min_area = int(rng.choice([0, 50, 400, 2000]))
        max_area = int(rng.choice([3000, 30000, 300000]))
        dist = int(rng.choice([0, 10, 35, 120, 2000]))
        n = int(rng.integers(0, 12))
        rects = clustered_rects(rng, n) if rng.random() < 0.5 else rand_rects(rng, n, span=500, smin=1, smax=200)
        b = np.zeros((max(n, 1), 4), np.int32); b[:n] = rects
        k = C.c_int(0)
        assert nv._lib.nv_debug_join_objects(b.ctypes.data, n, min_area, max_area, dist, C.byref(k)) == 0
        stats["merged"] += 0 < k.value < n
        yield b[:k.value]


def test_join_objects():
    """__join_objects with the element's own property values (set through g_object_set on the compiled reference element)."""
    stats = {"merged": 0}
    check("join_objects", join_objects_answers(stats))
    assert stats["merged"] > N_CASES // 10
