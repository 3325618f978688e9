#!/usr/bin/env python
"""bench.py — BASELINE.json's metric for the NUBOMEDIA-VCA detection hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE config 3, "Full-resolution 1920x1080 face detection (processing
width 1920, min window 24x24, scale 1.1)" — the configuration the metric's first half ("1080p face-cascade
frames/s per GPU") is quoted on.  A step = one pass of the face element's hot block
(kmsfacedetect.cpp:805-811: resize, BGR2GRAY, equalizeHist, detectMultiScale) over a batch of
`--batch` distinct synthetic 1080p BGR frames, each on its own per-stream context.

  value     whole-job frames/s with the frames already resident in HBM (nv_face_submit_device), device-timed
            with CUDA events on the contexts' own streams, max over ranks.
  e2e       the same through the reference-facing C-ABI call with HOST (pinned) frames:
            H2D copy of every frame and D2H of its rectangles inside the timed region.
  roofline  the dominant kernel (cascade stage evaluation): algorithmic bytes / event-timed duration
            against the measured HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline  the reference's CPU path (the same op sequence through cv2 4.13, the library the
            reference calls) timed on this box's host cores on a bounded sample.

Multi-GPU: one process per GPU (torchrun), streams sharded by rank, no data-path collective ("weak").
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "nubomedia-vca_b200", "python"))

import numpy as np  # noqa: E402

W, H = 1920, 1080
PARAMS = dict(width_to_process=1920, scale_factor=1.1, min_neighbors=3, min_size=(24, 24))
FACE_XML = os.path.join(ROOT, "nubomedia-vca_b200", "cascades", "haarcascade_frontalface_alt.xml")
WORKLOAD = "cfg3: 1920x1080 BGR, nubofacedetector hot block, processing width 1920, scale 1.1, min window 24x24, minNeighbors 3"
METRIC = "1080p face-cascade frames/s"


def load_synth():
    """nubovca/synth.py by file path: importing the package would dlopen libnubovca.so, which the reference arm must not."""
    import importlib.util
    if "nubovca_synth_standalone" in sys.modules:
        return sys.modules["nubovca_synth_standalone"]
    spec = importlib.util.spec_from_file_location("nubovca_synth_standalone",
                                                  os.path.join(ROOT, "nubomedia-vca_b200", "python", "nubovca", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["nubovca_synth_standalone"] = mod
    spec.loader.exec_module(mod)
    return mod


def make_frames(n, rank):
    synth = load_synth()
    return [synth.frame(W, H, 6, 3 + 100 * rank + i) for i in range(n)]


# (c) one `config` for both arms (the driver compares them); everything arm-specific goes to `config_detail`
CONFIG = {"workload": WORKLOAD,
          "frames": "distinct synthetic 1920x1080 BGR frames (6 procedural faces each, seeds 3 + 100*rank + i), cycled",
          "l2": "no flush needed: a step's working set (8 per-stream contexts x ~130 MB of integral images, plus the frames) exceeds the 126 MB L2"}


def rect_set(r):
    return sorted(tuple(int(v) for v in row) for row in r)


def cv2_rects(frames):
    """The CPU arm's rectangles for `frames` (cv2 4.13 through the reference's call sequence), untimed."""
    import cv2
    cv2.setNumThreads(os.cpu_count() or 1)
    cc = cv2.CascadeClassifier(FACE_XML)
    return [rect_set(cpu_face_step(cv2, cc, f)) for f in frames]


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation of the path = this OpenCV call sequence
# ------------------------------------------------------------------------------------------------
def cpu_face_step(cv2, cc, frame):
    """kmsfacedetect.cpp:805-811 with config-3 parameters."""
    aux = cv2.resize(frame, (W, H), interpolation=cv2.INTER_LINEAR)
    gray = cv2.cvtColor(aux, cv2.COLOR_BGR2GRAY)
    gray = cv2.equalizeHist(gray)
    return cc.detectMultiScale(gray, scaleFactor=PARAMS["scale_factor"], minNeighbors=PARAMS["min_neighbors"],
                               flags=0, minSize=PARAMS["min_size"])


def cpu_baseline(frames, budget_s=20.0, max_frames=40, warm=1):
    """Returns dict(value, unit, cores, kind, sample, ...) timed on the host cores."""
    try:
        import cv2
    except Exception:
        cv2 = None
    if cv2 is not None:
        cores = os.cpu_count() or 1
        cv2.setNumThreads(cores)
        cc = cv2.CascadeClassifier(FACE_XML)
        for i in range(warm):
            cpu_face_step(cv2, cc, frames[i % len(frames)])
        t0 = time.perf_counter(); n = 0
        while n < max_frames and (time.perf_counter() - t0 < budget_s or n < 2):
            cpu_face_step(cv2, cc, frames[n % len(frames)]); n += 1
        dt = time.perf_counter() - t0
        nthr = cv2.getNumThreads()
        cv2.setNumThreads(1)                              # SURVEY §8(d): also the single-thread figure
        t1 = time.perf_counter(); n1 = 0
        while n1 < 3 and (time.perf_counter() - t1 < 6.0 or n1 < 1):
            cpu_face_step(cv2, cc, frames[n1 % len(frames)]); n1 += 1
        dt1 = time.perf_counter() - t1
        cv2.setNumThreads(cores)
        return dict(value=n / dt, unit="frames/s", cores=nthr, kind="reference",
                    one_thread={"value": n1 / dt1, "unit": "frames/s", "sample": f"{n1} full cfg3 frames, {dt1:.1f} s"},
                    sample=f"{n} full cfg3 frames after {warm} warm-up, wall clock {dt:.1f} s",
                    via="cv2 %s call sequence of kmsfacedetect.cpp:805-811 (the reference C++ needs GStreamer/Kurento and "
                        "cannot be built here; its arithmetic is exactly these OpenCV calls)" % cv2.__version__,
                    host_cores=cores)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    oc = O.Cascade(FACE_XML)
    t0 = time.perf_counter(); n = 0
    while n < 8 and (time.perf_counter() - t0 < budget_s or n < 1):
        O.face_process(frames[n % len(frames)], oc, **PARAMS); n += 1
    dt = time.perf_counter() - t0
    return dict(value=n / dt, unit="frames/s", cores=1, kind="port",
                sample=f"{n} full cfg3 frames through oracle/nubo_oracle.c, wall clock {dt:.1f} s")


_CFG5_WORKER = r"""
import sys, time, importlib.util
import cv2, numpy as np
spec = importlib.util.spec_from_file_location("synth", sys.argv[1] + "/nubovca/synth.py")
synth = importlib.util.module_from_spec(spec); spec.loader.exec_module(synth)
cv2.setNumThreads(1)
cc = cv2.CascadeClassifier(sys.argv[2])
frames = [synth.frame(1280, 720, 3, 1000 + int(sys.argv[3]) * 2 + i) for i in range(2)]      # streams 2w, 2w+1 of SURVEY 8(d)
def step(f):                                         # kmsfacedetect.cpp:805-811 at width-to-process 640
    g = cv2.equalizeHist(cv2.cvtColor(cv2.resize(f, (640, 360), interpolation=cv2.INTER_LINEAR), cv2.COLOR_BGR2GRAY))
    return cc.detectMultiScale(g, scaleFactor=1.25, minNeighbors=3, flags=0, minSize=(32, 18))
step(frames[0])
t0 = time.perf_counter(); n = 0
while time.perf_counter() - t0 < float(sys.argv[4]):
    step(frames[n % 2]); n += 1
print(n / (time.perf_counter() - t0))
"""


def cpu_cfg5(seconds=6.0):
    """SURVEY §8(d): the cfg5 CPU side = min(cores, streams) single-threaded worker processes, each looping its
    streams' frames through the reference's call sequence; aggregate frames/s over the workers / 30."""
    try:
        import cv2  # noqa: F401
    except Exception:
        return None
    nw = min(os.cpu_count() or 1, 256)
    procs = [subprocess.Popen([sys.executable, "-c", _CFG5_WORKER, os.path.join(ROOT, "nubomedia-vca_b200", "python"),
                               FACE_XML, str(i), str(seconds)], stdout=subprocess.PIPE, text=True) for i in range(nw)]
    fps = 0.0
    for p_ in procs:
        out, _ = p_.communicate(timeout=120)
        fps += float(out.strip().splitlines()[-1])
    return {"frames_per_s": fps, "streams_at_30fps": fps / 30.0, "workers": nw, "threads_per_worker": 1,
            "sample": "%d worker processes x %.0f s of 1280x720 -> 640x360 frames" % (nw, seconds), "via": "cv2"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    frames = make_frames(min(8, max(1, args.steps)), 0)
    per = []
    base = None
    try:
        import cv2
        cv2.setNumThreads(os.cpu_count() or 1)
        cc = cv2.CascadeClassifier(FACE_XML)
        step = lambda f: cpu_face_step(cv2, cc, f)                      # noqa: E731
        kind, cores = "reference", cv2.getNumThreads()
        via = f"cv2 {cv2.__version__} call sequence of kmsfacedetect.cpp:805-811"
    except Exception:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle as O
        oc = O.Cascade(FACE_XML)
        step = lambda f: O.face_process(f, oc, **PARAMS)                # noqa: E731
        kind, cores, via = "port", 1, "oracle/nubo_oracle.c"
    for i in range(args.warmup):
        step(frames[i % len(frames)])
    t0 = time.perf_counter()
    for i in range(args.steps):
        t = time.perf_counter(); step(frames[i % len(frames)]); per.append(time.perf_counter() - t)
    dt = time.perf_counter() - t0
    v = args.steps / dt
    base = dict(value=v, unit="frames/s", cores=cores, kind=kind, via=via,
                sample=f"each step = 1 full cfg3 frame; {args.steps} steps after {args.warmup} warm-up")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/int32 integrals, f32 features, f64 stage sums", "data": "synthetic",
        "config": CONFIG, "config_detail": {"frames_per_step": 1}, "cpu_baseline": base,
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# algorithmic bytes (SURVEY.md §8d) from the plan the library actually built
# ------------------------------------------------------------------------------------------------
def algorithmic_bytes(levels, src_px, channels, proc_px, win=(20, 20)):
    P = sum(l["lw"] * l["lh"] for l in levels)
    Pp = sum((l["lw"] + 1) * (l["lh"] + 1) for l in levels)
    total = channels * src_px + 4 * proc_px + 2 * P + 16 * Pp
    cascade = 8 * Pp                    # the cascade kernels' compulsory read: sum + sqsum integrals once
    return dict(frame_total=total, cascade=cascade, pyramid_px=P, integral_px=Pp)


# ------------------------------------------------------------------------------------------------
# auxiliary measurements: the other BASELINE configs, each beside the same op sequence through cv2
# ------------------------------------------------------------------------------------------------
def _timeit(fn, n, warm=2):
    for _ in range(warm):
        fn()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    return n / (time.perf_counter() - t0)


def _pin(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def aux_other_configs(nv, local, world):
    """cfg1 (element defaults, one 640x480 stream), cfg2 (nested eye detection on one 720p stream, stand-in eye
    model: the mcs_* files are absent from this image) and cfg4 (tracker, 720p BGRA), frames/s of ONE stream
    through the element mirrors (page-locked host frames in, metadata out, one frame in flight: this is
    per-stream latency, not box throughput), next to cv2 on all host cores."""
    import shutil
    import tempfile
    from nubovca import synth
    out = {}
    cdir = tempfile.mkdtemp(prefix="nubovca_casc_")
    src = os.path.join(ROOT, "nubomedia-vca_b200", "cascades")
    shutil.copy(os.path.join(src, "haarcascade_frontalface_alt.xml"), cdir)
    for f in ("haarcascade_mcs_lefteye.xml", "haarcascade_mcs_righteye.xml"):
        shutil.copy(os.path.join(src, "haarcascade_eye.xml"), os.path.join(cdir, f))
    try:
        import cv2
        cv2.setNumThreads(os.cpu_count() or 1)
    except Exception:
        cv2 = None

    # cfg1
    f1 = _pin(synth.frame(640, 480, 4, 1))
    e = nv.Element("nubofacedetector", local, cdir)
    out["cfg1_face_640x480_defaults"] = {"frames_per_s": _timeit(lambda: e.process(f1), 300)}
    e.close()
    if cv2 is not None:
        cc = cv2.CascadeClassifier(os.path.join(cdir, "haarcascade_frontalface_alt.xml"))

        def cpu1():
            g = cv2.equalizeHist(cv2.cvtColor(cv2.resize(f1, (160, 120), interpolation=cv2.INTER_LINEAR), cv2.COLOR_BGR2GRAY))
            return cc.detectMultiScale(g, scaleFactor=1.25, minNeighbors=3, flags=0, minSize=(8, 6))
        out["cfg1_face_640x480_defaults"]["cpu_frames_per_s"] = _timeit(cpu1, 200)

    # cfg2: eye element, faces large enough for the 30x30 minimum at the 160-wide face stage
    f2 = _pin(synth.frame(1280, 720, 3, 2, smin=0.4, smax=0.6))
    e = nv.Element("nuboeyedetector", local, cdir)
    out["cfg2_eyes_in_faces_1280x720"] = {"frames_per_s": _timeit(lambda: e.process(f2), 100),
                                          "note": "haarcascade_eye.xml stands in for the absent mcs_lefteye/righteye models"}
    e.close()
    if cv2 is not None:
        ce = cv2.CascadeClassifier(os.path.join(cdir, "haarcascade_mcs_lefteye.xml"))

        def cpu2():
            g = cv2.equalizeHist(cv2.cvtColor(f2, cv2.COLOR_BGR2GRAY))
            faces = cc.detectMultiScale(cv2.resize(g, (160, 90), interpolation=cv2.INTER_LINEAR), scaleFactor=1.25,
                                        minNeighbors=3, flags=0, minSize=(30, 30))
            ef = cv2.equalizeHist(cv2.resize(g, (320, 180), interpolation=cv2.INTER_LINEAR))
            n = 0
            for (x, y, w, h) in faces:
                x, y, w, h = int(x * 2), int(y * 2), int(w * 2), int(h * 2)
                top, down = int(round(h * 0.25)), int(round(h * 0.40))
                for roi in (ef[y + top:y + h - down, x:x + w // 2], ef[y + top:y + h - down, x + w // 2:x + w]):
                    if roi.size:
                        n += len(ce.detectMultiScale(roi, scaleFactor=1.1, minNeighbors=2, flags=0, minSize=(20, 20)))
            return n
        out["cfg2_eyes_in_faces_1280x720"]["cpu_frames_per_s"] = _timeit(cpu2, 60)

    # cfg4: tracker
    seq = [_pin(f) for f in synth.tracker_sequence(1280, 720, 8, seed=4)]
    e = nv.Element("nubotracker", local, cdir)
    st = {"i": 0}

    def trk():
        st["i"] += 1
        return e.process(seq[st["i"] % len(seq)], pts_ns=33_300_000 * st["i"])
    out["cfg4_tracker_1280x720_bgra"] = {"frames_per_s": _timeit(trk, 300)}
    e.close()
    # the fused tracker kernel against the HBM roofline: algorithmic bytes 7 * S (SURVEY 8d: BGRA in 4, previous gray in 1,
    # gray out 1, mask / labels >= 1) over its CUDA-event time, isolated (one stream)
    tctx = nv.Context(local, 1280, 720)
    tctx.set_profile(True)
    kms = []
    for i in range(40):
        tctx.tracker_process(seq[i % len(seq)], 33.3 * (i + 1))
        if i >= 8:
            kms.append(tctx.tracker_kernel_ms())
    tctx.close()
    if kms:
        k_ms = statistics.median(kms)
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
        ab = 7 * 1280 * 720
        tj = {}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
        out["cfg4_tracker_1280x720_bgra"]["roofline"] = {
            "bound": "hbm", "kernel": "k_trk_fused<0> (one launch per frame)", "achieved": ab / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": ab / (k_ms * 1e-3) / 1e9 / peak, "kernel_ms": k_ms, "algorithmic_bytes_per_launch": ab,
            "bytes_moved_by_design": 8 * 1280 * 720, "traffic": tj.get("tracker_dram_bytes_per_frame")}
    if cv2 is not None:
        prev = {"g": cv2.cvtColor(seq[0], cv2.COLOR_BGRA2GRAY), "i": 0}

        def cpu4():
            prev["i"] += 1
            g = cv2.cvtColor(seq[prev["i"] % len(seq)], cv2.COLOR_BGRA2GRAY)
            m = cv2.threshold(cv2.absdiff(g, prev["g"]), 20, 255, cv2.THRESH_BINARY)[1]
            r = cv2.connectedComponentsWithStats(m, connectivity=4)
            prev["g"] = g
            return r
        out["cfg4_tracker_1280x720_bgra"]["cpu_frames_per_s"] = _timeit(cpu4, 200)
        out["cpu"] = {"cores": cv2.getNumThreads(), "via": "cv2 %s, the reference's call sequences" % cv2.__version__}
    # the same elements as concurrent streams: one host thread per stream (ctypes drops the GIL inside the library),
    # every stream its own element, contexts and CUDA streams — what a media server with several pipelines does
    import threading

    def concurrent(factory, frames_of, nstreams, nframes, yuv=None, **props):
        els = [nv.Element(factory, local, cdir) for _ in range(nstreams)]
        for e_ in els:
            for k, v in props.items():
                e_.set(k, v)

        def loop(i, n):
            fr = frames_of(i)
            for j in range(n):
                if yuv:
                    els[i].process_yuv(fr[j % len(fr)], yuv, pts_ns=33_300_000 * (j + 1))
                else:
                    els[i].process(fr[j % len(fr)], pts_ns=33_300_000 * (j + 1))
        for i in range(nstreams):
            loop(i, 3)
        th = [threading.Thread(target=loop, args=(i, nframes)) for i in range(nstreams)]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        dt = time.perf_counter() - t0
        for e_ in els:
            e_.close()
        return nstreams * nframes / dt

    NS = 8
    out["cfg2_eyes_in_faces_1280x720"]["frames_per_s_%d_streams" % NS] = concurrent("nuboeyedetector", lambda i: [f2], NS, 150)
    out["cfg4_tracker_1280x720_bgra"]["frames_per_s_%d_streams" % NS] = concurrent("nubotracker", lambda i: seq, NS, 300)
    # the same sequence handed over as NV12 planes (nv_element_transform_frame_yuv): 1.5 instead of 4 bytes per pixel
    seq_nv12 = [_pin(synth.to_yuv420(np.ascontiguousarray(f[..., :3]), "NV12")) for f in seq]
    pl_nv12 = [synth.yuv420_planes(b, 1280, 720, "NV12") for b in seq_nv12]
    out["cfg4_tracker_1280x720_bgra"]["frames_per_s_%d_streams_nv12" % NS] = concurrent("nubotracker", lambda i: pl_nv12, NS, 300, yuv="NV12")
    out["cfg1_face_640x480_defaults"]["frames_per_s_%d_streams" % NS] = concurrent("nubofacedetector", lambda i: [f1], NS, 300)
    shutil.rmtree(cdir, ignore_errors=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8, help="frames (= per-stream contexts) per step per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true", help="skip the cfg5 720p-streams auxiliary measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the rectangles of the last timed step, one DIR/faces_frame<i>.npy "
                                                           "(float64, rows x y w h) per frame of rank 0's batch")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import nubovca as nv
    if not torch.cuda.is_available() or nv.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: nubovca has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from nubovca import shard
    B = args.batch
    frames = make_frames(B, rank)
    casc = nv.Cascade(FACE_XML)
    ctxs = [nv.Context(local, W, H) for _ in range(B)]
    for c in ctxs:
        c.set_profile(True)
    # device-resident inputs (value) and pinned host inputs (e2e)
    d_frames = [torch.from_numpy(f).cuda() for f in frames]
    h_frames = [torch.from_numpy(f).pin_memory() for f in frames]
    h_np = [t.numpy() for t in h_frames]
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # A step = one pass of the hot path over the batch: every context takes one new frame.  The loop is software-
    # pipelined the way a streaming server runs it: a context's previous frame is collected right before its next
    # one is submitted, so the B streams stay out of phase (different kernels of different frames share the GPU) and
    # nothing drains between steps.  K steps = K x B frames submitted AND collected inside the timed region.
    pending = [False] * B
    out = [None] * B

    def run_steps(nsteps, submit, on_collect=None):
        for _ in range(nsteps):
            for i, c in enumerate(ctxs):
                if pending[i]:
                    out[i] = c.face_collect()
                    if on_collect:
                        on_collect(c)
                submit(i, c)
                pending[i] = True

    def drain(on_collect=None):
        for i, c in enumerate(ctxs):
            if pending[i]:
                out[i] = c.face_collect()
                pending[i] = False
                if on_collect:
                    on_collect(c)

    def submit_device(i, c):
        c.face_submit_device(casc, d_frames[i].data_ptr(), W, H, 3 * W, **PARAMS)

    def submit_host(i, c):
        c.face_submit(casc, h_np[i], **PARAMS)

    # ---- value: inputs resident in HBM -------------------------------------------------------
    run_steps(args.warmup, submit_device); drain()
    launches0 = sum(c.counters()["launches"] for c in ctxs)
    stage_acc = {}

    def acc_stage(c):
        for k, v in c.stage_times().items():
            stage_acc.setdefault(k, []).append(v)
    e0, e1s = nv.Event(), [nv.Event() for _ in ctxs]
    sampler = ClockSampler(local); sampler.start()
    barrier()
    ctxs[0].record(e0)
    run_steps(args.steps, submit_device, acc_stage); drain(acc_stage)
    for c, e in zip(ctxs, e1s):
        c.record(e)
    ms_dev = max(e0.elapsed_ms(e) for e in e1s)
    barrier()
    launches = sum(c.counters()["launches"] for c in ctxs) - launches0
    nfaces = [len(o) for o in out]
    out_d = list(out)

    # ---- e2e: host frames through the C ABI, copies inside the timed region ---------------------
    run_steps(args.warmup, submit_host); drain()
    barrier()
    t0 = time.perf_counter()
    ctxs[0].record(e0)
    run_steps(args.steps, submit_host); drain()
    for c, e in zip(ctxs, e1s):
        c.record(e)
    ms_e2e_dev = max(e0.elapsed_ms(e) for e in e1s)
    torch.cuda.synchronize()
    ms_e2e = max(ms_e2e_dev, 1e3 * (time.perf_counter() - t0))       # host copies count too
    barrier()
    clocks = sampler.stop()                       # sampled across both timed regions
    assert all((a == b).all() for a, b in zip(out_d, out))
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for i, o in enumerate(out):
            np.save(os.path.join(args.dump_outputs, f"faces_frame{i}.npy"), np.asarray(o, np.float64).reshape(-1, 4))
    # (a) the GPU's rectangles for this rank's frames against the CPU arm's (cv2, the reference's call sequence) in this run
    parity = None
    if rank == 0:
        try:
            exp = cv2_rects(frames)
            same = [rect_set(o) == e for o, e in zip(out, exp)]
            parity = {"frames": len(same), "identical": int(sum(same)), "rectangles": int(sum(len(e) for e in exp)),
                      "against": "cv2 %s, kmsfacedetect.cpp:805-811 call sequence, same frames, rectangle sets compared exactly" % __import__("cv2").__version__}
        except ImportError:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import oracle as O
            oc = O.Cascade(FACE_XML)
            exp = [rect_set(O.face_process(f, oc, **PARAMS)[0]) for f in frames[:2]]
            same = [rect_set(o) == e for o, e in zip(out, exp)]
            parity = {"frames": len(same), "identical": int(sum(same)), "rectangles": int(sum(len(e) for e in exp)), "against": "oracle/nubo_oracle.c (cv2 not importable)"}

    # isolated per-stage times: the same step with ONE stream in flight (no interleaving between contexts)
    iso_acc = {}
    for _ in range(3):
        for c, d in zip(ctxs[:2], d_frames[:2]):
            c.face_submit_device(casc, d.data_ptr(), W, H, 3 * W, **PARAMS)
            c.face_collect()
            for k, v in c.stage_times().items():
                iso_acc.setdefault(k, []).append(v)

    # auxiliary: BASELINE config 5 per GPU — 32 concurrent 1280x720 streams at the element's
    # width-to-process 640, host frames through the C ABI; streams@30fps = frames/s / 30
    aux = None
    if not args.no_aux:
        synth = load_synth()
        S5 = 32
        mine = shard.streams_of_rank(S5 * world, world, rank)
        f5 = [synth.frame(1280, 720, 3, 1000 + s) for s in mine]          # SURVEY 8(d): stream i uses seed 1000 + i
        h5 = [torch.from_numpy(f).pin_memory().numpy() for f in f5]
        c5 = [nv.Context(local, 1280, 720) for _ in mine]
        p5 = dict(width_to_process=640, scale_factor=1.25, min_neighbors=3, min_size=None)

        def run5(submit):
            def step5():
                for i, c in enumerate(c5):
                    submit(c, i)
                return [c.face_collect() for c in c5]
            for _ in range(3):
                step5()
            barrier()
            t5 = time.perf_counter()
            n5 = 10
            for _ in range(n5):
                step5()
            torch.cuda.synchronize()
            ms5 = 1e3 * (time.perf_counter() - t5)
            barrier()
            return shard.aggregate_throughput(len(c5) * n5, ms5, dist, "cuda")[0]
        fps5 = run5(lambda c, i: c.face_submit(casc, h5[i], **p5))
        aux = {"metric": "720p streams@30fps (cfg5: 1280x720 -> 640x360, sf 1.25, element defaults otherwise)",
               "streams_per_gpu_in_flight": S5, "frames_per_s": fps5, "streams_at_30fps": fps5 / 30.0,
               "timing": "host wall clock, H2D + D2H included"}
        # the same streams handed over as the decoder's NV12 planes (nv_face_submit_yuv: 1.5 instead of 3 bytes per
        # pixel across PCIe; result = the reference block on cvtColor(COLOR_YUV2BGR_NV12), tests/test_yuv_ingest.py)
        y5 = [_pin(synth.to_yuv420(f, "NV12")) for f in f5]
        pl5 = [synth.yuv420_planes(b, 1280, 720, "NV12") for b in y5]
        fps5y = run5(lambda c, i: c.face_submit_yuv(casc, pl5[i], "NV12", **p5))
        aux["nv12_ingest"] = {"frames_per_s": fps5y, "streams_at_30fps": fps5y / 30.0, "h2d_bytes_per_frame": 1280 * 720 * 3 // 2}
        for c in c5:
            c.close()
        # the same measurement from native host threads (tools/streams_bench.cpp: no interpreter between the calls;
        # what a media server's streaming threads do), BGR and NV12, checked by the number of rectangles found
        tool = os.path.join(ROOT, "nubomedia-vca_b200", "lib", "streams_bench")
        if os.path.exists(tool):
            import tempfile
            exp = [len(r) for r in (lambda c: [c.face_detect(casc, f, **p5) for f in f5])(nv.Context(local, 1280, 720))]
            iters, nthr = 200, 4
            nat = {}
            with tempfile.TemporaryDirectory(prefix="nubovca_s5_") as td:
                for fmt, blobs in (("bgr", f5), ("nv12", y5)):
                    path = os.path.join(td, fmt + ".raw")
                    with open(path, "wb") as fh:
                        for b in blobs:
                            fh.write(np.ascontiguousarray(b).tobytes())
                    barrier()
                    try:
                        r = subprocess.run([tool, "--frames-file", path, "--nframes", str(len(blobs)), "--fmt", fmt, "--xml", FACE_XML,
                                            "--gpu", str(local), "--streams", str(S5), "--threads", str(nthr), "--iters", str(iters)],
                                           capture_output=True, text=True, timeout=120)
                    except Exception as ex:                   # noqa: BLE001
                        r = subprocess.CompletedProcess([tool], 1, "", repr(ex))
                    # a failure here must not take the headline line down with it: every rank still joins the reduction
                    j = {"frames": 0, "seconds": 1.0, "rects": -1, "h2d_bytes_per_frame": 0}
                    err = None
                    if r.returncode == 0:
                        j = json.loads(r.stdout.strip().splitlines()[-1])
                    else:
                        err = r.stderr[-300:]
                    fps, _ = shard.aggregate_throughput(j["frames"], 1e3 * j["seconds"], dist, "cuda")
                    nat[fmt] = {"frames_per_s": fps, "streams_at_30fps": fps / 30.0, "h2d_bytes_per_frame": j["h2d_bytes_per_frame"]}
                    if fmt == "bgr":       # NV12 frames are a different image (quantised chroma): only the BGR count is pinned here
                        want = sum(exp[(s_ + it) % len(exp)] for s_ in range(S5) for it in range(iters))
                        nat[fmt]["rects_match_python_path"] = j["rects"] == want
                    if err:
                        nat[fmt]["error"] = err
            nat["host_threads_per_gpu"] = nthr
            nat["streams_per_gpu_in_flight"] = S5
            aux["native_host_threads"] = nat
        # the per-GPU ingest rate the figures above imply, and the same streams with the frames already in HBM: the compute
        # ceiling of a GPU at config 5, which separates "the kernels" from "getting the frames there" at every N
        aux["h2d_gb_per_s_per_gpu"] = {"bgr_python": fps5 / world * 1280 * 720 * 3 / 1e9, "nv12_python": fps5y / world * 1280 * 720 * 1.5 / 1e9}
        if "native_host_threads" in aux:
            for k_ in ("bgr", "nv12"):
                aux["h2d_gb_per_s_per_gpu"][k_ + "_native"] = aux["native_host_threads"][k_]["frames_per_s"] / world * \
                    aux["native_host_threads"][k_]["h2d_bytes_per_frame"] / 1e9
        c5 = [nv.Context(local, 1280, 720) for _ in mine]
        d5 = [torch.from_numpy(f).cuda() for f in f5]
        fps5d = run5(lambda c, i: c.face_submit_device(casc, d5[i].data_ptr(), 1280, 720, 3 * 1280, **p5))
        aux["device_resident"] = {"frames_per_s": fps5d, "streams_at_30fps": fps5d / 30.0,
                                  "note": "same 32 streams per GPU, frames already in HBM (nv_face_submit_device): no ingest"}
        for c in c5:
            c.close()
        del d5
        if rank == 0 and world == 1 and os.path.exists(tool):
            # the element's own call shape (VERDICT r1 #6): one synchronous nv_face_detect per buffer from T host threads, each
            # with its own streams, on PAGEABLE frames (what GStreamer hands an element), next to page-locked and
            # cudaHostRegister'ed memory.  C ABI, native threads, wall clock, copies included.
            import tempfile
            shaped = {}
            with tempfile.TemporaryDirectory(prefix="nubovca_shape_") as td:
                def blob(name, arrs):
                    path_ = os.path.join(td, name)
                    with open(path_, "wb") as fh:
                        for b_ in arrs:
                            fh.write(np.ascontiguousarray(b_).tobytes())
                    return path_, len(arrs)
                cases = {"cfg5_1280x720_w2p640": (blob("c5.raw", f5), ["--width", "1280", "--height", "720", "--width-to-process", "640"], 40),
                         "cfg1_640x480_defaults": (blob("c1.raw", [synth.frame(640, 480, 4, 1)]), ["--width", "640", "--height", "480", "--width-to-process", "160"], 200),
                         "cfg3_1920x1080_full": (blob("c3.raw", frames), ["--width", "1920", "--height", "1080", "--width-to-process", "1920",
                                                                        "--scale-factor", "1.1", "--min-size", "24"], 25)}
                for cname, ((path_, nfr), geo, iters_) in cases.items():
                    shaped[cname] = {}
                    for mem in ("pageable", "registered", "pinned"):
                        for thr in (1, 4, 32):
                            if mem == "registered" and thr != 4:
                                continue
                            try:
                                r = subprocess.run([tool, "--frames-file", path_, "--nframes", str(nfr), "--fmt", "bgr", "--xml", FACE_XML, "--gpu", str(local),
                                                    "--streams", str(max(thr, 4) if cname.startswith("cfg5") else thr), "--threads", str(thr), "--iters", str(iters_),
                                                    "--warmup", "3", "--sync", "1", "--memory", mem] + geo, capture_output=True, text=True, timeout=180)
                                shaped[cname]["%s_%dthr" % (mem, thr)] = json.loads(r.stdout.strip().splitlines()[-1])["frames_per_s"] if r.returncode == 0 else r.stderr[-200:]
                            except Exception as ex:           # noqa: BLE001
                                shaped[cname]["%s_%dthr" % (mem, thr)] = repr(ex)
            shaped["unit"] = "frames/s; one blocking nv_face_detect per buffer, T native host threads with their own streams"
            aux["element_shaped_sync_calls"] = shaped
        if rank == 0 and world == 1:
            try:                                         # auxiliary figures never take the headline line down
                aux["other_configs_one_stream"] = aux_other_configs(nv, local, world)
            except Exception as ex:                      # noqa: BLE001
                aux["other_configs_one_stream"] = {"error": repr(ex)}
            if not args.no_cpu_baseline:
                try:
                    aux["cpu_cfg5"] = cpu_cfg5()
                except Exception as ex:                  # noqa: BLE001
                    aux["cpu_cfg5"] = {"error": repr(ex)}

    total_frames = B * args.steps
    value, ms_dev = shard.aggregate_throughput(total_frames, ms_dev, dist, "cuda")
    e2e, ms_e2e = shard.aggregate_throughput(total_frames, ms_e2e, dist, "cuda")

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        levels = ctxs[0].levels()
        ab = algorithmic_bytes(levels, W * H, 3, W * H)
        med = {k: statistics.median(v) for k, v in stage_acc.items()}
        iso = {k: statistics.median(v) for k, v in iso_acc.items()}
        iso_casc = iso.get("cascade_stage0", 0) + iso.get("cascade_tiles", 0) + iso.get("cascade_tail", 0)
        traffic, onchip = None, None
        casc_names = "k_stage0_tiles<2> + k_stage0_tiles<1> + k_stage0_chain + k_cascade_classes<2> + k_cascade_wide<1, 128x64> + k_cascade_tail_fast"
        tpath = os.path.join(ROOT, "profiles", "traffic.json")          # counters from the committed ncu --set full capture
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic = tj.get("cascade_dram_bytes_per_frame")
            if tj.get("cascade_kernels"):
                casc_names = " + ".join(tj["cascade_kernels"])
            wf = tj.get("tile_shared_wavefronts_per_frame")
            wi = tj.get("tile_warp_instructions_per_frame")
            if wf and wi and iso.get("cascade_tiles", 0) > 0:
                # what actually bounds the bulk kernels (k_cascade_classes on ystep-2 levels, k_cascade_wide on ystep-1 levels): warp-instruction issue (4 per SM and
                # clock) first, the shared-memory pipe (one 128-byte wavefront per SM and clock) second
                clk = (clocks.get("sm_max_mhz") or 1965.0) * 1e6
                t = iso["cascade_tiles"] * 1e-3
                onchip = {"bound": "instruction issue", "achieved": wi / t / 1e9, "peak": 148 * 4 * clk / 1e9,
                          "unit": "G warp-instructions/s", "frac": wi / t / (148 * 4 * clk),
                          "warp_instructions_per_frame": wi,
                          "shared_memory": {"achieved": wf * 128 / t / 1e12, "peak": 148 * 128 * clk / 1e12, "unit": "TB/s",
                                            "frac": wf / t / (148 * clk), "wavefronts_per_frame": wf,
                                            "conflict_replays_per_frame": tj.get("tile_shared_bank_conflict_wavefronts_per_frame")},
                          "source": "counts from profiles/traffic.json (ncu), time = stage_ms_isolated.cascade_tiles"}
                fw = tj.get("frame_warp_instructions_per_frame")
                if fw and value > 0:
                    # the same bound for the timed region as a whole: every kernel's warp instructions of a frame x the frames
                    # one GPU finished per second in it (eight frames in flight: the kernels of different frames share the SMs)
                    onchip["timed_region"] = {"achieved": fw * (value / world) / 1e9, "frac": fw * (value / world) / (148 * 4 * clk),
                                              "unit": "G warp-instructions/s", "warp_instructions_per_frame": fw,
                                              "source": tj.get("frame_warp_instructions_source")}
        casc_ms = med.get("cascade_stage0", 0) + med.get("cascade_tiles", 0) + med.get("cascade_tail", 0)
        frame_ms = sum(med.values())
        achieved = ab["cascade"] / (casc_ms * 1e-3) / 1e9 if casc_ms > 0 else None
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8 pixels, int32/u32 integrals, f32 features, f64 stage sums", "data": "synthetic",
            "config": CONFIG,
            "config_detail": {"frames_per_step_per_gpu": B, "streams": "one CUDA stream + context per frame slot; a slot's previous frame is collected right before its next one is submitted",
                              "working_set_mb_per_context": (16 * ab["integral_px"]) >> 20,
                              "levels": len(levels), "windows_per_frame": ctxs[0].counters()["windows"],
                              "faces_found_per_frame": nfaces},
            "parity_in_run": parity,
            # whole-job figures: every rank runs the same batch shape, so bytes and launches are rank 0's times world
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": world * B * W * H * 3,
                    "d2h_bytes_per_step": world * B * (16 + 1024 * 16), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches) * world,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "cascade (" + casc_names + ")",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                         "traffic": traffic, "peak_source": peak_src,
                         "kernel_ms_isolated": iso_casc,
                         "achieved_isolated": ab["cascade"] / (iso_casc * 1e-3) / 1e9 if iso_casc > 0 else None,
                         "note": "kernel_ms is the median CUDA-event time inside the timed region, where the other "
                                 "contexts' kernels interleave on the GPU; kernel_ms_isolated is the same stage with one "
                                 "stream in flight.  The cascade re-reads integral patches from shared memory and is "
                                 "bound by instruction issue, so its HBM fraction is small by construction (DESIGN.md §4); "
                                 "`onchip` is the roofline that binds it.",
                         "algorithmic_bytes_per_launch": ab["cascade"], "kernel_ms": casc_ms,
                         "frame_algorithmic_bytes": ab["frame_total"], "frame_kernel_ms": frame_ms,
                         "frame_frac": ab["frame_total"] / (frame_ms * 1e-3) / 1e9 / peak if frame_ms > 0 else None},
            "stage_ms_median": med,
            "stage_ms_isolated": iso,
        }
        if onchip:
            line["roofline"]["onchip"] = onchip
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            if tj.get("tile_lts_bytes_per_frame") and iso.get("cascade_tiles", 0) > 0:
                # measured L2 and L1/TEX traffic of the bulk kernel (ncu lts__t_bytes.sum / l1tex__t_bytes.sum, profiles/) over
                # its isolated CUDA-event time, against the peaks ncu reports for this part in the same capture
                t = iso["cascade_tiles"] * 1e-3
                line["roofline"]["l2"] = {"achieved": tj["tile_lts_bytes_per_frame"] / t / 1e9, "unit": "GB/s",
                                          "bytes_per_frame": tj["tile_lts_bytes_per_frame"],
                                          "ncu_pct_of_peak_per_launch": tj.get("lts_ncu_pct_of_peak"), "source": tj.get("lts_source")}
                if tj.get("tile_l1tex_bytes_per_frame"):
                    line["roofline"]["l1tex"] = {"achieved": tj["tile_l1tex_bytes_per_frame"] / t / 1e9, "unit": "GB/s",
                                                 "bytes_per_frame": tj["tile_l1tex_bytes_per_frame"],
                                                 "ncu_pct_of_peak_per_launch": tj.get("l1tex_ncu_pct_of_peak")}
        if aux:
            line["aux"] = aux
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(frames)
        print(json.dumps(line), flush=True)
    for c in ctxs:
        c.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
