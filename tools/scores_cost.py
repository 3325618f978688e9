"""Cost of detection scores (nv_ctx_set_scores): the same calls with scores off and on, alternated within one process.

  - config 1 (640x480 -> 160x120, element defaults) and a 96x64 ROI detect: microseconds per blocking call
    (one stream, page-locked host frames, graph replay);
  - config 3 (1920x1080, processing width 1920, sf 1.1, min 24x24): frames/s of blocking calls on one context with the
    frame resident in HBM;
  - the candidate sort's kernel time (k_group_fused on the small plan, k_cand_sort on config 3), from torch.profiler.

Prints one JSON line.  Usage: python tools/scores_cost.py [rounds]"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nubomedia-vca_b200", "python"))
import nubovca as nv  # noqa: E402
from nubovca import synth  # noqa: E402
import torch  # noqa: E402

rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5


def pin(a):
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def per_call_us(fn, n, warm=20):
    for _ in range(warm):
        fn()
    t = time.perf_counter()
    for _ in range(n):
        fn()
    return 1e6 * (time.perf_counter() - t) / n


casc = nv.Cascade(os.path.join(ROOT, "nubomedia-vca_b200", "cascades", "haarcascade_frontalface_alt.xml"))
ctx = nv.Context(0, 1920, 1080)
f1 = pin(synth.frame(640, 480, 4, 1))
roi = pin(synth.frame(96, 64, 1, 5, smin=0.5, smax=0.9)[..., 0])
f3 = torch.from_numpy(synth.frame(1920, 1080, 6, 3)).cuda()


def cfg1():
    ctx.face_detect(casc, f1, 160, 1.25, 3, None)


def roi96():
    ctx.detect_multiscale(casc, roi, 1.1, 2, (20, 20))


def cfg3():
    ctx.face_submit_device(casc, f3.data_ptr(), 1920, 1080, 5760, 1920, 1.1, 3, (24, 24))
    ctx.face_collect()


res = {k: {"off": [], "on": []} for k in ("cfg1_us", "roi96x64_us", "cfg3_fps")}
for r in range(rounds):
    for mode in ("off", "on") if r % 2 == 0 else ("on", "off"):
        ctx.set_scores(mode == "on")
        res["cfg1_us"][mode].append(per_call_us(cfg1, 400))
        res["roi96x64_us"][mode].append(per_call_us(roi96, 400))
        res["cfg3_fps"][mode].append(1e6 / per_call_us(cfg3, 60, 5))

# kernel times of the candidate sort, scores off and on (separate profiled runs, not part of the timings above)
kern = {}
for mode in ("off", "on"):
    ctx.set_scores(mode == "on")
    for fn in (cfg1, cfg3):
        for _ in range(5):
            fn()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(50):
            cfg1()
        for _ in range(20):
            cfg3()
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        for name in ("k_group_fused", "k_cand_sort", "k_group"):
            if name + "<" in ev.key or ev.key.startswith(name + "("):
                kern.setdefault(f"{name}_us", {})[mode] = round(ev.device_time_total / max(ev.count, 1), 2)
ctx.close()

out = {k: {m: round(float(np.median(v)), 2) for m, v in d.items()} for k, d in res.items()}
out.update(kern)
out["gpu"] = torch.cuda.get_device_name(0)
print(json.dumps(out))
