"""Config-1 throughput of batched detection against the one-frame-per-call ways to reach the same work.

BASELINE config 1: 640x480 BGR frames processed at 160x120 with haarcascade_frontalface_alt (scale 1.25, 3 neighbours).
Variants, each over N frames per step:
  batch_pinned   nv_face_detect_batch on page-locked host frames (one call per step)
  batch_device   nv_face_detect_batch on a CUDA uint8 tensor [N, 480, 640, 3]
  loop_blocking  N blocking nv_face_detect calls on page-locked frames, one context
  inflight_pinned / inflight_device  N contexts: N face_submit / face_submit_device, then N face_collect, one thread
The variants alternate within every round (the host is shared); frames/s is the median over the rounds.  The card's name
and power limit are read in the same run and printed with the table.

    python tools/batch_throughput.py [--sizes 1,8,32,128] [--rounds 7] [--seconds 0.3] [--out FILE.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nubomedia-vca_b200", "python"))
import nubovca as nv  # noqa: E402
from nubovca import synth  # noqa: E402

W, H = 640, 480


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def pinned(shape):
    ptr = C.c_void_p()
    size = int(np.prod(shape))
    if nv._lib.nv_host_alloc(size, C.byref(ptr)) != 0:
        raise RuntimeError("nv_host_alloc failed")
    return np.ctypeslib.as_array((C.c_uint8 * size).from_address(ptr.value)).reshape(shape), ptr


def rate(step, n, seconds):
    step()                                                  # warm: plans, graphs
    step()
    k, t0 = 0, time.perf_counter()
    while True:
        step(); k += 1
        dt = time.perf_counter() - t0
        if dt >= seconds:
            return k * n / dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,8,32,128")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--seconds", type=float, default=0.3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if nv.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    casc = nv.Cascade("haarcascade_frontalface_alt.xml")
    sizes = [int(s) for s in a.sizes.split(",")]
    nmax = max(sizes)
    host, hptr = pinned((nmax, H, W, 3))
    for i in range(nmax):
        host[i] = synth.frame(W, H, 1 + i % 4, 2000 + i)
    dev = torch.from_numpy(np.ascontiguousarray(host)).cuda()
    torch.cuda.synchronize()
    bctx = nv.Context(0, W, H)
    sctx = nv.Context(0, W, H)
    ctxs = [nv.Context(0, W, H) for _ in range(nmax)]
    out = {"card": card(), "sizes": sizes, "rounds": a.rounds, "frames_per_s": {}}
    for n in sizes:
        hb, db = host[:n], dev[:n]
        ref = bctx.face_detect_batch(casc, hb)
        assert all((r == sctx.face_detect(casc, hb[i])).all() for i, r in enumerate(ref))

        def batch_pinned():
            bctx.face_detect_batch(casc, hb)

        def batch_device():
            bctx.face_detect_batch(casc, db)

        def loop_blocking():
            for i in range(n):
                sctx.face_detect(casc, hb[i])

        def inflight_pinned():
            for i in range(n):
                ctxs[i].face_submit(casc, hb[i])
            for i in range(n):
                ctxs[i].face_collect()

        stride = dev.stride(1)

        def inflight_device():
            for i in range(n):
                ctxs[i].face_submit_device(casc, dev[i].data_ptr(), W, H, stride)
            for i in range(n):
                ctxs[i].face_collect()

        variants = dict(batch_pinned=batch_pinned, batch_device=batch_device, loop_blocking=loop_blocking,
                        inflight_pinned=inflight_pinned, inflight_device=inflight_device)
        res = {k: [] for k in variants}
        for _ in range(a.rounds):
            for k, f in variants.items():
                res[k].append(rate(f, n, a.seconds))
        out["frames_per_s"][n] = {k: dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v))) for k, v in res.items()}
        print(f"N={n:4d} " + "  ".join(f"{k} {np.median(v):9.0f} [{min(v):.0f}-{max(v):.0f}]" for k, v in res.items()), flush=True)
    print("card, power limit:", out["card"])
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(out, open(a.out, "w"), indent=1)
    for c in ctxs + [bctx, sctx]:
        c.close()
    nv._lib.nv_host_free(hptr)


if __name__ == "__main__":
    main()
