"""Throughput of the batched tracker against the one-frame-per-call ways to track N streams, at 1280x720 BGRA.

Every stream is its own synth.tracker_sequence (seed 3000 + i, cfg4 parameters, 30 fps timestamps).  Variants, each over N
frames per step (one frame of every stream):
  batch_pinned      nv_tracker_process_batch on page-locked host frames (one call per step)
  batch_device      nv_tracker_process_batch on a CUDA uint8 tensor [N, 720, 1280, 4]
  loop_blocking     N blocking nv_tracker_process calls over N contexts, one thread, page-locked frames
  threads_pinned    N host threads, one context each, nv_tracker_process on page-locked frames
  threads_device    the same threads, on the device frames (nv_tracker_process_yuv cannot take BGRA device frames, so each
                    thread runs nv_tracker_process_batch with N = 1 on its own context: one launch, one synchronise)
With --yuv, the streams as NV12 (synth.to_yuv420) also run as
  batch_nv12_pinned / batch_nv12_device   nv_tracker_process_batch_yuv on page-locked host frames / a CUDA tensor
The variants alternate within every round (the host is shared); frames/s is the median over the rounds, with min and max.
The batched kernel's own time (nv_ctx_get_tracker_kernel_ms, CUDA events around the launch) is reported per N for the
device batch, from a separate profiled pass.  The card's name and power limit are read in the same run.

    python tools/tracker_batch_throughput.py [--sizes 1,8,32,128] [--rounds 5] [--seconds 0.3] [--yuv] [--out FILE.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nubomedia-vca_b200", "python"))
import nubovca as nv  # noqa: E402
from nubovca import synth  # noqa: E402

W, H, NF = 1280, 720, 4                                    # NF frames per stream, played in a loop


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
    step(); step()                                          # warm: slot buffers, frame slots
    k, t0 = 0, time.perf_counter()
    while True:
        step(); k += 1
        dt = time.perf_counter() - t0
        if dt >= seconds:
            return k * n / dt


class Threads:
    """n host threads, each running fn(i) once per step; the step ends when every thread has finished its frame."""
    def __init__(self, n, fn):
        self.n, self.fn = n, fn
        self.go = [threading.Event() for _ in range(n)]
        self.done = threading.Barrier(n + 1)
        self.stop = False
        self.err = None
        self.th = [threading.Thread(target=self._run, args=(i,), daemon=True) for i in range(n)]
        for t in self.th:
            t.start()

    def _run(self, i):
        while True:
            self.go[i].wait(); self.go[i].clear()
            if self.stop:
                return
            try:
                self.fn(i)
            except Exception as e:                          # reported by step()
                self.err = e
            self.done.wait()

    def step(self):
        for g in self.go:
            g.set()
        self.done.wait()
        if self.err:
            raise self.err

    def close(self):
        self.stop = True
        for g in self.go:
            g.set()
        for t in self.th:
            t.join()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,8,32,128")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seconds", type=float, default=0.3)
    ap.add_argument("--yuv", action="store_true", help="add the NV12 variants")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if nv.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    sizes = [int(s) for s in a.sizes.split(",")]
    nmax = max(sizes)
    host, hptr = pinned((NF, nmax, H, W, 4))                # frame f of every stream, stream by stream
    for i in range(nmax):
        for f, fr in enumerate(synth.tracker_sequence(W, H, NF, seed=3000 + i, noise=300)):
            host[f, i] = fr
    dev = torch.from_numpy(np.ascontiguousarray(host)).cuda()
    if a.yuv:
        yhost, yptr = pinned((NF, nmax, H * 3 // 2, W))
        for f in range(NF):
            for i in range(nmax):
                yhost[f, i] = synth.to_yuv420(np.ascontiguousarray(host[f, i, :, :, :3]), "NV12")
        ydev = torch.from_numpy(np.ascontiguousarray(yhost)).cuda()
    torch.cuda.synchronize()
    out = {"card": card(), "size": [W, H], "sizes": sizes, "rounds": a.rounds, "frames_per_s": {}, "kernel_ms": {}}
    bctx = nv.Context(0, W, H)
    ctxs = [nv.Context(0, W, H) for _ in range(nmax)]
    clock = {"f": 0}

    def ts():
        return 1000.0 + 33.3 * clock["f"]

    for n in sizes:
        # parity first: the device batch against N single contexts over one pass of the sequences
        bctx.tracker_reset_batch()
        for c in ctxs[:n]:
            c.tracker_reset()
        for f in range(NF):
            got = bctx.tracker_process_batch(dev[f, :n], [1000.0 + 33.3 * f] * n)
            for i in range(n):
                assert (got[i] == ctxs[i].tracker_process(host[f, i], 1000.0 + 33.3 * f)).all(), (n, f, i)

        def advance():
            clock["f"] += 1
            return clock["f"] % NF

        def batch_pinned():
            f = advance()
            bctx.tracker_process_batch(host[f, :n], [ts()] * n)

        def batch_device():
            f = advance()
            bctx.tracker_process_batch(dev[f, :n], [ts()] * n)

        def loop_blocking():
            f = advance()
            for i in range(n):
                ctxs[i].tracker_process(host[f, i], ts())

        th_pinned = Threads(n, lambda i: ctxs[i].tracker_process(host[clock["f"] % NF, i], ts()))
        th_device = Threads(n, lambda i: ctxs[i].tracker_process_batch(dev[clock["f"] % NF, i:i + 1], [ts()]))

        def threads_pinned():
            advance()
            th_pinned.step()

        def threads_device():
            advance()
            th_device.step()

        variants = dict(batch_pinned=batch_pinned, batch_device=batch_device, loop_blocking=loop_blocking,
                        threads_pinned=threads_pinned, threads_device=threads_device)
        if a.yuv:
            def batch_nv12_pinned():
                f = advance()
                bctx.tracker_process_batch_yuv(yhost[f, :n], "NV12", [ts()] * n)

            def batch_nv12_device():
                f = advance()
                bctx.tracker_process_batch_yuv(ydev[f, :n], "NV12", [ts()] * n)

            variants.update(batch_nv12_pinned=batch_nv12_pinned, batch_nv12_device=batch_nv12_device)
        res = {k: [] for k in variants}
        for _ in range(a.rounds):
            for k, fn in variants.items():
                res[k].append(rate(fn, n, a.seconds))
        th_pinned.close(); th_device.close()
        # the batched kernel alone: CUDA events around the launch, device frames
        bctx.set_profile(True)
        kms = []
        for _ in range(20):
            batch_device()
            kms.append(bctx.tracker_kernel_ms())
        bctx.set_profile(False)
        out["kernel_ms"][n] = dict(median=float(np.median(kms)), min=float(min(kms)), max=float(max(kms)))
        out["frames_per_s"][n] = {k: dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v))) for k, v in res.items()}
        print(f"N={n:4d} " + "  ".join(f"{k} {np.median(v):8.0f} [{min(v):.0f}-{max(v):.0f}]" for k, v in res.items())
              + f"  kernel {np.median(kms) * 1000:.0f} us", flush=True)
    print("card, power limit:", out["card"])
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)
    nv._lib.nv_host_free(hptr)
    if a.yuv:
        nv._lib.nv_host_free(yptr)


if __name__ == "__main__":
    main()
