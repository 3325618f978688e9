"""Randomised parity run of the nubotracker path (not part of the test suite): random frame sizes, strides, thresholds,
area / distance parameters, noise levels and timestamp gaps (history decay) over random sequences, through long-lived
contexts, against the CPU oracle.  Usage: python tools/fuzz_tracker.py [seconds] [seed] [--batch]
--batch: the batched tracker instead (nv_tracker_process_batch): random N, sizes, row pitches, per-slot parameters and
timestamp gaps, every slot against its own O.TrackerState; calls with fewer slots leave the higher slots waiting."""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "nubomedia-vca_b200", "python"), os.path.join(ROOT, "oracle")]
import nubovca as nv  # noqa: E402
import oracle as O  # noqa: E402
from nubovca import synth  # noqa: E402

BATCH = "--batch" in sys.argv
args = [a for a in sys.argv[1:] if a != "--batch"]
budget = float(args[0]) if len(args) > 0 else 60.0
seed = int(args[1]) if len(args) > 1 else 0
rng = np.random.default_rng(seed)
t0 = time.time()
nseq = nframes = bad = 0


def fuzz_batch():
    """One context, one frame size: random batch sizes over a few steps, every slot against its own oracle state."""
    global nframes, bad
    W = int(rng.integers(70, 700)) * 2; H = int(rng.integers(70, 380)) * 2
    nmax = int(rng.integers(1, 17)); steps = int(rng.integers(3, 9))
    pad = int(rng.choice([0, 0, 1, 3]))                                  # row pitch beyond W, in pixels
    seqs = [synth.tracker_sequence(W, H, steps, seed=int(rng.integers(1 << 30)), nsq=int(rng.integers(1, 5)),
                                   noise=int(rng.choice([0, 0, 20, 200, 2000]))) for _ in range(nmax)]
    prm = [dict(threshold=int(rng.choice([5, 20, 20, 60])), min_area=int(rng.choice([0, 50, 400])),
                max_area=int(rng.choice([3000, 30000, 10 ** 7])), distance=int(rng.choice([0, 35, 120]))) for _ in range(nmax)]
    ctx = nv.Context(0, W + pad, H)
    states = [O.TrackerState(W, H) for _ in range(nmax)]
    ts = [0.0] * nmax
    pos = [0] * nmax                                                      # next frame of each slot
    for _ in range(steps):
        n = int(rng.integers(1, nmax + 1))
        if any(pos[i] >= steps for i in range(n)):
            break
        wide = np.zeros((n, H, W + pad, 4), np.uint8)
        for i in range(n):
            wide[i, :, :W] = seqs[i][pos[i]]
            ts[i] += float(rng.choice([0.05, 33.3, 33.3, 100.0, 450.0]))   # stale history, and gaps beyond 200 ms
        got = ctx.tracker_process_batch(wide[:, :, :W], ts[:n], *[[p[k] for p in prm[:n]] for k in prm[0]])
        for i in range(n):
            exp, _, _ = states[i].process(seqs[i][pos[i]], ts[i], *prm[i].values())
            pos[i] += 1
            nframes += 1
            if got[i].shape != exp.shape or not (got[i] == exp).all():
                bad += 1
                print("MISMATCH", W, H, pad, n, i, prm[i], ts[i], got[i].tolist()[:4], exp.tolist()[:4], flush=True)
    ctx.close()


while BATCH and time.time() - t0 < budget:
    fuzz_batch()
    nseq += 1
while not BATCH and time.time() - t0 < budget:
    W = int(rng.integers(140, 700)) * 2; H = int(rng.integers(140, 380)) * 2
    n = int(rng.integers(3, 9))
    frames = synth.tracker_sequence(W, H, n, seed=int(rng.integers(1 << 30)), nsq=int(rng.integers(1, 5)),
                                    noise=int(rng.choice([0, 0, 20, 200, 2000])))
    thr = int(rng.choice([5, 20, 20, 60])); mina = int(rng.choice([0, 50, 400])); maxa = int(rng.choice([3000, 30000, 10 ** 7]))
    dist = int(rng.choice([0, 35, 120]))
    ctx = nv.Context(0, W, H)
    st = O.TrackerState(W, H)
    ts = 0.0
    for f in frames:
        ts += float(rng.choice([33.3, 33.3, 100.0, 450.0]))            # gaps beyond the 200 ms history window too
        a = ctx.tracker_process(f, ts, thr, mina, maxa, dist)
        b, _, _ = st.process(f, ts, thr, mina, maxa, dist)
        nframes += 1
        if a.shape != b.shape or not (a == b).all():
            bad += 1
            print("MISMATCH", W, H, thr, mina, maxa, dist, ts, a.tolist()[:4], b.tolist()[:4], flush=True)
    ctx.close()
    nseq += 1
print(f"fuzz_tracker{' --batch' if BATCH else ''}: {nseq} sequences, {nframes} frames, {bad} mismatches, seed {seed}, {time.time() - t0:.0f} s")
sys.exit(1 if bad else 0)
