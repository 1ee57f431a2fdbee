#!/usr/bin/env python
"""Randomised parity sweep (B200): random frame sizes and option sets through every window / level / box code path, faithful
arithmetic bit-for-bit against the C oracle, relaxed arithmetic bit-for-bit against oracle(144) where it is in effect, status and
vectors against the oracle's sampling.  usage: tools/fuzz_parity.py [cases=60] [seed=1]"""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tidalwave_b200 as tw
from oracle.oracle import FlowParam, RefOracle

n = int(sys.argv[1]) if len(sys.argv) > 1 else 60
rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 1)
O = RefOracle()
bad = 0


def draw_size():
    """Mostly ordinary frames; one in eight smaller than the window (a one-scale pyramid below 32 px), one in eight around
    the row-pitch classes: 2048 / 4096 (W = pitch: no padding after the last column) and above 4096 (runtime pitch, a multiple
    of 32 or ragged), short so the oracle stays fast."""
    r = int(rng.integers(8))
    if r == 0:
        w, h = int(rng.integers(1, 33)), int(rng.integers(1, 300))
        return (w, h) if rng.integers(2) else (h, w)
    if r == 1:
        if rng.integers(2):
            w = int(rng.choice([2048, 4096])) + int(rng.integers(-1, 2))
        else:
            w = 32 * int(rng.integers(129, 241)) + (int(rng.integers(1, 32)) if rng.integers(2) else 0)
        return w, int(rng.integers(16, 160))
    return int(rng.integers(33, 720)), int(rng.integers(33, 520))


for case in range(n):
    w, h = draw_size()
    kw = {}
    kind = int(rng.integers(6))
    if kind == 0:
        kw = dict(flags=0, winSize=int(rng.integers(2, 36)), polyN=int(rng.choice([5, 7])), polySigma=float(rng.choice([1.1, 1.5])))
    elif kind == 1:
        kw = dict(pyrLevels=int(rng.integers(0, 6)), pyrIterations=int(rng.integers(1, 4)))
    elif kind == 2:
        kw = dict(winSize=int(rng.choice([14, 15, 20, 30, 31, 40])), polyN=int(rng.choice([3, 5, 7])), polySigma=float(rng.choice([0.9, 1.1, 1.5])))
    elif kind == 3:
        kw = dict(pyrScale=float(rng.choice([0.5, 0.6, 0.8])), pyrLevels=int(rng.integers(1, 5)))
    batch = int(rng.integers(1, 4))
    opts = {"window_tiles": int(rng.integers(2)), "sparse_last": int(rng.integers(2)), "box_unfused": int(rng.integers(2)) if kind == 0 else 0,
            "polyexp_tma": int(rng.integers(2)), "level_generic": 1 if rng.integers(8) == 0 else 0, "tight_pitch": int(rng.integers(2))}
    thr, span = float(rng.choice([0.3, 0.6, 5.0])), int(rng.choice([7, 10, 16]))
    pairs = [tw.synth.make_pair("S" if rng.integers(2) else "T", w, h, int(rng.integers(1000)), defect=bool(rng.integers(2))) for _ in range(batch)]
    p = tw.OpticalFlowParameter(**kw)
    o = tw.OpticalFlow(0, 0, 0, batch)
    msg = None
    try:
        for name, v in opts.items():
            o.set_option(name, v)
        for arith in (0, 1):
            o.set_option("arithmetic", arith)
            relaxed = o.arithmetic_in_effect(p) == "relaxed"
            O.set_relax(144 if relaxed else 0)
            refs = [O.farneback(a, b, FlowParam(**kw)) for a, b in pairs]
            O.set_relax(0)
            res = o.calculate_batch(pairs, p, threshold=thr, span=span)
            for i in range(batch):
                status, vec = O.sample(refs[i], span, thr)
                if res[i]["status"] != status or [(v["x"], v["y"]) for v in res[i]["vector"]] != [(v[0], v[1]) for v in vec]:
                    msg = f"status/vectors differ (arith {arith}, pair {i})"
                if not opts["sparse_last"]:
                    fx, fy = o.batch_flow(i, w, h)
                    if not (np.array_equal(fx, refs[i][..., 0]) and np.array_equal(fy, refs[i][..., 1])):
                        msg = f"flow differs (arith {arith}, pair {i}): max {np.abs(fx - refs[i][..., 0]).max():.3g}"
    except Exception as e:  # noqa
        msg = "exception: " + str(e)
    o.close()
    if msg:
        bad += 1
        print("FAIL case", case, (w, h), kw, opts, "thr", thr, "span", span, "batch", batch, "->", msg, flush=True)
print("fuzz parity: %d cases, %d failures" % (n, bad))
sys.exit(1 if bad else 0)
