#!/usr/bin/env python
"""Cost of change regions (option "change_regions", tw_change_regions) at 1920x1080, batch 32, default options, on one GPU.

Four cases alternate in one process, each with the dense and the sparse last iteration ("sparse_last" 0 / 1):
  off          the option off, the bench's 32 seeded pairs at the default threshold (5)
  on           the option on, the same pairs and threshold
  worst        the option on at threshold 0: almost every sample point is suspicious, one big region per pair
  fragmented   the option on at threshold 0 with a mask on the single pixels of the grid points with an odd i or an odd j: up to
               96 x 54 isolated points, more than TW_MAX_CHANGE_REGIONS regions per pair
Every (case, sparse_last) has a context of its own, so each replays its own captured graph.  Reported per case:
  device_pairs_s   pairs/s of the device pass (the launch sequence replayed from its captured graph), from the CUDA events the
                   library records around it on its stream (tw_result.time; uploads and result copies excluded)
  kernels_ms       per step, event-timed per kernel family in an eager profiled run: the sample kernel and the region kernel
  pool_pairs_s     the dispatcher end to end (tw_pool_submit[_mask] / tw_pool_wait[_regions], host images, H2D + compute + D2H;
                   its contexts run the sparse last iteration).  At threshold 0 every answer carries about 20 k vectors, so there
                   the figure is bound by building the Python response dicts, not by the device
The card's name and power limit are read in the same run.

    python tools/change_regions_bench.py [--steps 30] [--rounds 3] [--pool-requests 640] [--out FILE]
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.mask_bench import B, H, W, card  # noqa: E402


def isolating_mask(span=10):
    """Nonzero only at the pixels of the grid points (i * span, j * span) with an odd i or an odd j."""
    import numpy as np
    m = np.zeros((H, W), np.uint8)
    ys, xs = np.mgrid[0:H:span, 0:W:span]
    odd = ((xs // span) % 2 == 1) | ((ys // span) % 2 == 1)
    m[ys[odd], xs[odd]] = 1
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--pool-requests", type=int, default=640)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import tidalwave_b200 as tw
    info = {"card": card(), "size": [W, H], "batch": B, "options": "default", "cases": {}}
    pairs = tw.synth.pool_pairs(B, W, H, seed0=100)
    mask = isolating_mask()
    # case -> (option, threshold, calculate_batch keywords)
    cases = {"off": (0, 5.0, {}), "on": (1, 5.0, {}), "worst": (1, 0.0, {}), "fragmented": (1, 0.0, {"ignore_mask": [mask] * B})}
    keys = [(name, sparse) for sparse in (0, 1) for name in cases]
    ctx = {}
    for name, sparse in keys:
        of = tw.OpticalFlow(0, W, H, B)
        of.set_option("sparse_last", sparse)
        of.set_option("change_regions", cases[name][0])
        ctx[name, sparse] = of

    def run(k):
        on, thr, kw = cases[k[0]]
        return ctx[k].calculate_batch(pairs, threshold=thr, **kw)

    answers = {}
    for k in keys:  # warm every graph
        for _ in range(args.warmup):
            r = run(k)
        answers[k] = {"suspicious": sum(x["status"] == "SUSPICIOUS" for x in r), "vectors": sum(x["n_vectors"] for x in r),
                      "regions": sum(x.get("n_regions", 0) for x in r)}
    dev = {k: [] for k in keys}
    for _ in range(args.rounds):
        for k in keys:
            step_s = []
            for _ in range(args.steps):
                r = run(k)
                step_s.append(sum(x["time"] for x in r))  # per-pair shares of the step's device time
            dev[k].append(B * len(step_s) / sum(step_s))
    fam = {}
    for k in keys:  # per-family kernel times, eager with events around every launch
        ctx[k].profile(True)
        for _ in range(args.steps):
            run(k)
        pr = ctx[k].profile_read()
        ctx[k].profile(False)
        fam[k] = {f: round(pr[f]["ms"] / args.steps, 4) for f in ("sample", "change_regions")}
    for of in ctx.values():
        of.close()

    pools = {name: tw.Pool([0], threshold=thr, batch=B, change_regions=bool(on)) for name, (on, thr, _) in cases.items()}

    def request(name, i):
        kw = {"ignore_mask": mask} if name == "fragmented" else {}
        return pools[name].request(*pairs[i % B], **kw)

    for name in cases:  # warm every pool path
        assert all(pools[name].wait(i)["status"] != "ERROR" for i in [request(name, i) for i in range(4 * B)])
    e2e = {name: [] for name in cases}
    for _ in range(args.rounds):
        for name in cases:
            gc.collect()  # the threshold-0 cases' answers (about 20 k vector dicts per pair) are freed outside the timed window
            t0 = time.perf_counter()
            ids = [request(name, i) for i in range(args.pool_requests)]
            res = [pools[name].wait(i) for i in ids]
            e2e[name].append(args.pool_requests / (time.perf_counter() - t0))
            assert all(x["status"] != "ERROR" for x in res)
            del res
    for p in pools.values():
        p.stop(); p.close()

    for name, (on, thr, _) in cases.items():
        c = {"change_regions": on, "threshold": thr, "pool_pairs_s": [round(v, 1) for v in e2e[name]]}
        for sparse in (0, 1):
            k = (name, sparse)
            c[f"sparse_last={sparse}"] = dict(device_pairs_s=[round(v, 1) for v in dev[k]], kernels_ms=fam[k], **answers[k])
            base = dev["off", sparse]
            c[f"sparse_last={sparse}"]["device_vs_off"] = round(sum(dev[k]) / sum(base), 4)
        info["cases"][name] = c
    print(json.dumps(info, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
