#!/usr/bin/env python
"""Cost of ignore masks (tw_compare_batch_mask & co.) at 1920x1080, batch 32, default options, on one GPU.

Three cases alternate in one process, on the same 32 seeded pairs: no mask; a mask on every pair covering about 5 % of the frame
(200 round spots of radius 13, seeded); and, for comparison, 32 regions of 200x100 per pair.  Reported per case:
  device_pairs_s   pairs/s of the device pass (the launch sequence replayed from its captured graph), from the CUDA events the
                   library records around it on its stream (tw_result.time; uploads and result copies excluded)
  kernels_ms       per step, event-timed per kernel family in an eager profiled run: the paint kernels and the sample kernel
  pool_pairs_s     the dispatcher end to end (tw_pool_submit[_mask] / tw_pool_wait, host images and masks, H2D + compute + D2H)
The card's name and power limit are read in the same run.

    python tools/mask_bench.py [--steps 30] [--rounds 3] [--pool-requests 640] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H, B = 1920, 1080, 32


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers below still stand; say that the card could not be read
        return {"error": str(e)}


def spots_mask(seed=7, n=200, r=13):
    import numpy as np
    rng = np.random.default_rng(seed)
    m = np.zeros((H, W), np.uint8)
    yy, xx = np.mgrid[-r:r + 1, -r:r + 1]
    disc = (xx * xx + yy * yy <= r * r).astype(np.uint8) * 255
    for x, y in zip(rng.integers(r, W - r, n), rng.integers(r, H - r, n)):
        m[y - r:y + r + 1, x - r:x + r + 1] |= disc
    return m


REGIONS = [(20 + 240 * (i % 8), 20 + 270 * (i // 8), 200, 100) for i in range(32)]


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
    mask = spots_mask()
    info["mask_fraction"] = round(float((mask != 0).mean()), 4)
    cases = {"none": {}, "mask_5pct": {"ignore_mask": mask}, "32x200x100": {"ignore": REGIONS}}
    batch = {name: {k: [v] * B for k, v in kw.items()} for name, kw in cases.items()}

    of = tw.OpticalFlow(0, W, H, B)
    answers = {}
    for name in cases:  # warm every graph key
        for _ in range(args.warmup):
            r = of.calculate_batch(pairs, **batch[name])
        answers[name] = [(x["status"], x["n_vectors"]) for x in r]
    dev = {name: [] for name in cases}
    for _ in range(args.rounds):
        for name in cases:
            step_s = []
            for _ in range(args.steps):
                r = of.calculate_batch(pairs, **batch[name])
                step_s.append(sum(x["time"] for x in r))  # per-pair shares of the step's device time
            dev[name].append(B * len(step_s) / sum(step_s))
    # per-family kernel times, eager with events around every launch
    fam = {}
    for name in cases:
        of.profile(True)
        for _ in range(args.steps):
            of.calculate_batch(pairs, **batch[name])
        pr = of.profile_read()
        of.profile(False)
        fam[name] = {k: round(pr[k]["ms"] / args.steps, 4) for k in ("mask_paint", "ignore_paint", "sample") if k in pr}
    of.close()

    pool = tw.Pool([0], batch=B)
    for kw in cases.values():  # warm every pool path: plan, graph keys, the staging buffer's growth for mask planes
        assert all(pool.wait(i)["status"] != "ERROR" for i in [pool.request(*pairs[i % B], **kw) for i in range(4 * B)])
    e2e = {name: [] for name in cases}
    for _ in range(args.rounds):
        for name, kw in cases.items():
            t0 = time.perf_counter()
            ids = [pool.request(*pairs[i % B], **kw) for i in range(args.pool_requests)]
            res = [pool.wait(i) for i in ids]
            e2e[name].append(args.pool_requests / (time.perf_counter() - t0))
            assert all(x["status"] != "ERROR" for x in res)
    pool.stop(); pool.close()

    for name in cases:
        info["cases"][name] = {"device_pairs_s": [round(v, 1) for v in dev[name]], "kernels_ms": fam[name],
                               "pool_pairs_s": [round(v, 1) for v in e2e[name]],
                               "suspicious": sum(s == "SUSPICIOUS" for s, _ in answers[name]),
                               "vectors": sum(n for _, n in answers[name])}
    base = sum(dev["none"]) / len(dev["none"])
    for name in cases:
        m = sum(dev[name]) / len(dev[name])
        info["cases"][name]["device_vs_none"] = round(m / base, 4)
    print(json.dumps(info, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
