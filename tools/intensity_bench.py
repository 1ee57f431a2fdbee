#!/usr/bin/env python
"""Cost of intensity cells (option "intensity_threshold", tw_intensity_cells) at 1920x1080, batch 32, default options, on one GPU.

Four cases alternate in one process, each with the dense and the sparse last iteration ("sparse_last" 0 / 1):
  off         the option off, the bench's 32 seeded pairs at the default threshold (5) and span (10)
  on          "intensity_threshold" = 16, the same pairs
  off_span1   the option off at span 1 (every pixel a sample point and a cell: 2 M cells per pair)
  on_span1    "intensity_threshold" = 16 at span 1
Every (case, sparse_last) has a context of its own, so each replays its own captured graph.  Reported per case:
  device_vs_off    device_pairs_s over the option-off case of the same span
  device_pairs_s   pairs/s of the device pass (the launch sequence replayed from its captured graph), from the CUDA events the
                   library records around it on its stream (tw_result.time; uploads and result copies excluded)
  kernels_ms       per step, event-timed per kernel family in an eager profiled run: the sample kernel, the "intensity" family
                   (the per-cell sums, the counts and the compaction) and the whole step (every family)
  intensity_share  the "intensity" family's share of the step
  hbm_floor_ms     the least time the intensity pass could take: reading E and T once (2 bytes per pixel per pair) at the data
                   sheet's 7.7 TB/s; hbm_floor_share = hbm_floor_ms / the family's time
The card's name and power limit are read in the same run.

    python tools/intensity_bench.py [--steps 30] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.mask_bench import B, H, W, card  # noqa: E402

HBM_BYTES_S = 7.7e12  # HGX B200 data sheet, one GPU


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import tidalwave_b200 as tw
    info = {"card": card(), "size": [W, H], "batch": B, "options": "default", "threshold": 5.0, "cases": {}}
    pairs = tw.synth.pool_pairs(B, W, H, seed0=100)
    cases = {"off": (0, 10), "on": (16, 10), "off_span1": (0, 1), "on_span1": (16, 1)}  # (intensity_threshold, span)
    keys = [(name, sparse) for sparse in (0, 1) for name in cases]
    ctx = {}
    for name, sparse in keys:
        of = tw.OpticalFlow(0, W, H, B)
        of.set_option("sparse_last", sparse)
        of.set_option("intensity_threshold", cases[name][0])
        ctx[name, sparse] = of

    def run(k):
        return ctx[k].calculate_batch(pairs, span=cases[k[0]][1], cap=1)

    answers = {}
    for k in keys:  # warm every graph
        for _ in range(args.warmup):
            r = run(k)
        answers[k] = {"suspicious": sum(x["status"] == "SUSPICIOUS" for x in r), "vectors": sum(x["n_vectors"] for x in r),
                      "intensity_cells": sum(x.get("n_intensity_cells", 0) for x in r)}
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
        fam[k] = {f: round(pr[f]["ms"] / args.steps, 4) for f in ("sample", "intensity")}
        fam[k]["step"] = round(sum(v["ms"] for v in pr.values()) / args.steps, 4)
    for of in ctx.values():
        of.close()

    floor_ms = B * 2.0 * W * H / HBM_BYTES_S * 1e3
    for name, (t, span) in cases.items():
        c = {"intensity_threshold": t, "span": span}
        for sparse in (0, 1):
            k = (name, sparse)
            d = dict(device_pairs_s=[round(v, 1) for v in dev[k]], kernels_ms=fam[k], **answers[k])
            d["device_vs_off"] = round(sum(dev[k]) / sum(dev["off" if span == 10 else "off_span1", sparse]), 4)
            if t:
                d["intensity_share"] = round(fam[k]["intensity"] / fam[k]["step"], 4)
                d["hbm_floor_ms"] = round(floor_ms, 4)
                d["hbm_floor_share"] = round(floor_ms / fam[k]["intensity"], 4)
            c[f"sparse_last={sparse}"] = d
        info["cases"][name] = c
    print(json.dumps(info, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
