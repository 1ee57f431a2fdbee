#!/usr/bin/env python
"""bench.py -- headline benchmark: image pairs/sec at 1920x1080 (BASELINE.json), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

A "step" = one pass of the whole hot path (pyramid, polynomial expansion, update-matrices, window blur + solve
iterations, span sampling + classification) over one batch of B (default 32) synthetic 1920x1080 pairs with the reference's
default options (BASELINE.json configs[1]; the batch is configs[4]'s work-queue unit).

  value         pairs/s with the batch already resident in HBM (device pass only, CUDA events on the library's stream; the
                launch sequence of a step replays as one captured CUDA graph, as it does for every API caller)
  e2e           BASELINE configs[4]: 10,000 pairs cycled from 64 distinct pinned HOST pairs through the dispatcher API
                (tw_pool_submit / tw_pool_wait), H2D + compute + D2H of the compact results inside the timed region
  roofline      dominant kernel family: algorithmic bytes (DESIGN.md section 4) / event-timed duration vs measured HBM peak
  variants      the other arithmetic / last-iteration forms of the same step (faithful, dense, faithful + dense)
  configs       BASELINE configs[2] (3840x2160, 5 levels, 5 iterations) and configs[3] (1280x2000 box window) device-resident,
                each against its own algorithmic-byte roofline (BASELINE.md section 2); configs[4] is the e2e leg
  cpu_baseline  the reference's CPU path (cv2 calcOpticalFlowFarneback, else the C oracle port) on this box's cores

Multi-GPU: pairs are independent => each rank runs its own shard (weak scaling), no data-path collective; torch.distributed
is used only for the barrier and the max-over-ranks of the timed region.  At N > 1 rank 0 additionally drives ONE in-process
dispatcher over all N GPUs (e2e_inprocess: the reference's Manager + Consumers shape) while the other ranks idle.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H = 1920, 1080
METRIC = "image pairs/sec at 1920x1080"
UNIT = "pairs/s"
# the SAME string in both arms (the driver compares config.workload)
WORKLOAD = ("configs[1]/[4]: synthetic 1920x1080 pairs (seeded S/T pool, true shift (-0.37,+0.61) px, every 8th with a defect), "
            "default options (threshold 5, span 10, pyrLevels 3, winSize 30, pyrIterations 3, polyN 7, polySigma 1.5, flags 256)")
# algorithmic HBM bytes per pair of the minimum-pass pipeline, SURVEY.md 8(d) / BASELINE.md section 2
B_ALG = {"cfg2": 859248000.0, "cfg3": 5251873920.0, "cfg4": 1060800000.0}


def measured_peaks():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "40"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, pw, reasons = [], None, [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1]); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # under load = samples in the top half of what we saw (idle samples at the edges are dropped)
        med = float(np.median([s for s in sm if s >= 0.5 * max(sm)])) if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


def make_pool(n: int, w: int = W, h: int = H, seed0: int = 100):
    import tidalwave_b200 as tw
    return tw.synth.pool_pairs(n, w, h, seed0=seed0)


def cpu_reference(pairs, n_pairs: int, workers: int):
    """The reference's CPU path on host cores: Farneback + sampling per pair, parallel ACROSS pairs like the
    reference's consumer pool (src/manager.cpp:55-59).  Returns (pairs/s, kind, description)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle.oracle import FlowParam, RefOracle, sample_numpy
    try:
        import cv2
        cv2.ipp.setUseIPP(False)
        cv2.setNumThreads(1)
        # what the reference itself executes on this path is this library call (src/opticalflow.cpp:83-85); its own code
        # around it (sampling, src/consumer.cpp:60-77) is restated in NumPy
        kind = "reference"
        impl = (f"cv2 {cv2.__version__} calcOpticalFlowFarneback (the reference's third-party Farneback implementation -- OpenCV, newer "
                "build than its 2.4.9 pin -- IPP off, 1 thread per pair) + the reference's sampling loop restated in NumPy")

        def one(i):
            a, b = pairs[i % len(pairs)]
            fl = cv2.calcOpticalFlowFarneback(a, b, None, 0.5, 3, 30, 3, 7, 1.5, 256)
            return sample_numpy(fl)[0]
    except Exception:
        os.environ.setdefault("OMP_NUM_THREADS", "1")
        O = RefOracle()
        kind = "port"
        impl = "oracle/farneback_ref.c (scalar C port of the same algorithm, 1 thread per pair) + sampling"

        def one(i):
            a, b = pairs[i % len(pairs)]
            return O.sample(O.farneback(a, b, FlowParam()))[0]
    one(0)  # warm
    t0 = time.perf_counter()
    with ThreadPoolExecutor(workers) as ex:
        list(ex.map(one, range(n_pairs)))
    dt = time.perf_counter() - t0
    return n_pairs / dt, kind, f"{n_pairs} pairs of the 1920x1080 pool, {workers} threads across pairs; {impl}"


def run_reference(args, rank):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    workers = cores
    pairs = make_pool(4)
    per_step = max(workers, 4)
    vals = []
    for s in range(args.warmup + args.steps):
        v, kind, desc = cpu_reference(pairs, per_step, workers)
        if s >= args.warmup:
            vals.append(v)
        if s == 0 and per_step / v > 60:  # keep the whole run within a few minutes
            per_step = max(workers // 2, 2)
    value = float(np.mean(vals))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * per_step / value, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "pairs_per_step": per_step, "where": "host CPU cores, no GPU"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": kind, "sample": desc},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


class Resident:
    """A batch of pairs resident in one context's HBM + the timing helpers around tw_batch_run."""

    def __init__(self, tw, lib, device, pairs, param, w, h):
        self.tw, self.lib, self.w, self.h, self.B = tw, lib, w, h, len(pairs)
        self.of = tw.OpticalFlow(device, w, h, self.B)
        self.cp = param.c()
        self.threshold, self.span = 5.0, 10
        npx = w * h
        self.pinned = []
        for a, b in pairs:
            pa = lib.tw_host_alloc(npx); pb = lib.tw_host_alloc(npx)
            C.memmove(pa, a.ctypes.data, npx); C.memmove(pb, b.ctypes.data, npx)
            self.pinned.append((pa, pb))
        ex = (C.c_void_p * self.B)(*[p[0] for p in self.pinned])
        tg = (C.c_void_p * self.B)(*[p[1] for p in self.pinned])
        self.check(lib.tw_batch_upload(self.of.ctx, self.B, ex, tg, w, h, w), "upload")
        self.check(lib.tw_sync(self.of.ctx), "sync")

    def check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what}: rc={rc} {self.of.last_error()}")

    def step(self):
        self.check(self.lib.tw_l2_flush(self.of.ctx), "flush")
        self.check(self.lib.tw_batch_run(self.of.ctx, self.B, self.w, self.h, C.byref(self.cp), self.threshold, self.span), "run")

    def timed(self, steps, warmup, dist):
        """-> device milliseconds of `steps` steps, max over ranks (barrier + stream sync on both sides)."""
        for _ in range(warmup):
            self.step()
        self.check(self.lib.tw_sync(self.of.ctx), "sync")
        dist.barrier()
        self.check(self.lib.tw_timer_start(self.of.ctx), "timer")
        for _ in range(steps):
            self.step()
        ms = C.c_float(0)
        self.check(self.lib.tw_timer_stop(self.of.ctx, C.byref(ms)), "timer")  # records + synchronises the stream
        dist.barrier()
        return dist.reduce_max(float(ms.value))

    def fetch(self):
        """-> (results, vectors, cap) of the last run as tw_batch_fetch hands them to a caller (pair i's vectors at i * cap)."""
        cap = ((self.w + self.span - 1) // self.span) * ((self.h + self.span - 1) // self.span)
        vec = (self.tw.tw_vector * (cap * self.B))()
        res = (self.tw.tw_result * self.B)()
        self.check(self.lib.tw_batch_fetch(self.of.ctx, self.B, vec, cap, res), "fetch")
        return res, vec, cap

    def statuses(self):
        return [r.status for r in self.fetch()[0]]

    def close(self):
        self.of.close()
        for pa, pb in self.pinned:
            self.lib.tw_host_free(pa); self.lib.tw_host_free(pb)


DUMP_BYTES = 60 << 20  # all files of --dump-outputs together, .npy headers included: below 64 MB however counted


def dump_outputs(out_dir, R, dense):
    """Writes what the last step of the timed pass handed its caller, as .npy files a second build's run can be compared with:
    status.npy and n_vectors.npy (one entry per pair), vectors.npy (pair, x, y, dx, dy per row, scan order) and, with the dense last
    iteration, flow.npy (pair, pixel, dx / dy) at the pixels listed in flow_pixels.npy (row-major indices).  The pixels, and the
    vectors if they would not fit, are a seeded sample so that the files stay within DUMP_BYTES."""
    os.makedirs(out_dir, exist_ok=True)
    res, vec, cap = R.fetch()
    n = [min(r.n_vectors, cap) for r in res]
    out = {"status": np.array([r.status for r in res], np.float64), "n_vectors": np.array([r.n_vectors for r in res], np.float64)}
    if dense:
        npx = R.w * R.h
        px = np.sort(np.random.default_rng(0).choice(npx, min(npx, (DUMP_BYTES // 2) // (8 * R.B)), replace=False))
        out["flow_pixels"] = px.astype(np.float64)
        out["flow"] = np.stack([np.stack([f.ravel()[px] for f in R.of.batch_flow(i, R.w, R.h)], 1) for i in range(R.B)])
    v = np.ctypeslib.as_array(vec).reshape(R.B, cap)
    rows = np.concatenate([np.stack([np.full(k, i, np.float64), v[i, :k]["x"], v[i, :k]["y"], v[i, :k]["dx"], v[i, :k]["dy"]], 1)
                           for i, k in enumerate(n)])
    room = (DUMP_BYTES - sum(a.nbytes for a in out.values())) // (5 * 8)
    if len(rows) > room:
        rows = rows[np.sort(np.random.default_rng(1).choice(len(rows), room, replace=False))]
    out["vectors"] = rows
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_pool(tw, lib, devices, B, cp, pinned, n_req, warm):
    """n_req pairs cycled from the pinned host pool through ONE dispatcher (tw_pool_*) over `devices`; -> (seconds, vectors)."""
    perr = C.create_string_buffer(256)
    dv = (C.c_int * len(devices))(*devices)
    pool = lib.tw_pool_create(dv, len(devices), W, H, B, C.byref(cp), 5.0, 10, 4096, perr, 256)
    if not pool:
        raise RuntimeError("tw_pool_create: " + perr.value.decode())
    rvec = (tw.tw_vector * 4096)()
    rres = tw.tw_result()
    P = len(pinned)

    def go(n):
        ids = [lib.tw_pool_submit(pool, pinned[i % P][0], W, H, pinned[i % P][1], W, H) for i in range(n)]
        nv = 0
        for i in ids:
            rc = lib.tw_pool_wait(pool, i, rvec, 4096, C.byref(rres))
            if rc != 0:
                raise RuntimeError(f"pool wait rc={rc} {rres.reason.decode()}")
            nv += min(rres.n_vectors, 4096)
        return nv
    try:
        go(warm)  # plans, buffers, graphs
        t0 = time.perf_counter()
        nv = go(n_req)
        dt = time.perf_counter() - t0
    finally:
        lib.tw_pool_destroy(pool)
    return dt, nv


def run_files_leg(tw, lib, device, B, cp, pairs, n_req=1536, n_png=768):
    """n_req pairs cycled from 16 distinct JPEG pairs on disk through tw_pool_submit_files (+ n_png pairs from the same images as
    PNG files); -> dict or None (no cv2 to write them)."""
    import shutil
    import tempfile
    try:
        import cv2
    except Exception:
        return None
    d = tempfile.mkdtemp(prefix="tw_bench_files_")
    try:
        paths = {"jpg": [], "png": [], "rgb.png": []}
        for i, (a, b) in enumerate(pairs[:16]):
            for ext, opt in (("jpg", [cv2.IMWRITE_JPEG_QUALITY, 90]), ("png", []), ("rgb.png", [])):
                pa, pb = os.path.join(d, f"e{i}.{ext}"), os.path.join(d, f"t{i}.{ext}")
                if ext == "rgb.png":  # colour-typed files (what browsers write): 3 bytes per pixel through inflate / filters / rgb -> gray
                    cv2.imwrite(pa, cv2.merge([a, a, a]), opt); cv2.imwrite(pb, cv2.merge([b, b, b]), opt)
                else:
                    cv2.imwrite(pa, a, opt); cv2.imwrite(pb, b, opt)
                paths[ext].append((pa.encode(), pb.encode()))
        perr = C.create_string_buffer(256)
        dv = (C.c_int * 1)(device)
        pool = lib.tw_pool_create(dv, 1, W, H, B, C.byref(cp), 5.0, 10, 4096, perr, 256)
        if not pool:
            return None
        threads = min(32, os.cpu_count() or 1)
        lib.tw_pool_set_decoders(pool, threads)
        rvec = (tw.tw_vector * 4096)()
        rres = tw.tw_result()

        def go(n, ext):
            pp = paths[ext]
            ids = [lib.tw_pool_submit_files(pool, *pp[i % len(pp)]) for i in range(n)]
            for i in ids:
                if lib.tw_pool_wait(pool, i, rvec, 4096, C.byref(rres)) != 0:
                    raise RuntimeError("file leg: " + rres.reason.decode())
        try:
            go(4 * B, "jpg")
            t0 = time.perf_counter()
            go(n_req, "jpg")
            dt = time.perf_counter() - t0
            go(B, "png")
            t0 = time.perf_counter()
            go(n_png, "png")
            dt_png = time.perf_counter() - t0
            go(B, "rgb.png")
            t0 = time.perf_counter()
            go(n_png // 2, "rgb.png")
            dt_rgb = time.perf_counter() - t0
        finally:
            lib.tw_pool_destroy(pool)
        return {"value": n_req / dt, "unit": UNIT, "pairs": n_req, "seconds": dt, "decoder_threads": threads,
                "api": "tw_pool_submit_files: %d pairs cycled from 16 distinct 1920x1080 JPEG pairs (cv2-written, quality 90) on disk; read + "
                       "decoded by tw_decode_gray on %d host threads (bit-identical to cv2.imread) into recycled page-locked buffers, then one "
                       "consumer on the GPU; bound by the host decode" % (n_req, threads),
                "png": {"value": n_png / dt_png, "unit": UNIT, "pairs": n_png, "seconds": dt_png,
                        "note": "the same images as 8-bit gray PNG files (cv2-written, default compression): zlib-inflate-bound; half of "
                                "the pool is band-limited noise texture, which PNG barely compresses"},
                "png_rgb": {"value": (n_png // 2) / dt_rgb, "unit": UNIT, "pairs": n_png // 2, "seconds": dt_rgb,
                            "note": "the same images as 8-bit RGB PNG files (three equal channels): 3 bytes per pixel through inflate, "
                                    "the row filters and the rgb -> gray conversion"}}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=32, help="pairs per step = the dispatcher's batch (16 -> 32: +3 %% pairs/s; 5.6 GB of device buffers)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the e2e, variants and configs legs (profilers)")
    ap.add_argument("--pool-consumers", type=int, default=1, help="e2e leg: consumer threads (contexts) per GPU")
    ap.add_argument("--e2e-pairs", type=int, default=10000, help="e2e leg: pairs per rank (BASELINE configs[4])")
    ap.add_argument("--arithmetic", default="default", choices=["default", "faithful"],
                    help="default = the library default (relaxed where validated: include/tidalwave_b200.h); faithful = the "
                         "oracle's operation order everywhere (bit-identical results)")
    ap.add_argument("--last", default="sparse", choices=["sparse", "dense"],
                    help="last iteration of the finest scale: 'sparse' = evaluated at the sampled positions only (what the dispatcher "
                         "does: the Response carries vectors, not the field; bit-identical vectors), 'dense' = full flow field")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the b200 arm; the reference arm keeps none")
    if args.impl == "b200":
        args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import tidalwave_b200 as tw
    dist = tw.dist.Dist()  # gloo barrier / max-reduce when launched by torch.distributed.run with N > 1; no-op at N = 1
    lib = tw.load()
    B = args.batch
    pairs = make_pool(B)  # every rank: same seeded pool, its own copy (weak scaling: B pairs per step per GPU)
    if args.arithmetic == "faithful":
        tw.set_default_arithmetic(False)  # contexts created from here on, the e2e pool's consumers included
    os.environ["TW_SPARSE_LAST"] = "1" if args.last == "sparse" else "0"  # the e2e pool's consumers
    param = tw.OpticalFlowParameter()
    R = Resident(tw, lib, local_rank, pairs, param, W, H)
    of = R.of
    of.set_option("sparse_last", 1 if args.last == "sparse" else 0)
    arithmetic = of.arithmetic_in_effect(param)
    npx = W * H

    # ---- headline: device-resident pass ----
    R.timed(0, args.warmup, dist)
    statuses = R.statuses()  # sanity: the warm-up results are real
    l0 = of.launch_count()
    sampler = ClockSampler(local_rank)
    try:
        elapsed_ms = R.timed(args.steps, 0, dist)
    finally:
        clocks = sampler.stop()  # also on failure: the sampler must not outlive this process
    launches = of.launch_count() - l0
    value = tw.dist.whole_job_throughput(B * args.steps, world, elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, R, args.last == "dense")

    # ---- per-kernel-family pass: the same steps again with a CUDA event pair around every launch (the graph replay above
    # has no per-kernel events; with profiling on the library issues the identical launch sequence eagerly) ----
    psteps = min(args.steps, 100)
    of.profile(True)
    prof_ms = R.timed(psteps, 0, dist)
    prof = of.profile_read()
    of.profile(False)

    # ---- roofline of the dominant kernel family ----
    peak, peak_src = measured_peaks()
    fams = {k: v for k, v in prof.items() if v["launches"] > 0}
    top = max(fams, key=lambda k: fams[k]["ms"])
    tv = fams[top]
    achieved = tv["alg_bytes"] / (tv["ms"] * 1e-3) / 1e9
    kernel_ms_total = sum(v["ms"] for v in fams.values())
    alg_total = sum(v["alg_bytes"] for v in fams.values())
    # DRAM traffic per launch of that family from the committed ncu --set full capture (same command line, same batch)
    traffic, traffic_src = None, None
    try:
        import glob
        # newest capture first: r2j is the set of the final commit, the others follow in reverse name order
        tfs = sorted(glob.glob(os.path.join(ROOT, "profiles", "r2*_traffic.json")), reverse=True)
        tfs.sort(key=lambda f: not os.path.basename(f).startswith("r2j_"))
        for tf in tfs:
            tj = json.load(open(tf))
            if tj.get("batch") == B and tj.get("arithmetic", "faithful") == arithmetic and top in tj:
                traffic = tj[top]["dram_bytes_per_launch"]
                traffic_src = "profiles/%s (ncu --set full: dram__bytes_read+write per launch)" % os.path.basename(tf)
                break
    except Exception:
        pass
    step_rate = B * args.steps / (elapsed_ms * 1e-3)  # this rank's pairs/s (= value / world)
    roofline = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "timed": "per-launch CUDA events on the library's stream over a second pass of %d steps (eager launches; the headline "
                         "pass replays a CUDA graph): %.3f ms/step" % (psteps, prof_ms / psteps), "avg_launch_ms": tv["ms"] / tv["launches"],
                "alg_bytes_per_launch": tv["alg_bytes"] / tv["launches"], "share_of_step": tv["ms"] / kernel_ms_total,
                "pipeline": {"alg_bytes_per_pair": alg_total / (B * psteps),
                             "alg_bytes_per_pair_survey": B_ALG["cfg2"],
                             "achieved": step_rate * alg_total / (B * psteps) / 1e9,
                             "frac": step_rate * alg_total / (B * psteps) / 1e9 / peak,
                             "frac_vs_survey_bytes": step_rate * B_ALG["cfg2"] / 1e9 / peak,
                             "note": "whole step (all kernels + launch gaps + the L2 flush) of the headline pass vs the HBM peak; "
                                     "alg_bytes_per_pair is what THIS step moves by the formula of SURVEY 8(d) (the sparse last iteration "
                                     "writes no finest-scale flow plane and reads M once: 859.2 -> 842.7 MB); frac_vs_survey_bytes charges the "
                                     "full 859.2 MB regardless"},
                "families": {k: {"ms_per_step": v["ms"] / psteps, "launches_per_step": v["launches"] / psteps,
                                 "GBps": (v["alg_bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 else None,
                                 "frac": (v["alg_bytes"] / (v["ms"] * 1e-3) / 1e9 / peak) if v["ms"] > 0 else None} for k, v in fams.items()},
                "families_note": "level_image is charged what the fused kernel moves: the u8 source ONCE for all four levels + the level "
                                 "images written (SURVEY's formula charges the source once per level)"}

    e2e = variants = configs = e2e_inprocess = e2e_files = None
    if not args.no_e2e:
        # ---- the other forms of the same step, beside the headline ----
        nv = max(20, args.steps // 4)
        variants = {}
        notes = {"faithful": "tw_set_option(arithmetic, 0): every kernel in the oracle's operation order, results bit-identical to "
                             "oracle/farneback_ref.c",
                 "relaxed": "tw_set_option(arithmetic, 1): direct-form fmaf window taps + mixed double/float poly-exp pass; <= 1.5e-4 px from "
                            "the faithful oracle at 1920x1080, status / vectors identical",
                 "sparse": "last iteration of the finest scale at the sampled positions only (the dispatcher's form; vectors bit-identical)",
                 "dense": "the whole flow field is produced (tw_flow / tw_batch_flow callers)"}
        for ar in ("relaxed", "faithful"):
            for la in ("sparse", "dense"):
                if ar == arithmetic and la == args.last:
                    continue
                of.set_option("arithmetic", 1 if ar == "relaxed" else 0)
                of.set_option("sparse_last", 1 if la == "sparse" else 0)
                ms = R.timed(nv, 3, dist)
                variants[f"{ar}_{la}"] = {"value": tw.dist.whole_job_throughput(B * nv, world, ms * 1e-3), "unit": UNIT, "ms_per_step": ms / nv,
                                          "note": notes[ar] + "; " + notes[la]}
        of.set_option("arithmetic", 1 if arithmetic == "relaxed" else 0)
        of.set_option("sparse_last", 1 if args.last == "sparse" else 0)
    R.close()

    if not args.no_e2e:
        # ---- e2e = BASELINE configs[4]: 10,000 pairs from 64 distinct pinned host pairs through the dispatcher ----
        POOL = 64
        pool_pairs = pairs + make_pool(POOL - B, seed0=100 + B) if POOL > B else pairs[:POOL]
        pinned = []
        for a, b in pool_pairs:
            pa = lib.tw_host_alloc(npx); pb = lib.tw_host_alloc(npx)
            C.memmove(pa, a.ctypes.data, npx); C.memmove(pb, b.ctypes.data, npx)
            pinned.append((pa, pb))
        cp = param.c()
        nc = max(1, args.pool_consumers)
        n_req = max(args.e2e_pairs // B * B, B * nc * 4)
        dist.barrier()
        dt, nvec = run_pool(tw, lib, [local_rank] * nc, B, cp, pinned, n_req, 2 * B * nc)
        dt = dist.reduce_max(dt)
        e2e = {"value": world * n_req / dt, "unit": UNIT, "h2d_bytes_per_step": 2 * npx * B,
               "d2h_bytes_per_step": int(4 * B + 24 * nvec * B / n_req), "pairs": n_req * world, "seconds": dt,
               "api": "tw_pool_submit/tw_pool_wait (configs[4]: %d pairs per GPU cycled from %d distinct pinned host pairs), %d consumer(s) per "
                      "GPU, batch %d" % (n_req, POOL, nc, B)}
        dist.barrier()
        if world > 1:
            # ONE in-process dispatcher over all N GPUs (rank 0), the reference's Manager + Consumers shape; other ranks idle
            if rank == 0:
                ndev = min(world, lib.tw_device_count())
                dti, _ = run_pool(tw, lib, [d for d in range(ndev) for _ in range(nc)], B, cp, pinned, n_req * ndev, 2 * B * nc * ndev)
                e2e_inprocess = {"value": n_req * ndev / dti, "unit": UNIT, "gpus": ndev, "pairs": n_req * ndev, "seconds": dti,
                                 "api": "one tw_pool in ONE process, %d consumer thread(s) on each of %d GPUs" % (nc, ndev)}
            dist.barrier()
        for pa, pb in pinned:
            lib.tw_host_free(pa); lib.tw_host_free(pb)

        # ---- file -> result: the reference's Manager::request takes two image PATHS (src/manager.cpp:68-78) and its consumers imread
        # them (src/opticalflow.cpp:37,44).  Same here: tw_pool_submit_files, decode on the pool's C++ threads (host code, bit-identical
        # to cv2.imread), then the same dispatcher.  This leg is bound by the host decode, not by the GPU. ----
        if world == 1:
            e2e_files = run_files_leg(tw, lib, local_rank, B, cp, pairs)

        # ---- BASELINE configs[2] and configs[3], device-resident, each against its own roofline (rank-local; N = 1 only) ----
        if world == 1:
            configs = {}
            for key, (w_, h_, b_, kw, gen) in {
                    "cfg3": (3840, 2160, 8, dict(pyrLevels=5, pyrIterations=5), [("T", 4), ("S", 5), ("T", 14), ("S", 15)]),
                    "cfg4": (1280, 2000, 32, dict(polyN=5, polySigma=1.1, winSize=15, flags=0), [("S", 3), ("T", 6)])}.items():
                made = {ks: tw.synth.make_pair(ks[0], w_, h_, ks[1], False) for ks in dict.fromkeys(gen)}
                prs = [made[ks] for ks in (gen * b_)[:b_]]  # the batch cycles through the distinct pairs
                p_ = tw.OpticalFlowParameter(**kw)
                Rc = Resident(tw, lib, local_rank, prs, p_, w_, h_)
                ns = 20
                ms = Rc.timed(ns, 3, dist)
                v_ = b_ * ns / (ms * 1e-3)
                Rc.of.profile(True)
                Rc.timed(5, 0, dist)
                pf = {k: v for k, v in Rc.of.profile_read().items() if v["launches"] > 0}
                Rc.of.profile(False)
                configs[key] = {"workload": "%dx%d, %s, batch %d" % (w_, h_, ", ".join(f"{k}={v}" for k, v in kw.items()), b_),
                                "value": v_, "unit": UNIT, "ms_per_pair": ms / ns / b_, "arithmetic": Rc.of.arithmetic_in_effect(p_),
                                "alg_bytes_per_pair": B_ALG[key], "roofline_pairs_per_s": peak * 1e9 / B_ALG[key],
                                "frac": v_ * B_ALG[key] / 1e9 / peak,
                                "families_ms_per_pair": {k: v["ms"] / 5 / b_ for k, v in pf.items()}}
                Rc.close()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        n_pairs = max(cores, 8)
        v, kind, desc = cpu_reference(pairs, n_pairs, cores)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": desc}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "pairs_per_step": B, "batch": B,
                           "arithmetic": ("relaxed (library default for this option family): direct-form fmaf Gaussian window taps + mixed "
                                          "double/float horizontal poly-exp pass; measured <= 1.5e-4 px from the faithful oracle at "
                                          "1920x1080 (bar 1e-2), status and vectors identical; tests/test_gpu_relaxed.py, "
                                          "tests/test_gpu_configs_fullsize.py; variants.faithful_* time the oracle's own arithmetic")
                           if arithmetic == "relaxed" else "faithful: the oracle's operation order, bit-identical results",
                           "last_iteration": ("sparse: the finest scale's last blur + solve runs only at the positions the reference samples "
                                              "(src/consumer.cpp:60-77), as in the dispatcher -- the Response carries vectors and status, never "
                                              "the field; vectors bit-identical to the dense path (tests/test_gpu_sparse_last.py); the dense form "
                                              "is timed in variants.*_dense") if args.last == "sparse" else "dense: full flow field",
                           "launch": "one CUDA graph replay per step (%d kernel nodes)" % (launches // max(args.steps, 1)),
                           "parallelism": "independent pairs per GPU, no collective",
                           "l2": "256 MB memset between steps (inside the timed region) + per-step intermediates >> 126 MB L2",
                           "timed_region_s": elapsed_ms * 1e-3},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_inprocess": e2e_inprocess, "e2e_files": e2e_files, "variants": variants, "configs": configs,
                "gpu_launches": int(launches), "clocks": clocks, "statuses": statuses}
        print(json.dumps(line), flush=True)
    dist.close()


if __name__ == "__main__":
    main()
