"""Every kernel path, stage by stage, bit for bit against the oracle (oracle/farneback_ref.c) in both arithmetics; the threshold
comparison of every place that counts or samples, at thresholds taken from the data; spans at and beyond the kernels' block edges.

"arithmetic" = 0 must equal the faithful oracle; "arithmetic" = 1 must equal oracle(144) where ``arithmetic_in_effect`` says
"relaxed" and the faithful oracle elsewhere.  Each path runs a batch of three different pairs (a screenshot with a defect, a
texture, another screenshot), so every kernel's ``blockIdx.z`` plane offsets are exercised.  When a stage differs, the failure
names the stage, the batch slot, the scale (0 = coarsest) and the first differing element."""
import math

import numpy as np
import pytest

from oracle.oracle import FlowParam, sample_numpy

pytestmark = pytest.mark.gpu

RELAX_BITS = 144  # what "arithmetic" = 1 runs where relaxed: direct-form fmaf window taps + mixed double/float poly-exp pass
THR, SPAN = 0.5, 10


def _pairs(tw, w, h, seed):
    return [tw.synth.make_pair("S", w, h, seed, defect=True), tw.synth.make_pair("T", w, h, seed + 1),
            tw.synth.make_pair("S", w, h, seed + 2)]


def _oracle_runs(oracle, pairs, kw, bits, dump=True):
    """[(flow, dump)] of the oracle for every pair, under relax bits `bits`."""
    oracle.set_relax(bits)
    try:
        out = []
        for a, b in pairs:
            d = {} if dump else None
            out.append((oracle.farneback(a, b, FlowParam(**kw), dump=d), d))
        return out
    finally:
        oracle.set_relax(0)


def _bits(o, p):
    return RELAX_BITS if o.arithmetic_in_effect(p) == "relaxed" else 0


def _same(got, want, what):
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    if np.array_equal(got, want):
        return
    bad = np.argwhere(got != want)
    i = tuple(int(v) for v in bad[0])
    pytest.fail(f"{what}: {len(bad)} of {got.size} values differ; first at {i}: got {got[i]!r}, oracle {want[i]!r}")


def _vec(resp):
    return [(v["x"], v["y"], v["dx"], v["dy"]) for v in resp["vector"]]


def _check_answer(oracle, resp, flow, span, thr, what, skip=()):
    """Status, count and vector list of one pair against oracle.sample (and its NumPy restatement) on `flow`; sample points in
    `skip` are left out (ignore regions)."""
    status, vec = oracle.sample(flow, span, thr)
    vec = [v for v in vec if (v[0], v[1]) not in skip]
    assert vec == [v for v in sample_numpy(flow, span, thr)[1] if (v[0], v[1]) not in skip], what
    assert resp["status"] == ("SUSPICIOUS" if vec else "OK"), f"{what}: status {resp['status']}, oracle {len(vec)} vectors"
    assert resp["n_vectors"] == len(vec) and _vec(resp) == [tuple(v) for v in vec], f"{what}: vectors differ"


# ------------------------------------------------------------------------------------------------------------------------------
# A1  path matrix
# ------------------------------------------------------------------------------------------------------------------------------
# id: (frame, options on top of the defaults, context switches)
CASES = {
    "default_fused": ((328, 264), {}, {}),
    "default_ragged": ((333, 217), {}, {}),
    "levels2": ((344, 232), dict(pyrLevels=2), {}),
    "deep_fused": ((640, 512), dict(pyrLevels=5, pyrIterations=2), {}),
    "deep_separable": ((650, 520), dict(pyrLevels=5, pyrIterations=2), {}),
    "scale06_l2": ((300, 220), dict(pyrScale=0.6, pyrLevels=2), {}),
    "scale06_l3": ((333, 217), dict(pyrScale=0.6, pyrLevels=3), {}),
    "scale08_l4": ((300, 220), dict(pyrScale=0.8, pyrLevels=4), {}),
    "levels0": ((300, 220), dict(pyrLevels=0), {}),
    "iters1": ((300, 220), dict(pyrIterations=1), {}),
    "iters0": ((300, 220), dict(pyrIterations=0, pyrLevels=2), {}),
    "win32": ((300, 220), dict(winSize=32), {}),
    "win33": ((300, 220), dict(winSize=33), {}),
    "win40": ((300, 220), dict(winSize=40), {}),
    "win61": ((300, 220), dict(winSize=61), {}),
    "win9": ((300, 220), dict(winSize=9), {}),
    "win12": ((300, 220), dict(winSize=12), {}),
    "win20": ((300, 220), dict(winSize=20), {}),
    "win15_n5": ((300, 220), dict(winSize=15, polyN=5, polySigma=1.1), {}),
    "win15_n7": ((300, 220), dict(winSize=15), {}),
    "poly3": ((300, 220), dict(polyN=3, polySigma=0.9), {}),
    "poly5": ((300, 220), dict(polyN=5, polySigma=1.1), {}),
    "box15": ((203, 157), dict(flags=0, winSize=15), {}),
    "box31": ((203, 157), dict(flags=0), {}),
    "box15_unfused": ((203, 157), dict(flags=0, winSize=15), dict(box_unfused=1)),
    "box31_unfused": ((203, 157), dict(flags=0), dict(box_unfused=1)),
    "pitch4096_win40": ((2049, 48), dict(winSize=40), {}),
    "pitch4096_scale08": ((2049, 48), dict(pyrScale=0.8), {}),
    "pitchrt_win40": ((4097, 40), dict(winSize=40), {}),
    "pitchrt_scale08": ((4097, 40), dict(pyrScale=0.8), {}),
}


@pytest.mark.parametrize("case", list(CASES))
def test_kernel_path_stage_by_stage(tw, oracle, case):
    """Kernels each case reaches, worked out from enqueue, build_plan (schedule, int_scale, fused_levels), launch_level_image_fast,
    launch_polyexp, launch_first_update, launch_gauss_iter and box_fused_ok.  "a / b": "arithmetic" 0 / 1 where 1 runs another
    kernel (relaxed_in_effect); one name: both arithmetics run it.  Levels coarsest first; "generic" = level_image_kernel,
    "ident" = level_ident_kernel, "pyr<S,K>" = level_pyr_kernel (exact S x down-scale, K-tap pre-blur), "fused" =
    level_fused_kernel (the four finest levels in one launch).  Up-sample = first_update_kernel's bilinear up-sample of the
    coarser flow, 2x unless noted.  Row pitch 2048 unless noted.

    | case              | level images                                     | poly-exp                 | window iteration               |
    |-------------------|--------------------------------------------------|--------------------------|--------------------------------|
    | default_fused     | fused (41x33, 82x66, 164x132, 328x264)           | fast<7> / mixed<7>       | gauss_iter2<15, fma 0 / 2>     |
    | default_ragged    | generic (83x54, 166x108; not exact), ident       | fast<7> / mixed<7>       | gauss_iter2<15, fma 0 / 2>     |
    | levels2           | pyr<4,9>, pyr<2,3>, ident (3 scales: unfused)    | fast<7> / mixed<7>       | gauss_iter2<15, fma 0 / 2>     |
    | deep_fused        | pyr<16,39> (40x32), fused (4 finest)             | fast<7> / mixed<7>       | gauss_iter2<15, fma 0 / 2>     |
    | deep_separable    | level_rows + level_cols (41x32, 39 taps),        | fast<7> / mixed<7>       | gauss_iter2<15, fma 0 / 2>     |
    |                   | generic (81x65, 162x130), pyr<2,3>, ident        |                          |                                |
    | scale06_l2 / _l3  | generic (2 / 3 levels), ident; up-sample 1/0.6   | fast<7> / mixed<7>       | gauss_iter2<15, fma 0 / 2>     |
    | scale08_l4        | generic (4 levels), ident; up-sample 1/0.8       | fast<7> / mixed<7>       | gauss_iter2<15, fma 0 / 2>     |
    | levels0           | ident (one scale, zero initial flow)             | fast<7> / mixed<7>       | gauss_iter2<15, fma 0 / 2>     |
    | iters1            | pyr<4,9>, pyr<2,3>, ident                        | fast<7> / mixed<7>       | gauss_iter2<15>, LAST only     |
    | iters0            | pyr<4,9>, pyr<2,3>, ident                        | fast<7> / mixed<7>       | none: first_update writes the  |
    |                   |                                                  |                          | flow; sample_kernel uncounted  |
    | win32/33/40/61    | pyr<4,9>, pyr<2,3>, ident                        | fast<7> / mixed<7>       | gauss_iter_generic fma 0 / 2   |
    | win9/12/20        | pyr<4,9>, pyr<2,3>, ident                        | fast<7>                  | gauss_iter_generic fma 0       |
    | win15_n5          | pyr<4,9>, pyr<2,3>, ident                        | fast<5>                  | gauss_iter2<7, fma 0>          |
    | win15_n7          | pyr<4,9>, pyr<2,3>, ident                        | fast<7>                  | gauss_iter2<7, fma 0>          |
    | poly3             | pyr<4,9>, pyr<2,3>, ident                        | polyexp_kernel (generic) | gauss_iter2<15, fma 0>         |
    | poly5             | pyr<4,9>, pyr<2,3>, ident                        | fast<5>                  | gauss_iter2<15, fma 0>         |
    | box15 / box31     | generic (51x39, 102x78), ident                   | fast<7>                  | box_ckpt + box_band (m 7 / 15) |
    | box*_unfused      | generic (51x39, 102x78), ident                   | fast<7>                  | box_vsum + box_hscan, then     |
    |                   |                                                  |                          | first_update (flow_in)         |
    | pitch4096_win40   | ident (one scale); pitch 4096                    | fast<7,4096> / mixed<7>  | gauss_iter_generic fma 0 / 2   |
    | pitch4096_scale08 | generic (1639x38), ident; first_update<4096>,    | fast<7,4096> / mixed<7>  | gauss_iter2<15, fma 0 / 2,     |
    |                   | up-sample 1/0.8; pitch 4096                      |                          | 4096>                          |
    | pitchrt_win40     | ident (one scale); run-time pitch 4128           | fast<7,0> / mixed<7>     | gauss_iter_generic fma 0 / 2   |
    | pitchrt_scale08   | generic (3278x32), ident; first_update<0>,       | fast<7,0> / mixed<7>     | gauss_iter2<15, fma 0 / 2, 0>  |
    |                   | up-sample 1/0.8; run-time pitch 4128             |                          |                                |

    Gaussian windows of radius 15 / 7 with pyrIterations > 0 count the pair's vectors in gauss_epilogue and run sample_kernel
    counted; the other cases run it uncounted.  The keep_levels plan is checked at every scale and slot: I0, I1, R0, R1, the
    input M of the last iteration and the flow after it; then the production plan, eager, captured and replayed: the final flow
    and the answer."""
    (w, h), kw, opts = CASES[case]
    pairs = _pairs(tw, w, h, 11 + 3 * list(CASES).index(case))
    p = tw.OpticalFlowParameter(**kw)
    iters = p.pyrIterations
    o = tw.OpticalFlow(0, w, h, 3)
    for k, v in opts.items():
        o.set_option(k, v)
    refs = {}
    try:
        for arith in (0, 1):
            o.set_option("arithmetic", arith)
            bits = _bits(o, p)
            if bits not in refs:
                refs[bits] = _oracle_runs(oracle, pairs, kw, bits)
            ref = refs[bits]
            tag = f"{case} arithmetic {arith} (oracle relax {bits})"
            nscales = 1 + max(k[1] for k in ref[0][1])
            o.debug_keep_levels(True)
            res = o.calculate_batch(pairs, p, threshold=THR, span=SPAN)
            for i, (flow, dump) in enumerate(ref):
                for s in range(nscales):
                    at = f"{tag}: slot {i} scale {s}"
                    for nm in ("I0", "I1"):
                        _same(o.debug_read(nm, s, i)[0], dump[(nm, s, 0)], f"{at} {nm}")
                    for nm in ("R0", "R1"):
                        _same(o.debug_read(nm, s, i).transpose(1, 2, 0), dump[(nm, s, 0)], f"{at} {nm}")
                    if iters > 0:
                        _same(o.debug_read("M", s, i).transpose(1, 2, 0), dump[("M", s, iters - 1)], f"{at} M (input of the last iteration)")
                        _same(o.debug_read("flow", s, i).transpose(1, 2, 0), dump[("flow", s, iters - 1)], f"{at} flow")
                    else:
                        _same(o.debug_read("flow", s, i).transpose(1, 2, 0), dump[("flow_init", s, 0)], f"{at} flow (first update)")
                with pytest.raises(RuntimeError):
                    o.debug_read("I0", nscales, i)  # the plan has exactly the oracle's scales
                _check_answer(oracle, res[i], flow, SPAN, THR, f"{tag}: slot {i} (keep_levels)")
            o.debug_keep_levels(False)
            for rep in ("eager", "captured", "replayed"):
                res = o.calculate_batch(pairs, p, threshold=THR, span=SPAN)
                for i, (flow, _) in enumerate(ref):
                    fx, fy = o.batch_flow(i, w, h)
                    _same(np.stack([fx, fy], -1), flow, f"{tag}: slot {i} final flow ({rep})")
                    _check_answer(oracle, res[i], flow, SPAN, THR, f"{tag}: slot {i} ({rep})")
    finally:
        o.close()


# ------------------------------------------------------------------------------------------------------------------------------
# A2  thresholds taken from the data
# ------------------------------------------------------------------------------------------------------------------------------
def _thresholds(L):
    """(t_lo, t_hi): the largest double with t_lo * t_lo < L and the smallest double with t_hi * t_hi >= L."""
    L = float(L)
    t = math.sqrt(L)
    while t * t < L:
        t = float(np.nextafter(t, math.inf))
    while float(np.nextafter(t, 0.0)) ** 2 >= L:
        t = float(np.nextafter(t, 0.0))
    t_lo = float(np.nextafter(t, 0.0))
    assert t_lo * t_lo < L <= t * t
    return t_lo, t


def _picks(flow, span, skip=()):
    """Sample points at the edges of the kernels' blocks, with their float32 length dx*dx + dy*dy: the largest length, the
    largest on a tile-column boundary (x % 96 == 0), on a tile-row boundary (y % 32 == 0), in the last sampled row and in the
    last sampled column (the boundaries at 0 only where the span reaches no other).  Points of length 0 (no threshold below
    them) and points in `skip` are passed over."""
    fx = flow[::span, ::span, 0]
    fy = flow[::span, ::span, 1]
    L = (fx * fx) + (fy * fy)
    assert L.dtype == np.float32
    ys, xs = np.mgrid[0:L.shape[0], 0:L.shape[1]] * span
    ok = L > 0
    for (x, y) in skip:
        ok &= ~((xs == x) & (ys == y))
    col, row = ok & (xs % 96 == 0), ok & (ys % 32 == 0)
    col = col & (xs > 0) if (col & (xs > 0)).any() else col  # an interior tile boundary where the span reaches one
    row = row & (ys > 0) if (row & (ys > 0)).any() else row
    out = {}
    for name, sel in (("largest", ok), ("tile column", col), ("tile row", row), ("last row", ok & (ys == ys.max())),
                      ("last column", ok & (xs == xs.max()))):
        if sel.any():
            k = np.argmax(np.where(sel, L, -1.0))
            out[name] = (int(xs.flat[k]), int(ys.flat[k]), np.float32(L.flat[k]))
    assert "largest" in out
    return out


# id: (options, context switches, span, how the sample kernel runs)
THRESHOLD_PATHS = {
    "dense_tile": (dict(), {}, 10, None),                      # gauss_iter2 epilogue counts, sample_kernel counted
    "sparse_rows3": (dict(), dict(sparse_last=1), 10, None),   # gauss_last_sparse3_kernel counts
    "sparse_row1": (dict(), dict(sparse_last=1), 7, None),     # gauss_last_sparse_kernel counts
    "strip_last": (dict(), dict(window_tiles=0), 10, None),    # strip kernel, LAST form, counts
    "generic_radius": (dict(winSize=40), {}, 10, None),        # gauss_iter_generic: not counted
    "box": (dict(flags=0), {}, 10, None),                      # box_band: not counted
    "ignore": (dict(), {}, 10, "ignore"),                      # sample_ignore_kernel, counted
    "mask": (dict(), {}, 10, "mask"),                          # sample_mask_kernel (all-zero mask), counted
}


@pytest.mark.parametrize("arith", [0, 1])
@pytest.mark.parametrize("path", list(THRESHOLD_PATHS))
def test_threshold_edges_from_data(tw, oracle, path, arith):
    """At t_lo a picked point is above the threshold, at t_hi it is not: every place that compares (double)len > thr2 -- the
    fused counts (tile epilogue, both sparse kernels, the strip kernel's LAST form) and sample_body -- must agree with the
    reference there, or a pair comes back with the wrong status or vector list.  The largest length decides OK / SUSPICIOUS and
    is where the sample kernels' early exit on a fused count of 0 must be right."""
    kw, opts, span, how = THRESHOLD_PATHS[path]
    if kw.get("flags") == 0 and arith == 1:
        pytest.skip("the box window runs the faithful kernels in both arithmetics")
    w, h = 500, 333
    pairs = _pairs(tw, w, h, 300)
    p = tw.OpticalFlowParameter(**kw)
    region = (0, 0, 1, 1)  # covers the sample point (0, 0) only
    skip = {(0, 0)} if how == "ignore" else set()
    dense_pairs = pairs
    if how == "ignore":  # the flow of an ignore run is the flow of the target painted with the expected pixels of the region
        a, b = pairs[0]
        b = b.copy()
        b[0:1, 0:1] = a[0:1, 0:1]
        dense_pairs = [(a, b)] + pairs[1:]
    o = tw.OpticalFlow(0, w, h, 3)
    try:
        o.set_option("arithmetic", arith)
        o.calculate_batch(dense_pairs, p, threshold=5.0, span=span)
        flows = [np.stack(o.batch_flow(i, w, h), -1) for i in range(3)]
        for k, v in opts.items():
            o.set_option(k, v)
        extra = {}
        if how == "ignore":
            extra = dict(ignore=[[region], [], []])
        elif how == "mask":
            extra = dict(ignore_mask=[np.zeros((h, w), np.uint8)] * 3)
        picks = _picks(flows[0], span, skip)
        exact = 0
        for name, (x, y, L) in picks.items():
            t_lo, t_hi = _thresholds(L)
            exact += t_hi * t_hi == float(L)
            for thr in (t_lo, t_hi):
                res = o.calculate_batch(pairs, p, threshold=thr, span=span, **extra)
                for i in range(3):
                    _check_answer(oracle, res[i], flows[i], span, thr, f"{path} arithmetic {arith}: {name} point ({x}, {y}) len {L!r} "
                                  f"threshold {thr!r} slot {i}", skip if i == 0 else ())
                got = [(v["x"], v["y"]) for v in res[0]["vector"]]
                assert ((x, y) in got) == (thr == t_lo), (name, thr)
                if name == "largest":
                    assert res[0]["status"] == ("SUSPICIOUS" if thr == t_lo else "OK") and (thr == t_lo or not got)
        assert exact > 0, "no picked length is the exact square of a double: a >= would go unnoticed"
    finally:
        o.close()


# ------------------------------------------------------------------------------------------------------------------------------
# A3  spans at and beyond the kernels' block edges
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arith", [0, 1])
def test_spans_at_block_edges(tw, oracle, arith):
    """Spans 1-3 (the sparse kernels cannot hold a CTA's samples: gauss_last_sparse_ok is false and the dense path runs), 4, the
    tile width 96 and its neighbours, the sparse CTA width 226 and its neighbours, a span taller than the frame (one sample row)
    and one wider than it (the single point (0, 0)); dense and sparse_last, against oracle.sample."""
    w, h = 333, 217
    pairs = _pairs(tw, w, h, 500)
    o = tw.OpticalFlow(0, w, h, 3)
    o.set_option("arithmetic", arith)
    p = tw.OpticalFlowParameter()
    ref = [f for f, _ in _oracle_runs(oracle, pairs, {}, _bits(o, p), dump=False)]
    try:
        for span in (1, 2, 3, 4, 95, 96, 97, 225, 226, 227, 300, 334):
            for thr in (0.0, 0.3):
                for sparse in (0, 1):
                    o.set_option("sparse_last", sparse)
                    res = o.calculate_batch(pairs, p, threshold=thr, span=span)
                    for i in range(3):
                        _check_answer(oracle, res[i], ref[i], span, thr, f"arithmetic {arith} span {span} threshold {thr} sparse {sparse} slot {i}")
                    if sparse and span >= 4:
                        with pytest.raises(RuntimeError):
                            o.batch_flow(0, w, h)  # the sparse kernel ran: no dense field
                    else:
                        for i in range(3):
                            _same(np.stack(o.batch_flow(i, w, h), -1), ref[i], f"arithmetic {arith} span {span} sparse {sparse} slot {i} flow")
    finally:
        o.close()
