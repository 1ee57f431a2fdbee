"""GPU tests of ignore regions (tw_compare_ignore, tw_compare_batch_ignore, tw_pipe_submit_ignore, tw_pool_submit*_ignore and
create()'s ignoreRegions / getIgnoreRegions).  The contract (include/tidalwave_b200.h): the answer for a pair with regions is the
plain answer for (expected, target painted with the expected pixels inside the regions) minus the vectors inside the regions --
bit for bit, in both arithmetics and on every window / box / sparse path.  That host-side restatement is the oracle here."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

from conftest import OPTS
from oracle.oracle import FlowParam

pytestmark = pytest.mark.gpu


def _box(r):
    if isinstance(r, dict):
        return r["x"], r["y"], r["width"], r["height"]
    return tuple(r)


def paint(a, b, regions):
    """b with a's pixels inside the regions (clipped to the frame)."""
    out = b.copy()
    h, w = a.shape
    for x, y, rw, rh in map(_box, regions or []):
        x0, y0, x1, y1 = max(x, 0), max(y, 0), min(x + rw, w), min(y + rh, h)
        if x0 < x1 and y0 < y1:
            out[y0:y1, x0:x1] = a[y0:y1, x0:x1]
    return out


def inside(v, regions):
    return any(x <= v[0] < x + rw and y <= v[1] < y + rh for x, y, rw, rh in map(_box, regions or []))


def vecs(resp):
    return [(v["x"], v["y"], v["dx"], v["dy"]) for v in resp["vector"]]


def drop(resp, regions):
    """(status, n_vectors, vectors) of a plain answer with the vectors inside the regions removed."""
    kept = [v for v in vecs(resp) if not inside(v, regions)]
    return ("SUSPICIOUS" if kept else "OK"), len(kept), kept


def answer(resp):
    return resp["status"], resp["n_vectors"], vecs(resp)


def _pairs(tw, w, h, seed=70):
    return [tw.synth.make_pair("S" if i % 2 == 0 else "T", w, h, seed + i, defect=(i == 0)) for i in range(3)]


def _lists(w, h):
    first = [None, [(40, 30, 80, 60)], [(10, 10, 100, 80), {"x": 60, "y": 50, "width": 120, "height": 90}]]  # none, one, overlapping
    second = [[(-20, h - 50, 90, 100)], [(0, 0, w, h)], [(w // 2, 0, 30, h), (0, h // 3, w, 20)]]  # partly outside, whole frame, a cross
    return first, second


@pytest.mark.parametrize("arith", [0, 1])
@pytest.mark.parametrize("sparse", [0, 1])
@pytest.mark.parametrize("opt,size", [("default", (333, 217)), ("cfg4", (300, 200)), ("g15n5", (300, 200)), ("cfg3", (512, 320))])
def test_equals_painted_compare(tw, arith, sparse, opt, size):
    w, h = size
    thr = 0.2
    pairs = _pairs(tw, w, h)
    p = tw.OpticalFlowParameter(**OPTS[opt])
    o, ref = tw.OpticalFlow(0, w, h, 3), tw.OpticalFlow(0, w, h, 3)
    for c in (o, ref):
        c.set_option("arithmetic", arith)
        c.set_option("sparse_last", sparse)
    nontrivial = 0
    for lists in _lists(w, h):
        want = [drop(r, g) for r, g in zip(ref.calculate_batch([(a, paint(a, b, g)) for (a, b), g in zip(pairs, lists)], p, thr), lists)]
        nontrivial += sum(n for _, n, _ in want)
        for rep in range(3):  # eager, capture, replay; the second list set replays the same graph key
            got = o.calculate_batch(pairs, p, thr, ignore=lists)
            assert [answer(r) for r in got] == want, (rep, lists)
            assert all((r["width"], r["height"]) == (w, h) for r in got)
    assert nontrivial > 0
    o.close(); ref.close()


def test_oracle_faithful(tw, oracle):
    a, b = tw.synth.make_pair("S", 480, 300, 33, defect=True)
    regions = [(100, 60, 120, 90), (300, 200, 500, 500)]
    o = tw.OpticalFlow(0, 480, 300, 1)
    o.set_option("arithmetic", 0)
    status, vec = oracle.sample(oracle.farneback(a, paint(a, b, regions), FlowParam()), span=10, threshold=0.2)
    kept = [tuple(v) for v in vec if not inside(v, regions)]
    got = o.calculate(a, b, threshold=0.2, ignore=regions)
    assert answer(got) == (("SUSPICIOUS" if kept else "OK"), len(kept), kept)
    assert kept and len(kept) < len(vec)
    o.close()


def test_dense_flow_is_painted_flow(tw):
    w, h = 320, 200
    pairs = _pairs(tw, w, h, 11)
    lists = [[(50, 40, 100, 70)], None, [(0, 0, 160, 200)]]
    o, ref = tw.OpticalFlow(0, w, h, 3), tw.OpticalFlow(0, w, h, 3)
    o.calculate_batch(pairs, ignore=lists)
    ref.calculate_batch([(a, paint(a, b, g)) for (a, b), g in zip(pairs, lists)])
    for i in range(3):
        fx, fy = o.batch_flow(i, w, h)
        rx, ry = ref.batch_flow(i, w, h)
        assert np.array_equal(fx, rx) and np.array_equal(fy, ry)
    o.close(); ref.close()


def test_no_regions_is_identity(tw):
    """*_ignore without regions (and regions wholly outside the frame) run exactly the plain launch sequence."""
    w, h = 333, 217
    pairs = _pairs(tw, w, h)
    a, b = pairs[0]
    plain, other = tw.OpticalFlow(0, w, h, 3), tw.OpticalFlow(0, w, h, 3)

    def strip(rs):
        return [{k: v for k, v in r.items() if k != "time"} for r in rs]

    for ignore in ([[], None, []], [[(w, 0, 10, 10)], [(-50, -50, 50, 400)], [(0, h + 3, w, 9)]]):
        for rep in range(3):
            l0, l1 = plain.launch_count(), other.launch_count()
            want = plain.calculate_batch(pairs, threshold=0.2)
            got = other.calculate_batch(pairs, threshold=0.2, ignore=ignore)
            assert strip(got) == strip(want)
            assert other.launch_count() - l1 == plain.launch_count() - l0
        l0, l1 = plain.launch_count(), other.launch_count()
        single = [plain.calculate(a, b, threshold=0.2), other.calculate(a, b, threshold=0.2, ignore=ignore[0])]
        assert strip(single[:1]) == strip(single[1:]) and other.launch_count() - l1 == plain.launch_count() - l0
    plain.close(); other.close()


def test_size_tolerance_path(tw):
    w, h = 320, 200
    a, _ = tw.synth.make_pair("S", w, h, 5, defect=True)
    _, big = tw.synth.make_pair("S", w + 3, h - 2, 5, defect=True)
    regions = [(30, 20, 90, 60), (200, 150, 200, 100)]
    o = tw.OpticalFlow(0, w + 8, h + 8, 1)
    lib = tw.load()
    resized = np.empty((h, w), np.uint8)
    big = np.ascontiguousarray(big)
    assert lib.tw_resize_target(o.ctx, big.ctypes.data, w + 3, h - 2, resized.ctypes.data, w, h) == 0
    want = drop(o.calculate(a, paint(a, resized, regions), threshold=0.3), regions)
    got = o.calculate(a, big, threshold=0.3, ignore=regions)
    assert answer(got) == want and (got["width"], got["height"]) == (w, h)
    o.close()


def _ptrs(imgs):
    return (C.c_void_p * len(imgs))(*[x.ctypes.data for x in imgs])


def test_pipe_batches_keep_their_lists(tw):
    w, h = 333, 217
    pairs = _pairs(tw, w, h)
    first, second = _lists(w, h)
    o, ref = tw.OpticalFlow(0, w, h, 3), tw.OpticalFlow(0, w, h, 3)
    want = [[answer(r) for r in ref.calculate_batch(pairs, threshold=0.2, ignore=g)] for g in (first, second, first)]
    lib = tw.load()
    p = tw.OpticalFlowParameter().c()
    ex, tg = _ptrs([a for a, _ in pairs]), _ptrs([b for _, b in pairs])
    keep = []

    def submit(lists):
        rs = [tw.api._rects(g) for g in lists]
        keep.append(rs)
        ig = (C.POINTER(tw.tw_rect) * 3)(*[C.cast(r, C.POINTER(tw.tw_rect)) if r is not None else None for r, _ in rs])
        nig = (C.c_int * 3)(*[k for _, k in rs])
        assert lib.tw_pipe_submit_ignore(o.ctx, 3, ex, tg, w, h, w, C.byref(p), 0.2, 10, ig, nig) == 0, o.last_error()

    cap = ((w + 9) // 10) * ((h + 9) // 10)

    def collect():
        vec = (tw.tw_vector * (3 * cap))()
        res = (tw.tw_result * 3)()
        assert lib.tw_pipe_collect(o.ctx, vec, cap, res) == 0
        return [answer(tw.api._response(res[i], (tw.tw_vector * cap).from_buffer(vec, i * cap * C.sizeof(tw.tw_vector)),
                                         min(res[i].n_vectors, cap), 10, 0.2)) for i in range(3)]

    got = []
    for lists in (first, second, first):  # two batches in flight with different lists, a third behind them; eager, capture, replay
        if lib.tw_pipe_pending(o.ctx) >= 2:
            got.append(collect())
        submit(lists)
    while lib.tw_pipe_pending(o.ctx):
        got.append(collect())
    assert got == want
    o.close(); ref.close()


def test_pool_mixed_requests(tw, tmp_path):
    cv2 = pytest.importorskip("cv2")
    w, h = 320, 200
    pairs = _pairs(tw, w, h, 40) + _pairs(tw, w, h, 50)
    files = []
    for i, (a, b) in enumerate(pairs[:3]):
        pa, pb = str(tmp_path / f"e{i}.png"), str(tmp_path / f"t{i}.png")
        cv2.imwrite(pa, a); cv2.imwrite(pb, b)
        files.append((pa, pb))
    _, big = tw.synth.make_pair("S", w - 4, h + 2, 40, defect=True)
    lists = [None, [(40, 30, 80, 60)], [(10, 10, 100, 80), (60, 50, 120, 90)], [(0, 0, w, h)], [(-5, 150, 400, 30)], []]
    jobs = []  # (kind, index, regions)
    for i in range(len(pairs)):
        jobs.append(("img", i, lists[i % len(lists)]))
    for i in range(3):
        jobs.append(("file", i, lists[(i + 1) % len(lists)]))
    jobs.append(("resize", 0, [(20, 20, 50, 50)]))
    jobs.append(("bad", 1, [(0, 0, 0, 10)]))
    o = tw.OpticalFlow(0, w, h, 1)

    def single(kind, i, regions):
        if kind == "resize":
            return o.calculate(pairs[0][0], big, threshold=0.2, ignore=regions)
        a, b = pairs[i]
        return o.calculate(a, b, threshold=0.2, ignore=regions)

    want = [single(*j) for j in jobs]
    assert want[-1]["status"] == "ERROR" and want[-1]["code"] == tw.api.BAD_PARAMETER
    pool = tw.Pool([0], threshold=0.2, batch=4)
    ids = [None] * len(jobs)

    def worker(k0):
        for k in range(k0, len(jobs), 3):
            kind, i, regions = jobs[k]
            if kind == "file":
                ids[k] = pool.request_files(*files[i], ignore=regions)
            elif kind == "resize":
                ids[k] = pool.request(pairs[0][0], big, ignore=regions)
            else:
                ids[k] = pool.request(*pairs[i], ignore=regions)

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(3)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    got = [pool.wait(i) for i in ids]
    rep = pool.report()
    pool.stop(); pool.close(); o.close()
    for g, wnt, job in zip(got, want, jobs):
        if wnt["status"] == "ERROR":
            assert g["status"] == "ERROR" and g["code"] == wnt["code"] and g["reason"].startswith("bad ignore region"), job
        else:
            assert answer(g) == answer(wnt) and (g["width"], g["height"]) == (wnt["width"], wnt["height"]), job
    assert rep == {"request": len(jobs), "data": len(jobs) - 1, "error": 1}
    assert sum(g["n_vectors"] for g in got if g["status"] != "ERROR") > 0


def test_validation(tw):
    w, h = 160, 120
    a, b = tw.synth.make_pair("S", w, h, 3, defect=True)
    o = tw.OpticalFlow(0, w, h, 2)
    base = o.calculate(a, b, threshold=0.2)
    for bad in ([(0, 0, 0, 10)], [(5, 5, 10, -1)], [(i, i, 4, 4) for i in range(33)]):
        r = o.calculate(a, b, threshold=0.2, ignore=bad)
        assert r["status"] == "ERROR" and r["code"] == tw.api.BAD_PARAMETER and r["reason"].startswith("bad ignore region"), bad
        rb = o.calculate_batch([(a, b), (a, b)], threshold=0.2, ignore=[None, bad])
        assert all(x["status"] == "ERROR" and x["code"] == tw.api.BAD_PARAMETER for x in rb)
    assert len(tw.api._rects([(0, 0, 1, 1)] * 32)[0]) == tw.MAX_IGNORE
    lib = tw.load()
    p = tw.OpticalFlowParameter().c()
    res = tw.tw_result()
    vec = (tw.tw_vector * 256)()
    rc = lib.tw_compare_ignore(o.ctx, a.ctypes.data, w, h, b.ctypes.data, w, h, C.byref(p), 0.2, 10, None, 1, vec, 256, C.byref(res))
    assert rc == tw.api.BAD_PARAMETER and res.reason.startswith(b"bad ignore region")
    nig = (C.c_int * 1)(2)
    rc = lib.tw_compare_batch_ignore(o.ctx, 1, _ptrs([a]), _ptrs([b]), w, h, w, C.byref(p), 0.2, 10, None, nig, vec, 256, C.byref(res))
    assert rc == tw.api.BAD_PARAMETER
    # the context still works, and a region wholly outside the frame is no region
    outside = o.calculate(a, b, threshold=0.2, ignore=[(w, 0, 5, 5), (-10, -10, 10, 500)])
    assert answer(outside) == answer(base) and base["n_vectors"] > 0
    with pytest.raises(ValueError):
        o.calculate(a, b, ignore=[(1, 2, 3)])
    o.close()


def test_user_story(tw):
    """A page whose changed part is declared ignorable comes back OK."""
    w, h, span = 320, 200, 10
    a, b = tw.synth.make_pair("S", w, h, 10, defect=True)  # seed chosen so that the defect's flow stays inside the grown box
    o = tw.OpticalFlow(0, w, h, 1)
    plain = o.calculate(a, b)
    assert plain["status"] == "SUSPICIOUS" and plain["n_vectors"] > 0
    xs, ys = [v["x"] for v in plain["vector"]], [v["y"] for v in plain["vector"]]
    box = {"x": min(xs) - 2 * span, "y": min(ys) - 2 * span, "width": max(xs) - min(xs) + 4 * span + 1,
           "height": max(ys) - min(ys) + 4 * span + 1}
    masked = o.calculate(a, b, ignore=[box])
    assert masked["status"] == "OK" and masked["n_vectors"] == 0 and masked["vector"] == []
    o.close()


def test_create_options(tw, tmp_path):
    cv2 = pytest.importorskip("cv2")
    w, h = 320, 200
    exp_dir, tgt_dir = tmp_path / "expected", tmp_path / "target"
    os.makedirs(exp_dir / "sub"); os.makedirs(tgt_dir / "sub")
    names = ["a.png", "b.png", "sub/c.png", "sub/d.png"]
    for i, n in enumerate(names):
        a, b = tw.synth.make_pair("S", w, h, 10 + i, defect=True)
        cv2.imwrite(str(exp_dir / n), a)
        cv2.imwrite(str(tgt_dir / n), b)
    common = [{"x": 0, "y": 0, "width": 40, "height": 30}]
    own = {"a.png": [{"x": 60, "y": 40, "width": 200, "height": 120}], "sub/c.png": [(100, 0, 50, 200)], "sub/d.png": [{"x": 1, "y": 2}]}
    data, errors, fin = [], [], []
    t = tw.create(str(tgt_dir), {"expectDir": str(exp_dir), "threshold": 0.5, "ignoreRegions": common,
                                 "getIgnoreRegions": lambda short: own.get(short)})
    t.on("data", data.append).on("error", errors.append).on("finish", fin.append)
    tw.run(t)
    assert fin == [{"request": 4, "data": 3, "error": 1}]
    assert len(errors) == 1 and errors[0]["reason"].startswith("bad ignore region")
    pool = tw.Pool([0], threshold=0.5)
    by_target = {d["target_image"]: d for d in data}
    for n in names[:3]:
        regions = common + (own.get(n) or [])
        want = pool.wait(pool.request_files(str(exp_dir / n), str(tgt_dir / n), ignore=regions))
        d = by_target[str(tgt_dir / n)]
        assert (d["status"], vecs(d)) == (want["status"], vecs(want)), n
    pool.stop(); pool.close()
    assert sum(len(d["vector"]) for d in data) > 0
