"""GPU tests of ignore masks (tw_compare_mask, tw_compare_batch_mask, tw_pipe_submit_mask, tw_pool_submit*_mask and create()'s
ignoreMaskDir / getIgnoreMaskPath).  The contract (include/tidalwave_b200.h): the answer for a pair with a mask (and regions) is the
plain answer for (expected, target painted with the expected pixels wherever the mask is nonzero or a region lies) minus the
vectors at those points -- bit for bit, in both arithmetics and on every window / box / sparse / strip path.  That host-side
restatement is the oracle here; the region helpers come from test_gpu_ignore."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

from conftest import OPTS
from test_gpu_ignore import _lists, _pairs, _ptrs, answer, inside, paint, vecs

pytestmark = pytest.mark.gpu


def mpaint(a, b, mask):
    """b with a's pixels where the mask is nonzero."""
    return b if mask is None else np.where(np.asarray(mask) != 0, a, b).astype(np.uint8)


def ignored(v, regions, mask):
    return inside(v, regions) or (mask is not None and bool(mask[v[1], v[0]]))


def want_batch(ref, pairs, lists, masks, p=None, thr=0.2):
    """The plain answers for the host-painted pairs, with the vectors at ignored points removed."""
    lists = lists or [None] * len(pairs)
    masks = masks or [None] * len(pairs)
    painted = [(a, mpaint(a, paint(a, b, g), m)) for (a, b), g, m in zip(pairs, lists, masks)]
    out = []
    for r, g, m in zip(ref.calculate_batch(painted, threshold=thr, **({"param": p} if p is not None else {})), lists, masks):
        kept = [v for v in vecs(r) if not ignored(v, g, m)]
        out.append((("SUSPICIOUS" if kept else "OK"), len(kept), kept))
    return out


def raster(regions, w, h):
    """The mask of a region list (clipped to the frame): 255 inside, 0 outside."""
    return paint(np.full((h, w), 255, np.uint8), np.zeros((h, w), np.uint8), regions)


def _masks(w, h, seed=3):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    r2 = (xx - 0.4 * w) ** 2 + (yy - 0.5 * h) ** 2
    disc = (r2 < (0.3 * min(w, h)) ** 2).astype(np.uint8) * 255
    ring = ((r2 < (0.45 * min(w, h)) ** 2) & (r2 > (0.2 * min(w, h)) ** 2)).astype(np.uint8) * rng.integers(1, 256, (h, w), dtype=np.uint8)
    spots = rng.random((h, w)) < 0.05  # bool, every 20th pixel
    band = np.zeros((h, w), bool)
    band[:, (w * 2) // 3:] = True  # the right third, up to the last column
    first = [None, disc, spots]
    second = [ring, None, band | spots]
    return first, second


@pytest.mark.parametrize("arith", [0, 1])
@pytest.mark.parametrize("sparse", [0, 1])
@pytest.mark.parametrize("opt,size", [("default", (333, 217)), ("cfg4", (300, 200)), ("g15n5", (300, 200)), ("cfg3", (512, 320)),
                                      ("strip", (512, 320))])
def test_equals_painted_compare(tw, arith, sparse, opt, size):
    w, h = size
    thr = 0.2
    pairs = _pairs(tw, w, h)
    p = tw.OpticalFlowParameter(**OPTS["default" if opt == "strip" else opt])
    o, ref = tw.OpticalFlow(0, w, h, 3), tw.OpticalFlow(0, w, h, 3)
    for c in (o, ref):
        c.set_option("arithmetic", arith)
        c.set_option("sparse_last", sparse)
        c.set_option("window_tiles", 0 if opt == "strip" else 1)
    masks = _masks(w, h)
    regions = ([None, [(40, 30, 80, 60)], None], [[(10, 10, 60, 40)], None, None])  # regions on some pair in both: one graph key
    nontrivial = 0
    for lists, mk in zip(regions, masks):
        want = want_batch(ref, pairs, lists, mk, p, thr)
        nontrivial += sum(n for _, n, _ in want)
        for rep in range(3):  # eager, capture, replay; the second mask set replays the same graph key
            got = o.calculate_batch(pairs, p, thr, ignore=lists, ignore_mask=mk)
            assert [answer(r) for r in got] == want, (rep, opt)
            assert all((r["width"], r["height"]) == (w, h) for r in got)
    assert nontrivial > 0
    o.close(); ref.close()


def test_mask_of_regions_and_union(tw):
    """A rasterised region list is that list; a mask plus regions is their union; an all-zero mask is no mask."""
    w, h = 333, 217
    pairs = _pairs(tw, w, h)
    o, ref = tw.OpticalFlow(0, w, h, 3), tw.OpticalFlow(0, w, h, 3)
    for lists in _lists(w, h):
        by_regions = [answer(r) for r in ref.calculate_batch(pairs, threshold=0.2, ignore=lists)]
        for rep in range(3):
            got = o.calculate_batch(pairs, threshold=0.2, ignore_mask=[raster(g, w, h) for g in lists])
            assert [answer(r) for r in got] == by_regions, rep
        a, b = pairs[2]
        assert answer(o.calculate(a, b, threshold=0.2, ignore_mask=raster(lists[2], w, h) > 0)) == by_regions[2]
    first, _ = _masks(w, h)
    lists = _lists(w, h)[0]
    want = want_batch(ref, pairs, lists, first)
    for rep in range(3):
        assert [answer(r) for r in o.calculate_batch(pairs, threshold=0.2, ignore=lists, ignore_mask=first)] == want
    plain = [answer(r) for r in ref.calculate_batch(pairs, threshold=0.2)]
    zeros = [np.zeros((h, w), np.uint8)] * 3
    for rep in range(3):
        assert [answer(r) for r in o.calculate_batch(pairs, threshold=0.2, ignore_mask=zeros)] == plain
    assert answer(o.calculate(*pairs[0], threshold=0.2, ignore_mask=zeros[0])) == plain[0]
    assert sum(n for _, n, _ in plain) > 0
    o.close(); ref.close()


def test_dense_flow_is_painted_flow(tw):
    w, h = 320, 200
    pairs = _pairs(tw, w, h, 11)
    masks = _masks(w, h)[0]
    o, ref = tw.OpticalFlow(0, w, h, 3), tw.OpticalFlow(0, w, h, 3)
    o.calculate_batch(pairs, ignore_mask=masks)
    ref.calculate_batch([(a, mpaint(a, b, m)) for (a, b), m in zip(pairs, masks)])
    for i in range(3):
        fx, fy = o.batch_flow(i, w, h)
        rx, ry = ref.batch_flow(i, w, h)
        assert np.array_equal(fx, rx) and np.array_equal(fy, ry)
    o.close(); ref.close()


def test_no_mask_is_identity(tw):
    """Without masks the plain and region-only launch sequences run unchanged; a mask adds exactly the paint launch."""
    w, h = 333, 217
    pairs = _pairs(tw, w, h)
    lists = _lists(w, h)[0]
    plain, other = tw.OpticalFlow(0, w, h, 3), tw.OpticalFlow(0, w, h, 3)

    def strip(rs):
        return [{k: v for k, v in r.items() if k != "time"} for r in rs]

    def launches(of, fn):
        l0 = of.launch_count()
        out = fn()
        return out, of.launch_count() - l0

    for rep in range(3):
        want, lw = launches(plain, lambda: plain.calculate_batch(pairs, threshold=0.2))
        got, lg = launches(other, lambda: other.calculate_batch(pairs, threshold=0.2, ignore_mask=[None] * 3))
        assert strip(got) == strip(want) and lg == lw
        want, lw = launches(plain, lambda: plain.calculate_batch(pairs, threshold=0.2, ignore=lists))
        got, lg = launches(other, lambda: other.calculate_batch(pairs, threshold=0.2, ignore=lists, ignore_mask=[None] * 3))
        assert strip(got) == strip(want) and lg == lw
    masks = _masks(w, h)[0]
    for rep in range(3):
        _, lp = launches(plain, lambda: plain.calculate_batch(pairs, threshold=0.2))
        _, lm = launches(other, lambda: other.calculate_batch(pairs, threshold=0.2, ignore_mask=masks))
        _, li = launches(plain, lambda: plain.calculate_batch(pairs, threshold=0.2, ignore=lists))
        _, lb = launches(other, lambda: other.calculate_batch(pairs, threshold=0.2, ignore=lists, ignore_mask=masks))
        assert (lm - lp, li - lp, lb - lp) == (1, 1, 2), rep
    # the C entry points with no mask return what their counterparts return
    lib = tw.load()
    p = tw.OpticalFlowParameter().c()
    a, b = pairs[0]
    cap = ((w + 9) // 10) * ((h + 9) // 10)
    res = [tw.tw_result() for _ in range(2)]
    vec = [(tw.tw_vector * cap)() for _ in range(2)]
    lib.tw_compare(plain.ctx, a.ctypes.data, w, h, b.ctypes.data, w, h, C.byref(p), 0.2, 10, vec[0], cap, C.byref(res[0]))
    lib.tw_compare_mask(other.ctx, a.ctypes.data, w, h, b.ctypes.data, w, h, C.byref(p), 0.2, 10, None, 0, None, vec[1], cap,
                        C.byref(res[1]))
    n = res[0].n_vectors
    assert n > 0 and (res[0].code, res[0].status, n) == (res[1].code, res[1].status, res[1].n_vectors)
    assert bytes(vec[0])[:n * C.sizeof(tw.tw_vector)] == bytes(vec[1])[:n * C.sizeof(tw.tw_vector)]
    plain.close(); other.close()


def test_size_tolerance_path(tw):
    """The target is resized to the expected size first; the mask is in expected-image pixels."""
    w, h = 320, 200
    a, _ = tw.synth.make_pair("S", w, h, 5, defect=True)
    _, big = tw.synth.make_pair("S", w + 3, h - 2, 5, defect=True)
    mask = _masks(w, h)[0][1]
    regions = [(200, 150, 200, 100)]
    o = tw.OpticalFlow(0, w + 8, h + 8, 1)
    lib = tw.load()
    resized = np.empty((h, w), np.uint8)
    big = np.ascontiguousarray(big)
    assert lib.tw_resize_target(o.ctx, big.ctypes.data, w + 3, h - 2, resized.ctypes.data, w, h) == 0
    r = o.calculate(a, mpaint(a, paint(a, resized, regions), mask), threshold=0.3)
    kept = [v for v in vecs(r) if not ignored(v, regions, mask)]
    got = o.calculate(a, big, threshold=0.3, ignore=regions, ignore_mask=mask)
    assert answer(got) == (("SUSPICIOUS" if kept else "OK"), len(kept), kept) and (got["width"], got["height"]) == (w, h)
    bad = o.calculate(a, big, threshold=0.3, ignore_mask=np.zeros((h - 2, w + 3), np.uint8))  # a mask of the target's size
    assert bad["status"] == "ERROR" and bad["code"] == tw.api.BAD_PARAMETER
    assert bad["reason"] == f"bad ignore mask: {w + 3}x{h - 2} mask for a {w}x{h} expected image"
    o.close()


@pytest.mark.parametrize("w", [2049, 4097])
def test_wide_frames_row_tails(tw, w):
    """No padding after the last column and a row pitch read at run time: the paint kernel's last vector of a row goes byte by
    byte."""
    h = 72
    pairs = [tw.synth.make_pair("S", w, h, 60 + i, defect=False) for i in range(2)]
    rng = np.random.default_rng(w)
    m0 = rng.random((h, w)) < 0.3
    m0[:, w - 5:] = True  # the row tail
    m1 = np.zeros((h, w), np.uint8)
    m1[::3, w - 20:] = 7
    m1[:, :40] = 1
    o, ref = tw.OpticalFlow(0, w, h, 2), tw.OpticalFlow(0, w, h, 2)
    want = want_batch(ref, pairs, None, [m0, m1], thr=0.05)
    assert sum(n for _, n, _ in want) > 0
    for rep in range(3):
        assert [answer(r) for r in o.calculate_batch(pairs, threshold=0.05, ignore_mask=[m0, m1])] == want, rep
    o.close(); ref.close()


def test_pipe_alternating_masks(tw):
    """Masked, unmasked and differently masked batches, two in flight; the staging buffer grows while one is in flight."""
    w, h = 333, 217
    pairs = _pairs(tw, w, h)
    first, second = _masks(w, h)
    o, ref = tw.OpticalFlow(0, w, h, 3), tw.OpticalFlow(0, w, h, 3)
    seq = [None, first, None, second, first, second]
    want = [[answer(r) for r in ref.calculate_batch(pairs, threshold=0.2, ignore_mask=m)] for m in seq]
    lib = tw.load()
    p = tw.OpticalFlowParameter().c()
    ex, tg = _ptrs([a for a, _ in pairs]), _ptrs([b for _, b in pairs])
    keep = []

    def submit(masks):
        if masks is None:
            mk = None
        else:
            arrs = [tw.api.mask_array(m) for m in masks]
            keep.append(arrs)
            mk = (C.c_void_p * 3)(*[m.ctypes.data if m is not None else None for m in arrs])
        assert lib.tw_pipe_submit_mask(o.ctx, 3, ex, tg, w, h, w, C.byref(p), 0.2, 10, None, None, mk) == 0, o.last_error()

    cap = ((w + 9) // 10) * ((h + 9) // 10)

    def collect():
        vec = (tw.tw_vector * (3 * cap))()
        res = (tw.tw_result * 3)()
        assert lib.tw_pipe_collect(o.ctx, vec, cap, res) == 0
        return [answer(tw.api._response(res[i], (tw.tw_vector * cap).from_buffer(vec, i * cap * C.sizeof(tw.tw_vector)),
                                         min(res[i].n_vectors, cap), 10, 0.2)) for i in range(3)]

    got = []
    for masks in seq:
        if lib.tw_pipe_pending(o.ctx) >= 2:
            got.append(collect())
        submit(masks)
    while lib.tw_pipe_pending(o.ctx):
        got.append(collect())
    assert got == want
    o.close(); ref.close()


def _write(cv2, path, img):
    assert cv2.imwrite(str(path), img)
    return str(path)


def test_pool_mixed_requests(tw, tmp_path):
    cv2 = pytest.importorskip("cv2")
    w, h = 320, 200
    pairs = _pairs(tw, w, h, 40) + _pairs(tw, w, h, 50)
    first, second = _masks(w, h)
    masks = [np.where(m != 0, 255, 0).astype(np.uint8) if m is not None else None for m in first + second]  # as PNG files keep them
    files = [(_write(cv2, tmp_path / f"e{i}.png", a), _write(cv2, tmp_path / f"t{i}.png", b)) for i, (a, b) in enumerate(pairs[:3])]
    mfiles = [_write(cv2, tmp_path / f"m{i}.png", m) if m is not None else None for i, m in enumerate(masks)]
    wrong = _write(cv2, tmp_path / "wrong.png", np.zeros((h, w + 1), np.uint8))
    junk = tmp_path / "junk.png"
    junk.write_bytes(b"\x89PNG not really")
    _, big = tw.synth.make_pair("S", w - 4, h + 2, 40, defect=True)
    lists = [None, [(40, 30, 80, 60)], [], [(0, 0, w // 2, h)]]
    jobs = []  # (kind, pair index, regions, mask index)
    for i in range(len(pairs)):
        jobs.append(("img", i, lists[i % 4], i % len(masks)))
    for i in range(3):
        jobs.append(("file", i, lists[(i + 1) % 4], (i + 1) % len(masks)))
    jobs.append(("resize", 0, [(20, 20, 50, 50)], 1))
    jobs.append(("wrong", 1, None, None))
    jobs.append(("junk", 2, [(1, 1, 5, 5)], None))
    o = tw.OpticalFlow(0, w, h, 1)

    def single(kind, i, regions, k):
        if kind in ("wrong", "junk"):
            return None
        a = pairs[0][0] if kind == "resize" else pairs[i][0]
        b = big if kind == "resize" else pairs[i][1]
        return o.calculate(a, b, threshold=0.2, ignore=regions, ignore_mask=masks[k] if k is not None else None)

    want = [single(*j) for j in jobs]
    pool = tw.Pool([0], threshold=0.2, batch=4)
    with pytest.raises(ValueError, match="bad ignore mask"):
        pool.request(*pairs[0], ignore_mask=np.zeros((h + 1, w), np.uint8))
    ids = [None] * len(jobs)

    def worker(k0):
        for k in range(k0, len(jobs), 3):
            kind, i, regions, mi = jobs[k]
            if kind == "file":
                ids[k] = pool.request_files(*files[i], ignore=regions, ignore_mask=mfiles[mi])
            elif kind == "wrong":
                ids[k] = pool.request_files(*files[i], ignore=regions, ignore_mask=wrong)
            elif kind == "junk":
                ids[k] = pool.request_files(*files[i], ignore=regions, ignore_mask=str(junk))
            elif kind == "resize":
                ids[k] = pool.request(pairs[0][0], big, ignore=regions, ignore_mask=masks[mi])
            else:
                ids[k] = pool.request(*pairs[i], ignore=regions, ignore_mask=masks[mi])

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(3)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    got = [pool.wait(i) for i in ids]
    rep = pool.report()
    pool.stop(); pool.close(); o.close()
    for g, wnt, job in zip(got, want, jobs):
        if job[0] == "wrong":
            assert (g["status"], g["code"], g["reason"]) == ("ERROR", tw.api.BAD_PARAMETER,
                                                             f"bad ignore mask: {w + 1}x{h} mask for a {w}x{h} expected image")
        elif job[0] == "junk":
            assert (g["status"], g["code"], g["reason"]) == ("ERROR", tw.api.BAD_IMAGE_FORMAT, f"Can't open {junk}")
        else:
            assert answer(g) == answer(wnt) and (g["width"], g["height"]) == (wnt["width"], wnt["height"]), job
    assert rep == {"request": len(jobs), "data": len(jobs) - 2, "error": 2}
    assert sum(g["n_vectors"] for g in got if g["status"] != "ERROR") > 0


def test_validation(tw):
    w, h = 160, 120
    a, b = tw.synth.make_pair("S", w, h, 3, defect=True)
    o = tw.OpticalFlow(0, w, h, 2)
    base = o.calculate(a, b, threshold=0.2)
    r = o.calculate(a, b, threshold=0.2, ignore_mask=np.zeros((h, w + 1), bool))
    assert (r["status"], r["code"], r["reason"]) == ("ERROR", tw.api.BAD_PARAMETER, f"bad ignore mask: {w + 1}x{h} mask for a {w}x{h} expected image")
    rb = o.calculate_batch([(a, b), (a, b)], threshold=0.2, ignore_mask=[None, np.zeros((h - 1, w), np.uint8)])
    assert all(x["status"] == "ERROR" and x["reason"].startswith("bad ignore mask") for x in rb)
    for bad in (np.zeros((h, w), np.float32), np.zeros((h, w, 1), np.uint8), [[0] * w] * h):
        with pytest.raises(ValueError, match="bad ignore mask"):
            o.calculate(a, b, ignore_mask=bad)
    assert answer(o.calculate(a, b, threshold=0.2)) == answer(base) and base["n_vectors"] > 0  # the context still works
    o.close()


def test_user_story(tw):
    """A page with 100 small changed spots in a non-rectangular layout (more than TW_MAX_IGNORE regions could name) is SUSPICIOUS;
    with a mask of the spots it is OK; a real change outside the mask makes it SUSPICIOUS again."""
    w, h, seed = 640, 400, 21
    P = tw.synth._PAD
    base, moved = tw.synth.canvas_screenshot(w, h, seed, defect=True)
    a, real = tw.synth._to_u8(base[P:P + h, P:P + w]), tw.synth._to_u8(moved[P:P + h, P:P + w])
    ys, xs = np.nonzero(a != real)  # the real change: one rectangle moved by 8 px
    rng = np.random.default_rng(5)
    b, mask = a.copy(), np.zeros((h, w), np.uint8)
    yy, xx = np.mgrid[-4:5, -4:5]
    disc = xx * xx + yy * yy <= 16
    for t in range(100):  # wavy rows of round spots, e.g. avatars or relative timestamps
        x = int(20 + (t % 20) * 30 + 10 * np.sin(t)); y = int(30 + (t // 20) * 70 + 25 * np.sin(0.7 * t + 1))
        if xs.min() - 40 < x < xs.max() + 40 and ys.min() - 40 < y < ys.max() + 40:
            x = (x + 300) % (w - 20)
        b[y - 4:y + 5, x - 4:x + 5][disc] = rng.integers(0, 120)
        mask[y - 4:y + 5, x - 4:x + 5] |= disc.astype(np.uint8)
    assert not (mask.astype(bool) & (a != real)).any() and ((a != b) <= mask.astype(bool)).all()
    o = tw.OpticalFlow(0, w, h, 1)
    plain = o.calculate(a, b)
    assert plain["status"] == "SUSPICIOUS" and plain["n_vectors"] > 0
    masked = o.calculate(a, b, ignore_mask=mask)
    assert masked["status"] == "OK" and masked["n_vectors"] == 0 and masked["vector"] == []
    b_real = np.where(mask != 0, b, real).astype(np.uint8)
    again = o.calculate(a, b_real, ignore_mask=mask)
    assert again["status"] == "SUSPICIOUS" and all(not mask[v["y"], v["x"]] for v in again["vector"])
    o.close()


def _tree(tw, cv2, root, names, w, h):
    exp_dir, tgt_dir = root / "expected", root / "target"
    for d in (exp_dir, tgt_dir):
        os.makedirs(d / "sub")
    for i, n in enumerate(names):
        a, b = tw.synth.make_pair("S", w, h, 10 + i, defect=True)
        _write(cv2, exp_dir / n, a)
        _write(cv2, tgt_dir / n, b)
    return exp_dir, tgt_dir


@pytest.mark.parametrize("how", ["ignoreMaskDir", "getIgnoreMaskPath"])
def test_create_options(tw, tmp_path, how):
    cv2 = pytest.importorskip("cv2")
    w, h = 320, 200
    names = ["a.png", "b.png", "sub/c.png", "sub/d.png"]
    exp_dir, tgt_dir = _tree(tw, cv2, tmp_path, names, w, h)
    mask_dir = tmp_path / "masks"
    os.makedirs(mask_dir / "sub")
    first, _ = _masks(w, h)
    _write(cv2, mask_dir / "a.png", first[1])                                # a.png: a disc; b.png: no mask file
    _write(cv2, mask_dir / "sub" / "c.png", np.where(first[2], 255, 0).astype(np.uint8))
    (mask_dir / "sub" / "d.png").write_bytes(b"not an image")                 # sub/d.png: undecodable
    common = [{"x": 0, "y": 0, "width": 40, "height": 30}]
    opts = {"expectDir": str(exp_dir), "threshold": 0.5, "ignoreRegions": common}
    if how == "ignoreMaskDir":
        opts["ignoreMaskDir"] = str(mask_dir)
    else:
        opts["ignoreMaskDir"] = None  # wrong-typed: no mask directory, so the callable decides
        opts["getIgnoreMaskPath"] = lambda short: str(mask_dir / short) if short != "b.png" else ""
    data, errors, fin = [], [], []
    t = tw.create(str(tgt_dir), opts)
    t.on("data", data.append).on("error", errors.append).on("finish", fin.append)
    tw.run(t)
    assert fin == [{"request": 4, "data": 3, "error": 1}]
    assert len(errors) == 1 and errors[0]["reason"] == f"Can't open {mask_dir / 'sub' / 'd.png'}"
    pool = tw.Pool([0], threshold=0.5)
    by_target = {d["target_image"]: d for d in data}
    for n in names[:3]:
        m = str(mask_dir / n) if n != "b.png" else None
        want = pool.wait(pool.request_files(str(exp_dir / n), str(tgt_dir / n), ignore=common, ignore_mask=m))
        d = by_target[str(tgt_dir / n)]
        assert (d["status"], vecs(d)) == (want["status"], vecs(want)), n
    unmasked = pool.wait(pool.request_files(str(exp_dir / "a.png"), str(tgt_dir / "a.png"), ignore=common))
    pool.stop(); pool.close()
    assert vecs(by_target[str(tgt_dir / "a.png")]) != vecs(unmasked)  # the mask did act
    assert sum(len(d["vector"]) for d in data) > 0
