"""GPU tests of change regions (tw_set_option "change_regions", tw_change_regions, tw_pool_set_change_regions /
tw_pool_wait_regions and create()'s changeRegions).  The contract (include/tidalwave_b200.h): a pair's regions are a function of
its vector list alone -- the 8-connected components of its suspicious span-grid points, in the order of their first points, with
clipped cell boxes, counts and peaks.  `regions_of` (test_change_regions_cpu, scipy.ndimage.label) restates it on the host, and
every answer here is compared with it applied to the same run's full vector list, bit for bit."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

from conftest import OPTS, golden_pair
from test_change_regions_cpu import regions_of
from test_gpu_ignore import _ptrs, answer, vecs

pytestmark = pytest.mark.gpu

MAX = 1024


def check(resp, w, h, span=10):
    """resp's regions against the oracle on resp's own vectors; returns the region count."""
    want = regions_of(vecs(resp), w, h, span)
    assert resp["n_regions"] == len(want)
    assert resp["regions"] == want[:MAX]
    if len(want) <= MAX:
        assert sum(r["n_vectors"] for r in resp["regions"]) == resp["n_vectors"]
    return len(want)


def regions(resp):
    return resp["n_regions"], resp["regions"]


def spots(a, seed, n=5, r=12):
    """a with n square patches, well apart, replaced by other content: n separate changed areas."""
    rng = np.random.default_rng(seed)
    b = a.copy()
    h, w = a.shape
    for k in range(n):
        x = int((k + 0.5) * w / n) - r
        y = int(rng.integers(r, h - 3 * r))
        b[y:y + 2 * r, x:x + 2 * r] = np.flipud(a[y + r:y + 3 * r, x:x + 2 * r])
    return b


def _pairs(tw, w, h, seed):
    """A page with several changed spots, a shifted page (one big change) and an unchanged flat page (OK: no gradient, no flow;
    an unchanged textured page can still show a vector near its border at a low threshold, in the oracle too)."""
    a, _ = tw.synth.make_pair("S", w, h, seed, defect=False)
    c, d = tw.synth.make_pair("T", w, h, seed + 1, defect=False)
    e = np.full((h, w), 200, np.uint8)
    return [(a, spots(a, seed)), (c, d), (e, e.copy())]


def _of(tw, w, h, n, **opts):
    o = tw.OpticalFlow(0, w, h, n)
    for k, v in dict(change_regions=1, **opts).items():
        o.set_option(k, v)
    return o


@pytest.mark.parametrize("arith", [0, 1])
@pytest.mark.parametrize("sparse", [0, 1])
@pytest.mark.parametrize("opt,size", [("default", (333, 217)), ("cfg4", (300, 200)), ("g15n5", (300, 200)), ("cfg3", (512, 320)),
                                      ("strip", (512, 320))])
def test_regions_match_oracle(tw, arith, sparse, opt, size):
    """Eager, captured and replayed runs, two pair sets on one graph key; OK and SUSPICIOUS pairs in one batch."""
    w, h = size
    p = tw.OpticalFlowParameter(**OPTS["default" if opt == "strip" else opt])
    o = _of(tw, w, h, 3, arithmetic=arith, sparse_last=sparse, window_tiles=0 if opt == "strip" else 1)
    many = 0
    for seed in (70, 90):
        pairs = _pairs(tw, w, h, seed)
        first = None
        for rep in range(3):
            got = o.calculate_batch(pairs, p, 0.2)
            counts = [check(r, w, h) for r in got]
            assert got[2]["status"] == "OK" and regions(got[2]) == (0, [])
            if first is None:
                first = [regions(r) for r in got]
            assert [regions(r) for r in got] == first, rep
            many += sum(c > 1 for c in counts)
    assert many > 0
    o.close()


def test_paths_give_identical_regions(tw):
    """Dense and sparse last iteration, tile and strip window kernels: the same vectors, so the same regions."""
    w, h = 512, 320
    pairs = _pairs(tw, w, h, 31)
    seen = []
    for sparse in (0, 1):
        for tiles in (1, 0):
            o = _of(tw, w, h, 3, sparse_last=sparse, window_tiles=tiles)
            got = o.calculate_batch(pairs, threshold=0.2)
            for r in got:
                check(r, w, h)
            seen.append([(answer(r), regions(r)) for r in got])
            o.close()
    assert all(s == seen[0] for s in seen) and seen[0][0][1][0] > 0


def test_ignored_points_and_a_mask_stripe(tw):
    """Ignored points are in no region; a mask stripe through one changed area (threshold 0: every moved point) splits it."""
    w, h, c = 320, 200, 16
    a, b = tw.synth.make_pair("S", w, h, 5, defect=True)
    o = _of(tw, w, h, 1)
    plain = o.calculate(a, b, threshold=0.0)
    check(plain, w, h)
    assert any(r["x"] < c * 10 and r["x"] + r["width"] > (c + 1) * 10 for r in plain["regions"])  # one area across column c
    mask = np.zeros((h, w), np.uint8)
    mask[:, c * 10 - 1:c * 10 + 2] = 1  # covers the sample points of grid column c
    lists = [(0, 0, 60, 40)]
    got = o.calculate(a, b, threshold=0.0, ignore=lists, ignore_mask=mask)
    check(got, w, h)
    assert not any(mask[v[1], v[0]] or (v[0] < 60 and v[1] < 40) for v in vecs(got))
    assert all(r["x"] + r["width"] <= c * 10 or r["x"] >= (c + 1) * 10 for r in got["regions"])  # nothing crosses the stripe
    assert any(r["x"] < c * 10 for r in got["regions"]) and any(r["x"] > c * 10 for r in got["regions"])
    o.close()


def test_more_regions_than_stored(tw):
    """1920x1080, span 10, threshold 0, a changed target and a mask on the single pixels of the grid points with an odd i or an odd
    j: up to 96 x 54 isolated points, each its own region."""
    w, h = 1920, 1080
    a, b = tw.synth.make_pair("S", w, h, 7, defect=True)
    mask = np.zeros((h, w), np.uint8)
    ys, xs = np.mgrid[0:h:10, 0:w:10]
    odd = ((xs // 10) % 2 == 1) | ((ys // 10) % 2 == 1)
    mask[ys[odd], xs[odd]] = 1
    o = _of(tw, w, h, 1)
    for rep in range(3):
        got = o.calculate(a, b, threshold=0.0, ignore_mask=mask)
        n = check(got, w, h)
        assert n == got["n_vectors"] > MAX and len(got["regions"]) == MAX
        assert all(r["n_vectors"] == 1 and (r["width"], r["height"]) == (10, 10) for r in got["regions"])
    o.close()


@pytest.mark.parametrize("w,h,span", [(1280, 8000, 10), (200, 150, 1), (1001, 77, 7), (333, 217, 10)])
def test_geometries(tw, w, h, span):
    pairs = [tw.synth.make_pair("S", w, h, 40 + i, defect=True) for i in range(2)]
    o = _of(tw, w, h, 2)
    n = 0
    for rep in range(3):
        for r in o.calculate_batch(pairs, threshold=0.2, span=span):
            n += check(r, w, h, span)
    assert n > 0
    o.close()


def test_size_tolerance_path(tw):
    """The target is resized to the expected size first; regions are in expected-image pixels."""
    w, h = 320, 200
    a, _ = tw.synth.make_pair("S", w, h, 5, defect=True)
    _, big = tw.synth.make_pair("S", w + 3, h - 2, 5, defect=True)
    o = _of(tw, w + 8, h + 8, 1)
    for rep in range(2):
        got = o.calculate(a, big, threshold=0.3)
        assert (got["width"], got["height"]) == (w, h) and check(got, w, h) > 0
    bad = o.calculate(a, np.zeros((h, w + 6), np.uint8), threshold=0.3)  # more than 5 px apart
    assert bad["status"] == "ERROR" and "regions" not in bad
    o.close()


def test_launch_count_key_and_pipe_refusal(tw):
    """Off: the launch count per run is a plain context's; on: one more.  Toggling keeps each key's graph right."""
    w, h = 333, 217
    pairs = _pairs(tw, w, h, 12)
    plain = tw.OpticalFlow(0, w, h, 3)
    o = tw.OpticalFlow(0, w, h, 3)

    def run(of):
        l0 = of.launch_count()
        out = of.calculate_batch(pairs, threshold=0.2)
        return out, of.launch_count() - l0

    def strip(rs):
        return [{k: v for k, v in r.items() if k not in ("time", "regions", "n_regions")} for r in rs]

    want = None
    for on in (0, 1, 0, 1, 0):
        o.set_option("change_regions", on)
        for rep in range(3):
            ref, lp = run(plain)
            got, lo = run(o)
            assert strip(got) == strip(ref) and lo - lp == on, (on, rep)
            assert all(("regions" in r) == bool(on) for r in got) and all("regions" not in r for r in ref)
            if on:
                for r in got:
                    check(r, w, h)
                want = want or [regions(r) for r in got]
                assert [regions(r) for r in got] == want
    lib = tw.load()
    reg = (tw.tw_change_region * 4)()
    n = C.c_int()
    assert lib.tw_change_regions(o.ctx, 0, reg, 4, C.byref(n)) == tw.api.BAD_PARAMETER  # the last batch ran without the option
    o.set_option("change_regions", 1)
    got = o.calculate_batch(pairs, threshold=0.2)
    assert lib.tw_change_regions(o.ctx, 3, reg, 4, C.byref(n)) == tw.api.BAD_PARAMETER  # out of range
    k = got[0]["n_regions"]
    assert k > 2 and lib.tw_change_regions(o.ctx, 0, reg, 2, C.byref(n)) == 0 and n.value == k  # 2 stored, the full count
    assert [(r.rect.x, r.rect.y, r.rect.width, r.rect.height, r.n_vectors) for r in reg[:2]] == \
           [(r["x"], r["y"], r["width"], r["height"], r["n_vectors"]) for r in got[0]["regions"][:2]]
    # toggling while a pipe batch is in flight is refused
    p = tw.OpticalFlowParameter().c()
    ex, tg = _ptrs([a for a, _ in pairs]), _ptrs([b for _, b in pairs])
    assert lib.tw_pipe_submit(o.ctx, 3, ex, tg, w, h, w, C.byref(p), 0.2, 10) == 0
    with pytest.raises(ValueError, match="change_regions"):
        o.set_option("change_regions", 0)
    cap = ((w + 9) // 10) * ((h + 9) // 10)
    assert lib.tw_pipe_collect(o.ctx, (tw.tw_vector * (3 * cap))(), cap, (tw.tw_result * 3)()) == 0
    o.set_option("change_regions", 0)
    plain.close(); o.close()


def test_pipe_two_batches_in_flight(tw):
    w, h = 333, 217
    batches = [_pairs(tw, w, h, s) for s in (50, 60, 70, 80)]
    o = _of(tw, w, h, 3)
    want = [[regions(r) for r in o.calculate_batch(pairs, threshold=0.2)] for pairs in batches]
    lib = tw.load()
    p = tw.OpticalFlowParameter().c()
    cap = ((w + 9) // 10) * ((h + 9) // 10)
    keep, got = [], []

    def collect():
        vec, res = (tw.tw_vector * (3 * cap))(), (tw.tw_result * 3)()
        assert lib.tw_pipe_collect(o.ctx, vec, cap, res) == 0
        out = []
        for i in range(3):
            r = tw.api._response(res[i], (tw.tw_vector * cap).from_buffer(vec, i * cap * C.sizeof(tw.tw_vector)),
                                 min(res[i].n_vectors, cap), 10, 0.2)
            r["regions"], r["n_regions"] = o.regions(i)
            check(r, w, h)
            out.append(regions(r))
        got.append(out)

    for pairs in batches:
        if lib.tw_pipe_pending(o.ctx) >= 2:
            collect()
        ex, tg = _ptrs([a for a, _ in pairs]), _ptrs([b for _, b in pairs])
        keep.append((ex, tg))
        assert lib.tw_pipe_submit(o.ctx, 3, ex, tg, w, h, w, C.byref(p), 0.2, 10) == 0
    while lib.tw_pipe_pending(o.ctx):
        collect()
    assert got == want and want[0] != want[1]
    o.close()


def _pgm(path, img):
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (img.shape[1], img.shape[0]) + np.ascontiguousarray(img).tobytes())
    return str(path)


def test_pool(tw, tmp_path):
    """A multi-threaded pool with image, path, resize and error requests; vector_cap = 1 still returns every region."""
    w, h = 320, 200
    pairs = _pairs(tw, w, h, 20) + _pairs(tw, w, h, 30)
    files = [(_pgm(tmp_path / f"e{i}.pgm", a), _pgm(tmp_path / f"t{i}.pgm", b)) for i, (a, b) in enumerate(pairs)]
    _, big = tw.synth.make_pair("S", w - 4, h + 2, 20, defect=True)
    o = _of(tw, w, h, 1)
    want = [o.calculate(a, b, threshold=0.2) for a, b in pairs] + [o.calculate(pairs[0][0], big, threshold=0.2)]
    assert all(check(r, w, h) >= 0 for r in want) and sum(r["n_regions"] > 1 for r in want) > 0
    o.close()
    for cap in (0, 1):
        pool = tw.Pool([0], threshold=0.2, batch=4, vector_cap=cap, change_regions=True)
        jobs = [("img", i) for i in range(len(pairs))] + [("file", i) for i in range(len(pairs))] + [("resize", 0), ("error", 0)]
        ids = [None] * len(jobs)

        def worker(k0):
            for k in range(k0, len(jobs), 3):
                kind, i = jobs[k]
                if kind == "img":
                    ids[k] = pool.request(*pairs[i])
                elif kind == "file":
                    ids[k] = pool.request_files(*files[i])
                elif kind == "resize":
                    ids[k] = pool.request(pairs[0][0], big)
                else:
                    ids[k] = pool.request(pairs[0][0], np.zeros((h + 9, w), np.uint8))

        threads = [threading.Thread(target=worker, args=(k,)) for k in range(3)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert pool.lib.tw_pool_set_change_regions(pool.pool, 0) == tw.api.BAD_PARAMETER  # after the first submit
        got = [pool.wait(i) for i in ids]
        pool.stop(); pool.close()
        for g, (kind, i) in zip(got, jobs):
            if kind == "error":
                assert g["status"] == "ERROR" and "regions" not in g
                continue
            wnt = want[-1] if kind == "resize" else want[i]
            assert regions(g) == regions(wnt) and g["n_vectors"] == wnt["n_vectors"], (cap, kind, i)
            if cap == 0:
                assert answer(g) == answer(wnt)
            else:
                assert len(g["vector"]) == min(1, g["n_vectors"])
    plain = tw.Pool([0], threshold=0.2)
    r = plain.wait(plain.request(*pairs[0]))
    plain.stop(); plain.close()
    assert "regions" not in r and "n_regions" not in r


def test_user_story_s2r2(tw, golden):
    """The reference's scenario2 fixture at its options: 24 vectors in 5 regions, the last one clipped at the bottom edge."""
    a, b = golden_pair(golden, tw, "s2r2")
    h, w = a.shape
    table = [(80, 70, 10, 10, 1), (130, 70, 20, 20, 4), (160, 70, 20, 47, 9), (110, 80, 10, 10, 1), (80, 100, 50, 17, 9)]
    for arith in (0, 1):
        o = _of(tw, w, h, 1, arithmetic=arith)
        for rep in range(3):
            r = o.calculate(a, b, threshold=5, span=10)
            assert r["n_vectors"] == 24 and r["n_regions"] == 5
            assert [(g["x"], g["y"], g["width"], g["height"], g["n_vectors"]) for g in r["regions"]] == table
            check(r, w, h)
        o.close()


def test_create(tw, tmp_path):
    names = ["a.pgm", "b.pgm", "sub/c.pgm"]
    for d in ("expected/sub", "target/sub"):
        os.makedirs(tmp_path / d)
    w, h = 320, 200
    for i, n in enumerate(names):
        a, b = tw.synth.make_pair("S", w, h, 10 + i, defect=True) if i != 1 else (np.full((h, w), 90, np.uint8),) * 2  # b: unchanged
        _pgm(tmp_path / "expected" / n, a)
        _pgm(tmp_path / "target" / n, b)
    events = {}
    for on in (None, True):
        opts = {"expectDir": str(tmp_path / "expected"), "threshold": 0.5}
        if on is not None:
            opts["changeRegions"] = on
        data = []
        t = tw.create(str(tmp_path / "target"), opts)
        t.on("data", data.append)
        tw.run(t)
        events[on] = sorted(data, key=lambda d: d["target_image"])
    keys = {"status", "span", "threshold", "expect_image", "target_image", "time", "height", "width", "vector"}
    assert all(set(d) == keys for d in events[None])
    assert all(set(d) == keys | {"regions", "n_regions"} for d in events[True])
    for d0, d1 in zip(events[None], events[True]):
        assert vecs(d0) == vecs(d1)
        d1 = dict(d1, n_vectors=len(d1["vector"]))
        check(d1, w, h)
    assert [d["n_regions"] > 0 for d in events[True]] == [True, False, True]
