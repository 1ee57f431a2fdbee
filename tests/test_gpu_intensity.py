"""GPU tests of intensity cells (tw_set_option "intensity_threshold", tw_intensity_cells, tw_pool_set_intensity /
tw_pool_wait_intensity and create()'s intensityThreshold).  The contract (include/tidalwave_b200.h): a pair's cells are a function
of (E, T, the flow at the sample points, the ignored set) alone.  `intensity_cells` (test_intensity_cpu) restates it on the host;
here it is fed the oracle's flow (faithful arithmetic, which is bit-identical to the oracle) or the device's own dense flow
(relaxed arithmetic), and every answer must equal it bit for bit."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

from conftest import OPTS
from oracle.oracle import FlowParam
from test_gpu_ignore import _ptrs, answer
from test_intensity_cpu import intensity_cells

pytestmark = pytest.mark.gpu

MAX = 4096


def cells(resp):
    return resp["n_intensity_cells"], resp["intensity_cells"]


def want(E, T, fx, fy, span, t, ignored=None):
    c = intensity_cells(E, T, fx, fy, span, t, ignored)
    return len(c), c[:MAX]


def _of(tw, w, h, n, t=16, **opts):
    o = tw.OpticalFlow(0, w, h, n)
    for k, v in dict(intensity_threshold=t, **opts).items():
        o.set_option(k, v)
    return o


def in_place(a, seed):
    """a with a moved-free change: one block darkened by 40 levels and one erased to white."""
    rng = np.random.default_rng(seed)
    b = a.copy()
    h, w = a.shape
    x, y = int(rng.integers(0, w // 2)), int(rng.integers(0, h // 2))
    b[y:y + h // 4, x:x + w // 4] = np.clip(b[y:y + h // 4, x:x + w // 4].astype(int) - 40, 0, 255)
    b[h - h // 5:h - h // 10, w - w // 4:w - w // 8] = 255
    return b


def _pairs(tw, w, h, seed):
    """A page with a moved block and an in-place change, a shifted page with an in-place change, an unchanged flat page."""
    a, b = tw.synth.make_pair("S", w, h, seed, defect=True)
    c, d = tw.synth.make_pair("T", w, h, seed + 1, defect=False)
    e = np.full((h, w), 200, np.uint8)
    return [(a, in_place(b, seed)), (c, in_place(d, seed + 2)), (e, e.copy())]


@pytest.mark.parametrize("opt,size", [("default", (1920, 1080)), ("default", (333, 217)), ("default", (4111, 120)),
                                      ("box31", (333, 217)), ("box31", (1001, 77))])
def test_faithful_matches_restatement_on_the_oracle_flow(tw, oracle, opt, size):
    """Faithful arithmetic: dense and sparse last iteration, tile and strip window kernels (Gaussian window), the box window;
    spans 1, 3, 10 and 16; each eager, captured and replayed."""
    w, h = size
    kw = OPTS[opt]
    p = tw.OpticalFlowParameter(**kw)
    pairs = _pairs(tw, w, h, 11)[:2]
    flows = [oracle.farneback(a, b, FlowParam(**kw)) for a, b in pairs]
    gauss = p.flags == 256
    forms = [(s, t) for s in (0, 1) for t in (1, 0)] if gauss else [(0, 1)]
    exps = {span: [want(a, b, f[..., 0], f[..., 1], span, 8) for (a, b), f in zip(pairs, flows)] for span in (1, 3, 10, 16)}
    hit = 0
    for sparse, tiles in forms:
        o = _of(tw, w, h, 2, t=8, arithmetic=0, sparse_last=sparse, window_tiles=tiles)
        for span, exp in exps.items():
            for rep in range(3):
                got = o.calculate_batch(pairs, p, 5.0, span)
                assert [cells(r) for r in got] == exp, (sparse, tiles, span, rep)
                assert all(r["status"] == ("SUSPICIOUS" if r["n_vectors"] or r["n_intensity_cells"] else "OK") for r in got)
            hit += sum(n for n, _ in exp)
        o.close()
    assert hit > 0


@pytest.mark.parametrize("span", [1, 3, 10, 16])
def test_relaxed_matches_restatement_on_the_device_flow(tw, span):
    w, h = 1920, 1080
    pairs = _pairs(tw, w, h, 21)
    o = _of(tw, w, h, 3)
    assert o.arithmetic_in_effect() == "relaxed"
    first = None
    for rep in range(3):
        got = o.calculate_batch(pairs, threshold=5.0, span=span)
        if first is None:
            for i, ((a, b), r) in enumerate(zip(pairs, got)):
                fx, fy = o.batch_flow(i, w, h)
                assert cells(r) == want(a, b, fx, fy, span, 16), i
            first = [cells(r) for r in got]
        assert [cells(r) for r in got] == first, rep
        assert got[0]["n_intensity_cells"] > 0 and got[1]["n_intensity_cells"] > 0 and cells(got[2]) == (0, [])
    o.close()


def _table(tw):
    """Five changes in place, none of which moves anything, on a seeded 1920x1080 synthetic page.  The first three are placed where
    the flow finds no vector at the default options (checked against the oracle), so they show what the flow alone misses."""
    a, _ = tw.synth.canvas_screenshot(1920, 1080, 3)
    E = np.clip(a[32:32 + 1080, 32:32 + 1920], 0, 255).astype(np.uint8)
    E[150:250, 1200:1400] = 200                          # a button
    out = {}
    T = E.copy(); T[200:400, 300:600] = np.clip(T[200:400, 300:600].astype(int) - 40, 0, 255); out["darkened block"] = T
    T = E.copy(); T[150:250, 1200:1400] = 128; out["button fill"] = T
    T = E.copy(); T[900:920, 800:860] = 255; out["erased content"] = T  # page content (mean 192) erased to white
    out["background"] = np.where(E == 255, 225, E).astype(np.uint8)
    out["darker page"] = np.clip(E.astype(int) - 30, 0, 255).astype(np.uint8)
    return E, out


def test_in_place_changes_are_suspicious(tw):
    E, cases = _table(tw)
    w, h = 1920, 1080
    off = tw.OpticalFlow(0, w, h, 1)
    on = _of(tw, w, h, 1, t=16)
    for name, T in cases.items():
        r0 = off.calculate(E, T)
        r1 = on.calculate(E, T)
        if name in ("darkened block", "button fill", "erased content"):
            assert r0["status"] == "OK" and r0["n_vectors"] == 0, name
        fx, fy = on.batch_flow(0, w, h)
        assert r1["status"] == "SUSPICIOUS" and r1["n_intensity_cells"] > 0, name
        assert cells(r1) == want(E, T, fx, fy, 10, 16), name
        assert answer(r1)[1:] == answer(r0)[1:], name  # the vectors do not change
    off.close(); on.close()


def test_ignored_changes_give_no_cells(tw):
    w, h = 640, 360
    a, _ = tw.synth.make_pair("S", w, h, 5)
    b = a.copy()
    b[100:180, 200:330] = np.clip(b[100:180, 200:330].astype(int) - 60, 0, 255)
    o = _of(tw, w, h, 1)
    plain = o.calculate(a, b)
    assert plain["n_intensity_cells"] > 0
    region = o.calculate(a, b, ignore=[(195, 95, 140, 90)])
    mask = np.zeros((h, w), np.uint8)
    mask[95:185, 195:335] = 1
    masked = o.calculate(a, b, ignore_mask=mask)
    assert cells(region) == cells(masked) == (0, []) and region["status"] == masked["status"] == "OK"
    # a mask over half the change: the restatement on the painted target with the ignored set
    half = np.zeros((h, w), np.uint8)
    half[:, :260] = 1
    got = o.calculate(a, b, ignore_mask=half)
    fx, fy = o.batch_flow(0, w, h)
    T = np.where(half != 0, a, b)
    assert cells(got) == want(a, T, fx, fy, 10, 16, half != 0) and got["n_intensity_cells"] > 0
    assert all(c["x"] + 10 > 260 for c in got["intensity_cells"])
    o.close()


def test_eager_and_replay_agree_with_new_images(tw):
    w, h = 512, 320
    o = _of(tw, w, h, 3)
    for seed in (30, 40, 50):
        pairs = _pairs(tw, w, h, seed)
        fresh = _of(tw, w, h, 3)
        ref = fresh.calculate_batch(pairs)  # an eager run on a new context
        fresh.close()
        got = o.calculate_batch(pairs)      # seed 30: eager; then captured and replayed with new images
        assert [cells(r) for r in got] == [cells(r) for r in ref] and [answer(r) for r in got] == [answer(r) for r in ref], seed
        for i, ((a, b), r) in enumerate(zip(pairs, got)):
            fx, fy = o.batch_flow(i, w, h)
            assert cells(r) == want(a, b, fx, fy, 10, 16)
    o.close()


def test_whole_page_change_reports_the_full_count(tw):
    w, h = 1920, 1080
    a, _ = tw.synth.make_pair("S", w, h, 9)
    b = np.clip(a.astype(int) + 60, 0, 255).astype(np.uint8)
    b = np.where(a > 195, a - 60, b).astype(np.uint8)
    o = _of(tw, w, h, 1)
    for rep in range(3):
        r = o.calculate(a, b)
        fx, fy = o.batch_flow(0, w, h)
        n, first = want(a, b, fx, fy, 10, 16)
        assert n > MAX and r["n_intensity_cells"] == n and r["intensity_cells"] == first and len(first) == MAX
        assert [(c["y"], c["x"]) for c in first] == sorted((c["y"], c["x"]) for c in first)
    o.close()


def test_launch_count_options_and_refusals(tw):
    """Off: every result and the launch count equal a context that never set the option; on: three more launches per run."""
    w, h = 333, 217
    pairs = _pairs(tw, w, h, 12)
    plain = tw.OpticalFlow(0, w, h, 3)
    o = tw.OpticalFlow(0, w, h, 3)

    def run(of):
        l0 = of.launch_count()
        out = of.calculate_batch(pairs)
        return out, of.launch_count() - l0

    def strip(rs):
        return [{k: v for k, v in r.items() if k not in ("time", "intensity_cells", "n_intensity_cells")} for r in rs]

    for t in (0, 16, 0, 40, 0):
        o.set_option("intensity_threshold", t)
        for rep in range(3):
            ref, lp = run(plain)
            got, lo = run(o)
            assert lo - lp == (3 if t else 0), (t, rep)
            assert all(("intensity_cells" in r) == bool(t) for r in got)
            if t:
                assert got[1]["status"] == "SUSPICIOUS" and got[1]["n_intensity_cells"] > 0  # an in-place change on a texture
                assert [r["n_vectors"] for r in got] == [r["n_vectors"] for r in ref]
            else:
                assert strip(got) == strip(ref)
    for bad in (-1, 256, 1000):
        with pytest.raises(ValueError, match="intensity_threshold"):
            o.set_option("intensity_threshold", bad)
    lib = tw.load()
    buf = (tw.tw_intensity_cell * 4)()
    n = C.c_int()
    assert lib.tw_intensity_cells(o.ctx, 0, buf, 4, C.byref(n)) == tw.api.BAD_PARAMETER  # the last batch ran without the option
    o.set_option("intensity_threshold", 16)
    got = o.calculate_batch(pairs)
    assert lib.tw_intensity_cells(o.ctx, 3, buf, 4, C.byref(n)) == tw.api.BAD_PARAMETER  # out of range
    k = got[1]["n_intensity_cells"]
    assert k > 2 and lib.tw_intensity_cells(o.ctx, 1, buf, 2, C.byref(n)) == 0 and n.value == k  # 2 stored, the full count
    assert [(c.x, c.y, c.n_pixels, c.residual) for c in buf[:2]] == \
           [(c["x"], c["y"], c["n_pixels"], c["residual"]) for c in got[1]["intensity_cells"][:2]]
    p = tw.OpticalFlowParameter().c()
    ex, tg = _ptrs([a for a, _ in pairs]), _ptrs([b for _, b in pairs])
    assert lib.tw_pipe_submit(o.ctx, 3, ex, tg, w, h, w, C.byref(p), 5.0, 10) == 0
    with pytest.raises(ValueError, match="intensity_threshold"):
        o.set_option("intensity_threshold", 0)
    cap = ((w + 9) // 10) * ((h + 9) // 10)
    assert lib.tw_pipe_collect(o.ctx, (tw.tw_vector * (3 * cap))(), cap, (tw.tw_result * 3)()) == 0
    o.set_option("intensity_threshold", 0)
    plain.close(); o.close()


def test_pipe_two_batches_in_flight(tw):
    w, h = 333, 217
    batches = [_pairs(tw, w, h, s) for s in (50, 60, 70, 80)]
    o = _of(tw, w, h, 3)
    exp = [[(r["status"], cells(r)) for r in o.calculate_batch(pairs)] for pairs in batches]
    lib = tw.load()
    p = tw.OpticalFlowParameter().c()
    cap = ((w + 9) // 10) * ((h + 9) // 10)
    keep, got = [], []

    def collect():
        vec, res = (tw.tw_vector * (3 * cap))(), (tw.tw_result * 3)()
        assert lib.tw_pipe_collect(o.ctx, vec, cap, res) == 0
        got.append([(tw.api.STATUS_NAMES[res[i].status], o.intensity_cells(i)) for i in range(3)])

    for pairs in batches:
        if lib.tw_pipe_pending(o.ctx) >= 2:
            collect()
        ex, tg = _ptrs([a for a, _ in pairs]), _ptrs([b for _, b in pairs])
        keep.append((ex, tg))
        assert lib.tw_pipe_submit(o.ctx, 3, ex, tg, w, h, w, C.byref(p), 5.0, 10) == 0
    while lib.tw_pipe_pending(o.ctx):
        collect()
    got = [[(s, (c[1], c[0])) for s, c in b] for b in got]
    assert got == exp and exp[0] != exp[1]
    o.close()


def _pgm(path, img):
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (img.shape[1], img.shape[0]) + np.ascontiguousarray(img).tobytes())
    return str(path)


def test_pool_and_create(tw, tmp_path):
    w, h = 320, 200
    pairs = _pairs(tw, w, h, 20) + _pairs(tw, w, h, 30)
    files = [(_pgm(tmp_path / f"e{i}.pgm", a), _pgm(tmp_path / f"t{i}.pgm", b)) for i, (a, b) in enumerate(pairs)]
    o = _of(tw, w, h, 1)
    exp = [o.calculate(a, b) for a, b in pairs]
    o.close()
    assert sum(r["n_intensity_cells"] > 0 for r in exp) >= 4
    for regions in (False, True):
        pool = tw.Pool([0], batch=4, intensity_threshold=16, change_regions=regions)
        jobs = [("img", i) for i in range(len(pairs))] + [("file", i) for i in range(len(pairs))] + [("error", 0)]
        ids = [None] * len(jobs)

        def worker(k0):
            for k in range(k0, len(jobs), 3):
                kind, i = jobs[k]
                if kind == "img":
                    ids[k] = pool.request(*pairs[i])
                elif kind == "file":
                    ids[k] = pool.request_files(*files[i])
                else:
                    ids[k] = pool.request(pairs[0][0], np.zeros((h + 9, w), np.uint8))

        threads = [threading.Thread(target=worker, args=(k,)) for k in range(3)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert pool.lib.tw_pool_set_intensity(pool.pool, 0) == tw.api.BAD_PARAMETER  # after the first submit
        got = [pool.wait(i) for i in ids]
        pool.stop(); pool.close()
        for g, (kind, i) in zip(got, jobs):
            if kind == "error":
                assert g["status"] == "ERROR" and "intensity_cells" not in g
                continue
            assert cells(g) == cells(exp[i]) and answer(g) == answer(exp[i]) and ("regions" in g) == regions, (kind, i)
    with pytest.raises(ValueError):
        tw.Pool([0], intensity_threshold=300)
    # create(): the same pairs from directories
    for d in ("expected", "target"):
        os.makedirs(tmp_path / d)
    for i, (a, b) in enumerate(pairs):
        _pgm(tmp_path / "expected" / f"{i}.pgm", a)
        _pgm(tmp_path / "target" / f"{i}.pgm", b)
    events = {}
    for t in (None, 16):
        opts = {"expectDir": str(tmp_path / "expected")}
        if t is not None:
            opts["intensityThreshold"] = t
        data = []
        c = tw.create(str(tmp_path / "target"), opts)
        c.on("data", data.append)
        tw.run(c)
        events[t] = sorted(data, key=lambda d: int(os.path.basename(d["target_image"]).split(".")[0]))
    assert all("intensity_cells" not in d for d in events[None])
    for d0, d1, r in zip(events[None], events[16], exp):
        assert d1["vector"] == d0["vector"] == r["vector"] and cells(d1) == cells(r) and d1["status"] == r["status"]
    assert any(d0["status"] == "OK" and d1["status"] == "SUSPICIOUS" for d0, d1 in zip(events[None], events[16]))
