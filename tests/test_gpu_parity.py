"""GPU parity tests (run on a B200 with -m gpu).  Everything goes through the C ABI (libtidalwave_b200.so).

Bar (BASELINE.json north_star): per-pixel flow within 1e-2 px max-abs and 1e-3 px RMS of the reference's CPU Farneback
path, classification (status + vector positions) identical.  This module pins the faithful arithmetic, which follows SURVEY
App. A's operation order: flows and per-stage tensors are compared with the oracle bit for bit; the cv2 goldens, another
build of the algorithm, within the tolerance."""
import numpy as np
import pytest

from conftest import OPTS, golden_pair
from oracle.oracle import FlowParam, sample_numpy

pytestmark = pytest.mark.gpu

TOL_MAX, TOL_RMS = 1e-2, 1e-3


@pytest.fixture(scope="module", autouse=True)
def _faithful_arithmetic(tw):
    """This module pins the FAITHFUL arithmetic (bit-identical to the oracle); the library default -- relaxed where
    validated -- is covered by tests/test_gpu_relaxed.py."""
    tw.set_default_arithmetic(False)
    yield
    tw.set_default_arithmetic(True)


@pytest.fixture(scope="module")
def of(tw):
    o = tw.OpticalFlow(0, 1920, 1080, 4)
    yield o
    o.close()


def _check_flow(fx, fy, ref, what):
    d = np.maximum(np.abs(fx - ref[..., 0]), np.abs(fy - ref[..., 1]))
    rms = float(np.sqrt(((fx - ref[..., 0]) ** 2 + (fy - ref[..., 1]) ** 2).mean() / 2))
    assert d.max() <= TOL_MAX and rms <= TOL_RMS, f"{what}: max {d.max():.3e} rms {rms:.3e}"
    return float(d.max())


def _vec_pos(resp):
    return [(v["x"], v["y"]) for v in resp["vector"]]


def test_reference_golden_cases(of, golden):
    """/root/reference/test/index.coffee:12-96 replayed through tw_compare."""
    thr, span = golden["options"]["threshold"], golden["options"]["span"]
    for case in golden["cases"]:
        a, b = golden["imgs"][case["expect"]], golden["imgs"][case["target"]]
        resp = of.calculate(a, b, threshold=thr, span=span)
        assert resp["status"] == case["status"]
        assert (resp["height"], resp["width"], resp["span"], resp["threshold"]) == (case["height"], case["width"], span, thr)
        assert _vec_pos(resp) == [(g["x"], g["y"]) for g in case["vector"]]
        for v, g in zip(resp["vector"], case["vector"]):
            assert abs(v["dx"] - g["dx"]) < 1e-3 and abs(v["dy"] - g["dy"]) < 1e-3


@pytest.mark.parametrize("name", ["s1", "s2r2", "S256", "T256", "Sdef"])
@pytest.mark.parametrize("opt", list(OPTS))
def test_flow_vs_oracle_and_cv2(of, tw, oracle, golden, name, opt):
    a, b = golden_pair(golden, tw, name)
    p = tw.OpticalFlowParameter(**OPTS[opt])
    rc, fx, fy, sec = of.calculateInternal(a, b, p)
    assert rc == 0, of.last_error()
    assert sec > 0
    ref = oracle.farneback(a, b, FlowParam(**OPTS[opt]))
    assert np.array_equal(fx, ref[..., 0]) and np.array_equal(fy, ref[..., 1]), f"{name}/{opt}: not bit-identical to the oracle"
    key = f"{name}__{opt}"
    if key in golden["flows"]:
        _check_flow(fx, fy, golden["flows"][key], f"{name}/{opt} vs cv2 golden")
    # classification identity
    resp = of.calculate(a, b, p)
    status, vec = oracle.sample(ref)
    assert resp["status"] == status
    assert _vec_pos(resp) == [(v[0], v[1]) for v in vec]
    flow = np.stack([fx, fy], -1)
    assert [(v["x"], v["y"], v["dx"], v["dy"]) for v in resp["vector"]] == sample_numpy(flow)[1]


@pytest.mark.parametrize("opt", ["default", "cfg4"])
def test_per_stage_parity(tw, oracle, golden, opt):
    """Stage-by-stage against the oracle's dump: level images, polynomial expansion, update-matrices input of the last
    iteration, per-scale flow."""
    a, b = golden_pair(golden, tw, "Sdef")
    of = tw.OpticalFlow(0, 320, 200, 1)
    of.debug_keep_levels(True)
    p = tw.OpticalFlowParameter(**OPTS[opt])
    rc, fx, fy, _ = of.calculateInternal(a, b, p)
    assert rc == 0
    dump = {}
    oracle.farneback(a, b, FlowParam(**OPTS[opt]), dump=dump)
    nscales = 1 + max(k[1] for k in dump)
    iters = p.pyrIterations
    for s in range(nscales):
        for nm in ("I0", "I1"):
            got = of.debug_read(nm, s)[0]
            np.testing.assert_array_equal(got, dump[(nm, s, 0)], err_msg=f"{nm} scale {s}")
        for nm in ("R0", "R1"):
            got = of.debug_read(nm, s).transpose(1, 2, 0)
            np.testing.assert_array_equal(got, dump[(nm, s, 0)], err_msg=f"{nm} scale {s}")
        got = of.debug_read("M", s).transpose(1, 2, 0)
        np.testing.assert_array_equal(got, dump[("M", s, iters - 1)], err_msg=f"M scale {s}")
        got = of.debug_read("flow", s).transpose(1, 2, 0)
        np.testing.assert_array_equal(got, dump[("flow", s, iters - 1)], err_msg=f"flow scale {s}")
    of.close()


@pytest.mark.parametrize("kw", [dict(winSize=20), dict(winSize=9, pyrIterations=2), dict(polyN=3, polySigma=0.9),
                                dict(pyrScale=0.8, pyrLevels=4), dict(pyrScale=0.6, pyrLevels=2, flags=0, winSize=12),
                                dict(pyrIterations=1), dict(pyrLevels=0), dict(pyrIterations=0, pyrLevels=2)])
def test_generic_kernel_paths(of, tw, oracle, kw):
    """Options outside the specialised kernels (window radius not 15/7, polyN not 5/7, pyrScale != 0.5, ...) take the
    generic kernels; they must match the oracle bit for bit too."""
    a, b = tw.synth.make_pair("S", 300, 220, 31, defect=True)
    rc, fx, fy, _ = of.calculateInternal(a, b, tw.OpticalFlowParameter(**kw))
    assert rc == 0, of.last_error()
    ref = oracle.farneback(a, b, FlowParam(**kw))
    assert np.array_equal(fx, ref[..., 0]) and np.array_equal(fy, ref[..., 1]), f"{kw}: not bit-identical to the oracle"
    for thr in (5.0, 0.5):
        resp = of.calculate(a, b, tw.OpticalFlowParameter(**kw), threshold=thr)
        status, vec = oracle.sample(ref, 10, thr)
        assert resp["status"] == status and [(v["x"], v["y"], v["dx"], v["dy"]) for v in resp["vector"]] == vec, thr


def test_kernel_variants_agree(tw, oracle):
    """The generic / unfused level-image kernels, the tight-pitch layout and both window kernels are alternative code paths for
    the same arithmetic: all bit-identical to the oracle.  The experimental options removed in round 2 answer TW_UNSUPPORTED."""
    a, b = tw.synth.make_pair("S", 480, 300, 33, defect=True)
    ref = oracle.farneback(a, b, FlowParam())
    for opt in (None, "level_generic", "level_unfused", "tight_pitch", "window_tiles=0", "window_tiles=1"):
        o = tw.OpticalFlow(0, 480, 300, 1)
        o.set_option("arithmetic", 0)
        if opt:
            name, _, val = opt.partition("=")
            o.set_option(name, int(val or 1))
        rc, fx, fy, _ = o.calculateInternal(a, b)
        assert rc == 0
        assert np.array_equal(fx, ref[..., 0]) and np.array_equal(fy, ref[..., 1]), opt
        o.close()
    o = tw.OpticalFlow(0, 480, 300, 1)
    for gone in ("gauss_fma", "update_fma", "gauss_scalar"):
        assert tw.load().tw_set_option(o.ctx, gone.encode(), 1) == 5 and tw.load().tw_set_option(o.ctx, gone.encode(), 0) == 0
    o.close()


def test_batch_equals_single(of, tw):
    pairs = [tw.synth.make_pair("S", 320, 200, 20 + i, defect=(i % 2 == 0)) for i in range(4)]
    single = [of.calculate(a, b) for a, b in pairs]
    batch = of.calculate_batch(pairs)
    for s, bt in zip(single, batch):
        assert s["status"] == bt["status"] and s["vector"] == bt["vector"]
    assert any(r["status"] == "SUSPICIOUS" for r in batch) and any(len(r["vector"]) > 0 for r in batch)


def test_known_shift_recovered(of, tw):
    """Synthetic texture with a known translation: the mean flow must recover (-0.37, +0.61)."""
    a, b = tw.synth.make_pair("T", 640, 360, 1)
    rc, fx, fy, _ = of.calculateInternal(a, b)
    assert rc == 0
    assert abs(float(fx[40:-40, 40:-40].mean()) + 0.37) < 0.05 and abs(float(fy[40:-40, 40:-40].mean()) - 0.61) < 0.05
    assert of.calculate(a, b)["status"] == "OK"


def test_identical_images_ok(of, golden):
    a = golden["imgs"]["s1_expected"]
    r = of.calculate(a, a.copy())
    assert r["status"] == "OK" and r["vector"] == [] and (r["height"], r["width"]) == (279, 280)


def test_error_codes(of, tw):
    """src/opticalflow.cpp:26-61 error behaviour at the C ABI."""
    a = np.zeros((100, 120), np.uint8)
    r = of.calculate(a, np.zeros((100, 126), np.uint8))
    assert r["status"] == "ERROR" and r["code"] == 3 and r["reason"] == "Don't match image size"
    assert of.calculate(a, np.zeros((100, 125), np.uint8))["status"] != "ERROR"  # within 5 px: resized, not an error
    r = of.calculate(a, np.zeros((106, 120), np.uint8))
    assert r["code"] == 3
    r = of.calculate(None, a)
    assert r["status"] == "ERROR" and r["code"] == 2 and r["reason"].startswith("Can't open")
    r = of.calculate(a, None)
    assert r["code"] == 2
    for bad in (dict(pyrScale=1.0), dict(flags=4), dict(flags=260), dict(polyN=0), dict(winSize=1), dict(pyrLevels=-1)):
        r = of.calculate(a, a, tw.OpticalFlowParameter(**bad))
        assert r["status"] == "ERROR" and r["code"] == 1, bad
    # the context survives errors
    assert of.calculate(a, a)["status"] == "OK"


@pytest.mark.parametrize("dw,dh", [(5, 0), (0, -5), (3, 4), (-2, -5), (-5, 5), (1, -1)])
def test_size_tolerance_resize_path(of, tw, oracle, dw, dh):
    """src/opticalflow.cpp:52-68: sizes within 5 px -> the target is bilinearly resized to the expected size first."""
    a, b0 = tw.synth.make_pair("S", 320, 200, 41, defect=True)
    rng = np.random.default_rng(5)
    b = rng.integers(0, 256, (200 + dh, 320 + dw), dtype=np.uint8)
    h0, w0 = min(200, 200 + dh), min(320, 320 + dw)
    b[:h0, :w0] = b0[:h0, :w0]
    resp = of.calculate(a, b)
    status, vec, flow = oracle.calculate(a, b)
    assert resp["status"] == status and (resp["height"], resp["width"]) == (200, 320)
    assert _vec_pos(resp) == [(v[0], v[1]) for v in vec]
    for v, g in zip(resp["vector"], vec):
        assert v["dx"] == g[2] and v["dy"] == g[3]


def test_vector_cap_truncates(of, golden):
    a, b = golden["imgs"]["s2_expected"], golden["imgs"]["s2_revision2"]
    r = of.calculate(a, b, cap=5)
    assert r["n_vectors"] == 24 and len(r["vector"]) == 5 and r["vector"][0]["x"] == 80


def test_threshold_and_span_options(of, oracle, golden):
    a, b = golden["imgs"]["s2_expected"], golden["imgs"]["s2_revision2"]
    ref = oracle.farneback(a, b, FlowParam())
    for thr, span in ((2.0, 7), (0.5, 1), (50.0, 10), (5.0, 3)):
        r = of.calculate(a, b, threshold=thr, span=span)
        status, vec = oracle.sample(ref, span, thr)
        assert r["status"] == status and _vec_pos(r) == [(v[0], v[1]) for v in vec], (thr, span)


def test_pool_dispatch(tw, golden):
    """Manager/Consumer semantics (src/manager.cpp:40-98): results independent of worker count / order; Report counters."""
    a, b = golden["imgs"]["s2_expected"], golden["imgs"]["s2_revision2"]
    s1 = golden["imgs"]["s1_expected"]
    pairs = [(a, b), (s1, s1), (a, a), (a, b), (a, np.zeros((200, 200), np.uint8)), (s1, s1), (a, b)]
    results = {}
    for devices, batch in (([0], 1), ([0, 0], 2), ([0, 0, 0], 4)):
        pool = tw.Pool(devices, batch=batch, max_w=280, max_h=279)
        ids = [pool.request(x, y) for x, y in pairs]
        out = [pool.wait(i) for i in ids]
        rep = pool.report()
        pool.stop()
        pool.close()
        assert rep == {"request": 7, "data": 6, "error": 1}
        results[(len(devices), batch)] = [(r["status"], r.get("vector")) for r in out]
    vals = list(results.values())
    assert vals[0] == vals[1] == vals[2]
    assert [s for s, _ in vals[0]] == ["SUSPICIOUS", "OK", "OK", "SUSPICIOUS", "ERROR", "OK", "SUSPICIOUS"]
    assert len(vals[0][0][1]) == 24


def test_pool_stop_drops_pending(tw, golden):
    s1 = golden["imgs"]["s1_expected"]
    pool = tw.Pool([0], batch=1, max_w=280, max_h=279)
    ids = [pool.request(s1, s1) for _ in range(50)]
    pool.stop()
    got = [pool.wait(i) for i in ids]
    rep = pool.report()
    assert rep["request"] == 50 and rep["data"] + sum(g is None for g in got) == 50
    assert pool.request(s1, s1) < 0
    pool.close()


def test_deterministic_and_context_independent(tw):
    """Same input -> bit-identical output, across repeats, across contexts and across batch slots (no atomics on the data path,
    no uninitialised reads)."""
    a, b = tw.synth.make_pair("S", 640, 360, 77, defect=True)
    o1 = tw.OpticalFlow(0, 640, 360, 3)
    o2 = tw.OpticalFlow(0, 640, 360, 1)
    rc, fx1, fy1, _ = o1.calculateInternal(a, b)
    rc, fx2, fy2, _ = o1.calculateInternal(a, b)
    rc, fx3, fy3, _ = o2.calculateInternal(a, b)
    assert np.array_equal(fx1, fx2) and np.array_equal(fy1, fy2) and np.array_equal(fx1, fx3) and np.array_equal(fy1, fy3)
    c, d = tw.synth.make_pair("T", 640, 360, 78)
    rb = o1.calculate_batch([(c, d), (a, b), (c, d)])
    fxb, fyb = o1.batch_flow(1, 640, 360)
    assert np.array_equal(fxb, fx1) and np.array_equal(fyb, fy1)
    assert rb[1] == {**o2.calculate(a, b), "time": rb[1]["time"]}
    o1.close(); o2.close()


def test_concurrent_contexts(tw):
    """Two consumers on the same GPU (two contexts / streams) running at once give the single-context answers."""
    import threading
    pairs = [tw.synth.make_pair("S", 480, 270, 90 + i, defect=(i % 2 == 0)) for i in range(6)]
    ref = tw.OpticalFlow(0, 480, 270, 1)
    want = [ref.calculate(a, b) for a, b in pairs]
    ref.close()
    out = [None, None]

    def work(k):
        o = tw.OpticalFlow(0, 480, 270, 2)
        res = []
        for _ in range(3):
            res = [o.calculate(a, b) for a, b in pairs]
        out[k] = res
        o.close()

    ts = [threading.Thread(target=work, args=(k,)) for k in range(2)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    for k in range(2):
        for w_, g in zip(want, out[k]):
            assert w_["status"] == g["status"] and w_["vector"] == g["vector"]


def test_pool_all_devices(tw, golden):
    """One process, one consumer per visible GPU (the reference's consumer i <-> GPU i, src/consumer.cpp:18-24): kernel
    attributes are per device, so every device must be able to launch every kernel.  (On a 1-GPU box this is devices=[0].)"""
    n = tw.load().tw_device_count()
    a, b = golden["imgs"]["s2_expected"], golden["imgs"]["s2_revision2"]
    pool = tw.Pool(list(range(n)) * 2, batch=2, max_w=180, max_h=117)
    ids = [pool.request(a, b) for _ in range(8 * n)]
    out = [pool.wait(i) for i in ids]
    rep = pool.report()
    pool.stop(); pool.close()
    assert rep == {"request": 8 * n, "data": 8 * n, "error": 0}
    assert all(r["status"] == "SUSPICIOUS" and len(r["vector"]) == 24 for r in out)


def test_pool_mixed_sizes_return_every_vector(tw):
    """Screenshot directories mix page sizes (index.js:33-73 feeds whatever the glob finds): a small OK pair followed by a larger
    SUSPICIOUS pair through one dispatcher with vector_cap = 0 must return EVERY vector of the larger pair, as the reference
    does (src/consumer.cpp:60-76) -- the capacity follows each request, not the first one."""
    small = tw.synth.make_pair("T", 200, 120, 3)
    big = tw.synth.make_pair("S", 960, 540, 100, defect=True)
    o = tw.OpticalFlow(0, 0, 0, 1)
    want_small, want_big = o.calculate(*small, threshold=0.3), o.calculate(*big, threshold=0.3)
    o.close()
    assert want_big["status"] == "SUSPICIOUS" and len(want_big["vector"]) > 24 * 12  # more than the small pair's whole grid
    pool = tw.Pool([0, 0], batch=2, threshold=0.3)  # max_w = max_h = vector_cap = 0
    ids = [pool.request(*small), pool.request(*big), pool.request(*small), pool.request(*big)]
    out = [pool.wait(i) for i in ids]
    pool.stop(); pool.close()
    for got, want in zip(out, (want_small, want_big, want_small, want_big)):
        assert got["status"] == want["status"] and got["vector"] == want["vector"] and got["n_vectors"] == len(got["vector"])


def test_context_size_bound_is_enforced(tw):
    """tw_create's max_w / max_h bound the images a context accepts; 0 = no bound."""
    a, b = tw.synth.make_pair("T", 200, 120, 3)
    o = tw.OpticalFlow(0, 160, 120, 1)
    r = o.calculate(a, b)
    assert r["status"] == "ERROR" and r["code"] == 1
    o.close()
    o = tw.OpticalFlow(0, 200, 120, 1)
    assert o.calculate(a, b)["status"] != "ERROR"
    o.close()


@pytest.mark.parametrize("size,seed,batch", [((1920, 1080), 100, 2), ((500, 333), 7, 3), ((97, 61), 9, 1), ((960, 540), 11, 1),
                                             ((40, 33), 3, 2), ((70, 130), 5, 1), ((64, 64), 6, 1), ((129, 72), 8, 2)])
def test_strip_window_kernel_bit_identical(tw, oracle, size, seed, batch):
    """The persistent strip window kernel ("window_tiles" = 0) and the tile kernel run the same arithmetic: bit-identical to
    each other and to the oracle in both arithmetics, on ragged strip / group geometry (w % 64 != 0, h % 8 != 0, frames narrower than
    one strip and shorter than one segment), with a defect
    (motion boundary: the global-memory gather path of the epilogue), on the last and the non-last iterations, batched."""
    w, h = size
    a, b = tw.synth.make_pair("S", w, h, seed, defect=True)
    pairs = [(a, b)] + [tw.synth.make_pair("T", w, h, seed + 1 + i) for i in range(batch - 1)]
    o = tw.OpticalFlow(0, w, h, batch)
    ref = {}
    for bits in (0, 144):
        oracle.set_relax(bits)
        ref[bits] = oracle.farneback(a, b, FlowParam())
    oracle.set_relax(0)
    for tiles in (1, 0):
        o.set_option("window_tiles", tiles)
        for arith, bits in ((0, 0), (1, 144)):
            o.set_option("arithmetic", arith)
            for _ in range(2):  # eager, then the captured graph
                res = o.calculate_batch(pairs, threshold=0.5)
                fx, fy = o.batch_flow(0, w, h)
                assert np.array_equal(fx, ref[bits][..., 0]) and np.array_equal(fy, ref[bits][..., 1]), (tiles, arith)
            status, vec = oracle.sample(ref[bits], 10, 0.5)
            assert res[0]["status"] == status and _vec_pos(res[0]) == [(v[0], v[1]) for v in vec]
    o.close()


@pytest.mark.gpu
def test_pipelined_batches_match_synchronous(tw):
    """tw_pipe_submit / tw_pipe_collect (two batches in flight: upload of k + 1 overlaps the kernels of k, results of k - 1 are read
    from a device snapshot) return exactly what tw_compare_batch returns, in submission order, across a change of batch size."""
    import ctypes as C
    lib = tw.load()
    w, h, B = 640, 360, 3
    batches = [[tw.synth.make_pair("S" if (i + j) % 2 else "T", w, h, 10 * i + j, defect=(j == 1)) for j in range(n)] for i, n in enumerate((3, 2, 3, 1, 3))]
    o = tw.OpticalFlow(0, w, h, B)
    o.set_option("sparse_last", 1)
    want = [o.calculate_batch(b, threshold=0.4) for b in batches]
    assert any(r["status"] == "SUSPICIOUS" for rs in want for r in rs)
    p = tw.OpticalFlowParameter().c()
    cap = ((w + 9) // 10) * ((h + 9) // 10)
    vec = (tw.tw_vector * (cap * B))()
    res = (tw.tw_result * B)()
    keep, got, pending = [], [], []

    def collect():
        n = pending.pop(0)
        assert lib.tw_pipe_collect(o.ctx, vec, cap, res) == 0, o.last_error()
        got.append([(res[i].status, res[i].n_vectors, [(vec[i * cap + k].x, vec[i * cap + k].y, vec[i * cap + k].dx, vec[i * cap + k].dy)
                                                       for k in range(min(res[i].n_vectors, cap))]) for i in range(n)])
    for b in batches:
        n = len(b)
        ex = (C.c_void_p * n)(*[x.ctypes.data for x, _ in b]); tg = (C.c_void_p * n)(*[y.ctypes.data for _, y in b])
        keep.append((b, ex, tg))
        if lib.tw_pipe_pending(o.ctx) == 2:
            collect()
        assert lib.tw_pipe_submit(o.ctx, n, ex, tg, w, h, w, C.byref(p), 0.4, 10) == 0, o.last_error()
        pending.append(n)
    while pending:
        collect()
    assert lib.tw_pipe_pending(o.ctx) == 0 and lib.tw_pipe_collect(o.ctx, vec, cap, res) != 0
    names = {0: "OK", 1: "SUSPICIOUS", 2: "ERROR"}
    for ws, gs in zip(want, got):
        assert len(ws) == len(gs)
        for wr, (st, nv, vs) in zip(ws, gs):
            assert wr["status"] == names[st] and len(wr["vector"]) == nv
            assert [(v["x"], v["y"], v["dx"], v["dy"]) for v in wr["vector"]] == vs
    o.close()


@pytest.mark.gpu
def test_pool_path_requests(tw, golden, tmp_path):
    """tw_pool_submit_files = Manager::request as the reference has it (two paths, src/manager.cpp:68-78): files read and decoded on
    the pool's C++ decoder threads; answers equal those of the image-based requests; the reference's error messages
    (src/opticalflow.cpp:20-61) for empty paths, unreadable files and mismatched sizes."""
    import os
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    s1 = os.path.join(gold, "jpg", "fixture_s1_capture1.jpg")
    s2e, s2r = os.path.join(gold, "png", "fixture_s2_expected.png"), os.path.join(gold, "png", "fixture_s2_revision2.png")
    (tmp_path / "junk.jpg").write_bytes(b"\xff\xd8\xff\xe0junk")
    pool = tw.Pool([0], batch=4)  # vector_cap = 0: every vector
    tw.load().tw_pool_set_decoders(pool.pool, 3)
    want = pool.wait(pool.request(tw.imread_gray(s2e), tw.imread_gray(s2r)))
    ids = [pool.request_files(*p) for p in ((s2e, s2r), (s1, s1), ("", s1), (s1, ""), (s2e, str(tmp_path / "junk.jpg")),
                                            (str(tmp_path / "missing.png"), s1), (s1, s2e), (s2e, s2r))]
    out = [pool.wait(i) for i in ids]
    rep = pool.report()
    pool.stop(); pool.close()
    assert want["status"] == "SUSPICIOUS" and len(want["vector"]) == 24
    for k in (0, 7):
        assert out[k]["status"] == "SUSPICIOUS" and out[k]["vector"] == want["vector"] and (out[k]["width"], out[k]["height"]) == (180, 117)
    assert out[1]["status"] == "OK" and (out[1]["width"], out[1]["height"]) == (280, 279)
    assert [o["status"] for o in out[2:7]] == ["ERROR"] * 5
    assert [o["reason"] for o in out[2:7]] == ["ExpectImagePath is empty.", "TargetImagePath is empty.", "Can't open " + str(tmp_path / "junk.jpg"),
                                              "Can't open " + str(tmp_path / "missing.png"), "Don't match image size"]
    assert rep == {"request": 9, "data": 4, "error": 5}


@pytest.mark.gpu
@pytest.mark.parametrize("size,kw", [((203, 157), dict(flags=0, winSize=2)), ((203, 157), dict(flags=0, winSize=9, polyN=5, polySigma=1.1)),
                                     ((330, 97), dict(flags=0, winSize=31)), ((97, 330), dict(flags=0, winSize=32)),
                                     ((203, 157), dict(flags=0, winSize=34)), ((64, 33), dict(flags=0, winSize=15))])
def test_box_window_fused_and_unfused_bit_identical(tw, oracle, size, kw):
    """The fused box iteration (band checkpoints + band kernel, window radius <= 16) and the three-launch form ("box_unfused", also the
    fall-back for larger radii: winSize 34 -> radius 17) follow App. A.6's running sums in the oracle's order: bit-identical to the
    oracle and to each other on ragged frames (w, h not multiples of 32), frames smaller than a band / a chunk, even and odd sizes."""
    w, h = size
    pairs = [tw.synth.make_pair("S", w, h, 3, defect=True), tw.synth.make_pair("T", w, h, 4)]
    ref = [oracle.farneback(a, b, FlowParam(**kw)) for a, b in pairs]
    o = tw.OpticalFlow(0, w, h, 2)
    p = tw.OpticalFlowParameter(**kw)
    for unfused in (0, 1):
        o.set_option("box_unfused", unfused)
        for _ in range(2):  # eager, then the captured graph
            res = o.calculate_batch(pairs, p, threshold=0.5)
            for i in range(2):
                fx, fy = o.batch_flow(i, w, h)
                assert np.array_equal(fx, ref[i][..., 0]) and np.array_equal(fy, ref[i][..., 1]), (unfused, i)
        status, vec = oracle.sample(ref[0], 10, 0.5)
        assert res[0]["status"] == status and _vec_pos(res[0]) == [(v[0], v[1]) for v in vec]
    o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("size,levels", [((500, 333), 5), ((700, 200), 4), ((130, 900), 5)])
def test_deep_pyramid_long_preblur_levels(tw, oracle, size, levels):
    """Deep pyramids put 39- / 79-tap pre-blurs in front of non-integer down-scales: the separable two-kernel level path
    (level_rows / level_cols) and the generic kernel ("level_generic") are bit-identical to the oracle."""
    w, h = size
    a, b = tw.synth.make_pair("S", w, h, 21, defect=True)
    kw = dict(pyrLevels=levels, pyrIterations=2)
    ref = oracle.farneback(a, b, FlowParam(**kw))
    for generic in (0, 1):
        o = tw.OpticalFlow(0, w, h, 1)
        o.set_option("arithmetic", 0)
        o.set_option("level_generic", generic)
        rc, fx, fy, _ = o.calculateInternal(a, b, tw.OpticalFlowParameter(**kw))
        assert rc == 0 and np.array_equal(fx, ref[..., 0]) and np.array_equal(fy, ref[..., 1]), generic
        o.close()


@pytest.mark.gpu
def test_plan_cache_switching_sizes(tw):
    """A context keeps the plans (buffers, tables, tensor maps, captured graph) of the sizes it has seen: switching back and forth between
    page sizes -- what a screenshot directory does -- gives the first-time answers again (graph replay included), also after evictions
    (more sizes than "plan_cache" holds) and with the cache turned off."""
    sizes = [(320, 200), (200, 320), (416, 240), (250, 250), (300, 180), (180, 300)]
    pairs = {sz: tw.synth.make_pair("S", sz[0], sz[1], 7 + i, defect=True) for i, sz in enumerate(sizes)}
    ref = {}
    o = tw.OpticalFlow(0, 0, 0, 2)
    for sz in sizes:
        rc, fx, fy, _ = o.calculateInternal(*pairs[sz])
        assert rc == 0
        ref[sz] = (fx.copy(), fy.copy(), o.calculate(*pairs[sz], threshold=0.5))
    o.close()
    for cache in (3, 0):
        o = tw.OpticalFlow(0, 0, 0, 2)
        o.set_option("plan_cache", cache)
        order = [0, 1, 0, 1, 0, 2, 3, 4, 5, 0, 1, 5, 0, 0, 1]
        for k in order:
            sz = sizes[k]
            rc, fx, fy, _ = o.calculateInternal(*pairs[sz])
            assert rc == 0 and np.array_equal(fx, ref[sz][0]) and np.array_equal(fy, ref[sz][1]), (cache, sz)
            r = o.calculate(*pairs[sz], threshold=0.5)
            assert r["status"] == ref[sz][2]["status"] and r["vector"] == ref[sz][2]["vector"]
        o.close()
