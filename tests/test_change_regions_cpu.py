"""CPU tests of change regions (include/tidalwave_b200.h, tw_change_regions): the struct layout and limit shared by the header and
the binding, the new entry points, the host oracle `regions_of` that the GPU tests compare the device against, and the parsing of
create()'s changeRegions."""
import ctypes as C
import re

import numpy as np
import pytest
from scipy import ndimage


def regions_of(vectors, w, h, span):
    """The change regions of a pair, restated on the host from its vector list ((x, y, dx, dy) in scan order): the 8-connected
    components of the suspicious span-grid points, labelled by scipy (first raster occurrence order), each with the bounding box of
    its cells clipped to the frame, its point count and its peak (largest f32(f32(dx * dx) + f32(dy * dy)), the earlier point on a
    tie).  Returns every region, as the binding's dicts."""
    nsx, nsy = (w + span - 1) // span, (h + span - 1) // span
    grid = np.zeros((nsy, nsx), bool)
    for x, y, _, _ in vectors:
        grid[y // span, x // span] = True
    labels, n = ndimage.label(grid, structure=np.ones((3, 3), int))
    out = [None] * n
    for x, y, dx, dy in vectors:
        k = labels[y // span, x // span] - 1
        fx, fy = np.float32(dx), np.float32(dy)
        ln = np.float32(np.float32(fx * fx) + np.float32(fy * fy))
        r = out[k]
        if r is None:
            out[k] = r = {"x0": x, "y0": y, "x1": x, "y1": y, "n_vectors": 0, "len": ln, "peak": (x, y, dx, dy)}
        r["x0"], r["y0"], r["x1"], r["y1"] = min(r["x0"], x), min(r["y0"], y), max(r["x1"], x), max(r["y1"], y)
        r["n_vectors"] += 1
        if ln > r["len"]:
            r["len"], r["peak"] = ln, (x, y, dx, dy)
    return [{"x": r["x0"], "y": r["y0"], "width": min(r["x1"] + span, w) - r["x0"], "height": min(r["y1"] + span, h) - r["y0"],
             "n_vectors": r["n_vectors"], "peak": dict(zip(("x", "y", "dx", "dy"), r["peak"]))} for r in out]


def _v(points, span, d=(1.0, 0.0)):
    """Vectors at grid points (i, j), in scan order."""
    return [(i * span, j * span, d[0], d[1]) for j, i in sorted((j, i) for i, j in points)]


def _rects(regs):
    return [(r["x"], r["y"], r["width"], r["height"], r["n_vectors"]) for r in regs]


def test_struct_layout_and_limit(tw):
    R = tw.tw_change_region
    assert C.sizeof(R) == 48
    assert (R.rect.offset, R.n_vectors.offset, R.peak.offset) == (0, 16, 24)
    src = open(tw.api.HEADER_PATH).read()
    assert int(re.search(r"#define\s+TW_MAX_CHANGE_REGIONS\s+(\d+)", src).group(1)) == tw.MAX_CHANGE_REGIONS == 1024


def test_abi_declares_exports_and_binds_the_region_entry_points(tw):
    src = re.sub(r"/\*.*?\*/", "", open(tw.api.HEADER_PATH).read(), flags=re.S)
    protos = {m.group(1): [a.strip() for a in m.group(2).split(",")] for m in re.finditer(r"\b(tw_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src)}
    lib = tw.load()
    for name, nargs in {"tw_change_regions": 5, "tw_pool_set_change_regions": 2, "tw_pool_wait_regions": 8}.items():
        assert name in tw.declared_symbols() and hasattr(lib, name), name
        assert len(protos[name]) == nargs == len(getattr(lib, name).argtypes), name
    assert protos["tw_pool_wait_regions"][:5] == protos["tw_pool_wait"]  # tw_pool_wait plus the regions


def test_diagonal_neighbours_join_and_a_knights_move_splits():
    s = 10
    assert _rects(regions_of(_v([(0, 0), (1, 1), (2, 2), (3, 1)], s), 100, 100, s)) == [(0, 0, 40, 30, 4)]
    assert _rects(regions_of(_v([(0, 0), (2, 1)], s), 100, 100, s)) == [(0, 0, 10, 10, 1), (20, 10, 10, 10, 1)]
    assert _rects(regions_of(_v([(2, 0), (1, 1)], s), 100, 100, s)) == [(10, 0, 20, 20, 2)]  # NE neighbour


def test_order_is_first_point_in_scan_order():
    s = 10
    # the region starting at (9, 3) comes before the one starting at (0, 4), although the latter lies left of its second point
    pts = [(5, 0), (5, 1), (1, 1), (2, 2), (9, 3), (8, 4), (0, 4), (0, 5)]
    regs = regions_of(_v(pts, s), 100, 100, s)
    assert _rects(regs) == [(50, 0, 10, 20, 2), (10, 10, 20, 20, 2), (80, 30, 20, 20, 2), (0, 40, 10, 20, 2)]
    # a U shape: one region whose first point is its top-left arm, although the other arm starts on the same row
    u = [(0, 0), (4, 0), (0, 1), (4, 1), (1, 2), (2, 2), (3, 2)]
    assert _rects(regions_of(_v(u, s), 100, 100, s)) == [(0, 0, 50, 30, 7)]


def test_rect_is_clipped_at_the_frame():
    s = 10
    # W = 95, H = 47: the last grid column is x = 90 (cell [90, 95)), the last row y = 40 (cell [40, 47))
    regs = regions_of(_v([(9, 4), (8, 3)], s), 95, 47, s)
    assert _rects(regs) == [(80, 30, 15, 17, 2)]
    # a frame narrower and lower than the span: one point, one cell, the whole frame
    assert _rects(regions_of([(0, 0, 3.0, 4.0)], 7, 4, s)) == [(0, 0, 7, 4, 1)]
    # a 1x1 frame
    regs = regions_of([(0, 0, -0.5, 2.0)], 1, 1, 1)
    assert regs == [{"x": 0, "y": 0, "width": 1, "height": 1, "n_vectors": 1, "peak": {"x": 0, "y": 0, "dx": -0.5, "dy": 2.0}}]
    assert regions_of([], 1, 1, 1) == []


def test_peak_is_the_longest_and_the_tie_goes_to_the_earlier_point():
    s = 10
    v = [(0, 0, 3.0, 4.0), (10, 0, -4.0, 3.0), (20, 0, 1.0, 1.0), (10, 10, 0.0, 6.0), (20, 10, -6.0, 0.0)]
    r = regions_of(v, 100, 100, s)
    assert len(r) == 1 and r[0]["peak"] == {"x": 10, "y": 10, "dx": 0.0, "dy": 6.0}
    r = regions_of(v[:3], 100, 100, s)
    assert r[0]["peak"] == {"x": 0, "y": 0, "dx": 3.0, "dy": 4.0}
    # the length is the float32 one: 1 + 2^-30 and 1 are equal in float32, so the earlier of the two wins
    assert regions_of([(0, 0, 1.0, 0.0), (10, 0, 1.0, 2.0 ** -15)], 100, 100, s)[0]["peak"]["dy"] == 0.0
    assert regions_of([(0, 0, 1.0, 2.0 ** -15), (10, 0, 1.0, 0.0)], 100, 100, s)[0]["peak"]["dy"] == 2.0 ** -15


def test_golden_s2r2_groups_into_five_regions(golden):
    """The reference's scenario2 fixture at its options (threshold 5, span 10, 180x117): 24 vectors, 5 regions."""
    case = next(c for c in golden["cases"] if c["target"] == "s2_revision2")
    v = [(p["x"], p["y"], p["dx"], p["dy"]) for p in case["vector"]]
    regs = regions_of(v, case["width"], case["height"], golden["options"]["span"])
    assert _rects(regs) == [(80, 70, 10, 10, 1), (130, 70, 20, 20, 4), (160, 70, 20, 47, 9), (110, 80, 10, 10, 1), (80, 100, 50, 17, 9)]
    assert sum(r["n_vectors"] for r in regs) == len(v) == 24


def test_create_change_regions_option(tw, tmp_path, monkeypatch):
    assert tw.TidalWave({"changeRegions": True}).changeRegions is True
    for off in ({}, {"changeRegions": False}, {"changeRegions": 1}, {"changeRegions": "true"}, {"changeRegions": None}):
        assert tw.TidalWave(off).changeRegions is False, off
    (tmp_path / "t").mkdir()
    (tmp_path / "t" / "a.png").write_bytes(b"x")
    made = []

    class StubPool:
        def __init__(self, *args, **kw):
            made.append(kw.get("change_regions"))
            self.pool = None

        def request_files(self, expected, target, ignore=None, ignore_mask=None):
            return 0

        def wait(self, rid):
            return {"status": "OK", "n_vectors": 0, "vector": [], "width": 1, "height": 1, "span": 10, "threshold": 5.0, "time": 0.0,
                    "regions": [], "n_regions": 0}

        def stop(self):
            pass

        def close(self):
            pass

    class StubLib:
        def tw_device_count(self):
            return 1

        def tw_pool_set_decoders(self, pool, n):
            return 0

    monkeypatch.setattr(tw.tidalwave, "Pool", StubPool)
    monkeypatch.setattr(tw.api, "load", lambda: StubLib())
    for opts, want in (({"changeRegions": True}, True), ({"changeRegions": "yes"}, False)):
        ev = []
        t = tw.create(str(tmp_path / "t"), dict(opts, getExpectedPath=lambda s: "/e/" + s))
        t.on("data", ev.append)
        tw.run(t)
        assert made[-1] is want and ev[0]["regions"] == [] and ev[0]["n_regions"] == 0  # what the pool answers is passed on
