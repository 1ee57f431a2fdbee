"""CPU tests of the ignore-region interface (include/tidalwave_b200.h, tw_compare_ignore): the struct layout and limit shared by
the header and the binding, the Python forms of a region, and the parsing of create()'s ignoreRegions / getIgnoreRegions."""
import ctypes as C
import re

import pytest


def test_rect_layout_and_limit(tw):
    assert C.sizeof(tw.tw_rect) == 16
    assert [f for f, _ in tw.tw_rect._fields_] == ["x", "y", "width", "height"]
    src = open(tw.api.HEADER_PATH).read()
    assert int(re.search(r"#define\s+TW_MAX_IGNORE\s+(\d+)", src).group(1)) == tw.MAX_IGNORE == 32


def test_region_forms(tw):
    assert tw.api.rect((1, 2, 3, 4)) == (1, 2, 3, 4)
    assert tw.api.rect([-5, 0, 10, 7]) == (-5, 0, 10, 7)
    assert tw.api.rect({"x": 1, "y": 2, "width": 3, "height": 4, "label": "clock"}) == (1, 2, 3, 4)
    for bad in ((1, 2, 3), {"x": 1, "y": 2, "width": 3}, (1, 2, 3.5, 4), (1, 2, True, 4), "0,0,1,1", None):
        with pytest.raises(ValueError, match="bad ignore region"):
            tw.api.rect(bad)
    rs, n = tw.api._rects([(1, 2, 3, 4), {"x": 5, "y": 6, "width": 7, "height": 8}])
    assert n == 2 and [(r.x, r.y, r.width, r.height) for r in rs] == [(1, 2, 3, 4), (5, 6, 7, 8)]
    assert tw.api._rects(None) == (None, 0) and tw.api._rects([]) == (None, 0)


def test_create_ignore_options(tw):
    seen = []

    def per_pair(short):
        seen.append(short)
        return {"a.png": [(10, 10, 5, 5)], "bad.png": [{"x": 1}], "odd.png": {"x": 1, "y": 1, "width": 1, "height": 1}}.get(short)

    t = tw.TidalWave({"ignoreRegions": [{"x": 0, "y": 0, "width": 100, "height": 20}], "getIgnoreRegions": per_pair})
    assert t.ignore_regions("a.png") == [(0, 0, 100, 20), (10, 10, 5, 5)]
    assert t.ignore_regions("other.png") == [(0, 0, 100, 20)]
    for short in ("bad.png", "odd.png"):
        with pytest.raises(ValueError, match="bad ignore region"):
            t.ignore_regions(short)
    assert seen == ["a.png", "other.png", "bad.png", "odd.png"]
    assert tw.TidalWave({}).ignore_regions("a.png") == []
    assert tw.TidalWave({"getIgnoreRegions": "not callable"}).ignore_regions("a.png") == []
    with pytest.raises(ValueError):
        tw.TidalWave({"ignoreRegions": 5}).ignore_regions("a.png")


def test_create_rejects_malformed_region_per_pair(tw, tmp_path):
    """A malformed region makes its pair an 'error' event; the other pairs are still requested (with their regions)."""
    (tmp_path / "t").mkdir()
    for n in ("a.png", "b.png"):
        (tmp_path / "t" / n).write_bytes(b"x")
    calls = []

    class StubPool:
        def request_files(self, expected, target, ignore=None):
            calls.append((expected.rsplit("/", 1)[-1], ignore))
            return len(calls) - 1

        def wait(self, rid):
            return {"status": "OK", "n_vectors": 0, "vector": [], "width": 1, "height": 1, "span": 10, "threshold": 5.0, "time": 0.0}

        def stop(self):
            pass

        def close(self):
            pass

    t = tw.create(str(tmp_path / "t"), {"getExpectedPath": lambda s: "/e/" + s,
                                        "getIgnoreRegions": lambda s: [(1, 2, 3, 4)] if s == "a.png" else [(0, 0)]})
    stub = StubPool()
    t._ensure_pool = lambda w, h: (setattr(t, "_pool", stub), stub)[1]
    ev = []
    t.on("data", lambda r: ev.append(("data", r["target_image"].rsplit("/", 1)[-1])))
    t.on("error", lambda r: ev.append(("error", r["reason"].split(":")[0]))).on("finish", lambda r: ev.append(("finish", r)))
    tw.run(t)
    assert calls == [("a.png", [(1, 2, 3, 4)])]
    assert ev == [("data", "a.png"), ("error", "bad ignore region"), ("finish", {"request": 2, "data": 1, "error": 1})]
