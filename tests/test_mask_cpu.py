"""CPU tests of the ignore-mask interface (include/tidalwave_b200.h, tw_compare_mask): the new entry points in the header, the
library and the binding, the Python forms of a mask and its size message, and create()'s ignoreMaskDir / getIgnoreMaskPath."""
import re

import numpy as np
import pytest

NEW = {  # entry point -> its parameter count in the header
    "tw_compare_mask": 16,
    "tw_compare_batch_mask": 16,
    "tw_pipe_submit_mask": 13,
    "tw_pool_submit_mask": 10,
    "tw_pool_submit_files_mask": 6,
}


def _prototypes(tw):
    src = re.sub(r"/\*.*?\*/", "", open(tw.api.HEADER_PATH).read(), flags=re.S)
    return {m.group(1): [a.strip() for a in m.group(2).split(",")] for m in re.finditer(r"\b(tw_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src)}


def test_abi_declares_exports_and_binds_the_mask_entry_points(tw):
    protos = _prototypes(tw)
    lib = tw.load()
    for name, nargs in NEW.items():
        assert name in tw.declared_symbols() and hasattr(lib, name), name
        assert len(protos[name]) == nargs == len(getattr(lib, name).argtypes), name
    assert protos["tw_compare_mask"][12] == "const uint8_t *mask"
    assert protos["tw_compare_batch_mask"][12] == protos["tw_pipe_submit_mask"][12] == "const uint8_t *const *mask"
    assert protos["tw_pool_submit_mask"][-1] == "const uint8_t *mask"
    assert protos["tw_pool_submit_files_mask"][3] == "const char *mask_path"
    # the *_mask entry points extend the *_ignore ones: the same leading parameters
    assert protos["tw_compare_mask"][:12] == protos["tw_compare_ignore"][:12]
    assert protos["tw_compare_batch_mask"][:12] == protos["tw_compare_batch_ignore"][:12]
    assert protos["tw_pipe_submit_mask"][:12] == protos["tw_pipe_submit_ignore"]


def test_mask_forms(tw):
    m = np.zeros((3, 4), bool)
    m[1, 2] = True
    u = tw.api.mask_array(m)
    assert u.dtype == np.uint8 and u.flags.c_contiguous and u.tolist() == [[0, 0, 0, 0], [0, 0, 1, 0], [0, 0, 0, 0]]
    v = np.arange(24, dtype=np.uint8).reshape(4, 6)[:, ::2]  # a strided view comes back contiguous, same values
    assert tw.api.mask_array(v).flags.c_contiguous and np.array_equal(tw.api.mask_array(v), v)
    assert tw.api.mask_array(None) is None
    for bad in (np.zeros((3, 4), np.float32), np.zeros((3, 4, 1), np.uint8), np.zeros(5, np.uint8), [[0, 1], [1, 0]], "mask.png"):
        with pytest.raises(ValueError, match="bad ignore mask"):
            tw.api.mask_array(bad)


def test_mask_size_message(tw):
    assert tw.api.mask_size_error((200, 321), (200, 320)) == "bad ignore mask: 321x200 mask for a 320x200 expected image"


def test_create_mask_options(tw, tmp_path):
    (tmp_path / "m" / "sub").mkdir(parents=True)
    (tmp_path / "m" / "a.png").write_bytes(b"x")
    (tmp_path / "m" / "sub" / "c.png").write_bytes(b"x")
    t = tw.TidalWave({"ignoreMaskDir": str(tmp_path / "m"), "getIgnoreMaskPath": lambda s: "/elsewhere/" + s})
    assert t.ignore_mask_path("a.png") == str(tmp_path / "m" / "a.png")
    assert t.ignore_mask_path("sub/c.png") == str(tmp_path / "m" / "sub" / "c.png")
    assert t.ignore_mask_path("b.png") is None  # no file there: no mask (the directory wins over the callable)
    seen = []

    def per_pair(short):
        seen.append(short)
        return {"a.png": "/m/a.png", "empty.png": "", "none.png": None, "odd.png": 5}.get(short)

    t = tw.TidalWave({"ignoreMaskDir": 7, "getIgnoreMaskPath": per_pair})  # wrong-typed directory: the callable decides
    assert [t.ignore_mask_path(s) for s in ("a.png", "empty.png", "none.png", "odd.png")] == ["/m/a.png", None, None, None]
    assert seen == ["a.png", "empty.png", "none.png", "odd.png"]
    for opts in ({}, {"ignoreMaskDir": ["x"]}, {"getIgnoreMaskPath": "not callable"}, {"ignoreMaskDir": None}):
        assert tw.TidalWave(opts).ignore_mask_path("a.png") is None, opts


def test_create_pairs_mask_files_and_regions(tw, tmp_path):
    """Each target takes the mask at its short path (if any) together with its regions; one pair's malformed region is still an
    'error' event of its own."""
    for d in ("t/sub", "m/sub"):
        (tmp_path / d).mkdir(parents=True)
    for n in ("a.png", "b.png", "sub/c.png", "sub/d.png"):
        (tmp_path / "t" / n).write_bytes(b"x")
    for n in ("a.png", "sub/c.png", "sub/d.png"):
        (tmp_path / "m" / n).write_bytes(b"x")
    calls = []

    class StubPool:
        def request_files(self, expected, target, ignore=None, ignore_mask=None):
            calls.append((expected.rsplit("/", 1)[-1], ignore, ignore_mask and ignore_mask[len(str(tmp_path)) + 1:]))
            return len(calls) - 1

        def wait(self, rid):
            return {"status": "OK", "n_vectors": 0, "vector": [], "width": 1, "height": 1, "span": 10, "threshold": 5.0, "time": 0.0}

        def stop(self):
            pass

        def close(self):
            pass

    t = tw.create(str(tmp_path / "t"), {"getExpectedPath": lambda s: "/e/" + s, "ignoreMaskDir": str(tmp_path / "m"),
                                        "ignoreRegions": [(0, 0, 10, 10)],
                                        "getIgnoreRegions": lambda s: [(0, 0)] if s == "sub/d.png" else [(5, 5, 2, 2)]})
    stub = StubPool()
    t._ensure_pool = lambda w, h: (setattr(t, "_pool", stub), stub)[1]
    ev = []
    t.on("data", lambda r: ev.append("data")).on("error", lambda r: ev.append(r["reason"].split(":")[0]))
    t.on("finish", lambda r: ev.append(r))
    tw.run(t)
    both = [(0, 0, 10, 10), (5, 5, 2, 2)]
    assert calls == [("a.png", both, "m/a.png"), ("b.png", both, None), ("c.png", both, "m/sub/c.png")]
    assert ev == ["data", "data", "data", "bad ignore region", {"request": 4, "data": 3, "error": 1}]
