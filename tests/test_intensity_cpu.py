"""CPU tests of intensity cells (include/tidalwave_b200.h, tw_intensity_cells): the struct layout and limit shared by the header and
the binding, the new entry points, the host restatement `intensity_cells` that the GPU tests compare the device against, and the
parsing of create()'s intensityThreshold."""
import ctypes as C
import re

import numpy as np


def intensity_cells(E, T, flowx, flowy, span, t, ignored=None):
    """The intensity cells of a pair, restated on the host.  E, T: u8 H x W (T as the flow saw it: resized, painted); flowx, flowy:
    the float32 flow, read at the sample points (i * span, j * span) only; ignored: bool H x W (regions and mask) or None.  Cell
    (i, j) covers [i * span, min(i * span + span, W)) x [j * span, min(j * span + span, H)); its shift is rint(clamp(flow, -W, W)),
    rint(clamp(flow, -H, H)) at its sample point, half to even, 0 for a non-finite component.  A pixel's residual is the least
    |E - T| over the 3 x 3 target pixels around its shifted position, clamped to the frame.  A cell with n > 0 pixels not ignored
    and residual sum S > t * n is an intensity cell.  Returns every such cell, in scan order, as the binding's dicts."""
    E = np.asarray(E, np.int32)
    T = np.asarray(T, np.int32)
    H, W = E.shape
    nsx, nsy = (W + span - 1) // span, (H + span - 1) // span

    def shift(f, lim):
        f = np.asarray(f, np.float32)[::span, ::span]
        c = np.clip(np.where(np.isfinite(f), f, np.float32(0)), np.float32(-lim), np.float32(lim))
        return np.rint(c).astype(np.int64)

    sx, sy = shift(flowx, W), shift(flowy, H)
    py, px = np.mgrid[0:H, 0:W]
    cy, cx = py // span, px // span
    qx, qy = px + sx[cy, cx], py + sy[cy, cx]
    r = np.full((H, W), 255, np.int64)
    for v in (-1, 0, 1):
        for u in (-1, 0, 1):
            r = np.minimum(r, np.abs(E - T[np.clip(qy + v, 0, H - 1), np.clip(qx + u, 0, W - 1)]))
    keep = np.ones((H, W), bool) if ignored is None else ~np.asarray(ignored, bool)
    ids = (cy * nsx + cx)[keep]
    S = np.bincount(ids, weights=r[keep].astype(np.float64), minlength=nsx * nsy).astype(np.int64)
    n = np.bincount(ids, minlength=nsx * nsy).astype(np.int64)
    hit = np.nonzero((n > 0) & (S > t * n))[0]
    return [{"x": int(i % nsx) * span, "y": int(i // nsx) * span, "n_pixels": int(n[i]), "residual": int(S[i])} for i in hit]


def _zero(E):
    return np.zeros(E.shape, np.float32), np.zeros(E.shape, np.float32)


def _page(h=40, w=60, seed=1):
    """Flat blocks with sharp edges, like a screenshot."""
    rng = np.random.default_rng(seed)
    E = np.full((h, w), 230, np.uint8)
    for _ in range(12):
        x, y = rng.integers(0, w - 8), rng.integers(0, h - 6)
        E[y:y + rng.integers(3, 10), x:x + rng.integers(4, 16)] = rng.integers(0, 200)
    return E


def test_struct_layout_and_limit(tw):
    Cc = tw.tw_intensity_cell
    assert C.sizeof(Cc) == 16
    assert (Cc.x.offset, Cc.y.offset, Cc.n_pixels.offset, Cc.residual.offset) == (0, 4, 8, 12)
    src = open(tw.api.HEADER_PATH).read()
    assert int(re.search(r"#define\s+TW_MAX_INTENSITY_CELLS\s+(\d+)", src).group(1)) == tw.MAX_INTENSITY_CELLS == 4096


def test_abi_declares_exports_and_binds_the_cell_entry_points(tw):
    src = re.sub(r"/\*.*?\*/", "", open(tw.api.HEADER_PATH).read(), flags=re.S)
    protos = {m.group(1): [a.strip() for a in m.group(2).split(",")] for m in re.finditer(r"\b(tw_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src)}
    lib = tw.load()
    for name, nargs in {"tw_intensity_cells": 5, "tw_pool_set_intensity": 2, "tw_pool_wait_intensity": 11}.items():
        assert name in tw.declared_symbols() and hasattr(lib, name), name
        assert len(protos[name]) == nargs == len(getattr(lib, name).argtypes), name
    assert protos["tw_pool_wait_intensity"][:8] == protos["tw_pool_wait_regions"]  # tw_pool_wait_regions plus the cells
    assert [a.split()[-1].lstrip("*") for a in protos["tw_intensity_cells"]] == ["ctx", "pair", "out", "cap", "n_cells"]


def test_flat_fill_change_is_flagged():
    E = _page()
    T = E.copy()
    T[10:20, 20:40] = np.clip(T[10:20, 20:40].astype(int) - 40, 0, 255)  # darkened in place: no motion
    cells = intensity_cells(E, T, *_zero(E), 10, 16)
    assert [(c["x"], c["y"]) for c in cells] == [(20, 10), (30, 10)]
    assert all(c["n_pixels"] == 100 and c["residual"] > 16 * 100 for c in cells)
    assert intensity_cells(E, E, *_zero(E), 10, 1) == []
    # the rule is strict: a uniform change of exactly t levels is not flagged, t - 1 is
    F = np.full((20, 20), 100, np.uint8)
    assert intensity_cells(F, F + 16, *_zero(F), 10, 16) == []
    assert len(intensity_cells(F, F + 16, *_zero(F), 10, 15)) == 4


def test_integer_translation_with_the_true_flow_gives_no_cells():
    E = _page(seed=2)
    E[:8], E[-8:], E[:, :8], E[:, -8:] = 230, 230, 230, 230  # a plain margin: what enters the frame matches what left it
    big = np.pad(E, 8, mode="edge")
    T = big[8 - 3:8 - 3 + E.shape[0], 8 + 5:8 + 5 + E.shape[1]]  # T(x, y) = E(x + 5, y - 3)
    fx, fy = np.full(E.shape, -5.0, np.float32), np.full(E.shape, 3.0, np.float32)  # E(p) = T(p + flow)
    assert intensity_cells(E, T, fx, fy, 10, 1) == []
    assert intensity_cells(E, T, *_zero(E), 10, 16) != []  # without the flow the same pair is all change


def test_half_pixel_shift_is_absorbed_by_the_3x3_minimum():
    E = np.zeros((20, 40), np.uint8)
    E[:, 20:] = 200                                       # a vertical step edge
    T = E.copy()
    T[:, 20] = 100                                        # the edge moved half a pixel: its column is half way
    fx, fy = np.full(E.shape, 0.5, np.float32), np.zeros(E.shape, np.float32)  # rounds to 0 (half to even)
    assert intensity_cells(E, T, fx, fy, 10, 0) == []
    fy[:] = -0.5
    assert intensity_cells(E, T, fx, fy, 10, 0) == []
    assert intensity_cells(E, T, *_zero(E), 10, 0) == []


def test_rounding_is_half_to_even():
    E = _page(seed=4)
    E[:, :8], E[:, -8:] = 230, 230
    T = np.roll(E, 3, axis=1)                             # E(x) = T(x + 3): the true shift is 3, and 2 .. 4 are absorbed

    def at(dx):
        return intensity_cells(E, T, np.full(E.shape, dx, np.float32), np.zeros(E.shape, np.float32), 10, 0)
    assert at(1.5) == at(2.5) == at(3.5) == at(4.5) == []  # 2, 2, 4, 4
    assert at(0.5) == at(0.0) == at(-0.5) != []            # 0
    assert at(5.5) == at(6.0) != [] and at(5.5) != at(5.0)  # 6, not 5


def test_ignored_pixels():
    E = np.full((20, 30), 50, np.uint8)
    T = E + 200                                           # every cell changed
    ign = np.zeros(E.shape, bool)
    ign[0:10, 0:10] = True                                # all of cell (0, 0) ignored: never flagged
    ign[0:10, 10:15] = True                               # half of cell (1, 0)
    cells = intensity_cells(E, T, *_zero(E), 10, 16, ign)
    assert cells[0] == {"x": 10, "y": 0, "n_pixels": 50, "residual": 50 * 200}
    assert [(c["x"], c["y"], c["n_pixels"]) for c in cells[1:]] == [(20, 0, 100), (0, 10, 100), (10, 10, 100), (20, 10, 100)]
    # a partly ignored cell uses its own n: a uniform change of 20 levels is a mean of 20 over its 50 pixels
    T2 = E + 20
    assert intensity_cells(E, T2, *_zero(E), 10, 19, ign)[0] == {"x": 10, "y": 0, "n_pixels": 50, "residual": 1000}
    assert intensity_cells(E, T2, *_zero(E), 10, 20, ign) == []
    assert intensity_cells(E, T2, *_zero(E), 10, 19, np.ones(E.shape, bool)) == []


def test_cells_are_cut_at_the_right_and_bottom_edges():
    E = np.full((23, 37), 10, np.uint8)
    T = E + 100
    cells = intensity_cells(E, T, *_zero(E), 10, 50)
    assert [(c["x"], c["y"], c["n_pixels"]) for c in cells] == [
        (0, 0, 100), (10, 0, 100), (20, 0, 100), (30, 0, 70),
        (0, 10, 100), (10, 10, 100), (20, 10, 100), (30, 10, 70),
        (0, 20, 30), (10, 20, 30), (20, 20, 30), (30, 20, 21)]
    assert all(c["residual"] == 100 * c["n_pixels"] for c in cells)
    # a span larger than the frame: one cell, the whole frame
    assert intensity_cells(E, T, *_zero(E), 64, 50) == [{"x": 0, "y": 0, "n_pixels": 23 * 37, "residual": 100 * 23 * 37}]


def test_shifts_are_clamped_at_the_frame():
    E = np.zeros((10, 10), np.uint8)
    T = np.zeros((10, 10), np.uint8)
    T[:, 9] = 200                                         # only the last column of the target is bright
    E[:, :] = 200
    fx = np.full(E.shape, 1e9, np.float32)                # clamped to W, then to the last column
    fy = np.full(E.shape, -1e9, np.float32)
    assert intensity_cells(E, T, fx, fy, 10, 0) == []
    fx[:] = -1e9                                          # the first column: all dark
    assert intensity_cells(E, T, fx, fy, 10, 0) == [{"x": 0, "y": 0, "n_pixels": 100, "residual": 100 * 200}]


def test_non_finite_flow_is_a_zero_shift():
    E = _page(seed=3)
    T = np.roll(E, 4, axis=1)
    zero = intensity_cells(E, T, *_zero(E), 10, 4)
    for bad in (np.nan, np.inf, -np.inf):
        fx = np.full(E.shape, bad, np.float32)
        fy = np.full(E.shape, bad, np.float32)
        assert intensity_cells(E, T, fx, fy, 10, 4) == zero != []
    # only the sample points matter
    fx, fy = _zero(E)
    fx[1::10, :] = 40.0
    assert intensity_cells(E, T, fx, fy, 10, 4) == zero


def test_create_intensity_threshold_option(tw, tmp_path, monkeypatch):
    for v, want in ((16, 16), (1, 1), (255, 255), (0, 0), (256, 0), (-3, 0), (16.0, 0), (True, 0), ("16", 0), (None, 0)):
        assert tw.TidalWave({"intensityThreshold": v}).intensityThreshold == want, v
    assert tw.TidalWave({}).intensityThreshold == 0
    (tmp_path / "t").mkdir()
    (tmp_path / "t" / "a.png").write_bytes(b"x")
    made = []

    class StubPool:
        def __init__(self, *args, **kw):
            made.append(kw.get("intensity_threshold"))
            self.pool = None

        def request_files(self, expected, target, ignore=None, ignore_mask=None):
            return 0

        def wait(self, rid):
            return {"status": "SUSPICIOUS", "n_vectors": 0, "vector": [], "width": 1, "height": 1, "span": 10, "threshold": 5.0,
                    "time": 0.0, "intensity_cells": [{"x": 0, "y": 0, "n_pixels": 1, "residual": 99}], "n_intensity_cells": 1}

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
    for opts, want in (({"intensityThreshold": 16}, 16), ({"intensityThreshold": 300}, 0)):
        ev = []
        t = tw.create(str(tmp_path / "t"), dict(opts, getExpectedPath=lambda s: "/e/" + s))
        t.on("data", ev.append)
        tw.run(t)
        assert made[-1] == want and ev[0]["n_intensity_cells"] == 1 and ev[0]["status"] == "SUSPICIOUS"
