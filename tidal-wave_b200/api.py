"""ctypes binding of include/tidalwave_b200.h + the host-side mirror of the reference's operator interface.

Mirrors, with the same names / argument meaning / error behaviour:
  * ``OpticalFlowParameter``      /root/reference/src/opticalflow.h:28-36 (defaults: src/broker.cpp:106-117)
  * ``OpticalFlow.calculate``     /root/reference/src/opticalflow.cpp:20-76 (decoded images instead of paths)
  * ``Consumer.run`` response     /root/reference/src/consumer.cpp:59-88 -> dict shaped like src/broker.cpp:161-188
  * ``Manager`` / ``TidalWave``   /root/reference/src/manager.cpp:40-98 -> ``Pool``

There is NO CPU fallback: importing works anywhere (symbol checks), but every compute call needs the CUDA
library and a B200; ``load()`` raises if libtidalwave_b200.so is missing.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TW_LIB") or os.path.join(_HERE, "libtidalwave_b200.so")  # TW_LIB: development builds (tools/timeline.py)
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "tidalwave_b200.h")

OK, BAD_PARAMETER, BAD_IMAGE_FORMAT, DONT_MATCH_SIZE, CUDA_ERROR, UNSUPPORTED = range(6)
STATUS_NAMES = {0: "OK", 1: "SUSPICIOUS", 2: "ERROR"}
MAX_IGNORE = 32  # TW_MAX_IGNORE: ignore regions per pair
MAX_CHANGE_REGIONS = 1024  # TW_MAX_CHANGE_REGIONS: change regions stored per pair
MAX_INTENSITY_CELLS = 4096  # TW_MAX_INTENSITY_CELLS: intensity cells stored per pair


class tw_flow_param(C.Structure):
    _fields_ = [("pyrScale", C.c_double), ("pyrLevels", C.c_int), ("winSize", C.c_int), ("pyrIterations", C.c_int),
                ("polyN", C.c_int), ("polySigma", C.c_double), ("flags", C.c_int)]


class tw_vector(C.Structure):
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("dx", C.c_double), ("dy", C.c_double)]


class tw_result(C.Structure):
    _fields_ = [("code", C.c_int), ("status", C.c_int), ("n_vectors", C.c_int), ("width", C.c_int), ("height", C.c_int),
                ("time", C.c_float), ("reason", C.c_char * 128)]


class tw_rect(C.Structure):
    """An ignore region in expected-image pixels: [x, x + width) x [y, y + height)."""
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("width", C.c_int), ("height", C.c_int)]


class tw_change_region(C.Structure):
    """A change region: the bounding box of a connected group of suspicious sample points (expected-image pixels), their count
    and the vector with the largest length among them (include/tidalwave_b200.h, tw_change_regions)."""
    _fields_ = [("rect", tw_rect), ("n_vectors", C.c_int), ("peak", tw_vector)]


class tw_intensity_cell(C.Structure):
    """An intensity cell: a span cell whose pixels changed where the flow found no motion -- its sample point, its n pixels that
    are not ignored and the sum S of their residuals (include/tidalwave_b200.h, tw_intensity_cells)."""
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("n_pixels", C.c_int), ("residual", C.c_int)]


def _cell_dicts(cells, n) -> list[dict]:
    return [{"x": c.x, "y": c.y, "n_pixels": c.n_pixels, "residual": c.residual} for c in cells[:n]]


def _region_dicts(regs, n) -> list[dict]:
    return [{"x": r.rect.x, "y": r.rect.y, "width": r.rect.width, "height": r.rect.height, "n_vectors": r.n_vectors,
             "peak": {"x": r.peak.x, "y": r.peak.y, "dx": r.peak.dx, "dy": r.peak.dy}} for r in regs[:n]]


def _int(v) -> int:
    if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
        raise ValueError(f"bad ignore region: {v!r} is not an integer")
    return int(v)


def rect(region) -> tuple:
    """An ignore region given as an ``(x, y, w, h)`` tuple or a ``{x, y, width, height}`` dict -> ``(x, y, w, h)`` ints.
    Raises ValueError for anything else; sizes and counts are checked by the library (TW_BAD_PARAMETER)."""
    if isinstance(region, dict):
        try:
            vals = [region[k] for k in ("x", "y", "width", "height")]
        except KeyError as e:
            raise ValueError(f"bad ignore region: {region!r} lacks {e.args[0]!r}") from None
    elif isinstance(region, (tuple, list)) and len(region) == 4:
        vals = list(region)
    else:
        raise ValueError(f"bad ignore region: {region!r} (an (x, y, w, h) tuple or an {{x, y, width, height}} dict)")
    return tuple(_int(v) for v in vals)


def _rects(regions):
    """-> (tw_rect array or None, count) for a list of regions (None or empty: no regions)."""
    rs = [rect(r) for r in (regions or [])]
    return ((tw_rect * len(rs))(*[tw_rect(*r) for r in rs]) if rs else None), len(rs)


def mask_size_error(mask_shape, expect_shape) -> str:
    """The library's reason for a mask of the wrong size (include/tidalwave_b200.h, tw_compare_mask)."""
    (mh, mw), (eh, ew) = mask_shape, expect_shape
    return f"bad ignore mask: {mw}x{mh} mask for a {ew}x{eh} expected image"


def mask_array(mask):
    """An ignore mask (2-D ``uint8`` or ``bool`` array in expected-image pixels, nonzero / True = ignore) -> a C-contiguous
    ``uint8`` array, or None for None.  Raises ValueError for anything else; the size is checked against the expected image by the
    callers (``mask_size_error``)."""
    if mask is None:
        return None
    if not isinstance(mask, np.ndarray) or mask.ndim != 2 or mask.dtype not in (np.uint8, np.bool_):
        raise ValueError(f"bad ignore mask: a 2-D uint8 or bool array expected, not {type(mask).__name__}"
                         + (f" {mask.dtype} {mask.shape}" if isinstance(mask, np.ndarray) else ""))
    return np.ascontiguousarray(mask.view(np.uint8) if mask.dtype == np.bool_ else mask)


@dataclass
class OpticalFlowParameter:
    pyrScale: float = 0.5
    pyrLevels: int = 3
    winSize: int = 30
    pyrIterations: int = 3
    polyN: int = 7
    polySigma: float = 1.5
    flags: int = 256

    def c(self) -> tw_flow_param:
        return tw_flow_param(self.pyrScale, self.pyrLevels, self.winSize, self.pyrIterations, self.polyN, self.polySigma,
                             self.flags)


_lib = None


def load() -> C.CDLL:
    """Loads the CUDA library; fails loudly (no fallback) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    u8pp = C.POINTER(C.c_void_p)
    L.tw_version.restype = C.c_char_p
    L.tw_last_error.restype = C.c_char_p
    L.tw_last_error.argtypes = [C.c_void_p]
    L.tw_create.restype = C.c_void_p
    L.tw_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]
    L.tw_destroy.argtypes = [C.c_void_p]
    L.tw_flow.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(tw_flow_param),
                          C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
    L.tw_compare.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                             C.POINTER(tw_flow_param), C.c_double, C.c_int, C.POINTER(tw_vector), C.c_int,
                             C.POINTER(tw_result)]
    L.tw_compare_batch.argtypes = [C.c_void_p, C.c_int, u8pp, u8pp, C.c_int, C.c_int, C.c_int, C.POINTER(tw_flow_param),
                                   C.c_double, C.c_int, C.POINTER(tw_vector), C.c_int, C.POINTER(tw_result)]
    rpp = C.POINTER(C.POINTER(tw_rect))
    L.tw_compare_ignore.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                    C.POINTER(tw_flow_param), C.c_double, C.c_int, C.POINTER(tw_rect), C.c_int,
                                    C.POINTER(tw_vector), C.c_int, C.POINTER(tw_result)]
    L.tw_compare_batch_ignore.argtypes = [C.c_void_p, C.c_int, u8pp, u8pp, C.c_int, C.c_int, C.c_int, C.POINTER(tw_flow_param),
                                          C.c_double, C.c_int, rpp, C.POINTER(C.c_int), C.POINTER(tw_vector), C.c_int,
                                          C.POINTER(tw_result)]
    L.tw_compare_mask.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                  C.POINTER(tw_flow_param), C.c_double, C.c_int, C.POINTER(tw_rect), C.c_int, C.c_void_p,
                                  C.POINTER(tw_vector), C.c_int, C.POINTER(tw_result)]
    L.tw_compare_batch_mask.argtypes = [C.c_void_p, C.c_int, u8pp, u8pp, C.c_int, C.c_int, C.c_int, C.POINTER(tw_flow_param),
                                        C.c_double, C.c_int, rpp, C.POINTER(C.c_int), u8pp, C.POINTER(tw_vector), C.c_int,
                                        C.POINTER(tw_result)]
    L.tw_pipe_submit.argtypes = [C.c_void_p, C.c_int, u8pp, u8pp, C.c_int, C.c_int, C.c_int, C.POINTER(tw_flow_param), C.c_double, C.c_int]
    L.tw_pipe_submit_ignore.argtypes = [C.c_void_p, C.c_int, u8pp, u8pp, C.c_int, C.c_int, C.c_int, C.POINTER(tw_flow_param),
                                        C.c_double, C.c_int, rpp, C.POINTER(C.c_int)]
    L.tw_pipe_submit_mask.argtypes = [C.c_void_p, C.c_int, u8pp, u8pp, C.c_int, C.c_int, C.c_int, C.POINTER(tw_flow_param),
                                      C.c_double, C.c_int, rpp, C.POINTER(C.c_int), u8pp]
    L.tw_change_regions.argtypes = [C.c_void_p, C.c_int, C.POINTER(tw_change_region), C.c_int, C.POINTER(C.c_int)]
    L.tw_intensity_cells.argtypes = [C.c_void_p, C.c_int, C.POINTER(tw_intensity_cell), C.c_int, C.POINTER(C.c_int)]
    L.tw_pipe_collect.argtypes = [C.c_void_p, C.POINTER(tw_vector), C.c_int, C.POINTER(tw_result)]
    L.tw_pipe_pending.argtypes = [C.c_void_p]
    L.tw_pipe_ready.argtypes = [C.c_void_p]
    L.tw_batch_upload.argtypes = [C.c_void_p, C.c_int, u8pp, u8pp, C.c_int, C.c_int, C.c_int]
    L.tw_batch_run.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(tw_flow_param), C.c_double, C.c_int]
    L.tw_batch_fetch.argtypes = [C.c_void_p, C.c_int, C.POINTER(tw_vector), C.c_int, C.POINTER(tw_result)]
    L.tw_resize_target.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]
    L.tw_decode_gray.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.tw_sync.argtypes = [C.c_void_p]
    L.tw_batch_flow.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.tw_host_alloc.restype = C.c_void_p
    L.tw_host_alloc.argtypes = [C.c_size_t]
    L.tw_host_free.argtypes = [C.c_void_p]
    L.tw_l2_flush.argtypes = [C.c_void_p]
    L.tw_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    L.tw_set_default_arithmetic.argtypes = [C.c_int]
    L.tw_arithmetic_in_effect.argtypes = [C.c_void_p, C.POINTER(tw_flow_param)]
    L.tw_timer_start.argtypes = [C.c_void_p]
    L.tw_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    L.tw_profile_enable.argtypes = [C.c_void_p, C.c_int]
    L.tw_profile_read.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_float), C.POINTER(C.c_int),
                                  C.POINTER(C.c_double)]
    L.tw_launch_count.restype = C.c_longlong
    L.tw_launch_count.argtypes = [C.c_void_p]
    L.tw_debug_read.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int),
                                C.POINTER(C.c_int)]
    L.tw_debug_keep_levels.argtypes = [C.c_void_p, C.c_int]
    L.tw_pool_create.restype = C.c_void_p
    L.tw_pool_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(tw_flow_param),
                                 C.c_double, C.c_int, C.c_int, C.c_char_p, C.c_int]
    L.tw_pool_submit.restype = C.c_longlong
    L.tw_pool_submit.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]
    L.tw_pool_submit_files.restype = C.c_longlong
    L.tw_pool_submit_files.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
    L.tw_pool_submit_ignore.restype = C.c_longlong
    L.tw_pool_submit_ignore.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                        C.POINTER(tw_rect), C.c_int]
    L.tw_pool_submit_files_ignore.restype = C.c_longlong
    L.tw_pool_submit_files_ignore.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.POINTER(tw_rect), C.c_int]
    L.tw_pool_submit_mask.restype = C.c_longlong
    L.tw_pool_submit_mask.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                      C.POINTER(tw_rect), C.c_int, C.c_void_p]
    L.tw_pool_submit_files_mask.restype = C.c_longlong
    L.tw_pool_submit_files_mask.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(tw_rect), C.c_int]
    L.tw_pool_set_decoders.argtypes = [C.c_void_p, C.c_int]
    L.tw_pool_peek.argtypes = [C.c_void_p, C.c_longlong, C.POINTER(tw_result)]
    L.tw_pool_wait.argtypes = [C.c_void_p, C.c_longlong, C.POINTER(tw_vector), C.c_int, C.POINTER(tw_result)]
    L.tw_pool_set_change_regions.argtypes = [C.c_void_p, C.c_int]
    L.tw_pool_wait_regions.argtypes = [C.c_void_p, C.c_longlong, C.POINTER(tw_vector), C.c_int, C.POINTER(tw_result),
                                       C.POINTER(tw_change_region), C.c_int, C.POINTER(C.c_int)]
    L.tw_pool_set_intensity.argtypes = [C.c_void_p, C.c_int]
    L.tw_pool_wait_intensity.argtypes = [C.c_void_p, C.c_longlong, C.POINTER(tw_vector), C.c_int, C.POINTER(tw_result),
                                         C.POINTER(tw_change_region), C.c_int, C.POINTER(C.c_int), C.POINTER(tw_intensity_cell),
                                         C.c_int, C.POINTER(C.c_int)]
    L.tw_pool_poll.argtypes = [C.c_void_p, C.c_longlong, C.POINTER(tw_vector), C.c_int, C.POINTER(tw_result)]
    L.tw_pool_report.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.tw_pool_stop.argtypes = [C.c_void_p]
    L.tw_pool_destroy.argtypes = [C.c_void_p]
    _lib = L
    return L


def set_default_arithmetic(relaxed: bool) -> None:
    """Process-wide default of the "arithmetic" option for contexts created afterwards (pool consumers included):
    False = faithful (SURVEY App. A operation order), True = relaxed where validated (include/tidalwave_b200.h)."""
    load().tw_set_default_arithmetic(1 if relaxed else 0)


def declared_symbols() -> list[str]:
    """Every function include/tidalwave_b200.h declares (for the export check)."""
    import re
    src = open(HEADER_PATH).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tw_[a-z0-9_]+)\s*\(", src)))


def imread_gray(path: str):
    """cv::imread(path, IMREAD_GRAYSCALE) (/root/reference/src/opticalflow.cpp:37,44) through tw_decode_gray: PNG / JPEG / PGM.
    Returns None (an "empty Mat") for a missing file or a format this build cannot decode bit-exactly (e.g. CMYK or
    arithmetic-coded JPEG)."""
    try:
        data = open(path, "rb").read()
    except OSError:
        return None
    L = load()
    w = C.c_int(); h = C.c_int()
    if not data or L.tw_decode_gray(data, len(data), None, 0, C.byref(w), C.byref(h)) != 0:
        return None
    out = np.empty((h.value, w.value), np.uint8)
    if L.tw_decode_gray(data, len(data), out.ctypes.data, out.size, C.byref(w), C.byref(h)) != 0:
        return None
    return out


def _u8(img) -> np.ndarray:
    a = np.ascontiguousarray(img, dtype=np.uint8)
    if a.ndim != 2:
        raise ValueError("8-bit single-channel image expected")
    return a


def _response(res: tw_result, vecs, n, span, threshold, expect_image="", target_image="") -> dict:
    """Response -> the object of Broker::convertResult (/root/reference/src/broker.cpp:161-188); error shape :57-70."""
    if res.status == 2:
        return {"status": "ERROR", "reason": res.reason.decode(), "code": res.code}
    return {"status": STATUS_NAMES[res.status], "span": span, "threshold": threshold, "expect_image": expect_image,
            "target_image": target_image, "time": float(res.time), "height": res.height, "width": res.width,
            "vector": [{"x": vecs[i].x, "y": vecs[i].y, "dx": vecs[i].dx, "dy": vecs[i].dy} for i in range(n)],
            "n_vectors": res.n_vectors}


class OpticalFlow:
    """One operator instance per consumer thread / device (src/consumer.cpp:27-35)."""

    def __init__(self, device: int = 0, max_w: int = 1920, max_h: int = 1080, max_batch: int = 1):
        self.lib = load()
        err = C.create_string_buffer(256)
        self.ctx = self.lib.tw_create(device, max_w, max_h, max_batch, err, 256)
        if not self.ctx:
            raise RuntimeError("tw_create failed: " + err.value.decode())
        self.max_batch = max_batch
        self.change_regions = False  # set_option("change_regions", 1): responses carry "regions" and "n_regions"
        self.intensity = 0  # set_option("intensity_threshold", t > 0): responses carry "intensity_cells" and "n_intensity_cells"

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.tw_destroy(self.ctx)
            self.ctx = None

    __del__ = close

    def set_option(self, name: str, value: int):
        if self.lib.tw_set_option(self.ctx, name.encode(), int(value)) != 0:
            raise ValueError(self.last_error())
        if name == "change_regions":
            self.change_regions = bool(value)
        if name == "intensity_threshold":
            self.intensity = int(value)

    def regions(self, pair: int = 0):
        """(regions as dicts, n_regions) of pair ``pair`` of the last answered batch (tw_change_regions); raises ValueError if that
        batch ran without the "change_regions" option."""
        regs = (tw_change_region * MAX_CHANGE_REGIONS)()
        n = C.c_int()
        if self.lib.tw_change_regions(self.ctx, pair, regs, MAX_CHANGE_REGIONS, C.byref(n)) != 0:
            raise ValueError(self.last_error())
        return _region_dicts(regs, min(n.value, MAX_CHANGE_REGIONS)), n.value

    def intensity_cells(self, pair: int = 0):
        """(intensity cells as dicts, n_cells) of pair ``pair`` of the last answered batch (tw_intensity_cells); raises ValueError if
        that batch ran without the "intensity_threshold" option."""
        cells = (tw_intensity_cell * MAX_INTENSITY_CELLS)()
        n = C.c_int()
        if self.lib.tw_intensity_cells(self.ctx, pair, cells, MAX_INTENSITY_CELLS, C.byref(n)) != 0:
            raise ValueError(self.last_error())
        return _cell_dicts(cells, min(n.value, MAX_INTENSITY_CELLS)), n.value

    def _with_regions(self, resp: dict, pair: int) -> dict:
        if self.change_regions and resp["status"] != "ERROR":
            resp["regions"], resp["n_regions"] = self.regions(pair)
        if self.intensity and resp["status"] != "ERROR":
            resp["intensity_cells"], resp["n_intensity_cells"] = self.intensity_cells(pair)
        return resp

    def last_error(self) -> str:
        return self.lib.tw_last_error(self.ctx).decode()

    def arithmetic_in_effect(self, param: "OpticalFlowParameter" = None) -> str:
        """'relaxed' or 'faithful': which kernels `param` runs on this context."""
        p = (param or OpticalFlowParameter()).c()
        return "relaxed" if self.lib.tw_arithmetic_in_effect(self.ctx, C.byref(p)) == 1 else "faithful"

    def calculateInternal(self, expectImg, targetImg, param: OpticalFlowParameter = OpticalFlowParameter()):
        """-> (code, flowx, flowy, seconds); src/opticalflow.cpp:78-119."""
        a, b = _u8(expectImg), _u8(targetImg)
        if a.shape != b.shape:
            raise ValueError("calculateInternal needs equal-size images (calculate() applies the size rule)")
        h, w = a.shape
        fx = np.empty((h, w), np.float32); fy = np.empty((h, w), np.float32)
        sec = C.c_float(0)
        p = param.c()
        rc = self.lib.tw_flow(self.ctx, a.ctypes.data, b.ctypes.data, w, h, w, C.byref(p), fx.ctypes.data, fy.ctypes.data,
                              C.byref(sec))
        return rc, fx, fy, sec.value

    def calculate(self, expectImg, targetImg, param: OpticalFlowParameter = OpticalFlowParameter(), threshold: float = 5.0,
                  span: int = 10, cap: int | None = None, expect_image: str = "", target_image: str = "", ignore=None,
                  ignore_mask=None) -> dict:
        """calculate + Consumer::run's sampling -> response dict (src/opticalflow.cpp:20-76, src/consumer.cpp:59-88).
        ignore: regions of the expected image left out of the comparison (``(x, y, w, h)`` tuples or ``{x, y, width, height}``
        dicts, at most MAX_IGNORE; include/tidalwave_b200.h, tw_compare_ignore).  ignore_mask: pixels of the expected image left
        out of the comparison, a 2-D ``uint8`` or ``bool`` array of the expected image's shape, nonzero = ignore (tw_compare_mask);
        a mask of another shape answers an ERROR response "bad ignore mask: ..."."""
        a = None if expectImg is None else _u8(expectImg)
        b = None if targetImg is None else _u8(targetImg)
        eh, ew = a.shape if a is not None else (0, 0)
        th, tw = b.shape if b is not None else (0, 0)
        if cap is None:
            cap = max(1, ((ew + span - 1) // max(span, 1)) * ((eh + span - 1) // max(span, 1))) if span > 0 else 1
        vec = (tw_vector * cap)()
        res = tw_result()
        p = param.c()
        m = mask_array(ignore_mask)
        if m is not None and a is not None and m.shape != a.shape:
            return {"status": "ERROR", "reason": mask_size_error(m.shape, a.shape), "code": BAD_PARAMETER}
        if m is not None:
            rs, nr = _rects(ignore)
            self.lib.tw_compare_mask(self.ctx, a.ctypes.data if a is not None else None, ew, eh,
                                     b.ctypes.data if b is not None else None, tw, th, C.byref(p), threshold, span, rs, nr,
                                     m.ctypes.data, vec, cap, C.byref(res))
        elif ignore is None:
            self.lib.tw_compare(self.ctx, a.ctypes.data if a is not None else None, ew, eh,
                                b.ctypes.data if b is not None else None, tw, th, C.byref(p), threshold, span, vec, cap,
                                C.byref(res))
        else:
            rs, nr = _rects(ignore)
            self.lib.tw_compare_ignore(self.ctx, a.ctypes.data if a is not None else None, ew, eh,
                                       b.ctypes.data if b is not None else None, tw, th, C.byref(p), threshold, span, rs, nr,
                                       vec, cap, C.byref(res))
        return self._with_regions(_response(res, vec, min(res.n_vectors, cap), span, threshold, expect_image, target_image), 0)

    def calculate_batch(self, pairs, param: OpticalFlowParameter = OpticalFlowParameter(), threshold: float = 5.0,
                        span: int = 10, cap: int | None = None, ignore=None, ignore_mask=None) -> list[dict]:
        """ignore: one region list (or None) per pair, as in calculate().  ignore_mask: one mask (or None) per pair, as in
        calculate(); a mask of another shape than the pairs' answers every pair with ERROR "bad ignore mask: ..." (as a bad region
        list does)."""
        n = len(pairs)
        imgs = [(_u8(a), _u8(b)) for a, b in pairs]
        h, w = imgs[0][0].shape
        if cap is None:
            cap = ((w + span - 1) // span) * ((h + span - 1) // span)
        ex = (C.c_void_p * n)(*[a.ctypes.data for a, _ in imgs])
        tg = (C.c_void_p * n)(*[b.ctypes.data for _, b in imgs])
        vec = (tw_vector * (cap * n))()
        res = (tw_result * n)()
        p = param.c()
        if ignore is not None and len(ignore) != n:
            raise ValueError("ignore: one region list per pair")
        if ignore_mask is not None and len(ignore_mask) != n:
            raise ValueError("ignore_mask: one mask (or None) per pair")
        masks = [mask_array(m) for m in ignore_mask] if ignore_mask is not None else None
        for m in masks or []:
            if m is not None and m.shape != (h, w):
                return [{"status": "ERROR", "reason": mask_size_error(m.shape, (h, w)), "code": BAD_PARAMETER} for _ in range(n)]
        if ignore is None and masks is None:
            self.lib.tw_compare_batch(self.ctx, n, ex, tg, w, h, w, C.byref(p), threshold, span, vec, cap, res)
        else:
            lists = [_rects(g) for g in ignore] if ignore is not None else None
            ig = (C.POINTER(tw_rect) * n)(*[C.cast(rs, C.POINTER(tw_rect)) if rs is not None else None for rs, _ in lists]) if lists else None
            nig = (C.c_int * n)(*[k for _, k in lists]) if lists else None
            if masks is None:
                self.lib.tw_compare_batch_ignore(self.ctx, n, ex, tg, w, h, w, C.byref(p), threshold, span, ig, nig, vec, cap, res)
            else:
                mk = (C.c_void_p * n)(*[m.ctypes.data if m is not None else None for m in masks])
                self.lib.tw_compare_batch_mask(self.ctx, n, ex, tg, w, h, w, C.byref(p), threshold, span, ig, nig, mk, vec, cap, res)
        out = []
        for i in range(n):
            sub = (tw_vector * cap).from_buffer(vec, i * cap * C.sizeof(tw_vector))
            out.append(self._with_regions(_response(res[i], sub, min(res[i].n_vectors, cap), span, threshold), i))
        return out

    def batch_flow(self, pair: int, w: int, h: int):
        fx = np.empty((h, w), np.float32); fy = np.empty((h, w), np.float32)
        rc = self.lib.tw_batch_flow(self.ctx, pair, fx.ctypes.data, fy.ctypes.data)
        if rc != 0:
            raise RuntimeError("tw_batch_flow: " + self.last_error())
        return fx, fy

    def debug_keep_levels(self, on: bool = True):
        self.lib.tw_debug_keep_levels(self.ctx, int(on))

    def debug_read(self, name: str, scale: int, pair: int = 0, max_floats: int = 5 * 4096 * 2304):
        buf = np.empty(max_floats, np.float32)
        w = C.c_int(); h = C.c_int()
        cn = self.lib.tw_debug_read(self.ctx, name.encode(), scale, pair, buf.ctypes.data, max_floats, C.byref(w), C.byref(h))
        if cn < 0:
            raise RuntimeError(f"tw_debug_read({name}, {scale}) -> {cn}")
        return buf[:cn * w.value * h.value].reshape(cn, h.value, w.value).copy()

    def profile(self, on: bool):
        self.lib.tw_profile_enable(self.ctx, int(on))

    def profile_read(self) -> dict:
        n = 16
        names = (C.c_char_p * n)(); ms = (C.c_float * n)(); ln = (C.c_int * n)(); by = (C.c_double * n)()
        k = self.lib.tw_profile_read(self.ctx, n, names, ms, ln, by)
        return {names[i].decode(): dict(ms=ms[i], launches=ln[i], alg_bytes=by[i]) for i in range(min(k, n))}

    def launch_count(self) -> int:
        return int(self.lib.tw_launch_count(self.ctx))


class Pool:
    """Manager + Consumer pool (src/manager.cpp:40-98): one consumer thread per entry of ``devices``."""

    def __init__(self, devices, param: OpticalFlowParameter = OpticalFlowParameter(), threshold: float = 5.0, span: int = 10,
                 max_w: int = 0, max_h: int = 0, batch: int = 1, vector_cap: int = 0, change_regions: bool = False,
                 intensity_threshold: int = 0):
        """max_w / max_h = 0: no bound on the image size; vector_cap = 0: every vector of every request is returned (the capacity
        follows each request's own sampling grid), > 0: at most that many (``n_vectors`` still holds the full count).
        change_regions: wait() answers also carry "regions" and "n_regions" (tw_pool_set_change_regions), whatever vector_cap is.
        intensity_threshold: t in 1 .. 255 gray levels adds "intensity_cells" and "n_intensity_cells" (tw_pool_set_intensity); 0 off."""
        self.lib = load()
        self.span, self.threshold, self.cap = span, threshold, vector_cap
        err = C.create_string_buffer(256)
        dv = (C.c_int * len(devices))(*devices)
        p = param.c()
        self.pool = self.lib.tw_pool_create(dv, len(devices), max_w, max_h, batch, C.byref(p), threshold, span, vector_cap,
                                            err, 256)
        if not self.pool:
            raise RuntimeError("tw_pool_create failed: " + err.value.decode())
        self.change_regions = bool(change_regions)
        if self.change_regions:
            if self.lib.tw_pool_set_change_regions(self.pool, 1) != OK:
                self.close()
                raise RuntimeError("tw_pool_set_change_regions refused: the pool has taken requests already")
        self.intensity = int(intensity_threshold)
        if self.intensity:
            if self.lib.tw_pool_set_intensity(self.pool, self.intensity) != OK:
                self.close()
                raise ValueError(f"tw_pool_set_intensity refused {intensity_threshold!r}: 0 (off) or 1 .. 255 gray levels")
        self._keep = {}

    def request(self, expectImg, targetImg, ignore=None, ignore_mask=None) -> int:
        """Manager::request (src/manager.cpp:68-78).  ignore / ignore_mask: regions and pixels left out of the comparison, as in
        OpticalFlow.calculate; a mask of another shape than the expected image raises ValueError "bad ignore mask: ..." (no
        request is made)."""
        a = None if expectImg is None else _u8(expectImg)
        b = None if targetImg is None else _u8(targetImg)
        eh, ew = a.shape if a is not None else (0, 0)
        th, tw = b.shape if b is not None else (0, 0)
        m = mask_array(ignore_mask)
        if m is not None and m.shape != (eh, ew):
            raise ValueError(mask_size_error(m.shape, (eh, ew)))
        if m is not None:
            rs, nr = _rects(ignore)
            rid = self.lib.tw_pool_submit_mask(self.pool, a.ctypes.data if a is not None else None, ew, eh,
                                               b.ctypes.data if b is not None else None, tw, th, rs, nr, m.ctypes.data)
        elif ignore is None:
            rid = self.lib.tw_pool_submit(self.pool, a.ctypes.data if a is not None else None, ew, eh,
                                          b.ctypes.data if b is not None else None, tw, th)
        else:
            rs, nr = _rects(ignore)
            rid = self.lib.tw_pool_submit_ignore(self.pool, a.ctypes.data if a is not None else None, ew, eh,
                                                 b.ctypes.data if b is not None else None, tw, th, rs, nr)
        if rid >= 0:
            self._keep[rid] = (a, b, m)
        return rid

    def request_files(self, expect_path: str, target_path: str, ignore=None, ignore_mask=None) -> int:
        """Manager::request with two image paths (src/manager.cpp:68-78): read + decoded on the pool's C++ decoder threads.
        ignore_mask: the path of a mask image (decoded to gray like the images, nonzero = ignore; include/tidalwave_b200.h,
        tw_pool_submit_files_mask) or None."""
        if ignore_mask is not None:
            rs, nr = _rects(ignore)
            return self.lib.tw_pool_submit_files_mask(self.pool, (expect_path or "").encode(), (target_path or "").encode(),
                                                      os.fsencode(ignore_mask), rs, nr)
        if ignore is None:
            return self.lib.tw_pool_submit_files(self.pool, (expect_path or "").encode(), (target_path or "").encode())
        rs, nr = _rects(ignore)
        return self.lib.tw_pool_submit_files_ignore(self.pool, (expect_path or "").encode(), (target_path or "").encode(), rs, nr)

    def wait(self, rid: int) -> dict | None:
        cap = self.cap
        if cap <= 0:  # all vectors: the request's own sampling grid (src/consumer.cpp:60-76)
            a = self._keep.get(rid, (None,))[0]
            if a is not None:
                eh, ew = a.shape
                cap = max(1, ((ew + self.span - 1) // self.span) * ((eh + self.span - 1) // self.span))
            else:  # path-based request: ask how many vectors there are
                info = tw_result()
                if self.lib.tw_pool_peek(self.pool, rid, C.byref(info)) < 0:
                    return None
                cap = max(1, info.n_vectors)
        vec = (tw_vector * cap)()
        res = tw_result()
        if not self.change_regions and not self.intensity:
            rc = self.lib.tw_pool_wait(self.pool, rid, vec, cap, C.byref(res))
        elif not self.intensity:
            regs = (tw_change_region * MAX_CHANGE_REGIONS)()
            nreg = C.c_int()
            rc = self.lib.tw_pool_wait_regions(self.pool, rid, vec, cap, C.byref(res), regs, MAX_CHANGE_REGIONS, C.byref(nreg))
        else:
            regs = (tw_change_region * MAX_CHANGE_REGIONS)() if self.change_regions else None
            nreg = C.c_int()
            cells = (tw_intensity_cell * MAX_INTENSITY_CELLS)()
            ncell = C.c_int()
            rc = self.lib.tw_pool_wait_intensity(self.pool, rid, vec, cap, C.byref(res), regs,
                                                 MAX_CHANGE_REGIONS if self.change_regions else 0, C.byref(nreg), cells,
                                                 MAX_INTENSITY_CELLS, C.byref(ncell))
        self._keep.pop(rid, None)
        if rc < 0:
            return None
        resp = _response(res, vec, min(res.n_vectors, cap), self.span, self.threshold)
        if self.change_regions and resp["status"] != "ERROR":
            resp["regions"], resp["n_regions"] = _region_dicts(regs, min(nreg.value, MAX_CHANGE_REGIONS)), nreg.value
        if self.intensity and resp["status"] != "ERROR":
            resp["intensity_cells"], resp["n_intensity_cells"] = _cell_dicts(cells, min(ncell.value, MAX_INTENSITY_CELLS)), ncell.value
        return resp

    def report(self) -> dict:
        a = C.c_int(); b = C.c_int(); c = C.c_int()
        self.lib.tw_pool_report(self.pool, C.byref(a), C.byref(b), C.byref(c))
        return {"request": a.value, "data": b.value, "error": c.value}  # src/broker.cpp:76-78

    def stop(self):
        if self.pool:
            self.lib.tw_pool_stop(self.pool)

    def close(self):
        if getattr(self, "pool", None):
            self.lib.tw_pool_destroy(self.pool)
            self.pool = None

    __del__ = close
