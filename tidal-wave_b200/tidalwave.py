"""JS-level API of the reference (SURVEY row f-3): ``create(targetDir, options)`` -> emitter of 'data' / 'error' / 'finish'.

Mirrors /root/reference/index.js:14-73 (directory pairing + lifecycle) and the option parsing of
Broker::createInstance (/root/reference/src/broker.cpp:101-123, typed defaults :106-117, wrong-typed keys silently fall back
to the default :190-209) on top of the dispatcher (tw_pool_*).  Two options of this port have no reference counterpart:
``ignoreRegions`` (a list of ``{x, y, width, height}`` in expected-image pixels, for every pair) and ``getIgnoreRegions(shortPath)``
(a callable like ``getExpectedPath`` returning a pair's own list, or something falsy): parts of the page that are expected to change
and are left out of the comparison (include/tidalwave_b200.h, tw_compare_ignore).  A pair's regions are the union of the two; a
malformed region makes that pair an 'error' event rather than a comparison of the region it asked to ignore.  Ignore masks (per-pixel,
nonzero = ignore, the expected image's size; tw_compare_mask) come from ``ignoreMaskDir`` (a directory holding a mask image at the same
short path as the target; a pair with no file there has no mask) or, if that is not a string, from ``getIgnoreMaskPath(shortPath)``
(a callable returning a mask path, or something falsy for none).  A pair's mask and regions are ignored together; a mask file that
cannot be decoded, or of another size than the expected image, makes that pair an 'error' event.  Wrong-typed values of these
options mean "no mask", as for the reference's options.  ``changeRegions`` (only ``True`` turns it on) adds ``regions`` and
``n_regions`` to every 'data' event: where the page changed, as connected groups of its suspicious sample points
(include/tidalwave_b200.h, tw_change_regions).  ``intensityThreshold`` (an integer from 1 to 255 gray levels; anything else
leaves it off) adds ``intensity_cells`` and ``n_intensity_cells`` to every 'data' event and makes a pair with intensity cells
SUSPICIOUS: the span cells whose pixels changed where the flow found no motion (tw_intensity_cells).  Files are decoded with ``imread_gray`` (PNG / JPEG / PGM,
bit-exact to cv::imread IMREAD_GRAYSCALE); a file that cannot be decoded becomes the reference's "Can't open <path>" error.
"""
from __future__ import annotations

import glob
import os

from .api import OpticalFlowParameter, Pool, imread_gray, rect


def _number(opts, key, default):
    v = opts.get(key, default)
    return float(v) if isinstance(v, (int, float)) and not isinstance(v, bool) else default  # getNumberOrDefault


def _int32(opts, key, default):
    v = opts.get(key, default)
    return int(v) if isinstance(v, int) and not isinstance(v, bool) else default  # getInt32OrDefault


class TidalWave:
    """The addon's ``TidalWave`` class (src/broker.cpp:29-42): ``calc(expected, target)``, ``dispose()``, events."""

    def __init__(self, options=None, devices=None, batch=8):
        o = options or {}
        self.threshold = _number(o, "threshold", 5.0)
        self.span = _int32(o, "span", 10)
        self.numThreads = _int32(o, "numThreads", 4)
        self.param = OpticalFlowParameter(
            pyrScale=_number(o, "pyrScale", 0.5), pyrLevels=_int32(o, "pyrLevels", 3), winSize=_int32(o, "winSize", 30),
            pyrIterations=_int32(o, "pyrIterations", 3), polyN=_int32(o, "polyN", 7), polySigma=_number(o, "polySigma", 1.5),
            flags=_int32(o, "flags", 256))
        self.ignoreRegions = o.get("ignoreRegions")
        self.getIgnoreRegions = o.get("getIgnoreRegions") if callable(o.get("getIgnoreRegions")) else None
        self.ignoreMaskDir = o.get("ignoreMaskDir") if isinstance(o.get("ignoreMaskDir"), str) else None
        self.getIgnoreMaskPath = o.get("getIgnoreMaskPath") if callable(o.get("getIgnoreMaskPath")) else None
        self.changeRegions = o.get("changeRegions") is True
        t = _int32(o, "intensityThreshold", 0)
        self.intensityThreshold = t if 1 <= t <= 255 else 0
        self._handlers = {"data": [], "error": [], "finish": []}
        self._pending = []   # (request id | None, expect path, target path, immediate error | None)
        self._report = {"request": 0, "data": 0, "error": 0}
        self._devices = devices
        self._batch = batch
        self._pool = None
        self._disposed = False

    # EventEmitter
    def on(self, event, fn):
        self._handlers[event].append(fn)
        return self

    def _emit(self, event, payload):
        for fn in self._handlers[event]:
            fn(payload)

    def _ensure_pool(self, w, h):
        if self._pool is None:
            import ctypes as C
            from .api import load
            ndev = max(1, load().tw_device_count())
            devices = self._devices or [i % ndev for i in range(max(1, self.numThreads))]  # consumer i <-> GPU i % count
            # screenshot directories mix page sizes: no size bound, and every vector of every pair comes back whatever its size
            self._pool = Pool(devices, self.param, self.threshold, self.span, max_w=0, max_h=0, batch=self._batch, vector_cap=0,
                              change_regions=self.changeRegions, intensity_threshold=self.intensityThreshold)
            load().tw_pool_set_decoders(self._pool.pool, max(1, self.numThreads))
        return self._pool

    def ignore_regions(self, shortPath) -> list:
        """The ignore regions of the pair whose target is ``shortPath`` (relative to targetDir): ``ignoreRegions`` followed by
        ``getIgnoreRegions(shortPath)``, as ``(x, y, w, h)`` tuples.  Raises ValueError for a malformed list or region."""
        regions = []
        for src in (self.ignoreRegions, self.getIgnoreRegions(shortPath) if self.getIgnoreRegions else None):
            if not src:
                continue
            if not isinstance(src, (list, tuple)):
                raise ValueError(f"bad ignore region: {src!r} is not a list of regions")
            regions += [rect(r) for r in src]
        return regions

    def ignore_mask_path(self, shortPath):
        """The ignore-mask file of the pair whose target is ``shortPath`` (relative to targetDir), or None: the file at the same short
        path under ``ignoreMaskDir`` if there is one there, else (without ``ignoreMaskDir``) what ``getIgnoreMaskPath(shortPath)``
        returns if it is a non-empty path."""
        if self.ignoreMaskDir is not None:
            path = os.path.abspath(os.path.join(self.ignoreMaskDir, shortPath))
            return path if os.path.isfile(path) else None
        if self.getIgnoreMaskPath is not None:
            path = self.getIgnoreMaskPath(shortPath)
            if isinstance(path, (str, os.PathLike)) and os.fspath(path):
                return os.fspath(path)
        return None

    def reject(self, expected: str, target: str, reason: str):
        """Counts a request that is answered with an 'error' event without being computed."""
        if self._disposed:
            return
        self._report["request"] += 1
        self._pending.append((None, expected, target, reason))

    def calc(self, expected: str, target: str, ignore=None, ignore_mask=None):
        """Broker::requestCalc -> Manager::request (src/broker.cpp:125-150, src/manager.cpp:68-78).  ignore: regions of the
        expected image left out of the comparison (see ignore_regions); ignore_mask: the path of a mask image (see
        ignore_mask_path) or None."""
        if self._disposed:
            return
        self._report["request"] += 1
        # OpticalFlow::calculate's checks, in its order (src/opticalflow.cpp:26-49)
        if not expected:
            self._pending.append((None, expected, target, "ExpectImagePath is empty.")); return
        if not target:
            self._pending.append((None, expected, target, "TargetImagePath is empty.")); return
        # Manager::request with the two paths: the imreads run on the dispatcher's C++ decoder threads (numThreads of them, as the
        # reference decodes inside its numThreads consumers, src/consumer.cpp:54), the pair joins the compute queue when both are in
        pool = self._ensure_pool(0, 0)
        if ignore_mask:
            rid = pool.request_files(expected, target, ignore=ignore or None, ignore_mask=ignore_mask)
        else:
            rid = pool.request_files(expected, target, ignore=ignore) if ignore else pool.request_files(expected, target)
        self._pending.append((rid, expected, target, None))

    def flush(self):
        """Delivers every outstanding answer as 'data' / 'error' events (the uv_async hop of src/manager.cpp:102-125)."""
        pending, self._pending = self._pending, []
        queued = pending  # (request id | None, expected, target, error message | None), in request order
        for rid, expected, target, err in queued:
            if err is None:
                r = self._pool.wait(rid)
                if r is None:
                    continue  # dropped by dispose()
                if r["status"] == "ERROR":
                    err = r["reason"]
            if err is not None:
                self._report["error"] += 1
                self._emit("error", {"status": "ERROR", "reason": err})  # src/broker.cpp:57-70
            else:
                self._report["data"] += 1
                if r.pop("n_vectors", len(r["vector"])) != len(r["vector"]):
                    raise RuntimeError("dispatcher returned a truncated vector list")  # cannot happen with vector_cap = 0
                r["expect_image"], r["target_image"] = expected, target
                self._emit("data", r)                                    # src/broker.cpp:44-55,161-188

    def dispose(self):
        """Broker::requestDispose -> Manager::stop -> 'finish' with the Report (src/broker.cpp:72-86,152-158)."""
        if self._disposed:
            return
        self.flush()
        self._disposed = True
        if self._pool is not None:
            self._pool.stop()
            self._pool.close()
            self._pool = None
        self._emit("finish", dict(self._report))


def create(targetDir, options=None, devices=None, batch=8) -> TidalWave:
    """index.js:14-31.  ``options`` must carry ``expectDir`` (string) or ``getExpectedPath`` (callable)."""
    options = options or {}
    t = TidalWave(options, devices=devices, batch=batch)
    if isinstance(options.get("expectDir"), str):
        def getExpectedPath(shortPath):
            return os.path.abspath(os.path.join(options["expectDir"], shortPath))
    elif callable(options.get("getExpectedPath")):
        getExpectedPath = options["getExpectedPath"]
    else:
        raise ValueError('An option must have "expectDir" or "getExpectedPath" property.')
    t._calc_all = lambda: _calc_all(t, targetDir, getExpectedPath)
    return t


def _calc_all(t: TidalWave, targetDir, getExpectedPath):
    """index.js:33-73: glob targetDir/**/*.*, map each file to its expected file, calc, dispose when all answered."""
    base = os.path.abspath(targetDir)
    for target in sorted(glob.glob(os.path.join(base, "**", "*.*"), recursive=True)):
        if not os.path.isfile(target):
            continue
        short = os.path.relpath(target, base)
        expected = getExpectedPath(short)
        if not expected:
            continue  # index.js:50-51
        try:
            regions = t.ignore_regions(short)
        except ValueError as e:
            t.reject(expected, target, str(e))
            continue
        t.calc(expected, target, regions, t.ignore_mask_path(short))  # FS.exists' answer is ignored by the reference too (index.js:57-58)
    t.dispose()
    return t


def run(t: TidalWave) -> dict:
    """Drives the pairing + lifecycle of a ``create()``d instance to completion; returns the final Report."""
    t._calc_all()
    return dict(t._report)
