"""bench.py --dump-outputs on the B200: the files hold what the timed pass computed, i.e. what a caller of the library gets for the
same seeded pairs (statuses and vectors; with the dense last iteration also the flow at the sampled pixels)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("last", ["sparse", "dense"])
def test_dump_outputs_match_the_api(tw, tmp_path, last):
    B = 2
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", str(B), "--no-e2e",
                          "--no-cpu", "--last", last, "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 2
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64e6
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert got["status"].tolist() == d["statuses"]

    pairs = tw.synth.pool_pairs(B, 1920, 1080, seed0=100)
    o = tw.OpticalFlow(0, 1920, 1080, B)
    want = o.calculate_batch(pairs)
    assert got["status"].tolist() == [{"OK": 0, "SUSPICIOUS": 1}[r["status"]] for r in want]
    assert got["n_vectors"].tolist() == [r["n_vectors"] for r in want]
    assert got["vectors"].tolist() == [[i, v["x"], v["y"], v["dx"], v["dy"]] for i, r in enumerate(want) for v in r["vector"]]
    assert len(got["vectors"]) > 0  # pair 0 carries a defect
    if last == "dense":
        px = got["flow_pixels"].astype(np.int64)
        for i in range(B):
            fx, fy = o.batch_flow(i, 1920, 1080)
            assert np.array_equal(got["flow"][i], np.stack([fx.ravel()[px], fy.ravel()[px]], 1))
    else:
        assert "flow" not in got
    o.close()
