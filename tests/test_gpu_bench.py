"""bench.py --dump-outputs: what the last timed update left for its caller, the same in every run of one command."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "1", "--warmup", "3", "--no-also",
           "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_hold_the_last_timed_update_and_repeat(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    line = _bench(a)
    _bench(b)
    assert line["steps"] == 1
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    assert len(names) == 21 and "bound.npy" in names          # the bound, 10 parameter tensors, their accumulators
    # one timed step: the bound the JSON line reports is the one that step returned
    assert float(np.load(a / "bound.npy")[0]) == pytest.approx(line["final_bound_per_datapoint"], rel=1e-7)
    total = 0
    for n in names:
        x, y = np.load(a / n), np.load(b / n)
        assert x.dtype == np.float32 and np.isfinite(x).all(), n
        np.testing.assert_allclose(x, y, rtol=1e-5, atol=1e-7, err_msg=n)
        total += x.nbytes
    assert total <= 64 << 20
