"""The large-batch step (config C3) ends either with ONE tail launch (split-K sums, bound, prior + Adagrad, weight
mirrors) or with five separate launches (`VAEB_TC_TAIL=0`, the structure L > 1, AdaDelta, NCCL and vaeb_gradients use).
Both run the same contractions and the same fused epilogues, so three updates must land on the same parameters whatever
the structure (what differs is the grouping of fp32 partial sums of the bound).  The default structure itself is held
against the fp64 oracle in tests/test_gpu_tc_step.py, tests/test_gpu_round2.py and tests/test_gpu_dp.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

VARIANTS = [
    ("tail-separate", {"VAEB_TC_TAIL": "0"}),
]


def _run(tmp_path, name, env, prec, rows):
    out = str(tmp_path / ("%s_%s.npz" % (name, prec)))
    e = dict(os.environ)
    e.pop("VAEB_TC_TAIL", None)
    e.update(env)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "c3_path_worker.py"), out, prec, str(rows)],
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=e)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return np.load(out)


@pytest.mark.parametrize("prec,rows", [("bf16x3", 4096), ("bf16", 2048)])
def test_launch_structures_agree(tmp_path, prec, rows):
    ref = _run(tmp_path, "default", {}, prec, rows)
    # fp32 tier: same operands, same MMAs; only summation groupings differ.  bf16 tier: one bf16 rounding of an
    # activation can flip with the grouping, so the comparison is at that tier's tolerance.
    rtol = 2e-5 if prec == "bf16x3" else 2e-2
    for name, env in VARIANTS:
        got = _run(tmp_path, name, env, prec, rows)
        np.testing.assert_allclose(got["bounds"], ref["bounds"], rtol=rtol, err_msg=name)
        for k in ref.files:
            if k[0] not in "pa":
                continue
            a, b = got[k], ref[k]
            scale = np.abs(b).max() + 1e-30
            # Adagrad's first steps are lr * sign(g) where |g| is tiny: compare on the tensor's scale
            assert np.abs(a - b).max() <= (2e-3 if prec == "bf16x3" else 5e-2) * scale, (name, k, np.abs(a - b).max(), scale)
        # fewer launches is the point of the fused tail
        assert int(ref["launches"]) < int(got["launches"]), name
