"""Adam (vaeb_set_adam) on the device against the fp64 Adam oracle of tests/adam_oracle.py (itself pinned against
torch.optim.Adam(maximize=True) in tests/test_adam_cpu.py): the fp32 per-layer path, update_many, checkpointing of the
optimizer state, the large-batch tail kernel against the five-launch structure, argument and state errors, and two
GPUs over NCCL and over peer memory.

Adam's first step moves every element by about +-lr whatever |g| is, so an element whose gradient is at rounding level
can step either way: parameter and moment comparisons are masked to elements whose oracle gradient is well above the
tensor's rounding (as in tests/test_gpu_activations.py)."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests import adam_oracle as A
from tests import adam_c3_worker as W
from vaeb_b200 import _lib

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-4
LR = 0.01


def _params(D, H, Z, continuous, seed, scale):
    rng = np.random.RandomState(seed)
    return [rng.normal(0, scale, s).astype(np.float32) for s in O.param_shapes(D, H, Z, continuous)]


def _check_state(m, o, p0, g_ref, names, rtol, step_tol):
    """Parameters (as the step from p0, on the scale of the three steps of size ~lr), m and v, masked to
    well-conditioned elements; and the step counter."""
    assert m.adam_step == o.adam_t
    mm, vv = m._get_buffer(_lib.BUF_ADA), m._get_buffer(_lib.BUF_ADAM_V)
    for a, b, q0, gr, ma, mb, va, vb, n in zip(m.get_params(), o.params, p0, g_ref, mm, o.ada, vv, o.adam_v, names):
        well = np.abs(gr) > 1e-2 * np.abs(gr).max()
        assert np.abs((a - q0) - (b - q0))[well].max() <= step_tol * 3 * LR, n
        # the moments on their tensor's scale (m of an element whose gradient changes sign can cancel to ~0)
        assert np.abs(ma - mb)[well].max() <= rtol * np.abs(mb).max(), "m " + n
        assert np.abs(va - vb)[well].max() <= rtol * np.abs(vb).max(), "v " + n


@pytest.mark.parametrize("continuous,est,L,D,H,Z,M", [
    (False, "LB", 1, 784, 500, 20, 100),      # C2 shape
    (True, "LB", 1, 560, 200, 2, 100),        # C1 shape, Gaussian decoder
    (False, "LA", 2, 40, 24, 3, 17),          # L > 1, ragged
])
def test_adam_per_layer_matches_oracle(continuous, est, L, D, H, Z, M):
    import vaeb_b200
    x = O.synthetic_mnist(2 * M, seed=5, D=D)
    if continuous:
        x = np.clip(np.random.RandomState(3).normal(0.5, 0.2, (2 * M, D)), 0.01, 0.99).astype(np.float32)
    params = _params(D, H, Z, continuous, 21, 0.05 if D > 100 else 0.2)
    rng = np.random.RandomState(9)
    eps = [rng.normal(size=(L, M, Z)).astype(np.float32) for _ in range(3)]
    m = vaeb_b200.VAEB(x, continuous, H, Z, M, L, LR, est == "LA", False, params, optimizer="adam")
    assert m.step_kernel_name() == "per-layer kernels"
    o = A.OracleAdamVAEB(x, continuous, H, Z, M, L=L, lr=LR, estimator=est, params=params)
    _, _, g_ref = o.grads(x[M:2 * M], eps[0])
    p0 = [q.copy() for q in o.params]
    for i, idx in enumerate((1, 0, 1)):
        ret_ref = o.update(idx, eps[i])
        assert float(m.update(idx, eps=eps[i])) == pytest.approx(ret_ref, rel=RTOL)
    _check_state(m, o, p0, g_ref, O.param_names(continuous), 1e-3, 2e-2)
    m.close()


def test_adam_update_many_matches_updates():
    import vaeb_b200
    D, H, Z, M = 784, 500, 20, 100
    x = O.synthetic_mnist(4 * M, seed=6)
    params = _params(D, H, Z, False, 4, 0.05)
    order = [2, 0, 3, 1, 2]
    a = vaeb_b200.VAEB(x, False, H, Z, M, 1, LR, False, False, params, optimizer="adam")
    b = vaeb_b200.VAEB(x, False, H, Z, M, 1, LR, False, False, params, optimizer="adam")
    ra = a.update_many(order)
    rb = [float(b.update(i)) for i in order]
    np.testing.assert_array_equal(np.asarray(ra, np.float32), np.asarray(rb, np.float32))
    for buf in (_lib.BUF_PARAMS, _lib.BUF_ADA, _lib.BUF_ADAM_V):
        for p, q in zip(a._get_buffer(buf), b._get_buffer(buf)):
            np.testing.assert_array_equal(p, q)
    assert a.adam_step == b.adam_step == len(order)
    a.close(); b.close()


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_adam_checkpoint_restores_state(precision):
    """Parameters, m, v, the Adam step and the Philox step counter copied into a fresh handle: one more update on
    each gives the same bits."""
    import vaeb_b200
    D, H, Z, M = 784, 500, 20, 1024 if precision != "fp32" else 100
    x = O.synthetic_mnist(2 * M, seed=7)
    params = _params(D, H, Z, False, 8, 0.05)
    a = vaeb_b200.VAEB(x, False, H, Z, M, 1, LR, False, False, params, optimizer="adam", precision=precision)
    for i in range(3):
        a.update(i % 2)
    b = vaeb_b200.VAEB(x, False, H, Z, M, 1, LR, False, False, params, optimizer="adam", precision=precision)
    b.set_params(a.get_params())
    b._set_buffer(_lib.BUF_ADA, a._get_buffer(_lib.BUF_ADA))
    b._set_buffer(_lib.BUF_ADAM_V, a._get_buffer(_lib.BUF_ADAM_V))
    b.adam_step = a.adam_step
    _lib.check(b._lib.vaeb_set_step_counter(b._h, 3))
    assert float(a.update(1)) == float(b.update(1))
    for buf in (_lib.BUF_PARAMS, _lib.BUF_ADA, _lib.BUF_ADAM_V):
        for p, q in zip(a._get_buffer(buf), b._get_buffer(buf)):
            np.testing.assert_array_equal(p, q)
    assert a.adam_step == b.adam_step == 4
    a.close(); b.close()


def _run_c3(tmp_path, name, env, prec, rows):
    out = str(tmp_path / ("%s_%s.npz" % (name, prec)))
    e = dict(os.environ)
    e.pop("VAEB_TC_TAIL", None)
    e.update(env)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "adam_c3_worker.py"), out, prec, str(rows)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=e)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return np.load(out)


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
def test_adam_large_batch_tail(tmp_path, prec):
    """16384 rows: the tail kernel's Adam against the five-launch structure (VAEB_TC_TAIL=0, flat Adam kernel) at the
    tolerances of tests/test_gpu_c3_paths.py, both against the oracle, and the launch counts against Adagrad's."""
    rows = 16384
    ref = _run_c3(tmp_path, "default", {}, prec, rows)
    sep = _run_c3(tmp_path, "separate", {"VAEB_TC_TAIL": "0"}, prec, rows)
    for r in (ref, sep):
        assert int(r["adam_launches"]) == int(r["adagrad_launches"])
        assert int(r["t"]) == 3
    assert int(ref["adam_launches"]) < int(sep["adam_launches"])
    rtol = 2e-5 if prec == "bf16x3" else 2e-2
    np.testing.assert_allclose(sep["bounds"], ref["bounds"], rtol=rtol)
    for k in ref.files:
        if k[0] not in "pmv" or not k[1:].isdigit():
            continue
        a, b = sep[k], ref[k]
        scale = np.abs(b).max() + 1e-30
        assert np.abs(a - b).max() <= (2e-3 if prec == "bf16x3" else 5e-2) * scale, (k, np.abs(a - b).max(), scale)
    # the oracle (fp64) on the same inputs
    x, params, eps, (D, H, Z) = W.inputs(rows)
    o = A.OracleAdamVAEB(x, False, H, Z, rows, L=1, lr=LR, params=params)
    # an entry is well conditioned when its gradient is large against its tensor's at EVERY step: Adam's step then
    # depends on gradient ratios that the precision's tier determines (the bf16 tier holds gradients to a few 1e-2
    # of the tensor's scale, so there 99.9 % of those entries are pinned)
    well_at, step_tol, mom_tol, share = (1e-2, 2e-2, 1e-3, 1.0) if prec == "bf16x3" else (1e-1, 0.25, 0.1, 0.999)
    rets, wells = [], None
    for i in range(3):
        _, _, g = o.grads(x[(i % 2) * rows:(i % 2 + 1) * rows], eps[i])
        w = [np.abs(t) > well_at * np.abs(t).max() for t in g]
        wells = w if wells is None else [a & b for a, b in zip(wells, w)]
        rets.append(o.update(i % 2, eps[i]))
    np.testing.assert_allclose(ref["bounds"], rets, rtol=1e-4 if prec == "bf16x3" else 1e-2)
    for i, (well, q0) in enumerate(zip(wells, params)):
        step = ref["p%d" % i] - q0
        err = np.abs(step - (o.params[i] - q0))[well]
        assert np.mean(err <= step_tol * 3 * LR) >= share, (i, err.max(), np.mean(err <= step_tol * 3 * LR))
        for key, r in (("m", o.ada[i]), ("v", o.adam_v[i])):
            got = ref["%s%d" % (key, i)]
            assert np.abs(got - r)[well].max() <= mom_tol * np.abs(r).max(), (key, i)


def test_adam_argument_and_state_errors():
    import vaeb_b200
    D, H, Z, M = 40, 24, 3, 8
    x = O.synthetic_mnist(2 * M, seed=1, D=D)
    params = _params(D, H, Z, False, 2, 0.2)
    m = vaeb_b200.VAEB(x, False, H, Z, M, 1, LR, False, False, params)
    h, lib = m._h, m._lib
    for b1, b2, e in ((1.0, 0.999, 1e-8), (-0.1, 0.999, 1e-8), (0.9, 1.0, 1e-8), (0.9, float("nan"), 1e-8),
                      (0.9, 0.999, 0.0), (0.9, 0.999, -1e-8), (0.9, 0.999, float("inf"))):
        assert lib.vaeb_set_adam(h, b1, b2, e) == 1, (b1, b2, e)
    assert lib.vaeb_set_adam_step(h, -1) == 1
    assert lib.vaeb_set_adam(h, 0.9, 0.999, 1e-8) == 0
    m.gradients(index=0)
    assert lib.vaeb_apply_update(h) == 1            # Adagrad only
    assert lib.vaeb_set_optimizer(h, _lib.OPT_ADAGRAD, 0.0) == 0
    assert lib.vaeb_apply_update(h) == 0
    m.close()
    # full VB
    f = vaeb_b200.VAEB(x, False, H, Z, M, 1, LR, False, True, params)
    assert f._lib.vaeb_set_adam(f._h, 0.9, 0.999, 1e-8) == 1
    f.close()
    with pytest.raises(ValueError):
        vaeb_b200.VAEB(x, False, H, Z, M, 1, LR, False, True, params, optimizer="adam")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("p2p", ["1", "0"])       # 1: the tail kernel over peer memory; 0: ncclAllReduce + flat Adam
def test_adam_data_parallel(tmp_path, p2p):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = tmp_path / "dp.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "adam_dp_worker.py"), str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, VAEB_DP_P2P=p2p))
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    res = json.load(open(out))
    assert res["ranks_bit_identical"] and res["adam_step"] == 2
    if p2p == "1":
        assert res["set_adam_after_export"] == 2           # VAEB_ESTATE: the peers mapped m without room for v
    assert res["bound_rel_err"] < 1e-4
    assert res["worst_rel_err"] < 5e-2
