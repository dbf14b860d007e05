"""Training with a weighted latent term (vaeb_set_kl_weight) on every update path, against the fp64 oracle of
tests/kl_oracle.py.  Every test first asserts which kernel runs (vaeb_step_kernel); each update is then compared with an
oracle restarted from the handle's own parameters and accumulators at the update's own beta_n: the returned bound (which
stays unweighted), the gradient recovered from the Adagrad accumulator increment (or read back with vaeb_gradients) and
the parameter step, at the fp32 tier, or at the tier of the tensor-core precision (tests/test_gpu_fused_step.py).
  1. the tensor-core step kernel (C2 L^B / L^A, C1, the VAEBfullbayes variant) at beta in {0, 0.25, 3};
  2. the fp32 step kernel at 1030 rows and at M = 100 with the tensor-core kernel switched off;
  3. the fp32 per-layer kernels: L = 2, the 64-row tiling, sigmoid, a deeper encoder, Adam and AdaDelta;
  4. the tensor-core per-layer path; 5. the large-batch path with and without the tail kernel, bf16, vaeb_gradients;
  6. a warm-up that ends inside one update_many launch; 7. the overflow hand-over of the Gaussian decoder during a
     warm-up; 8. the streaming entry point; 9. defaults, argument errors, profile_update; 10. two GPUs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests import adam_oracle as A
from tests import kl_oracle as K
from tests.test_gpu_adam import _free_port
from tests.test_gpu_fused_step import (BF16X3_TIER, C1, C2, FP32_TIER, FUSED, LAYERS, TC, _assert_gradient_from_increment,
                                       _data, _rand_params, _state)
from tests.util import assert_close_tensor, frey_trained_params

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FB = (560, 200, 10, True)                 # VAEBfullbayes.py's hard-coded shape
BF16_TIER = (3e-2, 1.0)                   # (gradient rtol, floor) of bf16 operands (tests/test_gpu_tc_step.py)


def _vaeb(shape, x, M, est="LB", params=None, L=1, **kw):
    import vaeb_b200
    D, H, Z, cont = shape
    return vaeb_b200.VAEB(x, cont, H, Z, M, L, 0.01, est == "LA", False, params, **kw)


def _oracle(m, xb, kl, est, variant="vaeb"):
    o = K.OracleKLVAEB(xb, m.continuous, m.n_hidden_units, m.n_latent, xb.shape[0], L=m.L, estimator=est,
                       params=m.get_params(), variant=variant, activation=m.activation, kl_weight=kl)
    return o


def _check(m, kernel, run, xb, eps, kl, est="LB", variant="vaeb", tier=FP32_TIER, bound_rtol=1e-4):
    """One Adagrad update run by `run()` against the oracle at KL weight `kl`, restarted from the handle's state."""
    rows = xb.shape[0]
    assert m.step_kernel_name(rows).startswith(kernel), (rows, m.step_kernel_name(rows))
    p0, a0 = _state(m)
    o = _oracle(m, xb, kl, est, variant)
    o.ada = [a.copy() for a in a0]
    sg, _, g = o.grads(xb, eps)
    fb = variant == "fullbayes"
    O.adagrad_update(o.params, o.ada, g, o.lr, 1e-6, p2_coeff=1e-6 if fb else 0.0)
    got = float(run())
    assert got == pytest.approx(sg if fb else sg / rows, rel=bound_rtol), (kernel, rows, kl)
    p1, a1 = _state(m)
    gtol, floor, thr = tier
    for q1, q0, qr, c1, c0, gr, n in zip(p1, p0, o.params, a1, a0, g, O.param_names(m.continuous, m.encoder_layers)):
        _assert_gradient_from_increment(c1, c0, gr, gtol, floor, "%s (%s, %d rows, beta %g)" % (n, kernel, rows, kl))
        well = np.abs(gr) > thr * np.abs(gr).max()
        assert well.mean() > 0.25, (n, well.mean())
        np.testing.assert_allclose((q1 - q0)[well], (qr - q0)[well], rtol=2e-3, atol=1e-7,
                                   err_msg="step %s (%s, %d rows, beta %g)" % (n, kernel, rows, kl))
    return got


def _check_gradients(m, kernel, xb, idx, eps, kl, est="LB", rtol=1e-4, floor=0.05):
    """vaeb_gradients (beta_{t+1}, t unchanged) against the oracle; the weighted and the unweighted oracle gradients must
    differ by more than the tolerance somewhere, so that the comparison sees the weight."""
    assert m.step_kernel_name(xb.shape[0]).startswith(kernel)
    t = m.kl_step
    g_ref = _oracle(m, xb, kl, est).grads(xb, eps)[2]
    g_one = _oracle(m, xb, 1.0, est).grads(xb, eps)[2]
    _, _, g = m.gradients(index=idx, eps=eps)
    assert m.kl_step == t
    seen = False
    for a, r, r1, n in zip(g, g_ref, g_one, O.param_names(m.continuous, m.encoder_layers)):
        assert_close_tensor(a, r, rtol, floor=floor, name="grad %s (beta %g)" % (n, kl))
        seen |= bool((np.abs(r - r1) > 4 * rtol * np.maximum(np.abs(r), floor * np.abs(r).max())).any())
    assert seen or kl == 1.0
    return g_ref


def _eps(rng, L, M, Z):
    return rng.normal(size=(L, M, Z)).astype(np.float32)


# ---- 1. the tensor-core step kernel ------------------------------------------------------------------------------------
@pytest.mark.parametrize("beta", [0.0, 0.25, 3.0])
@pytest.mark.parametrize("shape,est,variant", [
    pytest.param(C2, "LB", "vaeb", id="c2"), pytest.param(C2, "LA", "vaeb", id="c2-LA"),
    pytest.param(C1, "LB", "vaeb", id="c1"), pytest.param(FB, "LB", "fullbayes", id="fullbayes")])
def test_tensor_core_step_kernel(shape, est, variant, beta):
    """The kernel scales the three latent-term lines of its dz phase by beta_n and the whole gradient by w in its
    weight-gradient epilogues: for the VAEBfullbayes variant (w = 1/M) the update ascends w (grad loglik + beta grad aux)."""
    M = 100
    x = _data(shape, 2 * M)
    m = _vaeb(shape, x, M, est, _rand_params(shape, 3), variant=variant, kl_weight=beta)
    rng = np.random.RandomState(7)
    for idx in (1, 0):
        eps = _eps(rng, 1, M, shape[2])
        _check(m, TC, lambda: m.update(idx, eps=eps), x[idx * M:(idx + 1) * M], eps, beta, est, variant)
    assert m.kl_step == 2
    m.close()


# ---- 2. the fp32 step kernel --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("beta", [0.0, 3.0])
@pytest.mark.parametrize("shape,M,est,env", [
    pytest.param(C2, 1030, "LB", {}, id="c2-1030"), pytest.param(C2, 1030, "LA", {}, id="c2-1030-LA"),
    pytest.param(C1, 100, "LB", {"VAEB_B200_STEP_TC": "0"}, id="c1-100-no-tc")])
def test_fp32_step_kernel(monkeypatch, shape, M, est, env, beta):
    for k, v in env.items():
        monkeypatch.setenv(k, v)                                  # read when the handle is created
    x = _data(shape, 2 * M)
    m = _vaeb(shape, x, M, est, _rand_params(shape, 4), kl_weight=beta)
    rng = np.random.RandomState(M)
    for idx in (1, 0):
        eps = _eps(rng, 1, M, shape[2])
        _check(m, FUSED, lambda: m.update(idx, eps=eps), x[idx * M:(idx + 1) * M], eps, beta, est)
    m.close()


# ---- 3. the fp32 per-layer kernels ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,L,kw,est", [
    pytest.param(300, 2, {}, "LB", id="L2-300"),                              # latent_bwd_kernel<1>
    pytest.param(2048, 2, {}, "LA", id="L2-2048-LA"),                         # latent_bwd_kernel<8>
    pytest.param(2048, 1, {"activation": "sigmoid"}, "LB", id="sigmoid-2048"),  # the 64-row tiling (lb_latent_bwd_kernel)
    pytest.param(300, 1, {"encoder_layers": 2}, "LA", id="depth2-300"),
    pytest.param(300, 1, {"optimizer": "adam"}, "LB", id="adam-300"),
    pytest.param(2048, 1, {"optimizer": "adadelta"}, "LA", id="adadelta-2048")])
def test_fp32_per_layer(M, L, kw, est):
    beta, warmup = 3.0, 2
    x = _data(C2, 2 * M)
    params = _rand_params(C2, 5)
    if kw.get("encoder_layers", 1) == 2:                                      # W3_2, b3_2 after the reference's list
        base, extra = dict(zip(O.param_names(False), params)), np.random.RandomState(6)
        params = [base[n] if n in base else extra.normal(0, 0.05, s).astype(np.float32)
                  for n, s in zip(O.param_names(False, 2), O.param_shapes(784, 500, 20, False, 2))]
    m = _vaeb(C2, x, M, est, params, L=L, kl_weight=beta, kl_warmup=warmup, **kw)
    opt = kw.get("optimizer", "adagrad")
    rng = np.random.RandomState(9)
    for n, idx in enumerate((1, 0), 1):
        eps = _eps(rng, L, M, 20)
        xb = x[idx * M:(idx + 1) * M]
        kl = K.kl_weight_at(beta, warmup, n)
        if opt == "adagrad":
            _check(m, LAYERS, lambda: m.update(idx, eps=eps), xb, eps, kl, est)
            continue
        # Adam and AdaDelta: the gradient through vaeb_gradients, then the update against the rule
        g = _check_gradients(m, LAYERS, xb, idx, eps, kl, est)
        from vaeb_b200 import _lib
        p0 = [p.astype(np.float64) for p in m.get_params()]
        acc = [a.astype(np.float64) for a in m._get_buffer(_lib.BUF_ADA)]
        acc2 = [a.astype(np.float64) for a in m._get_buffer(_lib.BUF_ADA2)]
        ref = [p.copy() for p in p0]
        if opt == "adam":
            A.adam_update(ref, acc, acc2, g, n, 0.01)
        else:
            O.adadelta_update(ref, acc, acc2, g, 0.95, 1e-6)
        sg = _oracle(m, xb, kl, est).grads(xb, eps)[0]
        assert float(m.update(idx, eps=eps)) == pytest.approx(sg / M, rel=1e-4)
        for q1, q0, qr, gr, nm in zip(m.get_params(), p0, ref, g, O.param_names(False)):
            well = np.abs(gr) > 1e-3 * np.abs(gr).max()
            np.testing.assert_allclose((q1 - q0)[well], (qr - q0)[well], rtol=2e-3, atol=1e-7, err_msg=nm)
    assert m.kl_step == 2
    m.close()


# ---- 4-5. the tensor-core per-layer path and the large-batch path ---------------------------------------------------------
def test_tensor_core_per_layer_bf16x3():
    M, L, beta = 1152, 2, 0.25
    x = _data(C2, 2 * M)
    m = _vaeb(C2, x, M, "LB", _rand_params(C2, 8), L=L, precision="bf16x3", kl_weight=beta)
    rng = np.random.RandomState(10)
    for idx in (1, 0):
        eps = _eps(rng, L, M, 20)
        _check(m, LAYERS, lambda: m.update(idx, eps=eps), x[idx * M:(idx + 1) * M], eps, beta, tier=BF16X3_TIER)
    m.close()


def _check_c3_worker_state(r, x, params, eps):
    from vaeb_b200.model import kl_weight_at
    from tests.kl_worker import BETA, WARMUP
    H, Z, M = 500, 20, 4096
    gtol, floor, thr = BF16X3_TIER
    for k in range(3):
        xb = x[(k % 2) * M:(k % 2 + 1) * M]
        p0 = [r["p%d_%d" % (k, i)].astype(np.float64) for i in range(len(params))]
        a0 = [r["a%d_%d" % (k, i)].astype(np.float64) for i in range(len(params))]
        o = K.OracleKLVAEB(xb, False, H, Z, M, params=p0, kl_weight=float(kl_weight_at(BETA, WARMUP, k + 1)))
        o.ada = [a.copy() for a in a0]
        sg, _, g = o.grads(xb, eps[k])
        O.adagrad_update(o.params, o.ada, g, o.lr, 1e-6)
        assert float(r["bound%d" % k]) == pytest.approx(sg / M, rel=1e-4)
        for i, n in enumerate(O.param_names(False)):
            q1, c1 = r["p%d_%d" % (k + 1, i)].astype(np.float64), r["a%d_%d" % (k + 1, i)].astype(np.float64)
            _assert_gradient_from_increment(c1, a0[i], g[i], gtol, floor, "%s (update %d)" % (n, k + 1))
            well = np.abs(g[i]) > thr * np.abs(g[i]).max()
            np.testing.assert_allclose((q1 - p0[i])[well], (o.params[i] - p0[i])[well], rtol=2e-3, atol=1e-7,
                                       err_msg="step %s (update %d)" % (n, k + 1))
    assert int(r["kl_step"]) == 3


@pytest.mark.parametrize("tail", ["1", "0"])
def test_large_batch_over_a_warmup(tmp_path, tail):
    """bf16x3 at 4096 rows, beta_n = 1.25, 2.5, 2.5: the step that ends in the tail kernel and the one that launches the
    slice sum, the bound and Adagrad separately (VAEB_TC_TAIL is read once per process: a worker runs each)."""
    out = tmp_path / "c3.npz"
    env = dict(os.environ, VAEB_TC_TAIL=tail)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "kl_worker.py"), "c3", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    from tests.kl_worker import inputs
    x, params, eps = inputs(3)
    _check_c3_worker_state(dict(np.load(out)), x, params, eps)


def test_large_batch_bf16_and_gradients():
    """bf16 at 4096 rows at the bf16 tier, and vaeb_gradients at 4096 rows (bf16x3): beta_{t+1}, t unchanged."""
    M = 4096
    x = _data(C2, 2 * M)
    rng = np.random.RandomState(12)
    for prec, tol in (("bf16", BF16_TIER), ("bf16x3", (1e-4, 0.1))):
        m = _vaeb(C2, x, M, "LB", _rand_params(C2, 9), precision=prec, kl_weight=3.0, kl_warmup=4)
        m.kl_step = 1
        eps = _eps(rng, 1, M, 20)
        _check_gradients(m, LAYERS, x[M:], 1, eps, K.kl_weight_at(3.0, 4, 2), rtol=tol[0], floor=tol[1])
        sg = _oracle(m, x[M:], 1.0, "LB").grads(x[M:], eps)[0]
        assert float(m.update(1, eps=eps)) == pytest.approx(sg / M, rel=1e-2 if prec == "bf16" else 1e-4)
        assert m.kl_step == 2
        m.close()


# ---- 6. a warm-up that ends inside one launch -----------------------------------------------------------------------------
def test_warmup_inside_one_update_many_launch():
    """update_many of 7 updates from t = 2 with a warm-up of 4: beta_n = 3/4, 4/4, then 1 (times beta).  Bit-identical to
    7 update() calls on a twin handle, each of which matches the oracle at its own beta_n; replaying from t = 2 reproduces
    the parameters."""
    from vaeb_b200 import _lib
    M, Z, beta, warmup = 100, 20, 3.0, 4
    order = [1, 0, 1, 1, 0, 0, 1]
    x = _data(C2, 2 * M)
    params = _rand_params(C2, 11)
    m1, m2 = [_vaeb(C2, x, M, "LB", params, seed=10, kl_weight=beta, kl_warmup=warmup) for _ in range(2)]
    for m in (m1, m2):
        m.kl_step = 2
    assert m1.step_kernel_name().startswith(TC)
    b1 = m1.update_many(order)
    b2 = []
    for s, idx in enumerate(order):
        eps = O.philox_normal(10, 0, s, M * Z).reshape(1, M, Z)
        kl = K.kl_weight_at(beta, warmup, 3 + s)
        b2.append(_check(m2, TC, lambda: m2.update(idx), x[idx * M:(idx + 1) * M], eps, kl))
    np.testing.assert_array_equal(b1, np.array(b2, np.float32))
    end = m1.get_params()
    for p, q in zip(end, m2.get_params()):
        np.testing.assert_array_equal(p, q)
    for p, q in zip(m1._get_buffer(_lib.BUF_ADA), m2._get_buffer(_lib.BUF_ADA)):
        np.testing.assert_array_equal(p, q)
    assert m1.kl_step == 9 and m2.kl_step == 9
    # replay: the same state, step counter and KL step give the same parameters
    m1.set_params(params)
    m1._set_buffer(_lib.BUF_ADA, [np.zeros_like(p) for p in params])
    _lib.check(m1._lib.vaeb_set_step_counter(m1._h, 0))
    m1.kl_step = 2
    np.testing.assert_array_equal(m1.update_many(order), b1)
    for p, q in zip(m1.get_params(), end):
        np.testing.assert_array_equal(p, q)
    m1.close(); m2.close()


# ---- 7. the overflow hand-over during a warm-up ---------------------------------------------------------------------------
def test_overflow_hand_over_keeps_each_updates_weight():
    """The reference's trained Frey weights at lr = 0.01 leave the tensor-core kernel's operand range at the second
    update (tests/test_gpu_step_path.py): the fp32 kernel finishes the launch, and its updates must use their own
    beta_n, the same as update() one by one, each of which matches the oracle."""
    M, Z, beta, warmup = 100, 2, 0.5, 3
    order = [0, 1, 0, 1]
    params = frey_trained_params()
    x = O.synthetic_frey(300)[:2 * M]
    m1, m2 = [_vaeb(C1, x, M, "LB", params, seed=3, kl_weight=beta, kl_warmup=warmup) for _ in range(2)]
    assert m1.step_kernel_name().startswith(TC)
    l0 = m1.launch_count()
    a = m1.update_many(order)
    assert m1.launch_count() - l0 == 4        # mirror set-up (2), the tensor-core kernel, the fp32 kernel
    b = []
    for s, idx in enumerate(order):
        eps = O.philox_normal(3, 0, s, M * Z).reshape(1, M, Z)
        b.append(_check(m2, TC, lambda: m2.update(idx), x[idx * M:(idx + 1) * M], eps, K.kl_weight_at(beta, warmup, s + 1)))
    np.testing.assert_allclose(a, b, rtol=1e-5)
    for p, q, n in zip(m1.get_params(), m2.get_params(), O.param_names(True)):
        assert_close_tensor(p, q, 1e-4, name=n)
    assert m1.kl_step == 4
    m1.close(); m2.close()


# ---- 8. streaming --------------------------------------------------------------------------------------------------------
def test_streaming_updates_over_a_warmup():
    import vaeb_b200
    M, beta, warmup = 100, 2.0, 3
    order = [0, 1, 1, 0, 1]
    x = _data(C2, 2 * M)
    params = _rand_params(C2, 12)
    xp = vaeb_b200.pinned_empty((len(order) * M, x.shape[1]), np.float32)
    for k, i in enumerate(order):
        xp[k * M:(k + 1) * M] = x[i * M:(i + 1) * M]
    m1, m2 = [_vaeb(C2, x, M, "LB", params, seed=5, kl_weight=beta, kl_warmup=warmup) for _ in range(2)]
    assert m1.step_kernel_name().startswith(TC)
    for k in range(len(order)):
        m1.update_host_async(xp[k * M:(k + 1) * M])
    a = m1.collect()
    b = np.array([float(m2.update(i)) for i in order], np.float32)
    np.testing.assert_allclose(a, b, rtol=1e-5)
    for p, q, n in zip(m1.get_params(), m2.get_params(), O.param_names(False)):
        assert_close_tensor(p, q, 1e-4, name=n)
    assert m1.kl_step == m2.kl_step == len(order)
    # a ramp that differs from the constant weight must change the parameters (the comparison sees the weight)
    m3 = _vaeb(C2, x, M, "LB", params, seed=5)
    for i in order:
        m3.update(i)
    assert max(np.abs(p - q).max() for p, q in zip(m1.get_params(), m3.get_params())) > 1e-4
    m1.close(); m2.close(); m3.close()


# ---- 9. defaults, errors, profile_update ----------------------------------------------------------------------------------
@pytest.mark.parametrize("M,L,kw,kernel", [
    (100, 1, {}, TC), (1030, 1, {}, FUSED), (300, 2, {}, LAYERS), (4096, 1, {"precision": "bf16x3"}, LAYERS)])
def test_weight_one_is_bit_identical_to_no_weight(M, L, kw, kernel):
    x = _data(C2, 2 * M)
    params = _rand_params(C2, 13)
    m1 = _vaeb(C2, x, M, "LB", params, L=L, seed=4, **kw)
    m2 = _vaeb(C2, x, M, "LB", params, L=L, seed=4, **kw)
    m2.set_kl_weight(1.0, 0)
    assert m1.step_kernel_name().startswith(kernel)
    a = [float(m1.update(i)) for i in (1, 0)] + list(m1.update_many([0, 1]))
    b = [float(m2.update(i)) for i in (1, 0)] + list(m2.update_many([0, 1]))
    assert a == b
    for p, q in zip(m1.get_params(), m2.get_params()):
        np.testing.assert_array_equal(p, q)
    m1.close(); m2.close()


def test_argument_errors_and_full_vb():
    M = 100
    x = _data(C2, 2 * M)
    m = _vaeb(C2, x, M)
    for beta, warmup in ((-0.5, 0), (float("nan"), 0), (float("inf"), 0), (1.0, -1)):
        with pytest.raises(ValueError):
            m.set_kl_weight(beta, warmup)
    with pytest.raises(ValueError):
        m.kl_step = -1
    m.close()
    import vaeb_b200
    fvb = vaeb_b200.VAEB(x, False, 500, 20, M, 1, 0.01, False, True, _rand_params(C2, 1))
    with pytest.raises(ValueError):
        fvb.set_kl_weight(0.5, 0)
    fvb.close()
    with pytest.raises(ValueError):
        vaeb_b200.VAEB(x, False, 500, 20, M, 1, 0.01, False, True, _rand_params(C2, 1), kl_weight=0.5)


@pytest.mark.parametrize("M,kw,kernel", [(100, {}, TC), (2048, {"precision": "bf16x3"}, LAYERS)])
def test_profile_update_leaves_the_kl_step(M, kw, kernel):
    x = _data(C2, 2 * M)
    m = _vaeb(C2, x, M, "LB", _rand_params(C2, 14), kl_weight=0.5, kl_warmup=10, **kw)
    assert m.step_kernel_name().startswith(kernel)
    m.update(0)
    assert m.kl_step == 1
    m.profile_update(0, iters=3)
    assert m.kl_step == 1
    m.close()


# ---- 10. two GPUs --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("p2p", ["1", "0"])       # 1: the tail kernel over peer memory; 0: ncclAllReduce
def test_data_parallel_over_a_warmup(tmp_path, p2p):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = tmp_path / "dp.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "kl_worker.py"), "dp", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, VAEB_DP_P2P=p2p))
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    res = json.load(open(out))
    assert res["ranks_bit_identical"] and res["kl_step"] == 2
    assert res["bound_rel_err"] < 1e-4
    assert res["worst_step_err"] < 5e-2
