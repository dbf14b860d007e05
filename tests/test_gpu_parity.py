"""GPU parity tests proper: every number comes from the sm_100a kernels through the C-ABI
(ctypes) and is compared with the CPU oracle (fp64) on the same seeded inputs with injected
eps, with the committed golden vectors, and through size-independent properties at the
BASELINE.json sizes.

Tolerances (fp32 path, north star: 1e-4 relative):
  * per-datapoint bound, SGVB, log p(x):  |d| <= 1e-4 * |ref|
  * gradient / parameter tensors:         |d| <= 1e-4 * max(|ref|, 0.05*||ref||_inf)
    (tests/util.py:assert_close_tensor -- entries that are sums of cancelling terms have no
    meaningful purely-relative error)."""
import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests.util import assert_close_tensor, fingerprint, frey_trained_params, load_golden

pytestmark = pytest.mark.gpu

RTOL = 1e-4


def _model(x, continuous, H, Z, M, L=1, est="LB", params=None, **kw):
    import vaeb_b200
    return vaeb_b200.VAEB(x, continuous, H, Z, M, L, 0.01, est == "LA", est.startswith("FVB"), params,
                          sample_weights=(est == "FVB_SAMPLED"), **kw)


def _rand_params(D, H, Z, continuous, seed, scale=0.1):
    rng = np.random.RandomState(seed)
    return [rng.normal(0, scale, s).astype(np.float32) for s in O.param_shapes(D, H, Z, continuous)]


def _check_step(x, continuous, H, Z, M, L, est, params, seed):
    rng = np.random.RandomState(seed)
    eps = rng.normal(size=(L, M, Z)).astype(np.float32)
    m = _model(x, continuous, H, Z, M, L, est, params)
    o = O.OracleVAEB(x, continuous, H, Z, M, L=L, estimator=est, params=params, dtype=np.float64)
    idx = 1 if x.shape[0] >= 2 * M else 0
    xb = x[idx * M:(idx + 1) * M]
    sg_ref, rows_ref, g_ref = o.grads(xb, eps)
    sg, rows, g = m.gradients(index=idx, eps=eps)
    assert sg == pytest.approx(sg_ref, rel=RTOL)
    np.testing.assert_allclose(rows, rows_ref, rtol=RTOL)
    worst = 0.0
    for a, b, n in zip(g, g_ref, O.param_names(continuous)):
        worst = max(worst, assert_close_tensor(a, b, RTOL, name="grad " + n))
    # update(): pre-update value returned, Adagrad applied.  Two checks:
    #  (a) the Adagrad rule itself (VAEB.py:438-442).  update() runs a single-launch step kernel (the
    #      tensor-core one at C1/C2, M = 100; the fp32 FFMA one at the small ragged shapes, whose D is
    #      below the tensor-core kernel's minimum), whose gradient is summed in a different order than
    #      gradients()'s, so the rule is checked on the gradient the update itself used: after the first
    #      step ADA = g^2 exactly, hence
    #      |dp| = lr*sqrt(ADA)/(sqrt(ADA)+1e-6) must hold everywhere to fp32 rounding, sqrt(ADA) must
    #      agree with |g| of gradients() at the gradient tolerance, and dp carries the sign of g;
    #  (b) end-to-end against the oracle's own update where the step is well conditioned: the
    #      first Adagrad step is lr*g/(|g|+1e-6), whose sensitivity 1e-6/(|g|+1e-6)^2 blows any
    #      gradient rounding error up wherever |g| ~ 0, so entries with |g| below 1e-3*||g||_inf
    #      are excluded from (b) (they are covered by (a) and by the gradient parity above).
    p_old = [q.copy() for q in o.params]
    dev_old = [q.astype(np.float64) for q in m.get_params()]
    ret_ref = o.update(idx, eps)
    ret = m.update(idx, eps=eps)
    assert float(ret) == pytest.approx(ret_ref, rel=RTOL)
    new_params = m.get_params()
    for a, po, ada, gd, n in zip(new_params, dev_old, m._get_buffer(1), g, O.param_names(continuous)):
        ga = np.sqrt(ada.astype(np.float64))
        assert_close_tensor(ga, np.abs(np.asarray(gd, np.float64)), RTOL, name="sqrt(ada) " + n)
        dp = a.astype(np.float64) - po
        np.testing.assert_allclose(np.abs(dp), 0.01 * ga / (ga + 1e-6), rtol=1e-5, atol=2e-8, err_msg="adagrad rule " + n)
        well = np.abs(gd) > 1e-3 * np.abs(gd).max()
        assert np.array_equal(np.sign(dp[well]), np.sign(np.asarray(gd)[well])), "step sign " + n
    for a, b, gr, po, n in zip(new_params, o.params, g_ref, p_old, O.param_names(continuous)):
        well = np.abs(gr) > 1e-3 * np.abs(gr).max()
        np.testing.assert_allclose((a - po)[well], (b - po)[well], rtol=2e-3, atol=1e-7, err_msg="step " + n)
    # a second step from the device state (accumulators carried): compare the returned bound
    # with an oracle restarted from the device parameters
    o2 = O.OracleVAEB(x, continuous, H, Z, M, L=L, estimator=est, params=new_params, dtype=np.float64)
    eps2 = rng.normal(size=(L, M, Z)).astype(np.float32)
    assert float(m.update(0, eps=eps2)) == pytest.approx(o2.update(0, eps2), rel=RTOL)
    m.close()
    return worst


# ---- small and ragged shapes --------------------------------------------------------------
@pytest.mark.parametrize("continuous", [False, True])
@pytest.mark.parametrize("est,L", [("LB", 1), ("LB", 3), ("LA", 1), ("LA", 2)])
def test_step_small_ragged(continuous, est, L):
    D, H, Z, M = 37, 29, 3, 11      # nothing divides a tile
    x = np.random.RandomState(5).uniform(size=(3 * M, D)).astype(np.float32)
    _check_step(x, continuous, H, Z, M, L, est, _rand_params(D, H, Z, continuous, 7, 0.3), 11)


def test_step_single_row_and_unit_latent():
    D, H, Z, M = 16, 8, 1, 1
    x = np.random.RandomState(6).uniform(size=(4, D)).astype(np.float32)
    _check_step(x, False, H, Z, M, 1, "LB", _rand_params(D, H, Z, False, 8, 0.3), 12)


# ---- BASELINE configs at full width ------------------------------------------------------
def test_step_c1_frey_trained_weights_golden():
    """C1: Frey 560/200/2, M=100, Gaussian decoder, the reference's trained weights."""
    g = load_golden("golden_frey_z2.npz")
    x = O.synthetic_frey(300)
    params = frey_trained_params()
    for est in ("LB", "LA"):
        m = _model(x, True, 200, 2, 100, 1, est, params)
        sg, rows, grads = m.gradients(index=0, eps=g[est + "_eps"])
        assert sg == pytest.approx(float(g[est + "_sgvb"]), rel=RTOL)
        np.testing.assert_allclose(rows, g[est + "_per_row"], rtol=RTOL)
        fp, fr = fingerprint(grads), g[est + "_grad_fp"]
        for t in range(len(grads)):
            assert fp[t, 0] == pytest.approx(fr[t, 0], rel=RTOL, abs=RTOL * 0.05 * fr[t, 2] * np.sqrt(grads[t].size))
            assert fp[t, 1] == pytest.approx(fr[t, 1], rel=2 * RTOL)
            assert_close_tensor(fp[t, 2:], fr[t, 2:], RTOL, name="fingerprint %d" % t)
        ret = m.update(0, eps=g[est + "_eps"])
        assert float(ret) == pytest.approx(float(g[est + "_update_return"]), rel=RTOL)
        after = dict(zip(O.param_names(True), m.get_params()))
        for n in ("b3", "b4", "b5", "b1", "b2", "b6", "W4"):
            assert_close_tensor(after[n], g["%s_after_%s" % (est, n)], RTOL, name="after " + n)
        m.close()


def test_step_c1_frey_full_tensors():
    x = O.synthetic_frey(300)
    _check_step(x, True, 200, 2, 100, 1, "LB", frey_trained_params(), 21)


def test_step_c2_mnist_init_golden_and_full():
    """C2: MNIST 784/500/20, M=100, Bernoulli decoder, reference initialisation."""
    g = load_golden("golden_mnist_init.npz")
    x = O.synthetic_mnist(200)
    params = O.init_params(784, 500, 20, False)
    for est, L in (("LB", 1), ("LA", 2)):
        m = _model(x, False, 500, 20, 100, L, est)          # params=None: the model draws the init itself
        for a, b in zip(m.get_params(), params):
            np.testing.assert_array_equal(a, b)              # a1: same RandomState(10) draw order
        sg, rows, grads = m.gradients(index=0, eps=g[est + "_eps"])
        assert sg == pytest.approx(float(g[est + "_sgvb"]), rel=RTOL)
        np.testing.assert_allclose(rows, g[est + "_per_row"], rtol=RTOL)
        fp, fr = fingerprint(grads), g[est + "_grad_fp"]
        for t in range(len(grads)):
            assert_close_tensor(fp[t, 2:], fr[t, 2:], RTOL, name="fingerprint %d" % t)
        m.close()
    _check_step(x, False, 500, 20, 100, 1, "LB", _rand_params(784, 500, 20, False, 3, 0.05), 22)


def test_step_c2_trained_regime_large_weights():
    x = O.synthetic_mnist(200)
    _check_step(x, False, 500, 20, 100, 1, "LA", _rand_params(784, 500, 20, False, 4, 0.15), 23)


# ---- validate ---------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 37, 465])
def test_validate_ragged(n):
    x = O.synthetic_frey(500)
    params = frey_trained_params()
    m = _model(x[:200], True, 200, 2, 100, 1, "LB", params)
    o = O.OracleVAEB(x[:200], True, 200, 2, 100, params=params)
    eps = np.random.RandomState(n).normal(size=(1, n, 2)).astype(np.float32)
    before = m.get_params()
    val, rows = m.validate(x[:n], eps=eps, per_row=True)
    ref, rows_ref = o.validate(x[:n], eps)
    assert float(val) == pytest.approx(ref, rel=RTOL)
    np.testing.assert_allclose(rows, rows_ref, rtol=RTOL)
    for a, b in zip(before, m.get_params()):
        np.testing.assert_array_equal(a, b)                  # validate has no side effect on params
    m.close()


def test_validate_full_mnist_validation_set_is_sum_of_rows():
    x = O.synthetic_mnist(10000 + 100)
    m = _model(x[:100], False, 500, 20, 100, 1, "LB", _rand_params(784, 500, 20, False, 9, 0.05))
    val, rows = m.validate(x[100:], per_row=True)            # Philox eps, 10,000 rows in one call
    assert np.isfinite(rows).all()
    assert float(val) == pytest.approx(float(rows.astype(np.float64).sum()), rel=1e-5)
    # x*a - softplus(a) <= 0 and KL <= 0: every LB row is non-positive for the Bernoulli model
    assert (rows <= 0).all()
    m.close()


# ---- variants ------------------------------------------------------------------------------
def test_fullbayes_variant():
    D, H, Z, M = 40, 24, 5, 16
    x = np.random.RandomState(1).uniform(size=(2 * M, D)).astype(np.float32)
    params = _rand_params(D, H, Z, True, 2, 0.2)
    eps = np.random.RandomState(3).normal(size=(1, M, Z)).astype(np.float32)
    m = _model(x, True, H, Z, M, 1, "LB", params, variant="fullbayes")
    o = O.OracleVAEB(x, True, H, Z, M, params=params, variant="fullbayes")
    ret, ref = m.update(1, eps=eps), o.update(1, eps)
    assert float(ret) == pytest.approx(ref, rel=RTOL)       # the MEAN objective (VAEBfullbayes.py:142)
    for a, b, n in zip(m.get_params(), o.params, O.param_names(True)):
        assert_close_tensor(a, b, RTOL, name=n)
    ev = np.random.RandomState(4).normal(size=(1, 2 * M, Z)).astype(np.float32)
    assert float(m.validate(x, eps=ev)) == pytest.approx(o.validate(x, ev)[0], rel=RTOL)
    m.close()


@pytest.mark.parametrize("est", ["FVB", "FVB_SAMPLED"])
def test_full_variational(est):
    D, H, Z, M = 40, 24, 2, 16
    x = np.random.RandomState(1).uniform(size=(2 * M, D)).astype(np.float32)
    params = _rand_params(D, H, Z, False, 2, 0.2)
    eps = np.random.RandomState(3).normal(size=(1, M, Z)).astype(np.float32)
    zeta = [np.random.RandomState(10 + i).normal(size=p.shape).astype(np.float32) for i, p in enumerate(params)]
    m = _model(x, False, H, Z, M, 1, est, params)
    o = O.OracleVAEB(x, False, H, Z, M, params=params, estimator=est)
    z = zeta if est == "FVB_SAMPLED" else None
    sg, _, g = m.gradients(index=0, eps=eps, zeta=z)
    sg_ref, _, g_ref = o.grads(x[:M], eps, z)
    assert sg == pytest.approx(sg_ref, rel=RTOL)
    for i, (a, b) in enumerate(zip(g, g_ref)):
        assert_close_tensor(a, b, RTOL, name="fvp grad %d" % i)
    if est == "FVB":
        # SURVEY F5: faithful mode trains only the prior terms; MAP params untouched by update
        before = m.get_params()
        ret = m.update(0, eps=eps)
        assert float(ret) == pytest.approx(o.update(0, eps), rel=RTOL)
        for a, b in zip(before, m.get_params()):
            np.testing.assert_array_equal(a, b)
        fv = [p.get_value() for p in m.full_variational_params]
        for i, (a, b) in enumerate(zip(fv, o.fvp)):
            assert_close_tensor(a, b, RTOL, name="fvp %d" % i)
    ev = np.random.RandomState(4).normal(size=(1, 2 * M, Z)).astype(np.float32)
    if est == "FVB":
        assert float(m.validate(x, eps=ev)) == pytest.approx(o.validate(x, ev)[0], rel=RTOL)
    m.close()


def test_full_variational_rejects_L_gt_1():
    x = np.zeros((8, 6), np.float32)
    with pytest.raises(ValueError, match="L == 1"):
        _model(x, False, 4, 2, 4, 2, "FVB", _rand_params(6, 4, 2, False, 0))


def test_update_rejects_out_of_range_batch():
    x = np.zeros((8, 6), np.float32)
    m = _model(x, False, 4, 2, 4)
    with pytest.raises(ValueError, match="outside"):
        m.update(2)
    m.close()


# ---- Philox noise -----------------------------------------------------------------------
def test_philox_device_matches_cpu_restatement():
    import ctypes as C
    from vaeb_b200 import _lib
    m = _model(np.zeros((4, 6), np.float32), False, 4, 2, 4, seed=0x1234567890ABCDEF)
    out = np.empty(4099, np.float32)
    for stream, step, sample in ((0, 0, 0), (2, 7, 3), (1, 2 ** 31 + 5, 1)):
        _lib.check(m._lib.vaeb_philox_normal(m._h, stream, step, sample, 0, out.size, out.ctypes.data_as(C.c_void_p)))
        ref = O.philox_normal(0x1234567890ABCDEF, stream, step, out.size, sample)
        np.testing.assert_allclose(out, ref, rtol=0, atol=3e-6)
    m.close()


def test_update_with_philox_eps_matches_oracle_fed_the_same_draws():
    D, H, Z, M, L = 784, 500, 20, 100, 2
    x = O.synthetic_mnist(300)
    params = _rand_params(D, H, Z, False, 3, 0.05)
    m = _model(x, False, H, Z, M, L, "LB", params, seed=10)
    for step, idx in enumerate([2, 0, 1]):
        eps = np.stack([O.philox_normal(10, 0, step, M * Z, sample=l).reshape(M, Z) for l in range(L)])
        # the oracle restarts from the device parameters each step (Adagrad's first steps are
        # sign-like and ill-conditioned where g ~ 0, see _check_step)
        o = O.OracleVAEB(x, False, H, Z, M, L=L, params=m.get_params())
        assert float(m.update(idx)) == pytest.approx(o.update(idx, eps), rel=RTOL)
    m.close()


def test_update_many_equals_sequential_updates():
    x = O.synthetic_mnist(500)
    params = _rand_params(784, 500, 20, False, 3, 0.05)
    order = [3, 1, 4, 0, 2]
    m1 = _model(x, False, 500, 20, 100, 1, "LB", params)
    m2 = _model(x, False, 500, 20, 100, 1, "LB", params)
    a = np.array([float(m1.update(i)) for i in order], np.float32)
    b = m2.update_many(order)
    np.testing.assert_array_equal(a, b)                      # same kernels, same Philox counters: bit-identical
    for p, q in zip(m1.get_params(), m2.get_params()):
        np.testing.assert_array_equal(p, q)
    m1.close(); m2.close()


def test_update_host_equals_resident_update():
    x = O.synthetic_mnist(200)
    params = _rand_params(784, 500, 20, False, 3, 0.05)
    m1 = _model(x, False, 500, 20, 100, 1, "LB", params)
    m2 = _model(x[:100], False, 500, 20, 100, 1, "LB", params)
    assert float(m1.update(1)) == float(m2.update_host(x[100:200]))
    for p, q in zip(m1.get_params(), m2.get_params()):
        np.testing.assert_array_equal(p, q)
    m1.close(); m2.close()


def test_update_host_async_stream_equals_synchronous_updates():
    """vaeb_update_host_async + vaeb_collect: the pipelined host-input path (copy stream, staging ring,
    deferred readback) must give exactly the bounds and parameters of the synchronous calls."""
    import vaeb_b200
    xs = O.synthetic_mnist(1100)
    x = vaeb_b200.pinned_empty(xs.shape)                     # the streaming path needs page-locked host memory
    x[:] = xs
    params = _rand_params(784, 500, 20, False, 3, 0.05)
    m1 = _model(x[:100], False, 500, 20, 100, 1, "LB", params)
    m2 = _model(x[:100], False, 500, 20, 100, 1, "LB", params)
    order = [3, 1, 4, 0, 2, 9, 7, 8, 6, 5, 10]               # more steps than staging buffers
    a = np.array([float(m1.update_host(x[100 * i:100 * i + 100])) for i in order], np.float32)
    for i in order[:6]:
        m2.update_host_async(x[100 * i:100 * i + 100])
    b = list(m2.collect())
    for i in order[6:]:
        m2.update_host_async(x[100 * i:100 * i + 100])
    b += list(m2.collect())
    np.testing.assert_array_equal(a, np.array(b, np.float32))
    assert len(m2.collect()) == 0
    for p, q in zip(m1.get_params(), m2.get_params()):
        np.testing.assert_array_equal(p, q)
    # a non-fused configuration (L = 2) takes the per-layer path behind the same calls
    m3 = _model(x[:100], False, 500, 20, 100, 2, "LB", params)
    m4 = _model(x[:100], False, 500, 20, 100, 2, "LB", params)
    c = np.array([float(m3.update_host(x[100 * i:100 * i + 100])) for i in order[:5]], np.float32)
    for i in order[:5]:
        m4.update_host_async(x[100 * i:100 * i + 100])
    np.testing.assert_array_equal(c, m4.collect())
    for m in (m1, m2, m3, m4):
        m.close()


# ---- importance-sampled log p(x) ------------------------------------------------------------
def test_is_logpx_golden_and_oracle():
    g = load_golden("golden_frey_z2.npz")
    x = O.synthetic_frey(300)
    m = _model(x[:100], True, 200, 2, 100, 1, "LB", frey_trained_params())
    logp, logw = m.log_px(x[200:216], L=64, eps=g["is_eps"], return_weights=True)
    np.testing.assert_allclose(logw, g["is_logw"], rtol=RTOL)
    np.testing.assert_allclose(logp, g["is_logp"], rtol=RTOL)
    m.close()
    g = load_golden("golden_mnist_init.npz")
    x = O.synthetic_mnist(200)
    m = _model(x[:100], False, 500, 20, 100)
    logp, logw = m.log_px(x[100:108], L=32, eps=g["is_eps"], return_weights=True)
    np.testing.assert_allclose(logw, g["is_logw"], rtol=RTOL)
    np.testing.assert_allclose(logp, g["is_logp"], rtol=RTOL)
    m.close()


def test_is_logpx_philox_sharding_invariance_and_bound():
    x = O.synthetic_mnist(164)
    params = _rand_params(784, 500, 20, False, 3, 0.05)
    m = _model(x[:100], False, 500, 20, 100, params=params, seed=77)
    xt = x[100:164]
    full = m.log_px(xt, L=50)
    # sharded over "ranks" with global row offsets: identical numbers (SURVEY 8e)
    parts = np.concatenate([m.log_px(xt[a:b], L=50, row_offset=a) for a, b in ((0, 7), (7, 40), (40, 64))])
    np.testing.assert_array_equal(full, parts)
    # against the oracle fed the same Philox draws
    eps = np.stack([np.stack([O.philox_normal(77, 2, 0, (i + 1) * 20, sample=l)[i * 20:] for l in range(50)])
                    for i in range(8)])
    ref, _ = O.is_log_px([p.astype(np.float64) for p in params], xt[:8].astype(np.float64), eps.astype(np.float64), False)
    np.testing.assert_allclose(full[:8], ref, rtol=RTOL)
    # chunked path (rows > one chunk) agrees with the single-chunk path
    big = m.log_px(xt[:3], L=70000)
    assert np.isfinite(big).all() and np.all(big >= full[:3] - 5.0)
    m.close()


# ---- reconstruct and the AE-side dense layers ----------------------------------------------
@pytest.mark.parametrize("continuous", [False, True])
@pytest.mark.parametrize("n_samples", [0, 3])
def test_reconstruct(continuous, n_samples):
    D, H, Z = 40, 24, 5
    x = np.random.RandomState(1).uniform(size=(9, D)).astype(np.float32)
    params = _rand_params(D, H, Z, continuous, 2, 0.3)
    m = _model(x, continuous, H, Z, 3, params=params)
    eps = np.random.RandomState(3).normal(size=(n_samples, 9, Z)).astype(np.float32) if n_samples else None
    ref = O.reconstruct_mean([p.astype(np.float64) for p in params], x.astype(np.float64),
                             None if eps is None else eps.astype(np.float64), continuous)
    got = m.reconstruct(x, n_samples, eps=eps, sample_output=False)
    if continuous:
        np.testing.assert_allclose(got[0], ref[0], rtol=RTOL)
        np.testing.assert_allclose(got[1], ref[1], rtol=RTOL, atol=1e-6)
        one = m.reconstruct(x[0], n_samples, eps=None if eps is None else eps[:, :1])
        assert one.shape == (D,)
    else:
        np.testing.assert_allclose(got, ref, rtol=RTOL)
    m.close()


def test_mlp_forward_matches_construct_mlp():
    import vaeb_b200
    rng = np.random.RandomState(0)
    dims = [37, 50, 21, 9]
    Ws = [rng.normal(0, 0.3, (a, b)).astype(np.float32) for a, b in zip(dims, dims[1:])]
    bs = [rng.normal(0, 0.01, b).astype(np.float32) for b in dims[1:]]
    x = rng.uniform(size=(13, 37)).astype(np.float32)
    W64, b64 = [w.astype(np.float64) for w in Ws], [b.astype(np.float64) for b in bs]
    np.testing.assert_allclose(vaeb_b200.mlp_forward(x, Ws, bs), O.construct_mlp(x.astype(np.float64), W64, b64),
                               rtol=RTOL, atol=1e-6)
    hid = O.construct_mlp(x.astype(np.float64), W64[:-1], b64[:-1])
    np.testing.assert_allclose(vaeb_b200.mlp_forward(x, Ws, bs, act_last="sigmoid"),
                               O.out_to_probs(hid, W64[-1], b64[-1]), rtol=RTOL)
    np.testing.assert_allclose(vaeb_b200.mlp_forward(x, Ws, bs, act_last="identity"),
                               O.out_to_real(hid, W64[-1], b64[-1]), rtol=RTOL, atol=1e-6)


# ---- the driver: CLI -> train_model -> .trc / .mdl ---------------------------------------
def test_train_model_end_to_end(tmp_path, capsys):
    import vaeb_b200
    from vaeb_b200 import io
    trc, mdl = str(tmp_path / "t.trc"), str(tmp_path / "m.mdl")
    pgm = str(tmp_path / "manifold.pgm")
    args = vaeb_b200.parse_args(["--continuous", "--n_latent", "2", "--n_epochs", "3", "--trace_file", trc,
                                 "--save_file", mdl, "--synthetic", "--manifold_file", pgm])
    model, data = vaeb_b200.train_model(args)
    assert open(pgm, "rb").read().startswith(b"P5 200 280 255\n")     # 10 x 10 Frey tiles of 20 x 28 (freyFace.py:346-369)
    lines = open(trc).read().splitlines()
    assert lines[0] == "num_samples,L,Lvalid" and len(lines) == 1 + 2 * 3
    assert lines[1] == lines[2] and lines[1].startswith("1500,") and lines[5].startswith("4500,")
    lb = [float(l.split(",")[1]) for l in lines[1::2]]
    assert lb[-1] > lb[0]                                    # the bound improves over epochs
    out = capsys.readouterr().out
    assert "Epoch 0 : [Lower bound:" in out and "[Lower bound on validation set:" in out
    header, params = io.read_mdl(mdl)
    assert header["n_latent"] == 2 and header["continuous"] is True and len(params) == 12
    m2, _ = vaeb_b200.VAEB.load(mdl, data=data)
    for a, b in zip(m2.get_params(), model.get_params()):
        np.testing.assert_array_equal(a, b)
    # full-VB run on top of the saved MAP parameters (full_variational.sh)
    args = vaeb_b200.parse_args(["--continuous", "--n_latent", "2", "--n_epochs", "1", "--full_varational",
                                 "--vb_param_file", mdl, "--synthetic"])
    fv, _ = vaeb_b200.train_model(args, data=data)
    for a, b in zip(fv.get_params(), model.get_params()):
        np.testing.assert_array_equal(a, b)                  # F5: save() would write the untouched MAP params
    model.close(); m2.close(); fv.close()


def test_theano_eps_mode_reproduces_reference_stream_order():
    x = O.synthetic_frey(300)
    params = frey_trained_params()
    m = _model(x[:200], True, 200, 2, 100, 1, "LB", params, eps_mode="theano")
    o = O.OracleVAEB(x[:200], True, 200, 2, 100, params=params)
    s = O.TheanoRandomStreams(10, 1)
    # update, update, validate share one node state (VAEB.py:158): draws interleave in call order
    assert float(m.update(0)) == pytest.approx(o.update(0, s.draw(100, 2)), rel=RTOL)
    assert float(m.update(1)) == pytest.approx(o.update(1, s.draw(100, 2)), rel=RTOL)
    assert float(m.validate(x[200:])) == pytest.approx(o.validate(x[200:], s.draw(100, 2))[0], rel=RTOL)
    m.close()


def test_flat_adagrad_kernel_matches_numpy():
    """getUpdates (VAEB.py:426-444) + prior (VAEB.py:389-390) over the flat buffer, at the C2 size (P = 0.8 M, L2
    resident) and at a stream size beyond L2 (P = 19 M, ragged tail), against the same arithmetic in numpy fp32."""
    for Hh in (500, 12007):
        D, Z = 784, 20
        x = np.random.RandomState(3).uniform(size=(100, D)).astype(np.float32)
        m = _model(x, False, Hh, Z, 100)
        rng = np.random.RandomState(Hh)
        shapes = O.param_shapes(D, Hh, Z, False)
        p0 = [rng.normal(0, 0.1, s).astype(np.float32) for s in shapes]
        a0 = [rng.uniform(0, 2, s).astype(np.float32) for s in shapes]
        g0 = [rng.normal(0, 1, s).astype(np.float32) for s in shapes]
        import vaeb_b200._lib as L_
        for _ in range(2):            # twice: the accumulator written by the first pass feeds the second
            m._set_buffer(L_.BUF_PARAMS, p0); m._set_buffer(L_.BUF_ADA, a0); m._set_buffer(L_.BUF_GRADS, g0)
            m.apply_update()
            p1, a1 = m._get_buffer(L_.BUF_PARAMS), m._get_buffer(L_.BUF_ADA)
            for p, a, g, pn, an in zip(p0, a0, g0, p1, a1):
                gg = g - np.float32(1.0) * p
                ar = a + gg * gg
                pr = p + np.float32(0.01) * gg / (np.sqrt(ar) + np.float32(1e-6))
                np.testing.assert_allclose(an, ar, rtol=2e-6, atol=0)
                np.testing.assert_allclose(pn, pr, rtol=2e-6, atol=1e-7)
            p0, a0 = p1, a1
        m.close()


@pytest.mark.parametrize("continuous", [False, True])
def test_sampled_full_vb_update_fused_kernel_matches_oracle(continuous):
    """update() of the full-VB estimator with sampled weights (theta = mu + |sigma| zeta, VAEB.py:127-129 live in
    getFVBL :349-367) runs in the fused step kernel: phase 0 draws zeta (Philox stream 3, keyed by step and flat
    parameter index), every layer reads theta, the update epilogues apply Adagrad to mu and sigma.  The oracle is fed
    the same zeta / eps draws; three consecutive updates, then every variational parameter."""
    D, H, Z, M = 52, 36, 3, 24
    x = np.random.RandomState(1).uniform(size=(3 * M, D)).astype(np.float32)
    params = _rand_params(D, H, Z, continuous, 2, 0.2)
    m = _model(x, continuous, H, Z, M, 1, "FVB_SAMPLED", params, seed=10)
    o = O.OracleVAEB(x, continuous, H, Z, M, params=params, estimator="FVB_SAMPLED")
    total = sum(p.size for p in params)
    l0 = m.launch_count()
    for step, idx in enumerate([1, 0, 2]):
        flat = O.philox_normal(10, 3, step, total)
        zeta, k = [], 0
        for p in params:
            zeta.append(flat[k:k + p.size].reshape(p.shape)); k += p.size
        eps = np.random.RandomState(20 + step).normal(size=(1, M, Z)).astype(np.float32)
        got = float(m.update(idx, eps=eps))
        ref = o.update(idx, eps, zeta)
        assert got == pytest.approx(ref, rel=RTOL), step
    assert m.launch_count() - l0 == 3          # one fused launch per update
    fv = [p.get_value() for p in m.full_variational_params]
    for i, (a, b) in enumerate(zip(fv, o.fvp)):
        assert_close_tensor(a, b, RTOL, name="fvp %d" % i)
    m.close()


@pytest.mark.parametrize("continuous", [False, True])
def test_decode_and_manifold_grid_match_oracle_decoder(continuous):
    """vaeb_decode = the decoder alone (VAEB.py:253-265 / the compiled freyFace(z) of freyFace.py:237-244) on the
    10 x 10 quantile grid of the manifold renderer (freyFace.py:350-352), trained Frey weights for the Gaussian
    decoder."""
    from vaeb_b200 import manifold
    if continuous:
        D, H, Z = 560, 200, 2
        params = frey_trained_params()
    else:
        D, H, Z = 784, 500, 2
        params = _rand_params(D, H, Z, False, 5, 0.05)
    x = np.zeros((4, D), np.float32)
    m = _model(x, continuous, H, Z, 4, params=params)
    z = manifold.grid_points()
    p = O.as_dict([np.asarray(t, np.float64) for t in params], continuous)
    _, a, lv = O.decoder(p, z.astype(np.float64), continuous)
    y_ref = 1.0 / (1.0 + np.exp(-a))
    out = m.decode(z)
    if continuous:
        assert_close_tensor(out[0], y_ref, RTOL, name="mu_x")
        assert_close_tensor(out[1], lv, RTOL, name="log_sigma")
        assert m.freyFace(z[:1])[0].shape == (1, D)
    else:
        assert_close_tensor(out, y_ref, RTOL, name="y")
    faces, tiled = manifold.render(m)
    assert faces.shape == (100, D) and tiled.shape[0] == 280
    m.close()
