"""The fp32 single-launch step kernel (vaeb_b200/csrc/fused_step.cu) against the fp64 oracle at the row counts and shapes
it runs, and one handle whose minibatch size changes from update to update.
  1. Full width: C2 at 129, 1030 and 4096 rows, C1 (Gaussian decoder) at 300 and 2048 rows, the reference's Nz = 200
     model, a D % 4 != 0 input width, C2 at M = 100 with the tensor-core kernel switched off, full VB at the C4 shape
     and the VAEBfullbayes variant.  At these sizes the host planner splits each job over several rounds of CTA items,
     several tiles per warp group and k slices of a ragged row count, none of which the toy shapes of
     tests/test_gpu_parity.py reach.
  2. Philox noise past the first tile round, update_many of odd and even length, the parameter double buffer (read back
     three ways) and the streaming entry point.
  3. One handle through every update path in turn (tensor-core step kernel, fp32 step kernel, per-layer kernels, the
     large-batch tail), with the row count changing at every call: what each path re-plans or rebuilds when the size
     changes, and the operand mirrors another path left behind.
Every test first asserts which kernel runs (vaeb_step_kernel), then checks numbers.  Each update is compared with an fp64
oracle restarted from the handle's own state (parameters and accumulators), which makes a single Adagrad step well
posed however many steps came before.  Tolerances, the fp32 tier (DESIGN 3, tests/util.py): bounds 1e-4 relative; |g|
recovered from the accumulator increment within 1e-4 * max(|g|, 0.05 ||g||_inf); the parameter step within 2e-3 of the
oracle's where |g| > 1e-3 ||g||_inf."""
import ctypes as C

import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests.util import assert_close_tensor

pytestmark = pytest.mark.gpu

RTOL = 1e-4
TC, FUSED, LAYERS = "step_tc_kernel", "fused_step_kernel", "per-layer kernels"
C2 = (784, 500, 20, False)            # MNIST, Bernoulli decoder
C1 = (560, 200, 2, True)              # Frey Face, Gaussian decoder
# (gradient rtol, gradient floor, step mask) per tier.  bf16x3 (tests/test_gpu_tc_step.py): a hi + lo bf16 pair carries
# 16 mantissa bits, 2^-17 relative per operand, so gradients are held to 0.1 ||g||_inf, and a step is then determined to
# 2e-3 only where |g| > 1e-2 ||g||_inf.  A product of two pairs is off by up to 2^-16 of itself, so an entry g = sum of
# n terms is off by up to 2^-16 sum|terms|: in the state the large-batch steps of test_changing_minibatch_sizes_bf16x3
# reach, that bound is 1.1e-4 of the tier's scale at 3 of the 10^4 entries of the W1 gradient (sum|z da1| = 6.3 |g|),
# hence 1.5e-4 there
FP32_TIER, BF16X3_TIER = (RTOL, 0.05, 1e-3), (1.5e-4, 0.1, 1e-2)


def _rand_params(shape, seed, scale=0.05):
    D, H, Z, cont = shape
    rng = np.random.RandomState(seed)
    return [rng.normal(0, scale, s).astype(np.float32) for s in O.param_shapes(D, H, Z, cont)]


def _data(shape, n, seed=15485863):
    D, _, _, cont = shape
    return O.synthetic_frey(n, seed, D) if cont else O.synthetic_mnist(n, seed, D)


def _model(shape, x, M, est="LB", params=None, **kw):
    import vaeb_b200
    D, H, Z, cont = shape
    return vaeb_b200.VAEB(x, cont, H, Z, M, 1, 0.01, est == "LA", est.startswith("FVB"), params,
                          sample_weights=(est == "FVB_SAMPLED"), **kw)


def _split_flat(flat, params):
    out, k = [], 0
    for p in params:
        out.append(flat[k:k + p.size].reshape(p.shape)); k += p.size
    return out


def _state(m):
    """(the tensors an update moves, their Adagrad accumulators) in the oracle's order, float64."""
    from vaeb_b200 import _lib
    f64 = lambda ts: [t.astype(np.float64) for t in ts]
    if m._fvb:
        inter = lambda a, b: [t for pair in zip(a, b) for t in pair]
        return (f64(inter(m._get_buffer(_lib.BUF_VMU), m._get_buffer(_lib.BUF_VSIG))),
                f64(inter(m._get_buffer(_lib.BUF_ADA_MU), m._get_buffer(_lib.BUF_ADA_SIG))))
    return f64(m.get_params()), f64(m._get_buffer(_lib.BUF_ADA))


def _names(m):
    names = O.param_names(m.continuous)
    return [n + s for n in names for s in ("_mu", "_sigma")] if m._fvb else names


def _assert_gradient_from_increment(acc1, acc0, g, rtol, floor, name):
    """The gradient the update used, from its accumulator increment acc1 - acc0 = g^2: |sqrt(inc) - |g_ref|| <= t with
    t = rtol * max(|g_ref|, floor * ||g_ref||_inf), in the squared form (no cancellation in a square root), widened by
    one ulp of acc1 for the fp32 rounding of the sum acc0 + g^2."""
    g = np.abs(g)
    t = rtol * np.maximum(g, floor * g.max())
    inc = acc1 - acc0
    r = np.spacing(acc1.astype(np.float32)).astype(np.float64)
    bad = (inc < np.maximum(g - t, 0.0) ** 2 - r) | (inc > (g + t) ** 2 + r)
    if bad.any():
        i = np.unravel_index(np.argmax(bad), g.shape)
        raise AssertionError("|g| %s: %d entries off, first at %s: got %r ref %r (allowed %.3e)"
                             % (name, bad.sum(), i, np.sqrt(max(inc[i], 0.0)), g[i], t[i]))


def _step(m, kernel, run, xb, eps, est="LB", variant="vaeb", zeta=None, tier=FP32_TIER):
    """One update run by `run()` on the rows xb, checked against the fp64 oracle restarted from the handle's state: the
    returned bound, the gradient recovered from every accumulator, and the parameter step where it is well posed."""
    rows = xb.shape[0]
    assert m.step_kernel_name(rows).startswith(kernel), (rows, m.step_kernel_name(rows))
    p0, a0 = _state(m)
    o = O.OracleVAEB(xb, m.continuous, m.n_hidden_units, m.n_latent, rows, L=1, estimator=est,
                     params=m.get_params(), variant=variant)
    if o.fvp is not None:
        o.fvp = [p.copy() for p in p0]
    o.ada = [a.copy() for a in a0]
    sg, _, g = o.grads(xb, eps, zeta)
    ref = sg if variant == "fullbayes" else sg / rows             # (the variant's objective is a mean already)
    O.adagrad_update(o.fvp if o.fvp is not None else o.params, o.ada, g, o.lr, 1e-6,
                     p2_coeff=1e-6 if variant == "fullbayes" else 0.0)
    got = float(run())
    assert got == pytest.approx(ref, rel=RTOL), (kernel, rows, got, ref)
    p1, a1 = _state(m)
    gtol, floor, thr = tier
    for q1, q0, qr, c1, c0, gr, n in zip(p1, p0, o.fvp if o.fvp is not None else o.params, a1, a0, g, _names(m)):
        _assert_gradient_from_increment(c1, c0, gr, gtol, floor, "%s (%s, %d rows)" % (n, kernel, rows))
        well = np.abs(gr) > thr * np.abs(gr).max()
        assert well.mean() > 0.25, (n, well.mean())               # the compared subset is not vacuous
        np.testing.assert_allclose((q1 - q0)[well], (qr - q0)[well], rtol=2e-3, atol=1e-7,
                                   err_msg="step %s (%s, %d rows)" % (n, kernel, rows))
    return got


# ---- 1. the fp32 step kernel at full width ---------------------------------------------------------------------------
@pytest.mark.parametrize("shape,M,est,env", [
    pytest.param(C2, 129, "LB", {}, id="c2-129"),                  # the first row count past the tensor-core kernel
    pytest.param(C2, 1030, "LB", {}, id="c2-1030"),                # ragged, several rounds of items per CTA
    pytest.param(C2, 1030, "LA", {}, id="c2-1030-LA"),
    pytest.param(C2, 4096, "LB", {}, id="c2-4096"),                # the largest
    pytest.param(C1, 300, "LB", {}, id="c1-300"),                  # dual-N dec2, dual-K dgrad, W6
    pytest.param(C1, 2048, "LB", {}, id="c1-2048"),
    pytest.param((784, 500, 200, False), 100, "LB", {}, id="nz200"),   # heads too wide for the tensor-core kernel
    pytest.param((784, 500, 200, False), 100, "LA", {}, id="nz200-LA"),
    pytest.param((786, 500, 20, False), 100, "LB", {}, id="d786"),     # D % 4 != 0: 4-byte cp.async rows
    pytest.param(C2, 100, "LB", {"VAEB_B200_STEP_TC": "0"}, id="c2-100-no-tc"),
    pytest.param(C2, 100, "LA", {"VAEB_B200_STEP_TC": "0"}, id="c2-100-no-tc-LA"),
])
def test_fused_step_full_width(monkeypatch, shape, M, est, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)                                  # read when the handle is created
    x = _data(shape, 2 * M)
    m = _model(shape, x, M, est, _rand_params(shape, 3))
    rng = np.random.RandomState(M)
    for idx in (1, 0, 1):
        eps = rng.normal(size=(1, M, shape[2])).astype(np.float32)
        _step(m, FUSED, lambda: m.update(idx, eps=eps), x[idx * M:(idx + 1) * M], eps, est)
    m.close()


@pytest.mark.parametrize("est", ["FVB", "FVB_SAMPLED"])
def test_fused_step_full_vb(est):
    """C4's shape, 784-500-10, at 256 rows: every variational tensor and its accumulator; the sampled-weights oracle is
    fed the zeta of Philox stream 3 (keyed by the update's step and the flat parameter index)."""
    shape, M = (784, 500, 10, False), 256
    x = _data(shape, 2 * M)
    params = _rand_params(shape, 2)
    m = _model(shape, x, M, est, params, seed=10)
    total = sum(p.size for p in params)
    rng = np.random.RandomState(20)
    for step, idx in enumerate((1, 0, 1)):
        zeta = _split_flat(O.philox_normal(10, 3, step, total), params) if est == "FVB_SAMPLED" else None
        eps = rng.normal(size=(1, M, 10)).astype(np.float32)
        _step(m, FUSED, lambda: m.update(idx, eps=eps), x[idx * M:(idx + 1) * M], eps, est, zeta=zeta)
    if est == "FVB":
        for a, b in zip(m.get_params(), params):
            np.testing.assert_array_equal(a, b)                   # VAEB.py:119,352: the MAP parameters stay frozen
    m.close()


def test_fused_step_fullbayes_variant():
    """VAEBfullbayes.py at its hard-coded shape, 560-200-10 Gaussian: the mean objective (1/M weight), no weight prior,
    and the - lr * 1e-6 * p^2 term of its update."""
    shape, M = (560, 200, 10, True), 300
    x = _data(shape, 2 * M)
    m = _model(shape, x, M, "LB", _rand_params(shape, 4), variant="fullbayes")
    rng = np.random.RandomState(5)
    for idx in (1, 0, 1):
        eps = rng.normal(size=(1, M, 10)).astype(np.float32)
        _step(m, FUSED, lambda: m.update(idx, eps=eps), x[idx * M:(idx + 1) * M], eps, variant="fullbayes")
    m.close()


# ---- 2. noise, batching and the parameter double buffer --------------------------------------------------------------
def test_fused_step_philox_noise_past_the_first_tile_round():
    """eps = None: the kernel draws N(0,1) for row m, latent j from Philox (seed, stream 0, step, m * Z + j).  At 1030 rows
    the rows past the first round of encoder-head items are drawn by CTAs on their second and later items."""
    M, Z = 1030, 20
    x = _data(C2, 2 * M)
    m = _model(C2, x, M, params=_rand_params(C2, 6), seed=10)
    for step, idx in enumerate((1, 0, 1)):
        eps = O.philox_normal(10, 0, step, M * Z).reshape(1, M, Z)
        _step(m, FUSED, lambda: m.update(idx), x[idx * M:(idx + 1) * M], eps)
    m.close()


def test_fused_step_update_many_odd_and_even_equals_updates():
    M = 300
    x = _data(C2, 4 * M)
    params = _rand_params(C2, 7)
    m1, m2 = _model(C2, x, M, params=params, seed=5), _model(C2, x, M, params=params, seed=5)
    assert m1.step_kernel_name().startswith(FUSED)
    for order in ([2, 0, 3], [1, 3, 0, 2]):                      # odd, then even from the other parameter buffer
        a = m1.update_many(np.array(order, np.int32))
        b = np.array([float(m2.update(i)) for i in order], np.float32)
        np.testing.assert_array_equal(a, b)
        for p, q in zip(m1.get_params(), m2.get_params()):
            np.testing.assert_array_equal(p, q)
    m1.close(); m2.close()


def test_fused_step_parameter_double_buffer():
    """The fp32 step kernel writes the new parameters into the other half of a double buffer and the handle swaps the
    halves after an odd number of steps.  After update_many of three steps the re-queried device buffer, get_params()
    and validate() (per-layer kernels reading the parameter buffer) must agree; then gradients() and one more update."""
    from cuda.bindings import runtime as rt
    from vaeb_b200 import _lib
    M, Z = 300, 20
    x = _data(C2, 5 * M)
    m = _model(C2, x[:4 * M], M, params=_rand_params(C2, 8), seed=5)
    assert m.step_kernel_name().startswith(FUSED)
    m.update_many(np.array([2, 0, 3], np.int32))
    ptr, n = C.c_void_p(), C.c_int64()
    _lib.check(m._lib.vaeb_device_buffer(m._h, _lib.BUF_PARAMS, C.byref(ptr), C.byref(n)))
    flat = np.empty(n.value, np.float32)
    m.synchronize()
    (err,) = rt.cudaMemcpy(flat.ctypes.data, ptr.value, flat.nbytes, rt.cudaMemcpyKind.cudaMemcpyDeviceToHost)
    assert int(err) == 0
    params = m.get_params()
    got = np.concatenate([p.ravel() for p in params])
    np.testing.assert_array_equal(flat[:got.size], got)
    o = O.OracleVAEB(x, False, 500, Z, M, L=1, params=params)
    rng = np.random.RandomState(9)
    xv = x[4 * M:]
    ev = rng.normal(size=(1, M, Z)).astype(np.float32)
    assert float(m.validate(xv, eps=ev)) == pytest.approx(o.validate(xv, ev)[0], rel=RTOL)
    eg = rng.normal(size=(1, M, Z)).astype(np.float32)
    sg, _, g = m.gradients(index=1, eps=eg)
    sg_ref, _, g_ref = o.grads(x[M:2 * M], eg)
    assert sg == pytest.approx(sg_ref, rel=RTOL)
    for a, b, nm in zip(g, g_ref, O.param_names(False)):
        assert_close_tensor(a, b, RTOL, name="grad " + nm)
    eps = rng.normal(size=(1, M, Z)).astype(np.float32)
    _step(m, FUSED, lambda: m.update(0, eps=eps), x[:M], eps)
    m.close()


def test_fused_step_streaming_equals_update_host():
    """update_host_async at 300 rows: six minibatches are one launch for a full group of four and one for the remaining
    two; the same bounds and parameters as update_host one by one, bit for bit."""
    import vaeb_b200
    M, n = 300, 6
    x = _data(C2, n * M)
    xp = vaeb_b200.pinned_empty(x.shape, np.float32)
    xp[:] = x
    params = _rand_params(C2, 10)
    m1, m2 = _model(C2, x[:M], M, params=params, seed=3), _model(C2, x[:M], M, params=params, seed=3)
    assert m1.step_kernel_name().startswith(FUSED)
    for i in range(n):
        m1.update_host_async(xp[i * M:(i + 1) * M])
    a = m1.collect()
    b = np.array([float(m2.update_host(x[i * M:(i + 1) * M])) for i in range(n)], np.float32)
    np.testing.assert_array_equal(a, b)
    for p, q in zip(m1.get_params(), m2.get_params()):
        np.testing.assert_array_equal(p, q)
    m1.close(); m2.close()


# ---- 3. minibatch-size changes on one handle -------------------------------------------------------------------------
def test_changing_minibatch_sizes_fp32():
    """One fp32 C2 handle (resident data for M = 100) through: 100 (tensor-core kernel), 37 (its activation mirrors
    cleared for fewer rows), 300 (fp32 kernel, first plan; it swaps the parameter buffers), 100 (the tensor-core kernel's
    weight mirrors rebuilt from the swapped buffer), 5000 (per-layer kernels: 64-row latent tilings, flat Adagrad), 129
    and 300 (the fp32 kernel re-plans twice), 1 (tensor-core kernel); then update_many on the resident data and
    validate."""
    M, Z = 100, 20
    res = _data(C2, 2 * M)
    pool = _data(C2, 5000, seed=7)
    m = _model(C2, res, M, params=_rand_params(C2, 11), seed=10)
    rng = np.random.RandomState(12)
    steps = 0
    for rows, kernel in [(100, TC), (37, TC), (300, FUSED), (100, TC), (5000, LAYERS), (129, FUSED), (300, FUSED),
                         (1, TC)]:
        xb = pool[rng.randint(0, 5000 - rows + 1):][:rows]
        eps = rng.normal(size=(1, rows, Z)).astype(np.float32)
        _step(m, kernel, lambda: m.update_host(xb, eps=eps), xb, eps)
        steps += 1
    # two steps in one launch on the resident data (Philox noise of the handle's step counter), against a two-step oracle
    assert m.step_kernel_name().startswith(TC)
    p0, a0 = _state(m)
    o = O.OracleVAEB(res, False, 500, Z, M, L=1, params=m.get_params())
    o.ada = [a.copy() for a in a0]
    order = [1, 0]
    eps = [O.philox_normal(10, 0, steps + k, M * Z).reshape(1, M, Z) for k in range(2)]
    well = [np.ones(p.shape, bool) for p in p0]
    ref = []
    for i, e in zip(order, eps):
        _, _, g = o.grads(res[i * M:(i + 1) * M], e)
        for w, gr in zip(well, g):
            w &= np.abs(gr) > 1e-3 * np.abs(gr).max()
        ref.append(o.update(i, e))
    np.testing.assert_allclose(m.update_many(np.array(order, np.int32)), ref, rtol=RTOL)
    steps += 2
    p1, a1 = _state(m)
    for q1, q0, qr, c1, cr, w, n in zip(p1, p0, o.params, a1, o.ada, well, O.param_names(False)):
        np.testing.assert_allclose((q1 - q0)[w], (qr - q0)[w], rtol=2e-3, atol=2e-7, err_msg="step " + n)
        # at the mask's edge the gradient tolerance is 5e-3 of |g|, i.e. 1e-2 of g^2
        np.testing.assert_allclose(c1[w], cr[w], rtol=1e-2, err_msg="ADA " + n)
    xv = pool[:777]
    ev = rng.normal(size=(1, 777, Z)).astype(np.float32)
    assert float(m.validate(xv, eps=ev)) == pytest.approx(O.OracleVAEB(
        xv, False, 500, Z, M, params=m.get_params()).validate(xv, ev)[0], rel=RTOL)
    m.close()


def test_changing_minibatch_sizes_bf16x3():
    """bf16x3 C2 (the fp32 tier): 100 (tensor-core step kernel), 2048 (large-batch step; its tail writes the weight
    mirrors of the new parameters), 100 (the step kernel moves the parameters: those mirrors are stale now), 2048 (they
    must be rebuilt), 1500 (ragged last row block), 512 (per-layer tensor-core layers); then validate.  Each step also
    lands bit for bit where the same step lands on a fresh handle given the same parameters and accumulators: nothing
    another path left in the handle (operand mirrors, plans, workspaces sized for other row counts) leaks into it."""
    from vaeb_b200 import _lib
    M, Z = 100, 20
    res = _data(C2, M)
    pool = _data(C2, 4096, seed=8)
    m = _model(C2, res, M, params=_rand_params(C2, 13), precision="bf16x3")
    rng = np.random.RandomState(14)
    for rows, kernel in [(100, TC), (2048, LAYERS), (100, TC), (2048, LAYERS), (1500, LAYERS), (512, LAYERS)]:
        xb = pool[rng.randint(0, 4096 - rows + 1):][:rows]
        eps = rng.normal(size=(1, rows, Z)).astype(np.float32)
        fresh = _model(C2, res, M, params=m.get_params(), precision="bf16x3")
        fresh._set_buffer(_lib.BUF_ADA, m._get_buffer(_lib.BUF_ADA))
        got = _step(m, kernel, lambda: m.update_host(xb, eps=eps), xb, eps, tier=FP32_TIER if kernel == TC else BF16X3_TIER)
        assert got == float(fresh.update_host(xb, eps=eps)), rows
        for a, b in zip(m.get_params() + m._get_buffer(_lib.BUF_ADA), fresh.get_params() + fresh._get_buffer(_lib.BUF_ADA)):
            np.testing.assert_array_equal(a, b, err_msg="%d rows" % rows)
        fresh.close()
    xv = pool[:333]
    ev = rng.normal(size=(1, 333, Z)).astype(np.float32)
    assert float(m.validate(xv, eps=ev)) == pytest.approx(O.OracleVAEB(
        xv, False, 500, Z, M, params=m.get_params()).validate(xv, ev)[0], rel=RTOL)
    m.close()


def test_changing_minibatch_sizes_streaming():
    """update_host_async with a changing row count: a group holds minibatches of one size, so it is launched when the
    size changes, each group by the kernel of its size.  The same bounds and parameters as update_host one by one on a
    twin handle, bit for bit."""
    import vaeb_b200
    sizes = [100, 100, 100, 37, 300, 300, 300, 300, 300, 100, 5000]
    kernels = [TC, TC, TC, TC, FUSED, FUSED, FUSED, FUSED, FUSED, TC, LAYERS]
    x = _data(C2, sum(sizes), seed=9)
    xp = vaeb_b200.pinned_empty(x.shape, np.float32)
    xp[:] = x
    params = _rand_params(C2, 15)
    m1, m2 = _model(C2, x[:100], 100, params=params, seed=3), _model(C2, x[:100], 100, params=params, seed=3)
    cuts = np.cumsum([0] + sizes)
    for a, b, k in zip(cuts[:-1], cuts[1:], kernels):
        assert m1.step_kernel_name(b - a).startswith(k), (b - a, m1.step_kernel_name(b - a))
        m1.update_host_async(xp[a:b])
    got = m1.collect()
    ref = np.array([float(m2.update_host(x[a:b])) for a, b in zip(cuts[:-1], cuts[1:])], np.float32)
    np.testing.assert_array_equal(got, ref)
    for p, q in zip(m1.get_params(), m2.get_params()):
        np.testing.assert_array_equal(p, q)
    m1.close(); m2.close()
