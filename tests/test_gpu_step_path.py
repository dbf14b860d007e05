"""Which kernel runs an update (vaeb_step_kernel), and the entry points that launch the single-launch step kernels:
  * the choice for every precision, minibatch size, optimizer, activation, encoder depth, decoder and environment switch,
    and that it comes back when a setter is undone;
  * the overflow hand-over of the Gaussian decoder behind the staging ring of update_host_async, on a fresh handle;
  * vaeb_profile_update on each of the three ways an update runs: its phases, and a model it leaves untouched."""
import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests.util import assert_close_tensor, frey_trained_params

pytestmark = pytest.mark.gpu

TC, FUSED, LAYERS = "step_tc_kernel", "fused_step_kernel", "per-layer kernels"
MNIST = (784, 500, 20, False)          # C2
FREY = (560, 200, 2, True)             # C1: Gaussian decoder


def _model(shape, M, params=None, x=None, **kw):
    import vaeb_b200
    D, H, Z, cont = shape
    if x is None:
        x = O.synthetic_frey(8) if cont else O.synthetic_mnist(8)
    return vaeb_b200.VAEB(x, cont, H, Z, M, 1, 0.01, False, False, params, **kw)


def _rand_params(shape, seed):
    D, H, Z, cont = shape
    rng = np.random.RandomState(seed)
    return [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(D, H, Z, cont)]


@pytest.mark.parametrize("shape,M,kw,env,kernel", [
    (MNIST, 100, {}, {}, TC),
    (MNIST, 3000, {}, {}, FUSED),
    (MNIST, 100, {"precision": "bf16x3"}, {}, TC),
    (MNIST, 3000, {"precision": "bf16x3"}, {}, LAYERS),
    (MNIST, 100, {"precision": "bf16"}, {}, LAYERS),
    (MNIST, 3000, {"precision": "bf16"}, {}, LAYERS),
    (MNIST, 100, {"optimizer": "adadelta"}, {}, LAYERS),
    (MNIST, 3000, {"optimizer": "adadelta"}, {}, LAYERS),
    (MNIST, 100, {"optimizer": "adam"}, {}, LAYERS),
    (MNIST, 3000, {"optimizer": "adam"}, {}, LAYERS),
    (MNIST, 100, {"activation": "relu"}, {}, LAYERS),
    (MNIST, 3000, {"activation": "relu"}, {}, LAYERS),
    (MNIST, 100, {"encoder_layers": 2}, {}, LAYERS),
    (MNIST, 3000, {"encoder_layers": 2}, {}, LAYERS),
    (FREY, 100, {}, {}, TC),
    (FREY, 3000, {}, {}, FUSED),
    (FREY, 100, {"precision": "bf16x3"}, {}, LAYERS),     # no fp32 kernel could finish an overflowing step
    (MNIST, 100, {}, {"VAEB_B200_FUSED": "0"}, TC),
    (MNIST, 3000, {}, {"VAEB_B200_FUSED": "0"}, LAYERS),
    (FREY, 100, {}, {"VAEB_B200_FUSED": "0"}, LAYERS),
    (MNIST, 100, {}, {"VAEB_B200_STEP_TC": "0"}, FUSED),
    (MNIST, 100, {"precision": "bf16x3"}, {"VAEB_B200_STEP_TC": "0"}, LAYERS),
    (FREY, 100, {}, {"VAEB_B200_STEP_TC": "0"}, FUSED),
])
def test_step_kernel_selection(monkeypatch, shape, M, kw, env, kernel):
    for k, v in env.items():
        monkeypatch.setenv(k, v)                # read once, when the handle is created
    m = _model(shape, M, **kw)
    assert m.step_kernel_name().startswith(kernel), (kw, env, m.step_kernel_name())
    m.close()


def test_step_kernel_selection_by_rows():
    m = _model(MNIST, 100)
    for rows, kernel in [(1, TC), (128, TC), (129, FUSED), (4096, FUSED), (4097, LAYERS)]:
        assert m.step_kernel_name(rows).startswith(kernel), rows
    m.close()


def test_step_kernel_returns_when_a_setting_is_undone():
    from vaeb_b200 import _lib
    m = _model(MNIST, 100, optimizer="adam")
    assert m.step_kernel_name().startswith(LAYERS)
    _lib.check(m._lib.vaeb_set_optimizer(m._h, _lib.OPT_ADAGRAD, 0.95))
    assert m.step_kernel_name().startswith(TC)
    assert m.step_kernel_name(3000).startswith(FUSED)
    m.close()
    m = _model(MNIST, 100, activation="relu")
    assert m.step_kernel_name().startswith(LAYERS)
    _lib.check(m._lib.vaeb_set_hidden_activation(m._h, 1))        # tanh
    assert m.step_kernel_name().startswith(TC)
    assert m.step_kernel_name(3000).startswith(FUSED)
    m.close()


def test_streaming_updates_hand_an_overflowing_step_to_the_fp32_kernel():
    """The reference's trained Frey weights at lr = 0.01 explode at the second update (see test_gpu_step_kernel.py).  The
    first calls of a fresh handle are streaming updates: one launch of the tensor-core kernel for the group of four, which
    stops at the second update, and one of the fp32 kernel for the rest, with the update workspace no earlier call sized.
    Same bounds as update() one by one, parameters at the fp32 tier."""
    import vaeb_b200
    M, order = 100, [0, 1, 0, 1]
    params = frey_trained_params()
    x = O.synthetic_frey(300)[:2 * M]
    xp = vaeb_b200.pinned_empty((len(order) * M, x.shape[1]), np.float32)
    for k, i in enumerate(order):
        xp[k * M:(k + 1) * M] = x[i * M:(i + 1) * M]
    m1 = _model(FREY, M, params, x, seed=3)
    m2 = _model(FREY, M, params, x, seed=3)
    assert m1.step_kernel_name().startswith(TC)
    l0 = m1.launch_count()
    for k in range(len(order)):
        m1.update_host_async(xp[k * M:(k + 1) * M])
    a = m1.collect()
    # the tensor-core kernel (after its two set-up launches: activation mirrors, weight mirrors), then the fp32 kernel
    assert m1.launch_count() - l0 == 4
    b = np.array([float(m2.update(i)) for i in order], np.float32)
    np.testing.assert_allclose(a, b, rtol=1e-5)
    for p, q, n in zip(m1.get_params(), m2.get_params(), O.param_names(True)):
        assert_close_tensor(p, q, 1e-4, name=n)
    m1.close(); m2.close()


@pytest.mark.parametrize("M,precision,kernel,n_phases", [
    (100, "fp32", TC, 6),           # one stamp per grid barrier of the tensor-core kernel
    (300, "fp32", FUSED, 8),        # ... of the fp32 kernel
    # the per-layer launches of the 2048-row tensor-core path: enc1, enc2, dec1, dec2, dgrad h_d, dz, dgrad h_e, the
    # weight gradients and the tail (the tail of the update before wrote the weight mirrors)
    (2048, "bf16x3", LAYERS, 9),
])
def test_profile_update_leaves_the_model_as_it_was(M, precision, kernel, n_phases):
    x = O.synthetic_mnist(2 * M)
    m, twin = [_model(MNIST, M, _rand_params(MNIST, 4), x, precision=precision, seed=7) for _ in range(2)]
    assert m.step_kernel_name().startswith(kernel)
    m.update(0); twin.update(0)                 # accumulators that are not zero
    params, ada, launches = m.get_params(), m._get_buffer(1), m.launch_count()
    phases = m.profile_update(index=1, iters=5)
    assert len(phases) == n_phases, [p[0] for p in phases]
    ms = np.array([p[1] for p in phases])
    assert np.isfinite(ms).all() and (ms > 0).all(), phases
    for a, b in zip(m.get_params(), params):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(m._get_buffer(1), ada):
        np.testing.assert_array_equal(a, b)
    assert m.launch_count() == launches
    # the step counter: validate draws its noise from it
    assert float(m.validate(x)) == float(twin.validate(x))
    m.close(); twin.close()
