"""The tensor-core step kernel keeps two copies of its k-major [W4|W5] operand mirror: a step reads one while its
epilogue writes the updated weights into the other.  Which copy holds the current weights must follow the kernel's own
steps, not the parity of the Philox step counter -- validate and reconstruct advance that counter by one without
touching the mirrors.  Updates interleaved with validate calls must therefore match the fp64 oracle as updates alone
do, and bit for bit as a handle whose mirrors were rebuilt at that point."""
import numpy as np
import pytest

from oracle import vaeb_oracle as O

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("between", ["validate", "reconstruct"])
def test_step_kernel_after_counter_only_calls_matches_oracle(between):
    import vaeb_b200
    D, H, Z, M = 784, 500, 20, 100
    x = O.synthetic_mnist(4 * M, seed=21)
    rng = np.random.RandomState(4)
    params = [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(D, H, Z, False)]
    m = vaeb_b200.VAEB(x, False, H, Z, M, 1, 0.01, False, False, params)
    o = O.OracleVAEB(x, False, H, Z, M, L=1, params=params)
    assert m.step_kernel_name().startswith("step_tc_kernel")
    # each bound is computed with the parameters the previous update produced (Adagrad's first steps move every
    # element by about lr whatever its gradient, so the parameters themselves are compared through the bounds)
    for i in range(5):
        eps = rng.normal(size=(1, M, Z)).astype(np.float32)
        got, ref = float(m.update(i % 4, eps=eps)), o.update(i % 4, eps)
        assert abs(got - ref) <= 1e-4 * abs(ref), (i, got, ref)
        if between == "validate":
            m.validate(x[:64])
        else:
            m.reconstruct(x[:8], 1)
    m.close()


@pytest.mark.parametrize("between", ["validate", "reconstruct"])
def test_step_kernel_mirrors_after_counter_only_calls_equal_rebuilt_ones(between):
    """Bitwise: updates after a validate / reconstruct read the same [W4|W5] operands as a handle whose mirrors were
    rebuilt from the fp32 parameters at that point (set_params writes both copies)."""
    import vaeb_b200
    D, H, Z, M = 784, 500, 20, 100
    x = O.synthetic_mnist(4 * M, seed=21)
    rng = np.random.RandomState(4)
    params = [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(D, H, Z, False)]
    out = []
    for rebuild in (False, True):
        m = vaeb_b200.VAEB(x, False, H, Z, M, 1, 0.01, False, False, params)
        bounds = [float(m.update(0))]
        if between == "validate":
            m.validate(x[:64])
        else:
            m.reconstruct(x[:8], 1)
        if rebuild:
            m.set_params(m.get_params())
        bounds += [float(m.update(i)) for i in (1, 2, 3)]
        out.append((bounds, m.get_params(), m._get_buffer(1)))
        m.close()
    assert out[0][0] == out[1][0]
    for a, b in zip(out[0][1] + out[0][2], out[1][1] + out[1][2]):
        np.testing.assert_array_equal(a, b)
