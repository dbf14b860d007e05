"""tcgen05 / TMA building blocks on the B200: the generic bf16 GEMM in all four operand-major
combinations, ragged shapes, every UMMA N used by the step kernels."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _bf16_round(a):
    u = np.ascontiguousarray(a, np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


def _run(M, N, K, a_mn, b_mn, bn, seed=0):
    from vaeb_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(seed)
    A = rng.normal(size=(M, K)).astype(np.float32)
    B = rng.normal(size=(K, N)).astype(np.float32)
    Cm = np.empty((M, N), np.float32)
    _lib.check(lib.vaeb_tc_gemm_test(0, M, N, K, a_mn, b_mn, bn, A.ctypes.data_as(C.c_void_p),
                                     B.ctypes.data_as(C.c_void_p), Cm.ctypes.data_as(C.c_void_p)))
    ref = _bf16_round(A).astype(np.float64) @ _bf16_round(B).astype(np.float64)
    return Cm, ref


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("bn", [64, 128, 256])
def test_tc_gemm_majors(a_mn, b_mn, bn):
    Cm, ref = _run(256, 512, 192, a_mn, b_mn, bn)
    np.testing.assert_allclose(Cm, ref, rtol=2e-5, atol=2e-4)


@pytest.mark.parametrize("M,N,K", [(104, 504, 784), (128, 784, 504), (504, 784, 104), (8, 8, 8), (136, 72, 520)])
def test_tc_gemm_ragged_shapes(M, N, K):
    # the AEVB shapes: M=100->104, H=500->504, D=784; TMA zero-fills the out-of-bounds part of a box
    for a_mn, b_mn in ((0, 1), (0, 0), (1, 1)):
        Cm, ref = _run(M, N, K, a_mn, b_mn, 64, seed=M + N)
        np.testing.assert_allclose(Cm, ref, rtol=2e-5, atol=5e-4)


def test_tc_gemm_small_n_tile():
    Cm, ref = _run(128, 96, 256, 0, 0, 32)
    np.testing.assert_allclose(Cm, ref, rtol=2e-5, atol=2e-4)


# ---- importance-sampled log p(x) on the tensor cores (is_tc.cu), bf16 tier ---------------------------
def _is_case(D, H, Z, n, L, seed, scale, continuous=False):
    import vaeb_b200
    from oracle import vaeb_oracle as O
    rng = np.random.RandomState(seed)
    if continuous:
        x = np.clip(rng.normal(0.5, 0.2, (n, D)), 0.01, 0.99).astype(np.float32)
    else:
        x = (rng.uniform(size=(n, D)) * (rng.uniform(size=(n, D)) < 0.3)).astype(np.float32)
    params = [rng.normal(0, scale, s).astype(np.float32) for s in O.param_shapes(D, H, Z, continuous)]
    eps = rng.normal(size=(n, L, Z)).astype(np.float32)
    m = vaeb_b200.VAEB(x, continuous, H, Z, max(1, min(n, 4)), 1, 0.01, False, False, params, precision="bf16")
    lp, lw = m.log_px(x, L=L, eps=eps, return_weights=True)
    ref_lp, ref_lw = O.is_log_px([p.astype(np.float64) for p in params], x.astype(np.float64), eps.astype(np.float64),
                                 continuous)
    m.close()
    return lp, lw, ref_lp, ref_lw


@pytest.mark.parametrize("D,H,Z,n,L", [(784, 500, 20, 5, 300), (37, 29, 3, 4, 130), (560, 200, 2, 3, 128), (100, 64, 8, 2, 7)])
def test_is_logpx_tensor_core_matches_oracle(D, H, Z, n, L):
    lp, lw, ref_lp, ref_lw = _is_case(D, H, Z, n, L, 11, 0.08)
    # bf16 operands, fp32 accumulation: the 1e-2 tier (north star), per sample and per point
    np.testing.assert_allclose(lw, ref_lw, rtol=1e-2, atol=1e-2)
    np.testing.assert_allclose(lp, ref_lp, rtol=1e-2, atol=1e-2)


@pytest.mark.parametrize("D,H,Z,n,L", [(560, 200, 2, 5, 300), (784, 500, 20, 3, 130), (38, 29, 3, 4, 7)])
def test_is_logpx_tensor_core_gaussian_decoder(D, H, Z, n, L):
    """The importance-sampling kernel with the Gaussian decoder (VERDICT r1 item 6): the output sweep runs over the
    interleaved head [W2|W6]' (2 D columns), the epilogue folds pixel pairs (a_d, lv_d) into the log-density of
    VAEB.py:304-307.  C1's shape, the MNIST shape, a ragged one; bf16 tier."""
    lp, lw, ref_lp, ref_lw = _is_case(D, H, Z, n, L, 12, 0.08, continuous=True)
    np.testing.assert_allclose(lw, ref_lw, rtol=1e-2, atol=1e-2)
    np.testing.assert_allclose(lp, ref_lp, rtol=1e-2, atol=1e-2)
    # the Philox path (no injected noise, pipelined host input) agrees with itself across calls and stays finite
    import vaeb_b200
    from oracle import vaeb_oracle as O
    rng = np.random.RandomState(5)
    x = np.clip(rng.normal(0.5, 0.2, (700, D)), 0.01, 0.99).astype(np.float32)
    params = [rng.normal(0, 0.08, s).astype(np.float32) for s in O.param_shapes(D, H, Z, True)]
    m = vaeb_b200.VAEB(x[:4], True, H, Z, 4, 1, 0.01, False, False, params, precision="bf16")
    a = m.log_px(x, L=64)
    b = m.log_px(x[:300], L=64)
    assert np.isfinite(a).all()
    np.testing.assert_array_equal(a[:300], b)
    m.close()


def test_is_logpx_tensor_core_philox_sharding_invariance():
    import vaeb_b200
    from oracle import vaeb_oracle as O
    D, H, Z, n, L = 784, 500, 20, 12, 700
    rng = np.random.RandomState(2)
    x = (rng.uniform(size=(n, D)) * (rng.uniform(size=(n, D)) < 0.2)).astype(np.float32)
    params = [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(D, H, Z, False)]
    m = vaeb_b200.VAEB(x, False, H, Z, 4, 1, 0.01, False, False, params, precision="bf16")
    whole = m.log_px(x, L=L)
    parts = np.concatenate([m.log_px(x[:5], L=L, row_offset=0), m.log_px(x[5:], L=L, row_offset=5)])
    assert np.array_equal(whole, parts)                      # bit-identical for any sharding of the points
    m32 = vaeb_b200.VAEB(x, False, H, Z, 4, 1, 0.01, False, False, params, precision="fp32")
    ref = m32.log_px(x, L=L)                                 # same Philox draws, fp32 arithmetic
    np.testing.assert_allclose(whole, ref, rtol=1e-2)
    m.close(); m32.close()

