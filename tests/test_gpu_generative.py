"""The evaluation and generation entry points: encode (q(z|x) alone), validate_terms (the two terms of the per-row
bound) and sample (draws from p(z) p(x|z) on the device), against the fp64 oracle and against the library's own
validate / decode; and the CLI's --sample_file tile."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests import sample_oracle as S
from tests.util import assert_close_tensor

pytestmark = pytest.mark.gpu
RTOL = 1e-4
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _data(n, D, continuous, seed=5):
    if continuous:
        return np.clip(np.random.RandomState(seed).normal(0.5, 0.2, (n, D)), 0.01, 0.99).astype(np.float32)
    return O.synthetic_mnist(n, seed=seed, D=D)


def _params(D, H, Z, continuous, depth=1, seed=21, scale=None):
    rng = np.random.RandomState(seed)
    scale = scale or (0.05 if D > 100 else 0.2)
    return [rng.normal(0, scale, s).astype(np.float32) for s in O.param_shapes(D, H, Z, continuous, depth)]


def _p64(params, continuous):
    return O.as_dict([p.astype(np.float64) for p in params], continuous)


# ---- encode -------------------------------------------------------------------------------
@pytest.mark.parametrize("act,depth,continuous,D,H,Z,n,precision", [
    ("tanh", 1, False, 784, 500, 20, 1001, "fp32"),       # C2 shape, ragged n
    ("sigmoid", 3, True, 560, 200, 2, 1001, "fp32"),      # C1 shape, Gaussian decoder, deeper encoder
    ("relu", 1, False, 784, 500, 20, 40001, "fp32"),      # more rows than one 32768-row chunk
    ("relu", 3, False, 40, 24, 3, 77, "fp32"),
    ("tanh", 1, False, 784, 500, 20, 1001, "bf16"),       # the fp32 kernels serve every precision
])
def test_encode_matches_oracle(act, depth, continuous, D, H, Z, n, precision):
    import vaeb_b200
    params = _params(D, H, Z, continuous, depth)
    m = vaeb_b200.VAEB(_data(100, D, continuous), continuous, H, Z, 100, 1, 0.01, False, False, params,
                       activation=act, encoder_layers=depth, precision=precision)
    x = _data(n, D, continuous, seed=8)
    mu, lv = m.encode(x)
    assert mu.shape == (n, Z) and lv.shape == (n, Z)
    _, mu_ref, lv_ref = O.encoder(_p64(params, continuous), x.astype(np.float64), act)
    assert_close_tensor(mu, mu_ref, RTOL, name="mu")
    assert_close_tensor(lv, lv_ref, RTOL, name="log_var")
    m.close()


# ---- validate_terms --------------------------------------------------------------------------
@pytest.mark.parametrize("est,L,continuous,D,H,Z,n,precision", [
    ("LB", 1, False, 784, 500, 20, 2500, "fp32"),      # >= 2048 rows: the many-block finalize kernel
    ("LB", 3, False, 784, 500, 20, 301, "fp32"),
    ("LA", 1, True, 560, 200, 2, 301, "fp32"),
    ("LA", 3, False, 784, 500, 20, 2500, "fp32"),
    ("LB", 3, True, 560, 200, 2, 2500, "fp32"),
    ("LA", 2, False, 40, 24, 3, 77, "fp32"),
    ("LB", 1, False, 784, 500, 20, 2500, "bf16x3"),    # the tensor-core decoder layer feeds the same finalize
])
def test_validate_terms(est, L, continuous, D, H, Z, n, precision):
    import vaeb_b200
    params = _params(D, H, Z, continuous)
    m = vaeb_b200.VAEB(_data(100, D, continuous), continuous, H, Z, 100, L, 0.01, est == "LA", False, params,
                       precision=precision)
    x = _data(n, D, continuous, seed=8)
    eps = np.random.RandomState(9).normal(size=(L, n, Z)).astype(np.float32)
    _, rows = m.validate(x, eps=eps, per_row=True)
    ll, aux = m.validate_terms(x, eps=eps)
    s = ll + aux                                          # float32 sum
    if L & (L - 1) == 0:
        np.testing.assert_array_equal(s, rows)            # 1/L exact: the bound's fused multiply-add rounds once
    else:
        # the bound is fma(sum, 1/L, aux); loglik is sum * (1/L) rounded, so the float sum may differ in the last bit
        assert np.all(np.abs(s.astype(np.float64) - rows) <= np.spacing(np.abs(rows))), np.abs(s - rows).max()
    p = _p64(params, continuous)
    x64, e64 = x.astype(np.float64), eps.astype(np.float64)
    _, mu, ls = O.encoder(p, x64)
    ll_ref = np.zeros(n)
    la_ref = np.zeros(n)
    for l in range(L):
        z = O.reparam(mu, ls, e64[l])
        _, a, lv = O.decoder(p, z, continuous)
        ll_ref += O.log_px_given_z(x64, a, lv, continuous) / L
        prior = (-0.5 * O.LOG2PI - 0.5 * z ** 2).sum(axis=1)
        logq = (-0.5 * O.LOG2PI - 0.5 * ls - 0.5 * (z - mu) ** 2 / np.exp(ls)).sum(axis=1)
        la_ref += (prior - logq) / L
    aux_ref = la_ref if est == "LA" else O.kl_rows(mu, ls)
    np.testing.assert_allclose(ll, ll_ref, rtol=RTOL)
    assert_close_tensor(aux, aux_ref, RTOL, name="aux")
    m.close()


def test_validate_terms_full_vb():
    """Full-VB handles return the same two per-row terms; the weight-prior term is not per row."""
    import vaeb_b200
    D, H, Z, n = 784, 500, 20, 300
    params = _params(D, H, Z, False)
    m = vaeb_b200.VAEB(_data(100, D, False), False, H, Z, 100, 1, 0.01, False, True, params)
    x = _data(n, D, False, seed=8)
    eps = np.random.RandomState(9).normal(size=(1, n, Z)).astype(np.float32)
    _, rows = m.validate(x, eps=eps, per_row=True)
    ll, aux = m.validate_terms(x, eps=eps)
    np.testing.assert_array_equal(ll + aux, rows)
    m.close()


# ---- sample ----------------------------------------------------------------------------------
SEED, STEP = 10, 3


def _sample_model(continuous):
    import vaeb_b200
    D, H, Z = (560, 200, 2) if continuous else (784, 500, 20)
    params = _params(D, H, Z, continuous, scale=0.1)
    return vaeb_b200.VAEB(_data(100, D, continuous), continuous, H, Z, 100, 1, 0.01, False, False, params,
                          seed=SEED), params


@pytest.mark.parametrize("continuous", [False, True])
def test_sample_matches_oracle_and_decode(continuous):
    m, params = _sample_model(continuous)
    n, D, Z = 1001, m.input_size, m.n_latent
    z, mean, lv, x = m.sample(n, step=STEP, return_all=True)
    assert z.shape == (n, Z) and mean.shape == (n, D) and x.shape == (n, D) and (lv is None) == (not continuous)
    # z: the Philox normals of (seed, stream 5, step, sample 0); the project's RNG parity tolerance
    np.testing.assert_allclose(z, O.philox_normal(SEED, S.STREAM_SAMPLE, STEP, n * Z).reshape(n, Z), rtol=0, atol=3e-6)
    # the decoder outputs are decode(z)'s, bit for bit
    dec = m.decode(z)
    if continuous:
        np.testing.assert_array_equal(mean, dec[0])
        np.testing.assert_array_equal(lv, dec[1])
        eps = O.philox_normal(SEED, S.STREAM_SAMPLE, STEP, n * D, sample=1).reshape(n, D)
        np.testing.assert_allclose((x - mean) * np.exp(-0.5 * lv), eps, rtol=0, atol=1e-5)
    else:
        np.testing.assert_array_equal(mean, dec)
        assert set(np.unique(x)) <= {0.0, 1.0}
        u = S.philox_uniform(SEED, S.STREAM_SAMPLE, STEP, n * D, sample=1).reshape(n, D)
        np.testing.assert_array_equal(x, (u < mean).astype(np.float32))      # the same uniform, bit for bit
        _, _, _, x_ref = S.sample([p.astype(np.float64) for p in params], n, SEED, STEP, 0, False)
        y_ref = O.sigmoid(O.decoder(_p64(params, False), z.astype(np.float64), False)[1])
        far = np.abs(u - y_ref) >= 1e-5
        np.testing.assert_array_equal(x[far], x_ref[far])
    # the output pointers are optional
    assert np.array_equal(m.sample(n, step=STEP), x)
    m.close()


@pytest.mark.parametrize("continuous", [False, True])
def test_sample_does_not_depend_on_the_row_split(continuous):
    m, _ = _sample_model(continuous)
    n, k = 1001, 397
    whole = m.sample(n, step=STEP, return_all=True)
    lo = m.sample(k, step=STEP, row_offset=0, return_all=True)
    hi = m.sample(n - k, step=STEP, row_offset=k, return_all=True)
    for w, a, b in zip(whole, lo, hi):
        if w is not None:
            np.testing.assert_array_equal(w, np.concatenate([a, b]))
    other = m.sample(n, step=STEP + 1)
    assert not np.array_equal(other, whole[3])          # the step is part of the counter
    m.close()


def test_bernoulli_sample_frequencies():
    m, _ = _sample_model(False)
    n = (1 << 16) + 1001                                   # two 65536-row chunks
    _, mean, _, x = m.sample(n, step=STEP, return_all=True)
    freq = x.mean(axis=0, dtype=np.float64)
    p = mean.mean(axis=0, dtype=np.float64)
    sd = np.sqrt((mean.astype(np.float64) * (1 - mean)).sum(axis=0)) / n
    assert np.all(np.abs(freq - p) <= 5 * sd + 1e-12), np.max(np.abs(freq - p) / sd)
    m.close()


def test_cli_writes_sample_tile(tmp_path):
    out = tmp_path / "s.pgm"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "VAEB.py"), "--synthetic", "--n_epochs", "1",
                        "--sample_file", str(out)], cwd=str(tmp_path), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    data = out.read_bytes()
    header = b"P5 280 280 255\n"                            # 10 x 10 MNIST tiles of 28 x 28
    assert data.startswith(header) and len(data) == len(header) + 280 * 280
