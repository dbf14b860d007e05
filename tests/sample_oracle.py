"""CPU restatement of vaeb_sample's noise and draws (test infrastructure, beside oracle/vaeb_oracle.py, whose
Philox block function, normals and decoder it builds on): the Philox uniform of philox.cuh:philox_uniform1 and the
sampler's reference."""
import numpy as np

from oracle.vaeb_oracle import as_dict, decoder, philox4x32_10, philox_normal, sigmoid

STREAM_SAMPLE = 5      # VAEB_STREAM_SAMPLE, philox.cuh


def philox_bits(seed, stream, step, n_elems, sample=0, first=0):
    """The uint32 Philox output of flat elements first..first+n_elems-1 of (stream, step, sample): output e % 4 of
    group e // 4, with philox_normal's counter layout."""
    g = np.arange(first // 4, (first + n_elems + 3) // 4, dtype=np.uint64)
    ctr = np.empty((len(g), 4), dtype=np.uint32)
    ctr[:, 0] = (g & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    ctr[:, 1] = ((g >> np.uint64(32)).astype(np.uint32) & np.uint32(0x00FFFFFF)) | np.uint32((stream & 0xFF) << 24)
    ctr[:, 2] = np.uint32(sample & 0xFFFFFFFF)
    ctr[:, 3] = np.uint32(step & 0xFFFFFFFF)
    key = np.empty((len(g), 2), dtype=np.uint32)
    key[:, 0] = np.uint32(seed & 0xFFFFFFFF)
    key[:, 1] = np.uint32((seed >> 32) & 0xFFFFFFFF)
    r = philox4x32_10(ctr, key).reshape(-1)
    return r[first % 4:first % 4 + n_elems]


def philox_uniform(seed, stream, step, n_elems, sample=0, first=0):
    """fp32 U(0,1) of flat elements first.. of (stream, step, sample) (philox.cuh:philox_uniform1): the uniform
    ((r >> 8) + 0.5) * 2**-24 that philox_normal makes of the same element's uint32 output."""
    r = philox_bits(seed, stream, step, n_elems, sample, first)
    return ((r >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)


def sample(params, n, seed, step, row_offset, continuous, act="tanh"):
    """``vaeb_sample``: n draws from the generative model p(z) p(x|z) (AEVB Fig. 5) with the device's noise.  Global
    row r = row_offset + i: z[i, j] = Philox normal r*Z + j of (stream 5, step, sample 0); the draw of x uses element
    r*D + d of (stream 5, step, sample 1) -- Bernoulli x = (u < y), Gaussian x = y + exp(lv / 2) * eps: the variance of
    ``log_px_given_z`` (VAEB.py:302-313).  Returns (z, y, lv or None, x) in the dtype of the parameters."""
    p = as_dict(params, continuous)
    Z, D = p["W1"].shape[0], p["W2"].shape[1]
    dt = p["W1"].dtype
    z = philox_normal(seed, STREAM_SAMPLE, step, (row_offset + n) * Z, sample=0)[row_offset * Z:].reshape(n, Z)
    _, a, lv = decoder(p, z.astype(dt), continuous, act)
    y = sigmoid(a)
    if continuous:
        e = philox_normal(seed, STREAM_SAMPLE, step, (row_offset + n) * D, sample=1)[row_offset * D:].reshape(n, D)
        x = y + np.exp(0.5 * lv) * e
    else:
        u = philox_uniform(seed, STREAM_SAMPLE, step, n * D, sample=1, first=row_offset * D).reshape(n, D)
        x = (u < y).astype(dt)
    return z, y, lv, x
