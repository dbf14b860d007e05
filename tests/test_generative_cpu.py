"""CPU checks of the pieces behind vaeb_sample: the Philox uniform of tests/sample_oracle.py
(philox.cuh:philox_uniform1), its reference sampler and the 10 x 10 sample tile the CLI writes."""
import numpy as np

from oracle import vaeb_oracle as O
from tests import sample_oracle as S


def test_philox_bits_known_answers():
    # Random123 known-answer vectors of Philox4x32-10: counter 0, key 0 is element group 0 of (seed 0, stream 0,
    # step 0, sample 0); the all-ones and pi-digit vectors go through the block function directly
    np.testing.assert_array_equal(S.philox_bits(0, 0, 0, 4), [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8])
    r = O.philox4x32_10(np.full((1, 4), 0xFFFFFFFF, np.uint32), np.full((1, 2), 0xFFFFFFFF, np.uint32))[0]
    np.testing.assert_array_equal(r, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd])
    r = O.philox4x32_10(np.array([[0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]], np.uint32),
                        np.array([[0xa4093822, 0x299f31d0]], np.uint32))[0]
    np.testing.assert_array_equal(r, [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])


def test_philox_bits_counter_layout():
    # element e of (stream, step, sample) is output e % 4 of counter (g_lo, g_hi | stream << 24, sample, step),
    # g = e // 4, key (seed_lo, seed_hi) -- checked at a group index above 2^32
    seed, stream, step, sample = 0x123456789, 5, 77, 1
    g = (1 << 33) + 5
    ctr = np.array([[g & 0xFFFFFFFF, (g >> 32) | (stream << 24), sample, step]], np.uint32)
    key = np.array([[seed & 0xFFFFFFFF, seed >> 32]], np.uint32)
    want = O.philox4x32_10(ctr, key)[0]
    got = S.philox_bits(seed, stream, step, 4, sample=sample, first=4 * g)
    np.testing.assert_array_equal(got, want)
    # an unaligned window is the matching slice of an aligned one
    full = S.philox_bits(seed, stream, step, 40, sample=sample)
    np.testing.assert_array_equal(S.philox_bits(seed, stream, step, 29, sample=sample, first=7), full[7:36])


def test_philox_uniform_values_and_range():
    u = S.philox_uniform(0, 0, 0, 4)
    want = [((v >> 8) + 0.5) * 2.0 ** -24 for v in (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)]
    np.testing.assert_array_equal(u, np.float32(want))
    u = S.philox_uniform(10, 5, 3, 1 << 16, sample=1)
    assert u.dtype == np.float32 and u.min() > 0.0 and u.max() < 1.0
    assert abs(float(u.mean()) - 0.5) < 5 * np.sqrt(1 / 12 / u.size)


def test_philox_uniform_feeds_philox_normal():
    # the uniforms are the ones philox_normal's Box-Muller consumes: pairs (u0, u1) and (u2, u3) of each group
    n = 4 * 1000
    for seed, stream, step, sample in [(10, 0, 0, 0), (15485863, 2, 41, 7), (10, 5, 3, 1)]:
        u = S.philox_uniform(seed, stream, step, n, sample=sample).reshape(-1, 4)
        rad0 = np.sqrt(np.float32(-2.0) * np.log(u[:, 0]))
        rad1 = np.sqrt(np.float32(-2.0) * np.log(u[:, 2]))
        th0 = np.float32(2.0 * np.pi) * u[:, 1]
        th1 = np.float32(2.0 * np.pi) * u[:, 3]
        nrm = np.stack([rad0 * np.cos(th0), rad0 * np.sin(th0), rad1 * np.cos(th1), rad1 * np.sin(th1)], axis=-1)
        np.testing.assert_array_equal(nrm.reshape(-1).astype(np.float32),
                                      O.philox_normal(seed, stream, step, n, sample=sample))


def _params(D, H, Z, continuous, seed=3, scale=0.3):
    rng = np.random.RandomState(seed)
    return [rng.normal(0, scale, s) for s in O.param_shapes(D, H, Z, continuous)]


def test_oracle_sample_draws():
    D, H, Z, n = 30, 16, 3, 101
    for continuous in (False, True):
        params = _params(D, H, Z, continuous)
        z, y, lv, x = S.sample(params, n, 10, 4, 0, continuous)
        np.testing.assert_array_equal(z, O.philox_normal(10, S.STREAM_SAMPLE, 4, n * Z).reshape(n, Z))
        np.testing.assert_allclose(y, O.sigmoid(O.decoder(O.as_dict(params, continuous), z, continuous)[1]))
        if continuous:
            eps = O.philox_normal(10, S.STREAM_SAMPLE, 4, n * D, sample=1).reshape(n, D)
            np.testing.assert_allclose((x - y) * np.exp(-0.5 * lv), eps, atol=1e-12)
        else:
            assert lv is None and set(np.unique(x)) <= {0.0, 1.0}
            u = S.philox_uniform(10, S.STREAM_SAMPLE, 4, n * D, sample=1).reshape(n, D)
            np.testing.assert_array_equal(x, (u < y).astype(x.dtype))
        # rows keyed by their global index: a split into two calls gives the same draws
        k = 37
        a = S.sample(params, k, 10, 4, 0, continuous)
        b = S.sample(params, n - k, 10, 4, k, continuous)
        for whole, lo, hi in zip((z, y, lv, x), a, b):
            if whole is not None:
                np.testing.assert_array_equal(whole, np.concatenate([lo, hi]))


def test_sample_tile_is_a_mnist_sized_pgm(tmp_path):
    from vaeb_b200 import manifold

    class _Stub:
        continuous = False

        def sample(self, n, step=0, row_offset=0, return_all=False):
            rng = np.random.RandomState(step)
            mean = rng.uniform(size=(n, 784)).astype(np.float32)
            x = (mean > 0.5).astype(np.float32)
            return (None, mean, None, x) if return_all else x

    faces, tiled = manifold.render_samples(_Stub())
    assert faces.shape == (100, 784) and tiled.shape == (280, 280)
    np.testing.assert_array_equal(faces, _Stub().sample(100, return_all=True)[1])     # the decoder means
    path = str(tmp_path / "s.pgm")
    manifold.save_pgm(tiled, path)
    assert open(path, "rb").read().startswith(b"P5 280 280 255\n")
