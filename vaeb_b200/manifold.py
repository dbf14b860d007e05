"""Learned-manifold renderer (freyFace.py:346-369): decode a grid of latent points placed at Gaussian quantiles and
tile the decoded images.  Host side only -- the decoder pass is one `vaeb_decode` call for the whole grid (the
reference compiles a Theano function and calls it once per grid point)."""
from __future__ import annotations

from statistics import NormalDist

import numpy as np

# VAEBImage.py:7-11: data-item length -> image size, memory order, rotation
DIMENSIONS = {784: (28, 28), 560: (20, 28)}
ORDER = {784: "C", 560: "F"}
ROT90 = {784: 0, 560: -1}          # rotate(-90): one clockwise quarter turn


def grid_points(n=10, offset=0.9):
    """z[(ii, jj)] = (ppf((ii + offset)/n), ppf((jj + offset)/n)) -- freyFace.py:352 uses offset 0.9 (so the last
    quantile is 0.99, not a centred (ii + 0.5)/n grid); row-major over (ii, jj)."""
    q = [NormalDist().inv_cdf((i + offset) / n) for i in range(n)]
    return np.asarray([[q[ii], q[jj]] for ii in range(n) for jj in range(n)], np.float32)


def to_image(x):
    """One decoded row -> 2-D array in display orientation (VAEBImage.py:13-21, without the 1-x inversion)."""
    x = np.asarray(x)
    img = x.reshape(DIMENSIONS[x.size], order=ORDER[x.size])
    return np.rot90(img, ROT90[x.size]) if ROT90[x.size] else img


def render(model, n=10, offset=0.9, sample=False, rng=None):
    """(faces[n*n, D], tiled[n*h, n*w]) for a model with a 2-d latent space.  Gaussian decoder: the mean image, or
    with sample=True a draw y ~ N(mu, diag(exp(log_sigma)**2)) as freyFace.py:358-361 does (through a dense DxD
    covariance there; the diagonal draw is the same distribution)."""
    if model.n_latent != 2:
        raise ValueError("the manifold grid needs a 2-d latent space (freyFace.py:352)")
    out = model.decode(grid_points(n, offset))
    if model.continuous:
        mu, ls = out
        faces = mu
        if sample:
            rng = np.random if rng is None else rng
            faces = mu + np.exp(ls) * rng.standard_normal(mu.shape).astype(np.float32)
    else:
        faces = out
    return faces, tile(faces, n)


def tile(faces, n):
    """n x n data rows -> one 2-D image, row-major (VAEBImage.py:25-41)."""
    tiles = [to_image(f) for f in faces]
    return np.vstack([np.hstack(tiles[ii * n:(ii + 1) * n]) for ii in range(n)])


def render_samples(model, n=10, step=0):
    """(faces[n*n, D], tiled) of n*n random samples from the generative model (AEVB Fig. 5).  A Bernoulli model shows
    its decoder means, as the paper's figure does: the binary draws themselves make a poor image."""
    z, mean, lv, x = model.sample(n * n, step=step, return_all=True)
    faces = x if model.continuous else mean
    return faces, tile(faces, n)


def save_pgm(img, path):
    """8-bit greyscale dump with VAEBImage.save_image's (1 - x)*255 inversion; PGM needs no imaging library."""
    a = np.clip((1.0 - np.asarray(img, np.float64)) * 255.0, 0, 255).astype(np.uint8)
    with open(path, "wb") as f:
        f.write(b"P5 %d %d 255\n" % (a.shape[1], a.shape[0]))
        f.write(a.tobytes())


def save_image(x, filename):
    """VAEBImage.save_image (VAEBImage.py:13-21): one data row -> image file with the (1 - x)*255 inversion, in the
    dataset's orientation.  `.jpg` / `.png` go through PIL when it is installed (as in the reference); `.pgm` needs
    no imaging library.  Returns the 2-D uint8 array that was written."""
    x = np.asarray(x, np.float32).ravel()
    if x.size not in DIMENSIONS:
        raise ValueError("save_image knows MNIST (784) and Frey Face (560) rows, got %d values" % x.size)
    img = to_image(x)
    a = np.clip((1.0 - np.asarray(img, np.float64)) * 255.0, 0, 255).astype(np.uint8)
    if filename.lower().endswith(".pgm"):
        save_pgm(img, filename)
        return a
    try:
        from PIL import Image
    except ImportError as ex:                             # pragma: no cover
        raise RuntimeError("writing %s needs PIL; use a .pgm file name instead" % filename) from ex
    Image.fromarray(a).convert("RGB").save(filename)
    return a
