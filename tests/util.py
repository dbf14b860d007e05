import os

import numpy as np

from oracle import vaeb_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name)))


def frey_trained_params():
    # stored in two halves so that neither file exceeds 1 MB
    z = load_golden("frey_z2_trained_encoder.npz")
    z.update(load_golden("frey_z2_trained_decoder.npz"))
    return [z[n] for n in O.param_names(True)]


def fingerprint(grads):
    fp = []
    for g in grads:
        f = np.asarray(g, dtype=np.float64).ravel()
        idx = np.linspace(0, f.size - 1, 8).astype(int)
        fp.append(np.concatenate([[f.sum(), (f * f).sum(), np.abs(f).max()], f[idx]]))
    return np.stack(fp)


def assert_close_tensor(got, ref, rtol=1e-4, floor=0.05, name=""):
    """The stated fp32 tolerance (SURVEY.md 7 'hard parts'): |d| <= rtol*max(|ref|, floor*||ref||_inf).
    Gradients that are sums of cancelling terms make a purely relative bound ill-posed."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    scale = np.maximum(np.abs(ref), floor * (np.abs(ref).max() if ref.size else 0.0))
    err = np.abs(got - ref)
    bad = err > rtol * scale + 1e-30
    if bad.any():
        i = np.unravel_index(np.argmax(err / (scale + 1e-300)), err.shape)
        raise AssertionError("%s: max violation at %s: got %r ref %r (err %.3e, allowed %.3e)"
                             % (name, i, got[i], ref[i], err[i], rtol * scale[i]))
    return float((err / (scale + 1e-300)).max()) if err.size else 0.0
