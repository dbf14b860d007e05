"""Generates tests/golden/*.npz.  Run in the build container (needs /root/reference):
    python tests/golden/make_golden.py

frey_z2_trained_{encoder,decoder}.npz
                     -- the trained fp32 Frey weights the reference ships in
                        reconstruction_res/continuous_2.mdl (12 tensors, reference order),
                        extracted with the restricted unpickler (vaeb_b200/io.py); W3-W5, b3-b5
                        in the first file, W1, W2, W6, b1, b2, b6 in the second.
golden_frey_z2.npz   -- oracle (fp64) outputs for those weights on seeded synthetic
                        Frey-shaped rows with seeded eps: per-row bound, SGVB, gradient
                        fingerprints, parameters after one Adagrad step, IS estimates.
golden_mnist_init.npz-- the same for the reference initialisation (RandomState(10)) of the
                        MNIST-shaped Bernoulli model, LB and LA estimators.
The reference has no input/output vectors of its own (SURVEY.md 4, 8c): these files pin the
oracle against regressions and give the GPU tests committed numbers to hit."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import vaeb_oracle as O  # noqa: E402
from vaeb_b200 import io  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"


def fingerprint(grads):
    """Per tensor: [sum, sum of squares, max abs] + 8 entries at fixed strides."""
    fp = []
    for g in grads:
        f = g.ravel()
        idx = np.linspace(0, f.size - 1, 8).astype(int)
        fp.append(np.concatenate([[f.sum(), (f * f).sum(), np.abs(f).max()], f[idx]]))
    return np.stack(fp)


def case(params, x, M, continuous, estimator, L, seed, H, Z):
    rng = np.random.RandomState(seed)
    eps = rng.normal(size=(L, M, Z)).astype(np.float32)
    m = O.OracleVAEB(x, continuous, H, Z, M, L=L, estimator=estimator, params=params, dtype=np.float64)
    sgvb, per_row, grads = m.grads(x[:M], eps)
    ret = m.update(0, eps)
    out = {"eps": eps, "sgvb": np.float64(sgvb), "per_row": per_row, "grad_fp": fingerprint(grads),
           "update_return": np.float64(ret)}
    for n, p in zip(O.param_names(continuous), m.params):
        if n.startswith("b"):
            out["after_" + n] = p.astype(np.float32)
    out["after_W4"] = m.params[1].astype(np.float32)
    return out


def main():
    # ---- trained Frey weights -------------------------------------------------------
    header, params = io.read_mdl(os.path.join(REF, "reconstruction_res", "continuous_2.mdl"))
    assert header["continuous"] and header["n_latent"] == 2 and header["n_hidden_units"] == 200
    named = dict(zip(O.param_names(True), params))
    enc = ("W3", "W4", "W5", "b3", "b4", "b5")          # two halves, so that neither file exceeds 1 MB
    np.savez_compressed(os.path.join(HERE, "frey_z2_trained_encoder.npz"), **{n: named[n] for n in enc})
    np.savez_compressed(os.path.join(HERE, "frey_z2_trained_decoder.npz"),
                        **{n: p for n, p in named.items() if n not in enc})
    x = O.synthetic_frey(300)
    g = {"x_seed": np.int64(15485863)}
    for est in ("LB", "LA"):
        for k, v in case(params, x, 100, True, est, 1, 101, 200, 2).items():
            g["%s_%s" % (est, k)] = v
    eps_is = np.random.RandomState(102).normal(size=(16, 64, 2)).astype(np.float32)
    logp, logw = O.is_log_px([p.astype(np.float64) for p in params], x[200:216].astype(np.float64),
                             eps_is.astype(np.float64), True)
    g["is_eps"], g["is_logp"], g["is_logw"] = eps_is, logp, logw
    np.savez_compressed(os.path.join(HERE, "golden_frey_z2.npz"), **g)

    # ---- MNIST-shaped Bernoulli model at the reference initialisation -----------------
    D, H, Z, M = 784, 500, 20, 100
    params = O.init_params(D, H, Z, False)
    x = O.synthetic_mnist(200)
    g = {}
    for est, L in (("LB", 1), ("LA", 2)):
        for k, v in case(params, x, M, False, est, L, 103, H, Z).items():
            g["%s_%s" % (est, k)] = v
    eps_is = np.random.RandomState(104).normal(size=(8, 32, Z)).astype(np.float32)
    logp, logw = O.is_log_px([p.astype(np.float64) for p in params], x[100:108].astype(np.float64),
                             eps_is.astype(np.float64), False)
    g["is_eps"], g["is_logp"], g["is_logw"] = eps_is, logp, logw
    np.savez_compressed(os.path.join(HERE, "golden_mnist_init.npz"), **g)
    for f in sorted(os.listdir(HERE)):
        print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
