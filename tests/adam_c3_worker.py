"""Worker of tests/test_gpu_adam.py: three large-batch Adam updates (bf16x3 or bf16) on injected noise with whatever
launch structure the environment selects (VAEB_TC_TAIL is read once per process), then the same three updates with
Adagrad for the launch count.  Bounds, parameters, both moments, the Adam step and the launch counts go to an .npz."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vaeb_b200  # noqa: E402
from vaeb_b200 import _lib  # noqa: E402
from oracle import vaeb_oracle as O  # noqa: E402


def inputs(rows):
    D, H, Z = 784, 500, 20
    x = O.synthetic_mnist(2 * rows, seed=17)
    rng = np.random.RandomState(11)
    params = [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(D, H, Z, False)]
    eps = [rng.normal(size=(1, rows, Z)).astype(np.float32) for _ in range(3)]
    return x, params, eps, (D, H, Z)


def main():
    out, prec, rows = sys.argv[1], sys.argv[2], int(sys.argv[3])
    x, params, eps, (D, H, Z) = inputs(rows)
    res = {}
    for opt in ("adam", "adagrad"):
        m = vaeb_b200.VAEB(x, False, H, Z, rows, 1, 0.01, False, False, params, precision=prec, optimizer=opt)
        l0 = m.launch_count()
        bounds = [float(m.update(i % 2, eps=eps[i])) for i in range(3)]
        res[opt + "_launches"] = np.array(m.launch_count() - l0)
        if opt == "adam":
            res["bounds"] = np.array(bounds)
            res["t"] = np.array(m.adam_step)
            for i, a in enumerate(m.get_params()):
                res["p%d" % i] = a
            for i, a in enumerate(m._get_buffer(_lib.BUF_ADA)):
                res["m%d" % i] = a
            for i, a in enumerate(m._get_buffer(_lib.BUF_ADAM_V)):
                res["v%d" % i] = a
        m.close()
    np.savez(out, **res)


if __name__ == "__main__":
    main()
