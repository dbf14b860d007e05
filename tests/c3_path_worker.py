"""Worker of tests/test_gpu_c3_paths.py: three large-batch updates (bf16x3 or bf16) with whatever launch structure the
environment selects (VAEB_TC_TAIL is read once per process); bounds, parameters, Adagrad accumulators and the launch
count go to an .npz."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vaeb_b200  # noqa: E402
from vaeb_b200 import _lib  # noqa: E402
from vaeb_b200.data import synthetic_mnist  # noqa: E402


def main():
    out, prec, rows = sys.argv[1], sys.argv[2], int(sys.argv[3])
    D, H, Z = 784, 500, 20
    x = synthetic_mnist(2 * rows, seed=17)
    rng = np.random.RandomState(11)
    shapes = [(D, H), (H, Z), (H, Z), (Z, H), (H, D), (1, H), (1, Z), (1, Z), (1, H), (1, D)]
    params = [rng.normal(0, 0.05, s).astype(np.float32) for s in shapes]
    m = vaeb_b200.VAEB(x, False, H, Z, rows, 1, 0.01, False, False, params, precision=prec)
    bounds = [float(m.update(i % 2)) for i in range(3)]
    launches = m.launch_count()
    res = {"bounds": np.array(bounds), "launches": np.array(launches)}
    for i, a in enumerate(m.get_params()):
        res["p%d" % i] = a
    for i, a in enumerate(m._get_buffer(_lib.BUF_ADA)):
        res["a%d" % i] = a
    np.savez(out, **res)
    m.close()


if __name__ == "__main__":
    main()
