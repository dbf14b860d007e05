"""Throughput of the generation / evaluation entry points at the C2 shape (MNIST, D = 784, H = 500, Z = 20, fp32):
samples/s of `sample` for 10^6 samples (x only, and all four outputs) and rows/s of `encode` for 50 000 rows.  Host
clock around calls that end in a device synchronise (each entry point copies its outputs to the host), so the numbers
include the D2H copies; best of `reps` after one warm-up call at the timed size.  Prints one JSON line with the card's
name and power limit.  `python tools/time_sample.py [reps] [out.json]`"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import vaeb_b200  # noqa: E402
from vaeb_b200.data import synthetic_mnist  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def best(fn, reps):
    fn()                                    # warm-up: buffers sized, modules loaded
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts), float(np.median(ts))


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    x = synthetic_mnist(50000, seed=4242)
    m = vaeb_b200.VAEB(x[:100], False, 500, 20, 100, 1, 0.01, False, False)
    n_s = 1000000
    t_x, t_x_med = best(lambda: m.sample(n_s), reps)
    t_all, t_all_med = best(lambda: m.sample(n_s, return_all=True), reps)
    t_enc, t_enc_med = best(lambda: m.encode(x), reps)
    res = {"card": card(), "shape": "C2 D=784 H=500 Z=20 fp32",
           "sample_x_per_s": n_s / t_x, "sample_x_ms": 1e3 * t_x, "sample_x_ms_median": 1e3 * t_x_med,
           "sample_all_per_s": n_s / t_all, "sample_all_ms": 1e3 * t_all, "sample_all_ms_median": 1e3 * t_all_med,
           "encode_rows_per_s": len(x) / t_enc, "encode_ms": 1e3 * t_enc, "encode_ms_median": 1e3 * t_enc_med}
    m.close()
    line = json.dumps(res)
    print(line, flush=True)
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
