"""Cost of the KL weight (vaeb_set_kl_weight): the same updates with the constant weight 1 (nothing uploaded, the kernels
read no weights) against a running warm-up (a weight per update, uploaded with the batch order of every launch), in
alternation: C2 `update_many` at M = 100 on the tensor-core step kernel, the same with VAEB_B200_STEP_TC=0 (the fp32 step
kernel), and the C3 update (MNIST shape, 16384 rows, bf16x3, per-layer kernels and the tail).  Host clock around
`update_many` of `n` updates, which ends in a device synchronise; best and median of `reps`.  Prints one JSON line with
the card's name and power limit.  `python tools/time_kl.py [reps] [out.json]`"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def pair(rows, n, reps, **kw):
    """(constant weight 1, running warm-up): us per update, alternating the two handles rep by rep."""
    import vaeb_b200
    from vaeb_b200.data import synthetic_mnist
    x = synthetic_mnist(max(2 * rows, 600), seed=17)
    models = {"beta=1": vaeb_b200.VAEB(x, False, 500, 20, rows, 1, 0.01, False, False, **kw),
              "warm-up": vaeb_b200.VAEB(x, False, 500, 20, rows, 1, 0.01, False, False, kl_weight=1.0,
                                        kl_warmup=10 ** 9, **kw)}
    order = [i % (x.shape[0] // rows) for i in range(n)]
    kernel = models["beta=1"].step_kernel_name()
    ts = {k: [] for k in models}
    for m in models.values():
        m.update_many(order)                   # warm-up: buffers, tensor maps, modules
    for _ in range(reps):
        for k, m in models.items():
            t0 = time.perf_counter()
            m.update_many(order)
            ts[k].append(time.perf_counter() - t0)
    out = {"kernel": kernel}
    for k, m in models.items():
        out[k] = {"us_per_update": 1e6 * min(ts[k]) / n, "us_per_update_median": 1e6 * float(np.median(ts[k])) / n}
        m.close()
    return out


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7
    res = {"card": card()}
    res["c2_100_step_tc"] = pair(100, 600, reps)
    os.environ["VAEB_B200_STEP_TC"] = "0"      # read when a handle is created
    res["c2_100_fp32_step"] = pair(100, 600, reps)
    del os.environ["VAEB_B200_STEP_TC"]
    res["c3_16384_bf16x3"] = pair(16384, 20, reps, precision="bf16x3")
    line = json.dumps(res)
    print(line, flush=True)
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
