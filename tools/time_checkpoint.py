"""Cost of a checkpoint: host wall time of `save_checkpoint` (device-to-host copies of the state, npz write, fsync,
rename) and of `VAEB.resume` (read, constructor with data upload, state upload), at the C2 shape (MNIST 784-500-20,
M = 100, Adagrad: parameters + accumulators) and the C3 shape (16384 rows, bf16x3, with Adagrad and with Adam), plus
full VB at C2 (four more buffers), each on the 50,000 MNIST-shaped training rows and compared with the time of one
epoch of `update_many` at that shape.  Best and median of `reps`; the file goes to a temporary directory.  Prints one
JSON line with the card's name and power limit.  `python tools/time_checkpoint.py [reps] [out.json]`"""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def case(name, x, rows, reps, tmp, **kw):
    import vaeb_b200
    params = None
    if kw.get("fullVariational"):
        rng = np.random.RandomState(1)
        from oracle import vaeb_oracle as O
        params = [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(784, 500, 20, False)]
    fvb = kw.pop("fullVariational", False)
    m = vaeb_b200.VAEB(x, False, 500, 20, rows, 1, 0.01, False, fvb, params, **kw)
    order = np.arange(len(x) // rows, dtype=np.int32)
    m.update_many(order)                                   # warm-up
    t0 = time.perf_counter()
    m.update_many(order)
    epoch_s = time.perf_counter() - t0
    path = os.path.join(tmp, name + ".npz")
    save, res = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        m.save_checkpoint(path)
        save.append(time.perf_counter() - t0)
    m.close()
    for _ in range(reps):
        t0 = time.perf_counter()
        r = vaeb_b200.VAEB.resume(path, x)
        r.synchronize()
        res.append(time.perf_counter() - t0)
        r.close()
    return {"case": name, "bytes": os.path.getsize(path), "epoch_ms": 1e3 * epoch_s,
            "save_ms_best": 1e3 * min(save), "save_ms_median": 1e3 * float(np.median(save)),
            "resume_ms_best": 1e3 * min(res), "resume_ms_median": 1e3 * float(np.median(res))}


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    from vaeb_b200.data import synthetic_mnist
    x = synthetic_mnist(50000, seed=17)
    out = {"card": card(), "reps": reps, "cases": []}
    with tempfile.TemporaryDirectory() as tmp:
        out["cases"].append(case("C2 adagrad", x, 100, reps, tmp))
        out["cases"].append(case("C2 full VB", x, 100, reps, tmp, fullVariational=True))
        out["cases"].append(case("C3 bf16x3 adagrad", x[:49152], 16384, reps, tmp, precision="bf16x3"))
        out["cases"].append(case("C3 bf16x3 adam", x[:49152], 16384, reps, tmp, precision="bf16x3", optimizer="adam"))
    line = json.dumps(out)
    print(line)
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
