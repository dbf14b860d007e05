"""Cost of Adam against Adagrad.  (1) The flat optimizer kernels ("adam+prior (flat)" against "adagrad+prior (flat)",
CUDA events over repeated launches, vaeb_profile_update) on a handle of 12.9 M parameters (D = 784, H = 8192, Z = 20:
every pass streams its 360 MB from HBM, past the 126 MB L2), as algorithmic GB/s.  (2) The C3 update (MNIST shape,
16384 rows) with Adam and with Adagrad, bf16x3 and bf16, with the tail kernel and with VAEB_TC_TAIL=0 (read once per
process: each configuration runs in a process of its own): host clock around `update_many` of `n` updates, which ends
in a device synchronise; best and median of `reps`.  (3) When two GPUs are visible, the same update at 16384 global rows
on two GPUs under torchrun (tools/time_dp.py: 60 updates after 6 of warm-up), Adam against Adagrad, bf16x3 and bf16,
over peer memory (VAEB_DP_P2P=1: the tail kernel is the all-reduce) and over ncclAllReduce (VAEB_DP_P2P=0).  Prints one
JSON line with the card's name and power limit.  `python tools/time_adam.py [reps] [out.json]`"""
import json
import os
import re
import socket
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


def flat_pass():
    import vaeb_b200
    from vaeb_b200.data import synthetic_mnist
    D, H, Z, M = 784, 8192, 20, 256
    os.environ["VAEB_B200_FUSED"] = "0"     # Adagrad at this size would otherwise run the single-launch fp32 step
    x = synthetic_mnist(M, seed=3)
    out = {}
    for opt in ("adagrad", "adam"):
        m = vaeb_b200.VAEB(x, False, H, Z, M, 1, 0.01, False, False, optimizer=opt)
        for name, ms, _, by in m.profile_update(0, iters=50):
            if "(flat)" in name:
                out[opt] = {"phase": name, "us": 1e3 * ms, "GB_per_s": by / (ms * 1e-3) / 1e9, "bytes": by}
        m.close()
    return out


def c3(prec, opt, reps, n):
    import vaeb_b200
    from vaeb_b200.data import synthetic_mnist
    rows = 16384
    x = synthetic_mnist(2 * rows, seed=17)
    m = vaeb_b200.VAEB(x, False, 500, 20, rows, 1, 0.01, False, False, precision=prec, optimizer=opt)
    order = [i % 2 for i in range(n)]
    m.update_many(order)                    # warm-up: buffers, tensor maps, modules
    ts = []
    l0 = m.launch_count()
    for _ in range(reps):
        t0 = time.perf_counter()
        m.update_many(order)
        ts.append(time.perf_counter() - t0)
    launches = (m.launch_count() - l0) / (reps * n)
    m.close()
    return {"us_per_update": 1e6 * min(ts) / n, "us_per_update_median": 1e6 * float(np.median(ts)) / n,
            "launches_per_update": launches}


def two_gpus():
    """us per update on two GPUs, per (precision, optimizer, VAEB_DP_P2P); None on fewer GPUs."""
    import torch
    if torch.cuda.device_count() < 2:
        return None
    out = {}
    for p2p in ("1", "0"):
        for opt in ("adagrad", "adam"):
            s = socket.socket()
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
            s.close()
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                   "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "time_dp.py"), "bf16x3,bf16",
                   "16384", opt]
            r = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, VAEB_DP_P2P=p2p), cwd=ROOT)
            if r.returncode != 0:
                raise RuntimeError(r.stdout[-2000:] + r.stderr[-2000:])
            for line in r.stdout.splitlines():
                mt = re.match(r"(\S+) (\S+) global M=(\d+) on (\d+) GPUs \(p2p (\S+)\): ([\d.]+) us/update", line)
                if mt:
                    out["%s p2p=%s %s" % (mt.group(1), mt.group(5), mt.group(2))] = {"us_per_update": float(mt.group(6))}
    if len(out) != 8:
        raise RuntimeError("expected 8 two-GPU timings, got %s" % sorted(out))
    return out


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--c3":          # one configuration, in a process of its own
        print(json.dumps(c3(sys.argv[2], sys.argv[3], int(sys.argv[4]), int(sys.argv[5]))))
        return
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    res = {"card": card(), "flat_12.9M_params": flat_pass(), "c3_16384_rows": {}, "c3_16384_rows_2_gpus": None}
    for prec in ("bf16x3", "bf16"):
        for tail in ("1", "0"):
            for opt in ("adagrad", "adam"):
                env = dict(os.environ, VAEB_TC_TAIL=tail)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--c3", prec, opt, str(reps), "20"],
                                   capture_output=True, text=True, env=env, cwd=ROOT)
                if r.returncode != 0:
                    raise RuntimeError(r.stdout[-2000:] + r.stderr[-2000:])
                res["c3_16384_rows"]["%s tail=%s %s" % (prec, tail, opt)] = json.loads(r.stdout.strip().splitlines()[-1])
    res["c3_16384_rows_2_gpus"] = two_gpus() or "not measured: fewer than two GPUs visible"
    line = json.dumps(res)
    print(line, flush=True)
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
