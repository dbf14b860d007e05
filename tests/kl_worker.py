"""Worker of tests/test_gpu_kl_weight.py, for what has to be set before a process's first update.
  c3 OUT: three bf16x3 updates of 4096 rows over a KL warm-up, with the launch structure the environment selects
          (VAEB_TC_TAIL is read once per process): the state before and after every update and the bounds go to an .npz.
  dp OUT: one of WORLD_SIZE ranks under torchrun: two bf16x3 updates of ONE global minibatch of 4096 rows over a warm-up,
          data parallel (VAEB_DP_P2P=1: the tail kernel over peer memory; 0: ncclAllReduce).  Rank 0 writes whether the
          parameters are bit-identical on all ranks and the worst deviation from the fp64 oracle on the full batch."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vaeb_b200  # noqa: E402
from vaeb_b200 import _lib  # noqa: E402
from vaeb_b200.model import kl_weight_at  # noqa: E402
from oracle import vaeb_oracle as O  # noqa: E402
from tests import kl_oracle as K  # noqa: E402

D, H, Z, ROWS = 784, 500, 20, 4096
BETA, WARMUP = 2.5, 2


def inputs(n_updates):
    x = O.synthetic_mnist(2 * ROWS, seed=17)
    rng = np.random.RandomState(11)
    params = [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(D, H, Z, False)]
    eps = [rng.normal(size=(1, ROWS, Z)).astype(np.float32) for _ in range(n_updates)]
    return x, params, eps


def c3(out):
    x, params, eps = inputs(3)
    m = vaeb_b200.VAEB(x, False, H, Z, ROWS, 1, 0.01, False, False, params, precision="bf16x3",
                       kl_weight=BETA, kl_warmup=WARMUP)
    res = {}
    for k in range(3):
        for i, (p, a) in enumerate(zip(m.get_params(), m._get_buffer(_lib.BUF_ADA))):
            res["p%d_%d" % (k, i)], res["a%d_%d" % (k, i)] = p, a
        res["bound%d" % k] = np.array(float(m.update(k % 2, eps=eps[k])))
    for i, (p, a) in enumerate(zip(m.get_params(), m._get_buffer(_lib.BUF_ADA))):
        res["p3_%d" % i], res["a3_%d" % i] = p, a
    res["kl_step"] = np.array(m.kl_step)
    np.savez(out, **res)
    m.close()


def dp(out):
    import torch
    import torch.distributed as dist
    from vaeb_b200 import distributed as vd
    rank, world, local = vd.env_rank_world()
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    x, params, eps = inputs(2)
    x = x[:ROWS]
    per = ROWS // world
    lo = rank * per
    m = vaeb_b200.VAEB(x[lo:lo + per], False, H, Z, per, 1, 0.01, False, False, params, device=local,
                       precision="bf16x3", kl_weight=BETA, kl_warmup=WARMUP)
    vd.attach_data_parallel(m)
    rets = [float(m.update(0, eps=e[:, lo:lo + per])) for e in eps]
    state = m.get_params()
    flat = torch.from_numpy(np.concatenate([a.ravel() for a in state])).cuda()
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    same = all(bool(torch.equal(gathered[0], t)) for t in gathered)
    if rank == 0:
        o = K.OracleKLVAEB(x, False, H, Z, ROWS, L=1, params=params)
        g_ref, refs = [], []
        for n, e in enumerate(eps, 1):
            o.kl_weight = float(kl_weight_at(BETA, WARMUP, n))
            g_ref.append(o.grads(x, e)[2])
            refs.append(o.update(0, e))
        worst = 0.0
        for i, p0 in enumerate(params):           # the two steps together, where the gradients are well above the noise
            well = (np.abs(g_ref[0][i]) > 1e-2 * np.abs(g_ref[0][i]).max()) & \
                   (np.abs(g_ref[1][i]) > 1e-2 * np.abs(g_ref[1][i]).max())
            got, ref = state[i] - p0, o.params[i] - p0
            worst = max(worst, float(np.abs(got - ref)[well].max() / np.abs(ref)[well].max()))
        res = {"world": world, "ranks_bit_identical": same, "kl_step": m.kl_step, "worst_step_err": worst,
               "bound_rel_err": max(abs(a - b) / abs(b) for a, b in zip(rets, refs))}
        with open(out, "w") as f:
            json.dump(res, f)
    vd.close_data_parallel(m)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    {"c3": c3, "dp": dp}[sys.argv[1]](sys.argv[2])
