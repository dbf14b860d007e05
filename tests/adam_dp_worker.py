"""Worker of tests/test_gpu_adam.py: one of WORLD_SIZE ranks under torchrun.  Every rank owns a contiguous share of
ONE global minibatch of 4096 rows and runs two bf16x3 Adam updates data parallel (VAEB_DP_P2P=1: the tail kernel over
peer memory; 0: ncclAllReduce + the flat Adam kernel); with peer memory, vaeb_set_adam after the export must be a state
error.  The parameters and both moments must be bit-identical on all
ranks; rank 0 compares them with the fp64 Adam oracle on the full batch."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vaeb_b200  # noqa: E402
from vaeb_b200 import _lib  # noqa: E402
from vaeb_b200 import distributed as vd  # noqa: E402
from oracle import vaeb_oracle as O  # noqa: E402
from tests import adam_oracle as A  # noqa: E402


def main():
    out_path = sys.argv[1]
    rank, world, local = vd.env_rank_world()
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    D, H, Z, MG = 784, 500, 20, 4096
    per = MG // world
    x = O.synthetic_mnist(MG, seed=99)
    rng = np.random.RandomState(5)
    params = [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(D, H, Z, False)]
    eps = [rng.normal(size=(1, MG, Z)).astype(np.float32) for _ in range(2)]
    lo = rank * per
    m = vaeb_b200.VAEB(x[lo:lo + per], False, H, Z, per, 1, 0.01, False, False, params, device=local,
                       precision="bf16x3", optimizer="adam")
    vd.attach_data_parallel(m)
    export_rc = m._lib.vaeb_set_adam(m._h, 0.9, 0.999, 1e-8) if os.environ.get("VAEB_DP_P2P", "1") != "0" else None
    rets = [float(m.update(0, eps=e[:, lo:lo + per])) for e in eps]
    state = m.get_params() + m._get_buffer(_lib.BUF_ADA) + m._get_buffer(_lib.BUF_ADAM_V)
    flat = torch.from_numpy(np.concatenate([a.ravel() for a in state])).cuda()
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    same = all(bool(torch.equal(gathered[0], t)) for t in gathered)
    res = {"world": world, "p2p": os.environ.get("VAEB_DP_P2P", "1"), "ranks_bit_identical": same,
           "adam_step": m.adam_step, "set_adam_after_export": export_rc}
    if rank == 0:
        o = A.OracleAdamVAEB(x, False, H, Z, MG, L=1, params=params)
        _, _, g_ref = o.grads(x, eps[0])
        refs = [o.update(0, e) for e in eps]
        res["bound_rel_err"] = max(abs(a - b) / abs(b) for a, b in zip(rets, refs))
        worst = 0.0
        n = len(params)
        for i, (gr, p0) in enumerate(zip(g_ref, params)):
            well = np.abs(gr) > 1e-2 * np.abs(gr).max()
            got, ref = state[i] - p0, o.params[i] - p0
            worst = max(worst, float(np.abs(got - ref)[well].max() / (3 * 0.01)))
            for k, r in ((1, o.ada[i]), (2, o.adam_v[i])):
                a = state[k * n + i]
                worst = max(worst, float((np.abs(a - r)[well] / np.abs(r)[well]).max()))
        res["worst_rel_err"] = worst
        with open(out_path, "w") as f:
            json.dump(res, f)
    vd.close_data_parallel(m)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
