"""Worker of tests/test_gpu_checkpoint.py: one of WORLD_SIZE ranks under torchrun.  Every rank owns a contiguous share
of one global minibatch of 4096 rows and trains bf16x3 data parallel (VAEB_DP_P2P=1: the tail kernel over peer memory;
0: ncclAllReduce), with Adagrad and with Adam.  A: four updates without interruption.  B: two updates, a checkpoint
written by rank 0 (vaeb_b200.distributed.save_checkpoint), every rank closed, resumed from the file on its own shard,
attached again, two more updates.  Rank 0 reports whether B ends bit-identical to A on every rank and whether the
ranks agree with each other."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vaeb_b200  # noqa: E402
from vaeb_b200 import distributed as vd  # noqa: E402
from oracle import vaeb_oracle as O  # noqa: E402


def _flat_state(m):
    bufs = [a.ravel() for _, which in m._state_buffers() for a in m._get_buffer(which)]
    counters = np.array([m.step_counter, m.adam_step, m.kl_step], np.float32)
    return np.concatenate(bufs + [counters])


def main():
    out_path, tmp = sys.argv[1], sys.argv[2]
    rank, world, local = vd.env_rank_world()
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    D, H, Z, MG = 784, 500, 20, 4096
    per = MG // world
    x = O.synthetic_mnist(2 * MG, seed=99)
    lo = rank * per
    shard = np.concatenate([x[lo:lo + per], x[MG + lo:MG + lo + per]])     # two global minibatches
    rng = np.random.RandomState(5)
    params = [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(D, H, Z, False)]
    cases = []
    for opt in ("adagrad", "adam"):
        def make():
            return vaeb_b200.VAEB(shard, False, H, Z, per, 1, 0.01, False, False, params, device=local,
                                  precision="bf16x3", optimizer=opt)

        a = make()
        vd.attach_data_parallel(a)
        ra = [float(a.update(i % 2)) for i in range(4)]
        sa = _flat_state(a)
        vd.close_data_parallel(a)

        b = make()
        vd.attach_data_parallel(b)
        rb = [float(b.update(i % 2)) for i in range(2)]
        path = os.path.join(tmp, "dp_%s_%s.npz" % (opt, os.environ.get("VAEB_DP_P2P", "1")))
        vd.save_checkpoint(b, path)
        vd.close_data_parallel(b)
        b = vd.resume(path, shard, device=local)
        vd.attach_data_parallel(b)
        rb += [float(b.update(i % 2)) for i in range(2, 4)]
        sb = _flat_state(b)
        vd.close_data_parallel(b)

        same = bool(np.array_equal(sa, sb)) and ra == rb
        t = torch.from_numpy(sb).cuda()
        gathered = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        flags = [None] * world
        dist.all_gather_object(flags, same)
        cases.append({"optimizer": opt, "resumed_equals_uninterrupted": all(flags),
                      "ranks_bit_identical": all(bool(torch.equal(gathered[0], g)) for g in gathered)})
    if rank == 0:
        with open(out_path, "w") as f:
            json.dump({"world": world, "p2p": os.environ.get("VAEB_DP_P2P", "1"), "cases": cases}, f)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
