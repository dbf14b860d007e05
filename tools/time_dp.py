"""Data-parallel step time under torchrun:
python -m torch.distributed.run --nproc-per-node N tools/time_dp.py bf16x3 16384 [adagrad|adadelta|adam]"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
import vaeb_b200
from vaeb_b200 import distributed as vd
from vaeb_b200.data import synthetic_mnist
rank, world, local = vd.env_rank_world()
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
opt = sys.argv[3] if len(sys.argv) > 3 else "adagrad"
for prec in sys.argv[1].split(","):
    for MG in [int(v) for v in sys.argv[2].split(",")]:
        per = MG // world
        x = synthetic_mnist(per * 2, seed=3 + rank)
        m = vaeb_b200.VAEB(x, False, 500, 20, per, 1, 0.01, False, False, precision=prec, device=local, optimizer=opt)
        vd.attach_data_parallel(m)
        m.update_many(np.arange(6) % 2)
        torch.cuda.synchronize(); dist.barrier()
        k = 60
        t0 = time.perf_counter()
        out = m.update_many(np.arange(k) % 2)
        torch.cuda.synchronize(); dist.barrier()
        dt = (time.perf_counter() - t0) / k
        if rank == 0:
            print("%s %s global M=%d on %d GPUs (p2p %s): %.1f us/update (%.1f M datapoints/s) bound %.3f" %
                  (prec, opt, MG, world, os.environ.get("VAEB_DP_P2P", "1"), 1e6 * dt, MG / dt / 1e6, float(out[-1])),
                  flush=True)
        vd.close_data_parallel(m)
dist.barrier()
dist.destroy_process_group()
