"""Single-node multi-GPU plumbing: one process per GPU, `torch.distributed` for rendezvous,
NCCL (attached inside the C library) for the gradient all-reduce, plain sharding for the
importance-sampling estimator (SURVEY.md 8e).  Nothing here touches the data path."""
from __future__ import annotations

import os

import numpy as np


def env_rank_world():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def broadcast_bytes(payload, src=0):
    """Broadcast a bytes object from `src` through the default process group."""
    import torch.distributed as dist
    obj = [payload]
    dist.broadcast_object_list(obj, src=src)
    return obj[0]


def attach_data_parallel(model):
    """Give `model` (one per rank, built on this rank's GPU with batch_size = per-rank share)
    an NCCL communicator: afterwards every update all-reduces gradients and the bound.  The ranks must weight the
    latent term alike (set_kl_weight, kl_step) and stand at the same Philox step (a run resumed on every rank from the
    same checkpoint does)."""
    import torch.distributed as dist
    from .model import comm_unique_id
    rank, world = dist.get_rank(), dist.get_world_size()
    if world > 1:
        schedules = [None] * world
        dist.all_gather_object(schedules, (model.kl_weight, model.kl_warmup, model.kl_step))
        check_same_kl_weight(schedules)
        steps = [None] * world
        dist.all_gather_object(steps, model.step_counter)
        check_same_step_counter(steps)
    uid = comm_unique_id() if rank == 0 else None
    uid = broadcast_bytes(uid, 0)
    model.attach_comm(uid, rank, world)
    # ranks of one box map each other's buffers (CUDA IPC over NVLink): the tail kernel of a large-batch tensor-core
    # update then IS the gradient all-reduce (vaeb_comm_p2p_attach); VAEB_DP_P2P=0 keeps ncclAllReduce
    if 1 < world <= 8 and os.environ.get("VAEB_DP_P2P", "1") != "0" and getattr(model, "precision", "fp32") != "fp32":
        optimizers = [None] * world
        dist.all_gather_object(optimizers, getattr(model, "optimizer", "adagrad"))
        check_same_optimizer(optimizers)
        mine = model.p2p_export()
        handles = [None] * world
        dist.all_gather_object(handles, mine)
        model.p2p_attach(handles)
        dist.barrier()
    return rank, world


def check_same_optimizer(optimizers):
    """`optimizers`: every rank's update rule, in rank order.  Over peer memory the owner of a slice stores the updated
    parameters and accumulators into every rank's buffers, Adam's v right after m in the accumulator allocation: a rank
    whose allocation has no room for v (another rule) would be written past its end, so a mix is refused up front."""
    if len(set(optimizers)) > 1:
        raise ValueError("data parallel over peer memory needs the same optimizer on every rank, got %s" % (optimizers,))


def check_same_kl_weight(schedules):
    """`schedules`: every rank's (KL weight, warm-up, KL step), in rank order.  The summed gradient is the gradient of
    one objective only when every rank weights the latent term alike, so a mix is refused."""
    if len(set(schedules)) > 1:
        raise ValueError("data parallel needs the same KL weight, warm-up and KL step on every rank, got %s" % (schedules,))


def check_same_step_counter(steps):
    """`steps`: every rank's Philox step counter, in rank order.  Each rank draws its rows' noise from (seed, step,
    global row); ranks at different steps -- resumed from different checkpoints, say -- would not train one model."""
    if len(set(steps)) > 1:
        raise ValueError("data parallel needs the same step counter on every rank, got %s" % (steps,))


def save_checkpoint(model, path, driver_state=None):
    """Collective: the training state of a data-parallel model, written by rank 0 (the state is replicated) with the
    data fingerprint of every rank's shard.  Every rank returns once the file is in place."""
    import torch.distributed as dist
    from . import checkpoint
    rank, world = dist.get_rank(), dist.get_world_size()
    header, arrays = model.training_state()
    fps = [None] * world
    dist.all_gather_object(fps, model._data_fp)
    if rank == 0:
        header.update(world_size=world, data=fps)
        checkpoint.write(path, header, arrays, driver_state)
    dist.barrier()


def resume(path, x_shard, device, return_driver_state=False):
    """This rank's model from a checkpoint of save_checkpoint, on its own shard; attach_data_parallel afterwards."""
    import torch.distributed as dist
    from .model import VAEB
    return VAEB.resume(path, x_shard, device=device, rank=dist.get_rank(), world_size=dist.get_world_size(),
                       return_driver_state=return_driver_state)


def close_data_parallel(model):
    """Collective counterpart of model.close(): every rank stops using its peers' buffers (barrier) before any rank
    unmaps and frees its own (the exported allocations must outlive every importer's mapping)."""
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize()
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.barrier()
        _lib_detach(model)
        dist.barrier()
    model.close()


def _lib_detach(model):
    from . import _lib
    _lib.check(model._lib.vaeb_comm_detach(model._h))


def shard_rows(n, rank, world):
    """Contiguous block of rows owned by `rank` (SURVEY.md 8e: N/G points per GPU)."""
    per = (n + world - 1) // world
    lo = min(n, rank * per)
    return lo, min(n, lo + per)


def sharded_log_px(model, x, L, rank, world, gather=True):
    """IS estimator over the shard of x owned by this rank.  Philox counters are keyed by the
    GLOBAL row, so the concatenated result is identical for any world size."""
    lo, hi = shard_rows(len(x), rank, world)
    local = model.log_px(x[lo:hi], L=L, row_offset=lo) if hi > lo else np.empty(0, np.float32)
    if not gather or world == 1:
        return local
    import torch
    import torch.distributed as dist
    outs = [None] * world
    dist.all_gather_object(outs, local)
    return np.concatenate(outs)


def sharded_sample(model, n, rank, world, step=0, gather=True):
    """This rank's share of `n` samples from the generative model.  The Philox counters are keyed by the GLOBAL
    sample row, so the concatenated samples are identical for any world size."""
    lo, hi = shard_rows(n, rank, world)
    local = model.sample(hi - lo, step=step, row_offset=lo) if hi > lo else np.empty((0, model.input_size), np.float32)
    if not gather or world == 1:
        return local
    import torch.distributed as dist
    outs = [None] * world
    dist.all_gather_object(outs, local)
    return np.concatenate(outs)
