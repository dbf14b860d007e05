#!/usr/bin/env python
"""bench.py -- ELBO-gradient datapoints/s of the AEVB step on synthetic MNIST-shaped data.

Contract (driver): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line from rank 0.

HEADLINE (every N; changed in round 2 as VERDICT r1 item 3 asks -- round 1's headline was c2, which is now the
last entry of "also"): BASELINE.json configs[2] = "c3": MNIST Bernoulli 784-500-20, ONE global minibatch of
M = 16384 rows per step, split over the N ranks (16384/N rows each), bf16x3 tensor-core precision (bf16 hi+lo
operands, fp32 accumulation: the fp32 parity tier, 1e-4); when N > 1 the 3.26 MB gradient is summed inside the update's
tail kernel over NVLink peer memory (reduce-scatter, prior + Adagrad on the owner's slice, all-gather: tc_tail.cu;
VAEB_DP_P2P=0: ncclAllReduce + replicated Adagrad).  Total work per step is fixed => "scaling": "strong".

  value  device-resident: the rank's rows already in HBM (several minibatches, > L2 in total, visited in turn),
         K updates enqueued back to back, CUDA events on the launch stream, max over ranks.  The K timed updates
         start from the same state in every run (seeded data and parameters, W warm-up updates, Philox noise):
         --dump-outputs DIR writes what the last of them left for the caller -- its bound (bound.npy) and the
         parameters and Adagrad accumulators it wrote (param_<name>.npy, ada_<name>.npy; float32, 6.5 MB) -- so
         that two builds can be compared output for output.
  e2e    the reference-facing call with HOST inputs: every step copies ITS minibatch share from pinned host memory
         (H2D) and reads ITS bound back (D2H); streaming form (vaeb_update_host_async + vaeb_collect).
         e2e.sync_call: the synchronous call; e2e.u8_host: the same streaming call fed uint8 pixels (a quarter of the
         PCIe bytes, expanded on the device: exact for the reference's 8-bit data sets) -- reported beside, not as, e2e.
  roofline  tensor pipe: whole-step algorithmic flops (SURVEY 8d: 4,100,000 per datapoint) and the dominant kernel's
         own flops / its CUDA-event time (vaeb_profile_update), against the measured sustained bf16 peak.
  --impl reference  the reference's CPU path: it cannot run here (Python 2 + Theano), so this is the numpy fp32
         restatement in oracle/ (kind "port") on all BLAS threads of the host, same step (M = 16384 rows).
  also   c3 in plain bf16, c4 (full VB), c1 (Frey), the flat Adagrad pass vs HBM, then c5 (IS log p(x), sharded over
         the ranks) and c2 (M = 100, the reference's own hot loop; replicas when N > 1) LAST and compact.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D, H, Z, M, L = 784, 500, 20, 100, 1
N_TRAIN = 50000                      # c2: rows resident in HBM: 157 MB > the 126 MB L2
FLOPS_PER_DATAPOINT = 4100000        # SURVEY.md 8d (fwd 1,628,000 + bwd 2,472,000)
METRIC = "ELBO-gradient datapoints/sec (AEVB update, MNIST 784-500-20 Bernoulli, global M=16384, L=1)"
UNIT = "datapoints/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    # fallback stated in /opt/skills/guides/B200_PROFILING.md
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(object):
    """SM clock and throttle reasons sampled through NVML DURING the timed region (a thread in
    this process: spawning nvidia-smi in a loop contends with kernel launches for the driver)."""

    def __init__(self, index, period_s=0.01):
        self.index, self.period, self.rows, self.stop = index, period_s, [], threading.Event()
        self.max_mhz, self.t = None, None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            # the first NVML queries of a process take tens of ms inside the driver and serialise with a kernel
            # launch issued meanwhile (measured: +25..300 ms between the start event and the launch of the timed
            # kernel): pay for them here, before the timed region, and let the thread sleep before its first sample
            self._sample()
            self.rows = []
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        except Exception:
            self.t = None
        return self

    def _sample(self):
        nv = self.nv
        try:
            reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        self.rows.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)), int(reasons), time.perf_counter()))

    def _loop(self):
        while not self.stop.wait(self.period if self.rows else 0.02):
            try:
                self._sample()
            except Exception:
                pass

    def __exit__(self, *a):
        if self.t:
            try:
                self._sample()
            except Exception:
                pass
            self.stop.set()
            self.t.join(timeout=2)

    def summary(self, t0=None, t1=None):
        """Clocks / reasons of the samples taken in [t0, t1] (perf_counter), all samples if no window is given."""
        names = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}
        rows = [r for r in self.rows if (t0 is None or r[2] >= t0) and (t1 is None or r[2] <= t1)]
        if not rows:
            rows = self.rows[-1:]
        sm = [r[0] for r in rows]
        reasons = sorted({n for r in rows for bit, n in names.items() if r[1] & bit})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(sm)}


MG = 16384                           # c3: rows of the ONE global minibatch of a step
C3_PREC = "bf16x3"
C3_FLOPS_PER_STEP = MG * FLOPS_PER_DATAPOINT            # 67.17 GFLOP (SURVEY.md 8d)
WORKLOAD = ("c3: MNIST-shape Bernoulli VAE D=784 H=500 Z=20, global minibatch M=16384 rows per step split over the "
            "ranks, L=1, Adagrad, %s; one step = one update()" % C3_PREC)


def make_problem(seed=15485863):
    from vaeb_b200.data import synthetic_mnist
    return synthetic_mnist(N_TRAIN, seed=seed)


def reset_state(m, params, ada):
    """Puts back everything an update reads besides the data: parameters, Adagrad accumulators and the Philox step
    counter (0 after construction), so that what follows does not depend on how many updates ran before."""
    from vaeb_b200 import _lib
    m.set_params(params)
    m._set_buffer(_lib.BUF_ADA, ada)
    _lib.check(m._lib.vaeb_set_step_counter(m._h, 0))


def dump_outputs(out_dir, m, bounds):
    """The last timed update as its caller sees it: the bound it returned and the parameters and Adagrad
    accumulators it left on the device, as out_dir/<name>.npy (float32)."""
    from vaeb_b200 import _lib
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"bound": np.asarray(bounds[-1:], np.float32)}
    for p, v, a in zip(m.params, m.get_params(), m._get_buffer(_lib.BUF_ADA)):
        arrays["param_" + p.name], arrays["ada_" + p.name] = v, a
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------
def cpu_step_loop(x, rows, steps, warmup, budget_s=None, min_steps=2):
    """fp32 numpy restatement (oracle/vaeb_oracle.py) of the same update() on minibatches of `rows` rows."""
    from oracle import vaeb_oracle as O
    m = O.OracleVAEB(x, False, H, Z, rows, L=L, params=O.init_params(D, H, Z, False), dtype=np.float32)
    rng = np.random.RandomState(10)
    nb = x.shape[0] // rows
    for i in range(warmup):
        m.update(i % nb, rng.normal(size=(L, rows, Z)).astype(np.float32))
    t0 = time.perf_counter()
    done = 0
    for i in range(steps):
        # eps is drawn on the host inside the step, as the reference does (VAEB.py:42)
        m.update((warmup + i) % nb, rng.normal(size=(L, rows, Z)).astype(np.float32))
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s and done >= min_steps:
            break
    dt = time.perf_counter() - t0
    return done, dt


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        n = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(n) if n else 1
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to its workers; the reference arm is ONE process that may use every core
    # of the host whatever N is (VERDICT r1: the N >= 2 reference numbers ran single-threaded)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        pass
    from vaeb_b200.data import synthetic_mnist
    x = synthetic_mnist(2 * MG, seed=777)            # two global minibatches, visited in turn
    # a step of the reference arm is one whole update() on 16384 rows (~0.3-1 s of CPU work); cap the run at ~2 min
    done, dt = cpu_step_loop(x, MG, args.steps, min(args.warmup, 2), budget_s=120.0)
    val = done * MG / dt
    cores = blas_threads()
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": done, "warmup": min(args.warmup, 2), "ms_per_step": 1e3 * dt / done, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "host_cpus": os.cpu_count()},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d update() steps on 16384 rows each of the numpy fp32 restatement "
                                       "(oracle/vaeb_oracle.py); the reference itself needs Python 2 + Theano and "
                                       "cannot run here" % done},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# own arm
# ------------------------------------------------------------------------------------------
def run_own(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import vaeb_b200
    from vaeb_b200.data import synthetic_mnist, synthetic_frey
    from vaeb_b200 import _lib, distributed as vd
    stream = torch.cuda.current_stream()
    peaks = measured_peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        barrier()
        return max_over_ranks(a.elapsed_time(b))

    K, W = args.steps, max(args.warmup, 3)
    # ================= headline: c3, global M = 16384 split over the ranks ==========================================
    per = MG // world
    # resident rows: whole minibatches, > 160 MB in total per rank (the 126 MB L2 cannot hold them), visited in turn
    nb3 = max(3, -(-160 * 1024 * 1024 // (per * D * 4)))
    xs = synthetic_mnist(per * nb3, seed=777 + rank)
    m3 = vaeb_b200.VAEB(xs, False, H, Z, per, 1, 0.01, False, False, device=local, precision=args.precision, seed=10)
    m3.set_stream(stream.cuda_stream)
    if world > 1:
        vd.attach_data_parallel(m3)
    params0, ada0 = m3.get_params(), m3._get_buffer(_lib.BUF_ADA)

    def order3(n, start=0):
        return (np.arange(start, start + n) % nb3).astype(np.int32)

    m3.update_many(order3(max(W, 3)))                   # also sizes every per-launch buffer
    # clocks ramp up lazily: keep the device busy until two consecutive probes agree within 3 % (1..6 s)
    clocks = ClockSampler(local)
    clocks.__enter__()
    t_ramp = time.perf_counter()
    probe, last = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prev_ms, n_probe = None, 40
    while True:
        probe.record(stream)
        m3.update_many(order3(n_probe))
        last.record(stream)
        torch.cuda.synchronize()
        cur_ms = probe.elapsed_time(last)
        el = time.perf_counter() - t_ramp
        stop = (el >= 1.0 and prev_ms is not None and abs(cur_ms - prev_ms) <= 0.03 * prev_ms) or el >= 6.0
        if world > 1:                                   # every rank must leave the loop in the same iteration
            t = torch.tensor([1.0 if stop else 0.0], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            stop = bool(t.item() > 0.5) or el >= 12.0
        if stop:
            break
        prev_ms = cur_ms
    probe_ms_per_step = cur_ms / n_probe
    # the ramp ran as many updates as the clocks needed: start again from the initial state and replay the fixed
    # warm-up, so that the timed updates compute the same thing in every run
    barrier()
    reset_state(m3, params0, ada0)
    barrier()
    m3.update_many(order3(max(W, 3)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    order_k = order3(K, 1)
    barrier()
    l0 = m3.launch_count()
    t0 = time.perf_counter()
    e0.record(stream)
    elbos = m3.update_many(order_k)
    e1.record(stream)
    barrier()
    window = (t0, time.perf_counter())
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = m3.launch_count() - l0
    clocks.__exit__(None, None, None)
    clocks_summary = clocks.summary(*window)
    value = K * MG / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, m3, elbos)

    # ---- e2e: every step copies its minibatch share H2D from pinned host memory and reads its bound back D2H ----
    pinned = torch.empty((per * nb3, D), dtype=torch.float32, pin_memory=True)
    pinned.copy_(torch.from_numpy(xs))
    xp = pinned.numpy()
    Ke = min(K, 200)
    for b in order3(W):
        m3.update_host_async(xp[b * per:(b + 1) * per])
    m3.collect()
    barrier()
    e0.record(stream)
    got = 0
    for i, b in enumerate(order3(Ke, 1)):
        m3.update_host_async(xp[b * per:(b + 1) * per])
        if (i + 1) % 64 == 0:
            got += len(m3.collect())
    got += len(m3.collect())
    e1.record(stream)
    barrier()
    assert got == Ke
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    e2e = Ke * MG / (ms_e2e * 1e-3)
    # the synchronous call (H2D, update, D2H, host sync every step)
    Ks = min(K, 50)
    for b in order3(2):
        m3.update_host(xp[b * per:(b + 1) * per])
    barrier()
    e0.record(stream)
    for b in order3(Ks, 1):
        m3.update_host(xp[b * per:(b + 1) * per])
    e1.record(stream)
    barrier()
    ms_sync = max_over_ranks(e0.elapsed_time(e1))
    e2e_sync = Ks * MG / (ms_sync * 1e-3)
    # the same streaming call fed BYTES (the data sets of the reference are 8-bit pixels / 256: vaeb_update_host_async_u8
    # sends a quarter of the PCIe traffic and expands on the device, bit-identical to the float path on such data).
    # Reported beside the headline e2e, which keeps the float32 host buffers of the reference's loader.
    pinned8 = torch.empty((per * nb3, D), dtype=torch.uint8, pin_memory=True)
    pinned8.copy_(torch.from_numpy(np.minimum(np.floor(xs * 256.0), 255.0).astype(np.uint8)))
    xp8 = pinned8.numpy()
    for b in order3(W):
        m3.update_host_async(xp8[b * per:(b + 1) * per])
    m3.collect()
    barrier()
    e0.record(stream)
    got = 0
    for i, b in enumerate(order3(Ke, 1)):
        m3.update_host_async(xp8[b * per:(b + 1) * per])
        if (i + 1) % 64 == 0:
            got += len(m3.collect())
    got += len(m3.collect())
    e1.record(stream)
    barrier()
    assert got == Ke
    ms_u8 = max_over_ranks(e0.elapsed_time(e1))
    e2e_u8 = Ke * MG / (ms_u8 * 1e-3)

    # ---- roofline: whole step and the dominant kernel (per-kernel CUDA-event times, single GPU only) --------------
    tf_step = C3_FLOPS_PER_STEP / world / (ms / K * 1e-3) / 1e12          # per GPU
    peak_tf = peaks["bf16_tflops_sustained"]
    roofline = {"kernel": "whole c3 step (%d launches per update)" % round(launches / K), "bound": "tensor",
                "achieved": tf_step, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf_step / peak_tf,
                "traffic": None, "traffic_note": "per-kernel dram bytes: profiles/r2_c3_ncu_*.txt (ncu --set full)",
                "peak_source": peaks["source"] + " (sustained cuBLAS bf16, MEASURED_PEAKS.json: kernels timed inside a long step)",
                "flops_per_step": C3_FLOPS_PER_STEP, "flops_per_datapoint": FLOPS_PER_DATAPOINT,
                "note": "algorithmic flops (SURVEY 8d); bf16x3 issues three bf16 MMAs per algorithmic product"}
    if world == 1:
        try:
            phases = m3.profile_update(index=1, iters=20)
            tot = sum(p[1] for p in phases)
            gemm = [p for p in phases if p[2] > 0]
            dom = max(gemm, key=lambda p: p[1])
            dom_tf = dom[2] / (dom[1] * 1e-3) / 1e12
            # DRAM bytes of that kernel: NOT measured in this run -- dram__bytes_read.sum + dram__bytes_write.sum of one
            # `ncu --set full` capture of the same kernel at this size (profiles/r2_c3_ncu_full.txt)
            ncu_traffic = {"wgrad W2,W1,W4|W5,W3": 255.8e6, "dec2 h.W2+loglik": 107.9e6}
            traffic = None
            if args.precision == "bf16x3" and per == 16384:
                traffic = next((v for k, v in ncu_traffic.items() if dom[0].startswith(k)), None)
            roofline.update({"traffic": traffic,
                             "traffic_note": "from profiles/r2_c3_ncu_full.txt (one ncu --set full capture of this kernel at this size), "
                                             "not measured in this run" if traffic else roofline["traffic_note"],
                             "mma_level_frac": (3.0 if args.precision == "bf16x3" else 1.0) * dom_tf / peak_tf,
                             "mma_level_note": "bf16x3 issues three bf16 MMAs per algorithmic product: tensor-pipe work = 3 x the "
                                               "algorithmic rate (ncu: sm__pipe_tensor_cycles_active 74 % in this kernel)"})
            roofline.update({"kernel": dom[0] + " (dominant kernel of the step)", "achieved": dom_tf, "frac": dom_tf / peak_tf,
                             "ms_per_launch": dom[1], "flops_per_launch": dom[2], "share_of_step": dom[1] / tot,
                             "whole_step": {"achieved": tf_step, "frac": tf_step / peak_tf, "ms": ms / K},
                             "phases": [{"name": p[0][:40], "us": round(1e3 * p[1], 1), "share": round(p[1] / tot, 3),
                                         "tflops": round(p[2] / (p[1] * 1e-3) / 1e12, 1) if p[2] else None}
                                        for p in phases]})
        except Exception as ex:                          # profiling is evidence, never a reason to lose the line
            roofline["phases_error"] = str(ex)[:200]
    if world > 1:
        vd.close_data_parallel(m3)
    else:
        m3.close()
    del pinned, xp, xs

    # ================= also: the other configurations, c5 and c2 last ==============================================
    also = {}
    if not args.no_also:
        # c3 in plain bf16 (1e-2 tier)
        xs = synthetic_mnist(per * 3, seed=777 + rank)
        mb = vaeb_b200.VAEB(xs, False, H, Z, per, 1, 0.01, False, False, device=local, precision="bf16", seed=10)
        mb.set_stream(stream.cuda_stream)
        if world > 1:
            vd.attach_data_parallel(mb)
        mb.update_many(np.arange(6, dtype=np.int32) % 3)
        kb = 30
        msb = timed(lambda: mb.update_many(np.arange(kb, dtype=np.int32) % 3))
        tfb = MG * kb / (msb * 1e-3) * FLOPS_PER_DATAPOINT / 1e12
        also["c3_bf16"] = {"value": MG * kb / (msb * 1e-3), "unit": UNIT, "ms_per_step": msb / kb,
                           "frac_bf16_sustained_per_gpu": tfb / world / peak_tf}
        vd.close_data_parallel(mb) if world > 1 else mb.close()
        x = make_problem()
        # c4: full VB (VAEB.py --full_varational, getFVBL), MNIST Nz = 2 / 10, M = 100; replicas when N > 1
        for zz in (2, 10):
            m0 = vaeb_b200.VAEB(x[:200], False, H, zz, M, 1, 0.01, False, False, device=local, seed=10)
            p0 = m0.get_params()
            m0.close()
            for sampled in (False, True):
                m4 = vaeb_b200.VAEB(x[:5000], False, H, zz, M, 1, 0.01, False, True, p0, device=local, seed=10,
                                    sample_weights=sampled)
                m4.set_stream(stream.cuda_stream)
                m4.update_many(np.arange(50, dtype=np.int32) % 50)
                k4 = 1000
                ms4 = timed(lambda: m4.update_many(np.arange(k4, dtype=np.int32) % 50))
                also["c4_z%d_%s" % (zz, "sampled" if sampled else "faithful")] = {
                    "value": world * M * k4 / (ms4 * 1e-3), "unit": UNIT, "us_per_step": 1e3 * ms4 / k4}
                m4.close()
        # c1: Frey-shape Gaussian decoder 560-200-2, M = 100 (the reference's own CPU-runnable case)
        xf = synthetic_frey()[:1500]
        m1 = vaeb_b200.VAEB(xf, True, 200, 2, 100, 1, 0.01, False, False, device=local, seed=10)
        m1.set_stream(stream.cuda_stream)
        m1.update_many(np.arange(30, dtype=np.int32) % 15)
        k1 = 3000
        ms1 = timed(lambda: m1.update_many(np.arange(k1, dtype=np.int32) % 15))
        also["c1_frey"] = {"value": world * 100 * k1 / (ms1 * 1e-3), "unit": UNIT, "us_per_step": 1e3 * ms1 / k1}
        m1.close()
        # flat Adagrad pass against the HBM roofline on a stream-sized buffer (65 M parameters, 1.3 GB per launch)
        mo = vaeb_b200.VAEB(x[:200], False, 40000, Z, M, 1, 0.01, False, False, device=local, seed=10)
        mo.set_stream(stream.cuda_stream)
        ms_o, by_o = mo.profile_optimizer(iters=50)
        also["adagrad_flat"] = {"value": by_o / (ms_o * 1e-3) / 1e9, "unit": "GB/s",
                                "frac_hbm": by_o / (ms_o * 1e-3) / 1e9 / peaks["hbm_gbs"]}
        mo.close()
        # c5: importance-sampled log p(x), 10,000 points x L = 5000, points sharded over the ranks; host x in, host
        # log p out.  Tensor-core estimator (bf16, 1e-2 tier) at full size; fp32 estimator (1e-4 tier) on 1000 points
        L5 = 5000
        for prec, n_pts in (("fp32", 1000), ("bf16", 10000)):
            xt = synthetic_mnist(n_pts, seed=4242)
            m5 = vaeb_b200.VAEB(xt[:100], False, H, Z, 100, 1, 0.01, False, False, device=local, seed=10, precision=prec)
            m5.set_stream(stream.cuda_stream)
            vd.sharded_log_px(m5, xt, L5, rank, world, gather=False)          # warm-up at the timed size
            res5 = {}
            ms5 = timed(lambda: res5.update(lp=vd.sharded_log_px(m5, xt, L5, rank, world, gather=False)))
            sps = n_pts * L5 / (ms5 * 1e-3)
            also["c5_is_" + prec] = {"value": sps, "unit": "samples/s", "ms": ms5, "points": n_pts, "L": L5,
                                     "frac_bf16_sustained_per_gpu": sps * 804000 / 1e12 / world / peak_tf,
                                     "mean_logpx_rank0": float(np.mean(res5["lp"]))}
            m5.close()
        # c2: the reference's own hot loop (BASELINE configs[1]): M = 100, single-launch step kernel; replicas if N > 1
        m2 = vaeb_b200.VAEB(x, False, H, Z, M, L, 0.01, False, False, device=local, seed=10 + rank)
        m2.set_stream(stream.cuda_stream)
        nb = N_TRAIN // M
        rng = np.random.RandomState(15485863 + rank)
        k2 = 2000

        def order2(n):                                  # np.random.shuffle(batch_order) per epoch (VAEB.py:574)
            return np.concatenate([rng.permutation(nb) for _ in range(-(-n // nb))])[:n].astype(np.int32)
        m2.update_many(order2(k2))
        t_r = time.perf_counter()
        while time.perf_counter() - t_r < 1.0:
            m2.update_many(order2(1000))
        o2 = order2(k2)
        assert len(o2) == k2
        ms2 = timed(lambda: m2.update_many(o2))
        pin2 = torch.empty((N_TRAIN, D), dtype=torch.float32, pin_memory=True)
        pin2.copy_(torch.from_numpy(x))
        xp2 = pin2.numpy()
        for b in o2[:8]:
            m2.update_host_async(xp2[b * M:(b + 1) * M])
        m2.collect()

        def stream2():
            for b in o2:
                m2.update_host_async(xp2[b * M:(b + 1) * M])
            m2.collect()
        ms2e = timed(stream2)
        n_params = sum(int(np.prod(sh)) for sh in m2._shapes)
        by2 = 20.0 * n_params + 4.0 * M * D
        also["c2_m100"] = {"value": world * k2 * M / (ms2 * 1e-3), "unit": UNIT, "us_per_step": 1e3 * ms2 / k2,
                           "e2e": world * k2 * M / (ms2e * 1e-3), "e2e_us_per_step": 1e3 * ms2e / k2,
                           "hbm_frac": by2 * k2 / (ms2 * 1e-3) / 1e9 / peaks["hbm_gbs"],
                           "kernel": m2.step_kernel_name() if hasattr(m2, "step_kernel_name") else "fused_step_kernel"}
        m2.close()

    line = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            xc = synthetic_mnist(2 * MG, seed=777)
            done, dt = cpu_step_loop(xc, MG, 1000, 1, budget_s=15.0)
            cpu = {"value": done * MG / dt, "unit": UNIT, "cores": blas_threads(), "kind": "port",
                   "sample": "%d update() steps on 16384 rows (%.1f s) of the numpy fp32 restatement in oracle/" % (done, dt)}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": {"fp32": "f32", "bf16x3": "bf16x3 (bf16 hi+lo operands, fp32 accumulate: the fp32 parity tier)",
                          "bf16": "bf16"}[args.precision],
                "data": "synthetic",
                "config": {"workload": WORKLOAD, "rows_per_gpu": per, "rows_resident_per_gpu": per * nb3,
                           "l2": "inputs larger than L2: %d minibatches (%.0f MB) resident per GPU, visited in turn"
                                 % (nb3, per * nb3 * D * 4 / 1e6),
                           "eps": "Philox4x32-10 on device", "precision": args.precision,
                           "collective": ("none (1 GPU)" if world == 1 else
                                          "ncclAllReduce(sum) of the flat gradient + bound" if os.environ.get("VAEB_DP_P2P", "1") == "0" else
                                          "inside the tail kernel, over peer memory (CUDA IPC / NVLink): reduce-scatter by peer "
                                          "loads, prior + Adagrad on the owner's slice, all-gather by peer stores (tc_tail.cu)"),
                           "launch_structure": "seven layer launches (VAEB_TC_CHAIN=1: one chain launch, tc_chain.cu), one weight-"
                                               "gradient launch, slice sum + bound + Adagrad (N > 1: one tail launch that is also the collective, tc_tail.cu)"},
                "clocks": clocks_summary, "warmup_probe_ms_per_step": probe_ms_per_step,
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": per * D * 4 * world, "d2h_bytes_per_step": 4 * world,
                        "steps": Ke, "ms_per_step": ms_e2e / Ke,
                        "h2d_gbs_per_gpu": per * D * 4 / (ms_e2e / Ke * 1e-3) / 1e9,
                        "bound": "host-to-device copy of the minibatch (PCIe): the step itself takes ms_per_step of the headline",
                        "api": "VAEB.update_host_async + collect (pinned host minibatch per step, H2D on a copy stream "
                               "overlapping the previous step, 4-byte D2H of every bound)",
                        "sync_call": {"value": e2e_sync, "ms_per_step": ms_sync / Ks, "steps": Ks},
                        "u8_host": {"value": e2e_u8, "ms_per_step": ms_u8 / Ke, "steps": Ke,
                                    "h2d_bytes_per_step": per * D * world,
                                    "note": "same call, minibatch as uint8 pixels (x = byte / 256, what mnist.pkl.gz holds), "
                                            "expanded on the device; bit-identical updates on byte-valued data "
                                            "(tests/test_gpu_async.py); not the headline e2e"}},
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
                "final_bound_per_datapoint": float(np.mean(elbos[-5:])), "also": also}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the side measurements (c1, c2, c4, c5, Adagrad)")
    ap.add_argument("--precision", default=C3_PREC, choices=["fp32", "bf16x3", "bf16"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the bound, parameters and Adagrad accumulators of the last timed update as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "own":
        ap.error("--dump-outputs writes the outputs of --impl own")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
