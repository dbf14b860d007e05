"""Save and resume the complete training state (VAEB.save_checkpoint / VAEB.resume) on one B200.

Every case runs the same schedule three times: twice without interruption (A, A2) and once (B) saved to a checkpoint
after the first n1 updates (directly, or after a validate, which advances the step counter without an update), closed,
resumed into a fresh handle, and continued.  A and A2 must agree
bit for bit first -- otherwise the path is not reproducible and resume cannot be judged -- and then A and B: the n2
bounds, a following validate (it draws from the step counter), every state buffer and the three counters.  The resumed
handle rebuilds state an uninterrupted run keeps: the fp16 hi/lo weight images of the tensor-core step kernel, the
bf16 mirrors of the large-batch path, the parameter double buffer of the single-launch kernels and the sampled
full-VB weights.  Each case also asserts which update path it runs, so the matrix covers all three."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import vaeb_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TC, FUSED, LAYERS = "step_tc_kernel", "fused_step_kernel", "per-layer kernels"


def _frey(n, D=560, seed=3):
    rng = np.random.RandomState(seed)
    return np.clip(0.5 + 0.2 * rng.normal(size=(n, D)), 0, 1).astype(np.float32)


# name -> (D, H, Z, M, continuous, L, genericEstimator, fullVariational, keywords, driver, expected kernel)
CASES = {
    "c2_adagrad": (784, 500, 20, 100, False, 1, False, False, {}, "many", TC),
    "c1_gaussian": (560, 200, 2, 100, True, 1, False, False, {}, "many", TC),
    "fused_z32": (784, 500, 32, 100, False, 1, False, False, {}, "many", FUSED),
    "layers_L2_LA": (784, 500, 20, 100, False, 2, True, False, {}, "many", LAYERS),
    "relu_enc3_adadelta": (784, 256, 20, 100, False, 1, False, False,
                           dict(activation="relu", encoder_layers=3, optimizer="adadelta"), "many", LAYERS),
    "relu_enc3_adam": (784, 256, 20, 100, False, 1, False, False,
                       dict(activation="relu", encoder_layers=3, optimizer="adam"), "many", LAYERS),
    "kl_warmup_mid_ramp": (784, 500, 20, 100, False, 1, False, False, dict(kl_weight=0.5, kl_warmup=10), "many", TC),
    "fullbayes_variant": (784, 500, 20, 100, False, 1, False, False, dict(variant="fullbayes"), "many", TC),
    "bf16x3_2048_adagrad": (784, 500, 20, 2048, False, 1, False, False, dict(precision="bf16x3"), "update", LAYERS),
    "bf16x3_2048_adam": (784, 500, 20, 2048, False, 1, False, False, dict(precision="bf16x3", optimizer="adam"),
                         "update", LAYERS),
    "bf16_2048": (784, 500, 20, 2048, False, 1, False, False, dict(precision="bf16"), "update", LAYERS),
    "fvb_100": (784, 500, 20, 100, False, 1, False, True, {}, "many", TC),
    "fvb_sampled_100": (784, 500, 20, 100, False, 1, False, True, dict(sample_weights=True), "many", TC),
    "fvb_2048": (784, 500, 20, 2048, False, 1, False, True, dict(precision="bf16x3"), "update", LAYERS),
    "fvb_sampled_2048": (784, 500, 20, 2048, False, 1, False, True, dict(precision="bf16x3", sample_weights=True),
                         "update", LAYERS),
    "theano_interleaved": (784, 500, 20, 100, False, 1, False, False, dict(eps_mode="theano"), "theano", TC),
    "host_async": (784, 500, 20, 100, False, 1, False, False, {}, "async", TC),
}
N1, N2, NB = 3, 3, 4      # updates before and after the checkpoint, minibatches in the data


def _data(case):
    D, H, Z, M, cont = CASES[case][:5]
    x = _frey(NB * M + 256, D) if cont else O.synthetic_mnist(NB * M + 256, seed=11, D=D)
    return x[:NB * M], x[NB * M:]


def _model(case, x):
    import vaeb_b200
    D, H, Z, M, cont, L, la, fvb, kw, _, _ = CASES[case]
    rng = np.random.RandomState(8)
    params = None
    if fvb:
        params = [rng.normal(0, 0.05, s).astype(np.float32) for s in O.param_shapes(D, H, Z, cont)]
    return vaeb_b200.VAEB(x, cont, H, Z, M, L, 0.01, la, fvb, params, **kw)


def _updates(case, m, x, xv, first):
    """n updates in the case's driver; returns their bounds (and, for eps_mode='theano', reconstructions)."""
    import vaeb_b200
    drv = CASES[case][9]
    M = m.batch_size
    order = np.array([0, 2, 1] if first else [3, 1, 2], dtype=np.int32)
    if drv == "many":
        return [m.update_many(order)]
    if drv == "update":
        return [np.array([float(m.update(int(i))) for i in order], np.float32)]
    if drv == "theano":
        out = []
        for i in order:
            out.append(np.asarray(m.update(int(i))))
            out.append(np.asarray(m.validate(xv[:64])))
            out.append(m.reconstruct(xv[:8], 2))
        return out
    xb = vaeb_b200.pinned_empty((len(order) * M, m.input_size), np.float32)
    for k, i in enumerate(order):
        xb[k * M:(k + 1) * M] = x[i * M:(i + 1) * M]
        m.update_host_async(xb[k * M:(k + 1) * M])
    return [m.collect()]


def _state(m):
    s = {"%s.%d" % (name, i): a for name, which in m._state_buffers() for i, a in enumerate(m._get_buffer(which))}
    s["step"], s["adam_step"], s["kl_step"] = m.step_counter, m.adam_step, m.kl_step
    return s


def _run(case, tmp_path, resume, before):
    import vaeb_b200
    x, xv = _data(case)
    m = _model(case, x)
    kernel = m.step_kernel_name()
    first = _updates(case, m, x, xv, True)
    v1 = float(m.validate(xv)) if before == "validate" else None
    if resume:
        path = str(tmp_path / ("%s.npz" % case))
        m.save_checkpoint(path)
        m.close()
        m = vaeb_b200.VAEB.resume(path, x)
        assert m.step_kernel_name() == kernel
    second = _updates(case, m, x, xv, False)
    v2 = float(m.validate(xv))
    st = _state(m)
    m.close()
    return kernel, first, v1, second, v2, st


def _assert_same(a, b):
    ka, fa, v1a, sa, v2a, sta = a
    kb, fb, v1b, sb, v2b, stb = b
    assert ka == kb
    for p, q in zip(fa + sa, fb + sb):
        np.testing.assert_array_equal(p, q)
    assert v1a == v1b and v2a == v2b
    assert sorted(sta) == sorted(stb)
    for k in sta:
        np.testing.assert_array_equal(sta[k], stb[k], err_msg=k)


@pytest.mark.parametrize("before", ["update", "validate"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_resume_is_bit_identical(case, before, tmp_path):
    a = _run(case, tmp_path, False, before)
    assert a[0].startswith(CASES[case][10]), a[0]
    _assert_same(a, _run(case, tmp_path, False, before))          # the path itself is reproducible
    _assert_same(a, _run(case, tmp_path, True, before))           # and resume continues it bit for bit
    if "kl_warmup" in case:
        assert a[5]["kl_step"] == N1 + N2 < CASES[case][8]["kl_warmup"]
    if "adam" in case:
        assert a[5]["adam_step"] == N1 + N2


def test_resume_refuses_other_data(tmp_path):
    import vaeb_b200
    x, xv = _data("c2_adagrad")
    m = _model("c2_adagrad", x)
    m.update_many(np.arange(2, dtype=np.int32))
    path = str(tmp_path / "c.npz")
    m.save_checkpoint(path)
    m.close()
    y = x.copy()
    y[5, 7] += 0.5
    with pytest.raises(ValueError, match="fingerprint"):
        vaeb_b200.VAEB.resume(path, y)
    with pytest.raises(ValueError, match="world_size"):
        vaeb_b200.VAEB.resume(path, x, rank=0, world_size=2)


def test_step_counter_getter_tracks_updates_and_async():
    x, xv = _data("c2_adagrad")
    m = _model("c2_adagrad", x)
    assert m.step_counter == 0
    m.update_many(np.arange(3, dtype=np.int32))
    m.validate(xv)
    assert m.step_counter == 4
    import vaeb_b200
    xb = vaeb_b200.pinned_empty((100, 784), np.float32)
    xb[:] = x[:100]
    m.update_host_async(xb)
    assert m.step_counter == 5            # the getter launches the pending streaming update first
    with pytest.raises(ValueError, match="collect"):
        m.save_checkpoint("/nonexistent/never-written.npz")
    m.collect()
    m.step_counter = 17
    assert m.step_counter == 17
    m.close()


def test_cli_resume_matches_uninterrupted_run(tmp_path):
    """main() with --synthetic for 4 epochs, against: 2 epochs with --checkpoint_file; a resumed run that gets to epoch 3
    and stops before its next checkpoint (its trace lines stay behind); a second resume from the epoch-2 checkpoint to
    4.  The trace files and the saved parameters are identical."""
    code = ("import sys; sys.path.insert(0, %r); from vaeb_b200 import cli; cli.main(sys.argv[1:])" % ROOT)
    common = ["--synthetic", "--continuous", "--n_latent", "2", "--hidden_unit", "200", "--batch_size", "100",
              "--checkpoint_every", "1"]

    def run(*extra):
        r = subprocess.run([sys.executable, "-c", code, *common, *extra], cwd=str(tmp_path), capture_output=True,
                           text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        return r.stdout

    run("--n_epochs", "4", "--trace_file", "a.trc", "--save_file", "a.mdl")
    run("--n_epochs", "2", "--trace_file", "b.trc", "--checkpoint_file", "b.npz")
    run("--n_epochs", "3", "--trace_file", "b.trc", "--resume_file", "b.npz", "--checkpoint_file", "later.npz")
    assert (tmp_path / "b.trc").read_text().count("\n") == 1 + 2 * 3
    out = run("--n_epochs", "4", "--trace_file", "b.trc", "--resume_file", "b.npz", "--checkpoint_file", "b.npz",
              "--save_file", "b.mdl")
    assert "Epoch 2 :" in out and "Epoch 0 :" not in out
    a, b = (tmp_path / "a.trc").read_text(), (tmp_path / "b.trc").read_text()
    assert a.count("\n") == 1 + 2 * 4 and a == b
    from vaeb_b200 import io
    _, pa = io.read_mdl(str(tmp_path / "a.mdl"))
    _, pb = io.read_mdl(str(tmp_path / "b.mdl"))
    for p, q in zip(pa, pb):
        np.testing.assert_array_equal(p, q)
    bad = subprocess.run([sys.executable, "-c", code, *common, "--n_epochs", "5", "--resume_file", "b.npz",
                          "--learning_rate", "0.02"], cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert bad.returncode != 0 and "learning_rate" in bad.stderr


def test_two_gpus_resume(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import json
    import socket
    for p2p in ("1", "0"):
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
        s.close()
        out = tmp_path / ("dp_%s.json" % p2p)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
               "--master-addr", "127.0.0.1", "--master-port", str(port),
               os.path.join(ROOT, "tests", "checkpoint_dp_worker.py"), str(out), str(tmp_path)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=dict(os.environ, VAEB_DP_P2P=p2p))
        assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
        res = json.load(open(out))
        assert len(res["cases"]) == 2
        for c in res["cases"]:
            assert c["resumed_equals_uninterrupted"] and c["ranks_bit_identical"], c
