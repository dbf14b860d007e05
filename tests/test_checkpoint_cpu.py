"""The checkpoint file (vaeb_b200/checkpoint.py) without a device: the npz / JSON round trip, the host RNG states, every
refusal, the atomic write, the CLI options and the driver state of the training loop."""
import json
import os

import numpy as np
import pytest

from vaeb_b200 import checkpoint as ck
from vaeb_b200 import cli
from vaeb_b200.rng import RandomStreams


def _header(x, world=1):
    return dict(vaeb_version=106, args={"hidden_units": 8, "learning_rate": 0.01, "adam_betas": [0.9, 0.999]},
                tensors=[["W3", [6, 8]], ["b3", [8]]], buffers=["params"], world_size=world,
                data=[ck.data_fingerprint(x)] * world, theano_nodes=0)


def _arrays():
    rng = np.random.RandomState(1)
    return {"params.W3": rng.normal(size=(6, 8)).astype(np.float32), "params.b3": rng.normal(size=8).astype(np.float32),
            "counter.step": np.array(4000000000, np.uint32), "counter.adam_step": np.array(7, np.int64),
            "counter.kl_step": np.array(3, np.int64)}


def test_round_trip_of_arrays_header_and_driver_state(tmp_path):
    x = np.random.RandomState(0).uniform(size=(10, 6)).astype(np.float32)
    path = str(tmp_path / "c.npz")
    arrays = _arrays()
    ck.write(path, _header(x), arrays, driver_state={"epoch": 12, "note": "x", "order": np.arange(5)})
    header, got, driver = ck.read(path)
    assert header["format_version"] == ck.FORMAT_VERSION and header["args"]["adam_betas"] == [0.9, 0.999]
    assert header["data"][0] == ck.data_fingerprint(x)
    assert sorted(got) == sorted(arrays)
    for k in arrays:
        assert got[k].dtype == arrays[k].dtype
        np.testing.assert_array_equal(got[k], arrays[k])
    assert driver["epoch"] == 12 and driver["note"] == "x"
    np.testing.assert_array_equal(driver["order"], np.arange(5))
    with np.load(path, allow_pickle=False) as z:           # readable without pickle
        json.loads(str(z["header"][()]))


def test_random_streams_and_numpy_state_round_trip(tmp_path):
    s = RandomStreams(seed=10)
    nodes = [s.new_node() for _ in range(3)]
    s.normal(nodes[1], (3, 5))
    s.nodes[2].standard_normal()            # an odd number of normals leaves a cached Gaussian behind
    np.random.seed(123)
    np.random.standard_normal()
    arrays = {}
    ck.pack_random_state(arrays, "seedgen", s.gen_seedgen.get_state())
    for k, nd in enumerate(s.nodes):
        ck.pack_random_state(arrays, "node%d" % k, nd.get_state())
    drv = cli.loop_state(2, np.array([3, 1, 2]))
    path = str(tmp_path / "r.npz")
    ck.write(path, _header(np.zeros((2, 6), np.float32)), arrays, driver_state=drv)
    _, got, driver = ck.read(path)
    expect = [s.normal(k, (4, 2)) for k in range(3)] + [s.gen_seedgen.randint(2 ** 30)]
    t = RandomStreams(seed=99)
    t.gen_seedgen.set_state(ck.unpack_random_state(got, "seedgen"))
    for k in range(3):
        r = np.random.RandomState()
        r.set_state(ck.unpack_random_state(got, "node%d" % k))
        t.nodes.append(r)
    again = [t.normal(k, (4, 2)) for k in range(3)] + [t.gen_seedgen.randint(2 ** 30)]
    for a, b in zip(expect, again):
        np.testing.assert_array_equal(a, b)
    want = np.random.standard_normal(4)
    np.random.seed(0)
    np.random.set_state(ck.random_state_tuple(driver["np_random_keys"], driver["np_random_aux"]))
    np.testing.assert_array_equal(np.random.standard_normal(4), want)
    assert driver["epoch"] == 2
    np.testing.assert_array_equal(driver["batch_order"], [3, 1, 2])


def test_unknown_format_version_is_refused(tmp_path):
    path = str(tmp_path / "v.npz")
    np.savez(path, header=np.array(json.dumps({"format_version": 99, "arrays": {}})))
    with pytest.raises(ValueError, match="format_version"):
        ck.read(path)


def test_missing_array_is_refused(tmp_path):
    path = str(tmp_path / "m.npz")
    ck.write(path, _header(np.zeros((2, 6), np.float32)), _arrays())
    with np.load(path, allow_pickle=False) as z:
        kept = {k: z[k] for k in z.files if k != "params.b3"}
    np.savez(path, **kept)
    with pytest.raises(ValueError, match="params.b3"):
        ck.read(path)
    with pytest.raises(ValueError, match="counter.step"):
        ck.require({}, "counter.step")


def test_shape_mismatches_are_refused(tmp_path):
    path = str(tmp_path / "s.npz")
    ck.write(path, _header(np.zeros((2, 6), np.float32)), _arrays())
    with np.load(path, allow_pickle=False) as z:
        kept = {k: z[k] for k in z.files}
    kept["params.W3"] = np.zeros((6, 9), np.float32)
    np.savez(path, **kept)
    with pytest.raises(ValueError, match="params.W3"):
        ck.read(path)
    header = _header(np.zeros((2, 6), np.float32))
    with pytest.raises(ValueError, match="W3"):
        ck.check_tensors(header, [("W3", (6, 9)), ("b3", (8,))])
    with pytest.raises(ValueError, match="tensors"):
        ck.check_tensors(header, [("W3", (6, 8))])
    ck.check_tensors(header, [("W3", (6, 8)), ("b3", (8,))])
    with pytest.raises(ValueError, match="W3"):
        ck.require(_arrays(), "params.W3", (6, 9))


def test_data_and_world_size_mismatches_are_refused():
    x = np.random.RandomState(0).uniform(size=(10, 6)).astype(np.float32)
    header = _header(x)
    ck.check_compatible(header, data=ck.data_fingerprint(x), rank=0, world_size=1)
    y = x.copy()
    y[3, 2] = np.nextafter(y[3, 2], np.float32(2))         # one ulp in one element
    with pytest.raises(ValueError, match="fingerprint.*sha256"):
        ck.check_compatible(header, data=ck.data_fingerprint(y), rank=0, world_size=1)
    with pytest.raises(ValueError, match="fingerprint.*N"):
        ck.check_compatible(header, data=ck.data_fingerprint(x[:9]), rank=0, world_size=1)
    with pytest.raises(ValueError, match="world_size"):
        ck.check_compatible(header, data=ck.data_fingerprint(x), rank=0, world_size=2)


def test_a_writer_that_fails_halfway_leaves_the_old_file(tmp_path, monkeypatch):
    path = str(tmp_path / "a.npz")
    ck.write(path, _header(np.zeros((2, 6), np.float32)), _arrays())
    before = open(path, "rb").read()
    real = np.savez

    def broken(f, **kw):
        real(f, **kw)
        f.write(b"partial")
        raise OSError("disk full")

    monkeypatch.setattr(np, "savez", broken)
    arrays = _arrays()
    arrays["params.W3"] = arrays["params.W3"] + 1
    with pytest.raises(OSError, match="disk full"):
        ck.write(path, _header(np.zeros((2, 6), np.float32)), arrays)
    assert open(path, "rb").read() == before
    assert os.listdir(str(tmp_path)) == ["a.npz"]


def test_object_arrays_are_refused(tmp_path):
    with pytest.raises(TypeError, match="pickle"):
        ck.write(str(tmp_path / "o.npz"), {}, {"bad": np.array([{}, 1], dtype=object)})
    assert os.listdir(str(tmp_path)) == []


def test_parse_args_of_the_checkpoint_options():
    a = cli.parse_args([])
    assert (a["checkpoint_file"], a["checkpoint_every"], a["resume_file"]) == ("", 100, "")
    a = cli.parse_args(["--checkpoint_file", "c.npz", "--checkpoint_every", "5", "--resume_file", "r.npz"])
    assert (a["checkpoint_file"], a["checkpoint_every"], a["resume_file"]) == ("c.npz", 5, "r.npz")


def test_resume_refuses_other_model_shaping_options():
    args = cli.parse_args(["--n_latent", "2", "--continuous"])
    saved = cli.model_args(args, 1500)
    cli.check_resume_args(saved, cli.model_args(args, 1500))
    other = cli.model_args(cli.parse_args(["--n_latent", "2", "--continuous", "--learning_rate", "0.02"]), 1500)
    with pytest.raises(ValueError, match="learning_rate"):
        cli.check_resume_args(saved, other)
    other = cli.model_args(cli.parse_args(["--n_latent", "2", "--continuous", "--kl_warmup", "3"]), 1500)
    with pytest.raises(ValueError, match="kl_warmup"):
        cli.check_resume_args(saved, other)


def test_written_files_get_the_umask_mode_or_keep_the_replaced_ones(tmp_path):
    old = os.umask(0o022)
    try:
        path = str(tmp_path / "p.npz")
        ck.write(path, _header(np.zeros((2, 6), np.float32)), _arrays())
        assert os.stat(path).st_mode & 0o777 == 0o644
        os.chmod(path, 0o640)
        ck.write(path, _header(np.zeros((2, 6), np.float32)), _arrays())
        assert os.stat(path).st_mode & 0o777 == 0o640
    finally:
        os.umask(old)


def test_resume_rewinds_the_trace_to_the_checkpoint(tmp_path):
    from vaeb_b200 import io
    trace = str(tmp_path / "t.trc")
    io.trace_header(trace)
    io.trace_line(trace, 1500, -1.5, -2.5)
    at_checkpoint = cli.loop_state(1, np.arange(3), trace)["trace_bytes"]
    kept = open(trace).read()
    io.trace_line(trace, 3000, -1.0, -2.0)           # an epoch after the checkpoint, before the run stopped
    cli.rewind_trace(trace, at_checkpoint)
    assert open(trace).read() == kept
    with pytest.raises(ValueError, match="shorter"):
        cli.rewind_trace(trace, at_checkpoint + 1)
    cli.rewind_trace(str(tmp_path / "new.trc"), -1)  # no trace at the checkpoint: a fresh file
    assert open(str(tmp_path / "new.trc")).read() == "num_samples,L,Lvalid\n"
