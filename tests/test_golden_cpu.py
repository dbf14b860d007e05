"""CPU checks: the oracle reproduces the committed golden vectors; host logic (CLI parser,
.mdl/.trc layout, RandomStreams emulation, sharding); the C-ABI library loads and exports every
symbol include/vaeb_b200.h declares."""
import os
import re

import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests.util import GOLDEN, fingerprint, frey_trained_params, load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run_case(params, x, M, continuous, est, L, eps, H, Z):
    m = O.OracleVAEB(x, continuous, H, Z, M, L=L, estimator=est, params=params, dtype=np.float64)
    sgvb, per_row, grads = m.grads(x[:M], eps)
    ret = m.update(0, eps)
    return sgvb, per_row, grads, ret, m


@pytest.mark.parametrize("est", ["LB", "LA"])
def test_oracle_reproduces_golden_frey(est):
    g = load_golden("golden_frey_z2.npz")
    x = O.synthetic_frey(300)
    sgvb, per_row, grads, ret, m = _run_case(frey_trained_params(), x, 100, True, est, 1, g[est + "_eps"], 200, 2)
    assert sgvb == pytest.approx(float(g[est + "_sgvb"]), rel=1e-12)
    np.testing.assert_allclose(per_row, g[est + "_per_row"], rtol=1e-11)
    np.testing.assert_allclose(fingerprint(grads), g[est + "_grad_fp"], rtol=1e-9, atol=1e-12)
    assert ret == pytest.approx(float(g[est + "_update_return"]), rel=1e-12)
    np.testing.assert_allclose(m.params[1].astype(np.float32), g[est + "_after_W4"], rtol=1e-6)


def test_oracle_reproduces_golden_mnist_and_is():
    g = load_golden("golden_mnist_init.npz")
    params = O.init_params(784, 500, 20, False)
    x = O.synthetic_mnist(200)
    for est, L in (("LB", 1), ("LA", 2)):
        sgvb, per_row, grads, ret, _ = _run_case(params, x, 100, False, est, L, g[est + "_eps"], 500, 20)
        assert sgvb == pytest.approx(float(g[est + "_sgvb"]), rel=1e-12)
        np.testing.assert_allclose(fingerprint(grads), g[est + "_grad_fp"], rtol=1e-9, atol=1e-12)
    logp, logw = O.is_log_px([p.astype(np.float64) for p in params], x[100:108].astype(np.float64),
                             g["is_eps"].astype(np.float64), False)
    np.testing.assert_allclose(logp, g["is_logp"], rtol=1e-12)
    np.testing.assert_allclose(logw, g["is_logw"], rtol=1e-12)


def test_trained_weights_fixture_is_the_reference_layout():
    ps = frey_trained_params()
    assert [p.shape for p in ps] == O.param_shapes(560, 200, 2, True)
    assert all(p.dtype == np.float32 for p in ps)
    assert np.abs(ps[0]).max() > 0.1           # trained, not the 0.01-sigma initialisation


# ---- host logic ---------------------------------------------------------------------------
def test_cli_parser_matches_reference_defaults(capsys):
    from vaeb_b200 import cli
    a = cli.parse_args([])
    # VAEB.py:25-36
    assert (a["seed"], a["n_latent"], a["n_epochs"], a["batch_size"], a["L"], a["hidden_unit"]) == \
        (15485863, 10, 2000, 100, 1, -1)
    assert a["learning_rate"] == 0.01 and a["trace_file"] == "" and a["save_file"] == "" and a["load_file"] == ""
    assert a["continuous"] is False and a["generic_estimator"] is False and a["full_varational"] is False
    a = cli.parse_args(["--continuous", "--n_latent", "2", "--learning_rate", "0.5", "--full_varational",
                        "--vb_param_file", "m.mdl", "-generic_estimator", "-n_epochs", "3"])
    assert a["continuous"] and a["n_latent"] == 2 and a["learning_rate"] == 0.5 and a["full_varational"]
    assert a["vb_param_file"] == "m.mdl"
    # single-dash spellings (scripts/LAvsLB.sh:8,16) are NOT understood by the reference parser
    assert a["generic_estimator"] is False and a["n_epochs"] == 2000
    assert "Have unused args: ['-generic_estimator', '-n_epochs', '3']" in capsys.readouterr().out
    cli.print_args({"a": 1})
    out = capsys.readouterr().out
    assert out.startswith("Parameters used:\n" + "-" * 38 + "\n\ta: 1\n")


def test_mdl_roundtrip_and_legacy_layouts(tmp_path):
    from vaeb_b200 import io
    params = [np.random.RandomState(i).normal(size=s).astype(np.float32)
              for i, s in enumerate(O.param_shapes(12, 7, 3, False))]
    header = dict(n_hidden_units=7, n_latent=3, continuous=False, learning_rate=0.01, batch_size=5,
                  prng=np.random.RandomState(10), sigmaInit=0.01, L=1, genericEstimator=True)
    f = str(tmp_path / "m.mdl")
    io.write_mdl(f, header, params)
    h2, p2 = io.read_mdl(f)
    assert h2["genericEstimator"] is True and h2["n_latent"] == 3 and h2["continuous"] is False
    for a, b in zip(params, p2):
        np.testing.assert_array_equal(a, b)
    # the 8-object header the reference's current `save` writes (VAEB.py:193-200)
    import pickle
    f8 = str(tmp_path / "m8.mdl")
    with open(f8, "wb") as fh:
        for k in ["n_hidden_units", "n_latent", "continuous", "learning_rate", "batch_size", "prng", "sigmaInit", "L"]:
            pickle.dump(header[k], fh, protocol=2)
        for p in params:
            pickle.dump(p, fh, protocol=2)
    h3, p3 = io.read_mdl(f8)
    assert h3["genericEstimator"] is False and len(p3) == 10


def test_restricted_unpickler_never_imports_foreign_classes(tmp_path):
    import pickle
    from vaeb_b200 import io

    f = str(tmp_path / "evil.mdl")
    marker = tmp_path / "pwned"
    with open(f, "wb") as fh:
        fh.write(b"cos\nsystem\n(S'echo pwned > " + str(marker).encode() + b"'\ntR.")
    with pytest.raises(Exception):
        io.read_mdl(f)
    assert not marker.exists()


def test_trace_layout(tmp_path):
    from vaeb_b200 import io
    f = str(tmp_path / "t.trc")
    io.trace_header(f)
    io.trace_line(f, 1500, 84290.38083781234, 75975.2662633)
    io.trace_line(f, 1500, 84290.38083781234, 75975.2662633)
    # full_vb_res/continuous_2.trc:1-3 of the reference
    assert open(f).read() == "num_samples,L,Lvalid\n1500,84290.3808378,75975.2662633\n1500,84290.3808378,75975.2662633\n"
    assert io.py2_float(-61.0923518288) == "-61.0923518288" and io.py2_float(2.0) == "2.0"


def test_random_streams_emulation_matches_oracle_copy():
    from vaeb_b200.rng import RandomStreams
    s = RandomStreams(10)
    nodes = [s.new_node() for _ in range(2)]
    o = O.TheanoRandomStreams(10, n_nodes=2)
    for _ in range(3):
        a = np.stack([s.normal(n, (5, 4)) for n in nodes])
        np.testing.assert_array_equal(a, o.draw(5, 4))
    gen = np.random.RandomState(10)
    first = np.random.RandomState(int(gen.randint(2 ** 30))).normal(0, 1, (5, 4)).astype(np.float32)
    np.testing.assert_array_equal(RandomStreams(10).normal(RandomStreams(10).new_node() * 0 + 0, (5, 4)) if False else first,
                                  O.TheanoRandomStreams(10, 1).draw(5, 4)[0])


def test_shard_rows_cover_exactly():
    from vaeb_b200.distributed import shard_rows
    for n in (1, 7, 10000, 10001):
        for world in (1, 2, 3, 8):
            spans = [shard_rows(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))


def test_synthetic_data_matches_oracle_generator():
    from vaeb_b200 import data
    np.testing.assert_array_equal(data.synthetic_mnist(50), O.synthetic_mnist(50))
    np.testing.assert_array_equal(data.synthetic_frey(50), O.synthetic_frey(50))
    x = data.synthetic_mnist(2000)
    assert 0.17 < (x > 0).mean() < 0.21 and x.min() >= 0 and x.max() <= 1


# ---- the C-ABI library -------------------------------------------------------------------
def test_library_exports_every_declared_symbol():
    from vaeb_b200 import _lib
    header = open(os.path.join(ROOT, "include", "vaeb_b200.h")).read()
    declared = set(re.findall(r"\b(vaeb_[a-z_0-9]+)\s*\(", header))
    declared -= {"vaeb_handle", "vaeb_config"}
    assert declared, "no declarations found"
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), "library does not export " + name
    assert declared == set(_lib.EXPORTS), (declared ^ set(_lib.EXPORTS))
    assert lib.vaeb_version() >= 100


def test_no_cpu_fallback_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    import vaeb_b200
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        vaeb_b200.VAEB(np.zeros((10, 8), np.float32), False, 4, 2, 5, 1, 0.01, False, False)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "vaeb_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_persistent_layer_tile_schedule_covers_every_tile_once():
    """The persistent tensor-core layer kernel's tile order (tc_layers.cu TileSeq: full tiles round-robin, sliver column
    tiles to the CTAs with fewer full tiles).  Host arithmetic exported through vaeb_diag_tile_schedule: for every shape
    the three warp roles of a CTA walk the same list, and over the grid every tile must appear exactly once."""
    import ctypes as C
    from vaeb_b200 import _lib
    lib = _lib.load()
    cap = 4096
    tm, tn, n = (C.c_int32 * cap)(), (C.c_int32 * cap)(), C.c_int32()
    shapes = [(16384, 784, 256), (8192, 784, 256), (16384, 500, 256), (16384, 1120, 256), (16384, 560, 256),
              (128, 784, 256), (5000, 272, 256), (16384, 784, 128), (300, 130, 64), (16384, 40, 64), (77777, 784, 256),
              (16384, 1040, 256)]
    for rows, N, bn in shapes:
        tiles_m, tiles_n = -(-rows // 128), -(-N // bn)
        for grid in sorted({1, 7, 148, min(148, tiles_m * tiles_n)}):
            seen, per_cta = {}, []
            for cta in range(grid):
                assert lib.vaeb_diag_tile_schedule(rows, N, bn, grid, cta, cap, tm, tn, C.byref(n)) == 0
                per_cta.append(n.value)
                for i in range(n.value):
                    assert 0 <= tm[i] < tiles_m and 0 <= tn[i] < tiles_n
                    key = (tm[i], tn[i])
                    assert key not in seen, (rows, N, bn, grid, key)
                    seen[key] = cta
            assert len(seen) == tiles_m * tiles_n, (rows, N, bn, grid, len(seen))
            sliver = tiles_n > 1 and (N - (tiles_n - 1) * bn) * 4 <= bn
            if not sliver:                         # plain round-robin: tile t on CTA t % grid
                assert all(seen[(t // tiles_n, t % tiles_n)] == t % grid for t in range(tiles_m * tiles_n))
            else:                                  # no CTA holds more than one full tile above the others
                full = [sum(1 for (a, b), c in seen.items() if c == cta and b < tiles_n - 1) for cta in range(grid)]
                assert max(full) - min(full) <= 1
    assert lib.vaeb_diag_tile_schedule(128, 784, 256, 4, 4, cap, tm, tn, C.byref(n)) != 0      # cta out of range


def test_mdl_round_trip_carries_deeper_encoder_layers(tmp_path):
    """.mdl files (VAEB.py:204-226 layout) of deeper encoders: the extra (W3_k, b3_k) tensors follow the reference's list and
    read_mdl infers the depth from their number; the reference's 10 / 12 tensor files still read as depth 1."""
    from vaeb_b200 import io as vio
    hdr = {"n_hidden_units": 9, "n_latent": 3, "continuous": True, "learning_rate": 0.01, "batch_size": 7, "prng": None,
           "sigmaInit": 0.01, "L": 1, "genericEstimator": False}
    rng = np.random.RandomState(4)
    for depth in (1, 2, 4):
        params = [rng.normal(size=s).astype(np.float32) for s in O.param_shapes(12, 9, 3, True, depth)]
        f = str(tmp_path / ("d%d.mdl" % depth))
        vio.write_mdl(f, hdr, params)
        h2, p2 = vio.read_mdl(f)
        assert h2["encoder_layers"] == depth and len(p2) == 12 + 2 * (depth - 1)
        for a, b in zip(params, p2):
            np.testing.assert_array_equal(a, b)
    bad = str(tmp_path / "bad.mdl")
    vio.write_mdl(bad, hdr, params[:13])                     # an odd number of extra tensors is not a model
    with pytest.raises(ValueError):
        vio.read_mdl(bad)
