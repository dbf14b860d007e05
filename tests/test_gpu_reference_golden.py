"""The CUDA path (through the C-ABI) against golden vectors produced by the reference's OWN source
(tests/golden/make_reference_golden.py).  Same inputs, same initial parameters, the same noise the
reference drew, injected call by call.  fp32 tier of the north star: returned bounds within 1e-4
relative; parameters / Adagrad accumulators within 1e-4 * max(|ref|, 0.05 * ||ref||_inf)."""
import numpy as np
import pytest

from tests.util import assert_close_tensor, frey_trained_params, load_golden

pytestmark = pytest.mark.gpu

NAMES_D = ["W3", "W4", "W5", "W1", "W2", "b3", "b4", "b5", "b1", "b2"]
NAMES_C = ["W3", "W4", "W5", "W1", "W2", "W6", "b3", "b4", "b5", "b1", "b2", "b6"]


def fp16(t):
    f = np.asarray(t, np.float64).ravel()
    idx = np.linspace(0, f.size - 1, 16).astype(int)
    return np.concatenate([[f.sum(), (f * f).sum(), np.abs(f).max()], f[idx]])


def _sub(g, prefix):
    return {k[len(prefix) + 2:]: v for k, v in g.items() if k.startswith(prefix + "__")}


def _replay(c, params0, generic=False, full_var=False, **kw):
    import vaeb_b200
    cont = bool(c["continuous"])
    m = vaeb_b200.VAEB(c["x"], cont, int(c["H"]), int(c["Z"]), int(c["M"]), int(c.get("L", 1)), float(c["lr"]),
                       generic, full_var, [np.asarray(p, np.float32) for p in params0], **kw)
    rets = [float(m.update(int(i), eps=c["eps_update_%d" % k])) for k, i in enumerate(c["order"])]
    nv = c["eps_validate"].shape[1]
    val = float(m.validate(c["x"][:nv], eps=c["eps_validate"]))
    return m, np.array(rets), val


def _check_state(m, c, names, step_atol=0.0):
    """step_atol: Adagrad normalises every step to magnitude <= lr whatever |g| is, so a gradient entry
    that is a sum of cancelling terms (fp32 relative error up to ~1e-3 of the entry) moves its
    parameter by up to 1e-3*lr per update; the trained-weights cases allow exactly that on top."""
    for n, p, a in zip(names, m.get_params(), [t.get_value() for t in m.ADA]):
        if "fp_final_" + n in c:
            np.testing.assert_allclose(fp16(p)[:3], c["fp_final_" + n][:3], rtol=2e-4, err_msg=n)
            ref = c["fp_final_" + n][3:]
            assert np.all(np.abs(fp16(p)[3:] - ref) <= 1e-4 * np.maximum(np.abs(ref), 0.05 * np.abs(ref).max()) + step_atol), n
        else:
            ref = np.asarray(c["final_" + n], np.float64)
            err = np.abs(p.astype(np.float64) - ref)
            assert np.all(err <= 1e-4 * np.maximum(np.abs(ref), 0.05 * np.abs(ref).max()) + step_atol), (n, err.max())
            assert_close_tensor(a, c["ada_" + n], 1e-3 if step_atol else 2e-4, 0.05, "ada " + n)


@pytest.mark.parametrize("case", ["disc_LB_L1", "disc_LA_L2", "cont_LB_L2", "cont_LA_L1"])
def test_cuda_matches_reference_vaeb_small(case):
    c = _sub(load_golden("ref_vaeb_small.npz"), case)
    names = NAMES_C if bool(c["continuous"]) else NAMES_D
    m, rets, val = _replay(c, [c["init_" + n] for n in names], generic=bool(c["generic"]))
    np.testing.assert_allclose(rets, c["update_returns"], rtol=1e-4)
    assert val == pytest.approx(float(c["validate_return"]), rel=1e-4)
    _check_state(m, c, names)
    m.close()


@pytest.mark.parametrize("case", ["disc_LB_L1", "cont_LA_L1"])
def test_cuda_matches_reference_adadelta(case):
    """getAdaDeltaUpdates (VAEB.py:449-469) on the device: six updates, then validate."""
    c = _sub(load_golden("ref_adadelta_small.npz"), case)
    names = NAMES_C if bool(c["continuous"]) else NAMES_D
    m, rets, val = _replay(c, [c["init_" + n] for n in names], generic=bool(c["generic"]), optimizer="adadelta")
    np.testing.assert_allclose(rets, c["update_returns"], rtol=1e-4)
    assert val == pytest.approx(float(c["validate_return"]), rel=1e-4)
    for n, p in zip(names, m.get_params()):
        # an AdaDelta step is sqrt(dx_ac + 1e-6) * g / sqrt(g_ac + 1e-6) ~ 1e-3 * sign(g) at first: entries whose
        # gradient is a sum of cancelling terms move by up to that much differently (cf. _check_state)
        ref = np.asarray(c["final_" + n], np.float64)
        err = np.abs(p.astype(np.float64) - ref)
        assert np.all(err <= 1e-4 * np.maximum(np.abs(ref), 0.05 * np.abs(ref).max()) + 6e-6), (n, err.max())
    m.close()


@pytest.mark.parametrize("est", ["LB", "LA"])
def test_cuda_matches_reference_frey_trained(est):
    """C1 shape (560-200-2, M=100) with the trained weights the reference ships."""
    g = load_golden("ref_vaeb_frey_trained.npz")
    c = dict(_sub(g, est), x=g["x"])               # both estimators ran on the same rows, stored once
    m, rets, val = _replay(c, frey_trained_params(), generic=(est == "LA"))
    np.testing.assert_allclose(rets, c["update_returns"], rtol=1e-4)
    assert val == pytest.approx(float(c["validate_return"]), rel=1e-4)
    _check_state(m, c, NAMES_C, step_atol=1e-3 * 0.01 * len(c["order"]))
    m.close()


@pytest.mark.parametrize("precision,rtol", [("fp32", 1e-4), ("bf16x3", 1e-4), ("bf16", 1e-2)])
def test_cuda_matches_reference_mnist_init(precision, rtol):
    """C2 shape (784-500-20, M=100) from the reference's own initialisation (params=None: the
    host mirror must reproduce the RandomState(10) draw order, VAEB.py:50-125)."""
    import vaeb_b200
    c = load_golden("ref_vaeb_mnist_init.npz")
    m = vaeb_b200.VAEB(c["x"], False, 500, 20, 100, 1, 0.01, False, False, precision=precision)
    ret = float(m.update(1, eps=c["eps_update_0"]))
    val = float(m.validate(c["x"][:200], eps=c["eps_validate"]))
    assert ret == pytest.approx(float(c["update_returns"][0]), rel=rtol)
    assert val == pytest.approx(float(c["validate_return"]), rel=rtol)
    if precision != "bf16":
        _check_state(m, c, NAMES_D)
    m.close()


def test_cuda_matches_reference_full_variational():
    """getFVBL through the kernels: M * (data term) + theta prior; only (mu_vb, sigma_vb) move."""
    c = load_golden("ref_fvb_small.npz")
    c["continuous"], c["L"] = False, 1
    p0 = [c["init_" + n] for n in NAMES_D]
    m, rets, val = _replay(c, p0, full_var=True)
    np.testing.assert_allclose(rets, c["update_returns"], rtol=1e-4)
    assert val == pytest.approx(float(c["validate_return"]), rel=1e-4)
    fv = [t.get_value() for t in m.full_variational_params]
    for i, n in enumerate(NAMES_D):
        assert_close_tensor(fv[2 * i], c["final_mu_" + n], 1e-4, 0.05, "mu " + n)
        assert_close_tensor(fv[2 * i + 1], c["final_sigma_" + n], 1e-4, 0.05, "sigma " + n)
    for p, n in zip(m.get_params(), NAMES_D):
        np.testing.assert_array_equal(p, c["init_" + n].astype(np.float32))     # MAP parameters untouched (F5)
    m.close()


@pytest.mark.parametrize("tag", ["disc", "cont"])
def test_cuda_matches_reference_fullbayes_variant(tag):
    c = _sub(load_golden("ref_fullbayes_small.npz"), tag)
    names = NAMES_C if bool(c["continuous"]) else NAMES_D
    m, rets, val = _replay(c, [c["init_" + n] for n in names], variant="fullbayes")
    np.testing.assert_allclose(rets, c["update_returns"], rtol=1e-4)
    assert val == pytest.approx(float(c["validate_return"]), rel=1e-4)
    _check_state(m, c, names)
    m.close()


def test_cuda_mlp_forward_matches_reference_construct_mlp():
    """degenerate-vae/mlp.py:66-74 ConstructMLP, logpdf.py:46-47 OutToProbs, :72-73 OutToReal."""
    import vaeb_b200.model as M
    g = load_golden("ref_ae_primitives.npz")
    Ws = [g["mlp_W%d" % i] for i in range(3)]
    bs = [g["mlp_b%d" % i] for i in range(3)]
    np.testing.assert_allclose(M.mlp_forward(g["Y"], Ws, bs, "tanh"), g["mlp_out"], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(M.mlp_forward(g["Y"], Ws[:1], bs[:1], "sigmoid"), g["out_to_probs"], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(M.mlp_forward(g["Y"], Ws[:1], bs[:1], "identity"), g["out_to_real"], rtol=1e-4, atol=1e-6)
