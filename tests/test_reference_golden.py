"""The numpy oracle against golden vectors produced by the reference's OWN source
(tests/golden/make_reference_golden.py: /root/reference/VAEB.py, VAEBfullbayes.py and
degenerate-vae/{logpdf,mlp,infalg}.py executed on the Theano stand-in tests/golden/theano_shim.py,
float64).  Inputs, initial parameters and the noise of every call are read from the fixture; the
oracle must reproduce every returned bound and every parameter / accumulator after the updates."""
import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests.util import frey_trained_params, load_golden

RTOL = 1e-9     # float64 on both sides; summation orders differ


def fp16(t):
    f = np.asarray(t, np.float64).ravel()
    idx = np.linspace(0, f.size - 1, 16).astype(int)
    return np.concatenate([[f.sum(), (f * f).sum(), np.abs(f).max()], f[idx]])


def _sub(g, prefix):
    return {k[len(prefix) + 2:]: v for k, v in g.items() if k.startswith(prefix + "__")}


def _replay(c, params0, estimator, variant="vaeb", optimizer="adagrad"):
    cont = bool(c["continuous"])
    names = O.param_names(cont)
    H, Z, M, L = int(c["H"]), int(c["Z"]), int(c["M"]), int(c.get("L", 1))
    x = c["x"].astype(np.float64)
    m = O.OracleVAEB(x, cont, H, Z, M, L=L, lr=float(c["lr"]), estimator=estimator, params=params0,
                     dtype=np.float64, variant=variant, optimizer=optimizer)
    rets = [m.update(int(i), c["eps_update_%d" % k]) for k, i in enumerate(c["order"])]
    nv = c["eps_validate"].shape[1]
    val = m.validate(x[:nv], c["eps_validate"])[0]
    return m, names, np.array(rets), val


@pytest.mark.parametrize("case", ["disc_LB_L1", "disc_LA_L2", "cont_LB_L2", "cont_LA_L1"])
def test_oracle_matches_reference_vaeb_small(case):
    """VAEB.py update()/validate() for both decoders x both estimators x L in {1,2}: 4 Adagrad
    updates (pre-update outputs, VAEB.py:408-415) and one validate (VAEB.py:418-422)."""
    c = _sub(load_golden("ref_vaeb_small.npz"), case)
    cont = bool(c["continuous"])
    p0 = [c["init_" + n] for n in O.param_names(cont)]
    m, names, rets, val = _replay(c, p0, "LA" if bool(c["generic"]) else "LB")
    np.testing.assert_allclose(rets, c["update_returns"], rtol=RTOL)
    assert val == pytest.approx(float(c["validate_return"]), rel=RTOL)
    for n, p, a in zip(names, m.params, m.ada):
        np.testing.assert_allclose(p, c["final_" + n], rtol=1e-8, atol=1e-12, err_msg=n)
        np.testing.assert_allclose(a, c["ada_" + n], rtol=1e-8, atol=1e-14, err_msg="ada " + n)


@pytest.mark.parametrize("case", ["disc_LB_L1", "cont_LA_L1"])
def test_oracle_matches_reference_adadelta(case):
    """getAdaDeltaUpdates (VAEB.py:449-469) swapped in for getUpdates, as un-commenting VAEB.py:404 does:
    six updates (rho = 0.95, eps = 1e-6) and one validate."""
    c = _sub(load_golden("ref_adadelta_small.npz"), case)
    cont = bool(c["continuous"])
    p0 = [c["init_" + n] for n in O.param_names(cont)]
    m, names, rets, val = _replay(c, p0, "LA" if bool(c["generic"]) else "LB", optimizer="adadelta")
    np.testing.assert_allclose(rets, c["update_returns"], rtol=RTOL)
    assert val == pytest.approx(float(c["validate_return"]), rel=RTOL)
    for n, p in zip(names, m.params):
        np.testing.assert_allclose(p, c["final_" + n], rtol=1e-8, atol=1e-12, err_msg=n)


def test_oracle_init_matches_reference_draw_order():
    """initialize_params (VAEB.py:50-125): RandomState(10), the discarded duplicate W3/W4 block,
    float32 cast -- at the real MNIST and Frey shapes."""
    g = load_golden("ref_init_fingerprints.npz")
    for tag, (D, H, Z, cont) in {"mnist": (784, 500, 20, False), "frey": (560, 200, 2, True)}.items():
        ps = O.init_params(D, H, Z, cont)
        for n, p in zip(O.param_names(cont), ps):
            assert p.dtype == np.float32
            np.testing.assert_allclose(fp16(p), g["%s__fp_%s" % (tag, n)], rtol=1e-12, atol=0, err_msg=tag + n)


@pytest.mark.parametrize("est", ["LB", "LA"])
def test_oracle_matches_reference_frey_trained(est):
    """Frey shape (560-200-2, M=100) with the trained weights the reference ships: 2 updates + validate."""
    g = load_golden("ref_vaeb_frey_trained.npz")
    c = dict(_sub(g, est), x=g["x"])               # both estimators ran on the same rows, stored once
    m, names, rets, val = _replay(c, [p.astype(np.float64) for p in frey_trained_params()], est)
    np.testing.assert_allclose(rets, c["update_returns"], rtol=RTOL)
    assert val == pytest.approx(float(c["validate_return"]), rel=RTOL)
    for n, p, a in zip(names, m.params, m.ada):
        if "fp_final_" + n in c:
            np.testing.assert_allclose(fp16(p), c["fp_final_" + n], rtol=1e-8, atol=1e-12, err_msg=n)
            np.testing.assert_allclose(fp16(a), c["fp_ada_" + n], rtol=1e-8, atol=1e-12, err_msg="ada " + n)
        else:
            np.testing.assert_allclose(p, c["final_" + n], rtol=1e-8, atol=1e-12, err_msg=n)
            np.testing.assert_allclose(a, c["ada_" + n], rtol=1e-8, atol=1e-14, err_msg="ada " + n)


def test_oracle_matches_reference_mnist_init():
    """MNIST shape (784-500-20, M=100), the reference's own initialisation: update(1) + validate."""
    c = load_golden("ref_vaeb_mnist_init.npz")
    p0 = [p.astype(np.float64) for p in O.init_params(784, 500, 20, False, dtype=np.float64)]
    m, names, rets, val = _replay(c, p0, "LB")
    np.testing.assert_allclose(rets, c["update_returns"], rtol=RTOL)
    assert val == pytest.approx(float(c["validate_return"]), rel=RTOL)
    for n, p, a in zip(names, m.params, m.ada):
        if "fp_final_" + n in c:
            np.testing.assert_allclose(fp16(p), c["fp_final_" + n], rtol=1e-8, atol=1e-12, err_msg=n)
        else:
            np.testing.assert_allclose(p, c["final_" + n], rtol=1e-8, atol=1e-12, err_msg=n)


def test_oracle_matches_reference_full_variational():
    """fullVariational=True (getFVBL VAEB.py:349-367; SURVEY F5): the bound carries M * (data term)
    + theta prior, only the (mu_vb, sigma_vb) pairs move, the MAP parameters stay put."""
    c = load_golden("ref_fvb_small.npz")
    c["continuous"], c["L"] = False, 1
    p0 = [c["init_" + n] for n in O.param_names(False)]
    m, names, rets, val = _replay(c, p0, "FVB")
    np.testing.assert_allclose(rets, c["update_returns"], rtol=RTOL)
    assert val == pytest.approx(float(c["validate_return"]), rel=RTOL)
    for i, n in enumerate(names):
        np.testing.assert_allclose(m.fvp[2 * i], c["final_mu_" + n], rtol=1e-8, atol=1e-12, err_msg="mu " + n)
        np.testing.assert_allclose(m.fvp[2 * i + 1], c["final_sigma_" + n], rtol=1e-8, atol=1e-12, err_msg="sigma " + n)
        np.testing.assert_array_equal(m.params[i], c["final_map_" + n])
        np.testing.assert_array_equal(c["final_map_" + n], c["init_" + n])


@pytest.mark.parametrize("tag", ["disc", "cont"])
def test_oracle_matches_reference_fullbayes_variant(tag):
    """VAEBfullbayes.py:121-201: mean objective, no weight prior, the extra -lr*1e-6*p**2 term."""
    c = _sub(load_golden("ref_fullbayes_small.npz"), tag)
    cont = bool(c["continuous"])
    p0 = [c["init_" + n] for n in O.param_names(cont)]
    m, names, rets, val = _replay(c, p0, "LB", variant="fullbayes")
    np.testing.assert_allclose(rets, c["update_returns"], rtol=RTOL)
    assert val == pytest.approx(float(c["validate_return"]), rel=RTOL)
    for n, p, a in zip(names, m.params, m.ada):
        np.testing.assert_allclose(p, c["final_" + n], rtol=1e-8, atol=1e-12, err_msg=n)
        np.testing.assert_allclose(a, c["ada_" + n], rtol=1e-8, atol=1e-14, err_msg="ada " + n)


def test_oracle_matches_reference_ae_primitives():
    """degenerate-vae/logpdf.py:46-47,72-73,85-86,112-114; mlp.py:66-91,157-159; infalg.py:148-164."""
    g = load_golden("ref_ae_primitives.npz")
    assert float(g["bernoulli_kat"]) == pytest.approx(-0.0603014090604, rel=1e-11)      # logpdf.py:119-123
    assert float(O.lpdf_bernoulli(np.array([[0, 0, 1], [0, 0, 1.]]), np.array([[.01, .01, .99]] * 2))) == \
        pytest.approx(float(g["bernoulli_kat"]), rel=1e-13)
    Y, P, MU, LS2 = g["Y"], g["P"], g["MU"], g["LS2"]
    assert float(O.lpdf_bernoulli(Y, P)) == pytest.approx(float(g["bernoulli"]), rel=1e-12)
    assert float(O.lpdf_indep_normal(Y, MU, LS2)) == pytest.approx(float(g["indep_normal"]), rel=1e-12)
    Ws = [g["mlp_W%d" % i] for i in range(3)]
    bs = [g["mlp_b%d" % i] for i in range(3)]
    np.testing.assert_allclose(O.construct_mlp(Y, Ws, bs), g["mlp_out"], rtol=1e-12)
    assert float(O.normal_prior(Ws + bs, 0.7)) == pytest.approx(float(g["normal_prior"]), rel=1e-12)
    assert float(O.gauss_dkl(MU, np.exp(LS2), P, g["s21"])) == pytest.approx(float(g["gauss_dkl"]), rel=1e-12)
    np.testing.assert_allclose(O.out_to_probs(Y, Ws[0], bs[0]), g["out_to_probs"], rtol=1e-12)
    np.testing.assert_allclose(O.out_to_real(Y, Ws[0], bs[0]), g["out_to_real"], rtol=1e-12)
    # AdaGrad.construct: two ascent steps on the toy objective of the generator
    th = [g["ag_theta0_0"].copy(), g["ag_theta0_1"].copy()]
    ada = [np.zeros_like(t) for t in th]
    objs = []
    for _ in range(2):
        objs.append(-3.0 * ((th[0] - 0.5) ** 2).sum() - 0.25 * (((th[1] + 1.0) ** 2) * th[1]).sum())
        grads = [-6.0 * (th[0] - 0.5), -0.25 * (2.0 * (th[1] + 1.0) * th[1] + (th[1] + 1.0) ** 2)]
        O.adagrad_update(th, ada, grads, float(g["ag_eta"]), 1e-6)
    np.testing.assert_allclose(objs, g["ag_obj"], rtol=1e-12)
    np.testing.assert_allclose(th[0], g["ag_theta2_0"], rtol=1e-12)
    np.testing.assert_allclose(th[1], g["ag_theta2_1"], rtol=1e-12)


def ae_params_from_fixture(c, continuous, prefix):
    """VAEB-ordered parameter list from a ref_ae_baselines fixture (W5, b5 are not part of an AE: zeros)."""
    H, Z = c["init_W4"].shape
    out = []
    for n in O.param_names(continuous):
        if n == "W5":
            out.append(np.zeros((H, Z)))
        elif n == "b5":
            out.append(np.zeros(Z))
        else:
            out.append(np.array(c[prefix + n], dtype=np.float64))
    return out


@pytest.mark.parametrize("tag,kind,cont", [("deg_binary", "degenerate", False), ("deg_cont", "degenerate", True),
                                           ("vanilla", "vanilla", False)])
def test_oracle_matches_reference_ae_baselines(tag, kind, cont):
    """ConstructAE of degenerate-vae/ae.py:41-117 (binary and cont outputs) and vanilla-ae/ae.py:45-104: five
    `train(idx)` calls on gathered minibatches (the last one ragged), then reconstruct / encode / decode."""
    c = _sub(load_golden("ref_ae_baselines.npz"), tag)
    m = O.OracleAE(c["x"].astype(np.float64), cont, ae_params_from_fixture(c, cont, "init_"), kind=kind)
    rets = [m.train(row[row >= 0]) for row in c["idx"]]
    np.testing.assert_allclose(rets, c["train_returns"], rtol=RTOL)
    for n, p in zip(O.param_names(cont), m.params):
        if n in ("W5", "b5"):
            assert not p.any()
        else:
            np.testing.assert_allclose(p, c["final_" + n], rtol=1e-8, atol=1e-12, err_msg=n)
    x6 = c["x"][:6].astype(np.float64)
    np.testing.assert_allclose(m.forward(x6, "reconstruct"), c["reconstruct"], rtol=1e-10)
    np.testing.assert_allclose(m.forward(x6, "encode"), c["encode"], rtol=1e-10, atol=1e-14)
    np.testing.assert_allclose(m.forward(c["encode"], "decode"), c["decode"], rtol=1e-10)
