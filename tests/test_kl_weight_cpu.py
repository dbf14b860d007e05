"""The KL weight on the CPU: the oracle's weighted gradient against torch.autograd (fp64) of loglik + beta * aux - prior,
its identity at beta = 1, the warm-up schedule of vaeb_set_kl_weight as the Python side computes it, and the CLI's two
options."""
import math

import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests import kl_oracle as K

torch = pytest.importorskip("torch")


def _act(a, act):
    return {"tanh": torch.tanh, "sigmoid": torch.sigmoid, "relu": torch.relu}[act](a)


def _torch_terms(tp, names, x, eps, continuous, estimator, act, depth):
    """Per-row (loglik, aux) of getLB / getLA (VAEB.py:315-346), written from the reference's expressions; deeper
    encoders as replic.tex:46-57 builds them."""
    p = dict(zip(names, tp))
    x = torch.as_tensor(x)
    h = _act(x @ p["W3"] + p["b3"], act)
    for k in range(2, depth + 1):
        h = _act(h @ p["W3_%d" % k] + p["b3_%d" % k], act)
    mu, ls = h @ p["W4"] + p["b4"], h @ p["W5"] + p["b5"]
    L = eps.shape[0]
    loglik, aux = 0, 0
    for l in range(L):
        z = mu + torch.exp(0.5 * ls) * torch.as_tensor(eps[l])
        hd = _act(z @ p["W1"] + p["b1"], act)
        y = torch.sigmoid(hd @ p["W2"] + p["b2"])
        if continuous:
            lv = hd @ p["W6"] + p["b6"]
            loglik = loglik + (-0.5 * math.log(2 * math.pi) - 0.5 * lv - 0.5 * (x - y) ** 2 / torch.exp(lv)).sum(1)
        else:
            loglik = loglik + (x * torch.log(y) + (1 - x) * torch.log(1 - y)).sum(1)
        if estimator == "LA":
            prior = (-0.5 * math.log(2 * math.pi) - 0.5 * z ** 2).sum(1)
            logq = (-0.5 * math.log(2 * math.pi) - 0.5 * ls - 0.5 * (z - mu) ** 2 / torch.exp(ls)).sum(1)
            aux = aux + (prior - logq)
    if estimator == "LB":
        return loglik / L, 0.5 * (1 + ls - mu ** 2 - torch.exp(ls)).sum(1)
    return loglik / L, aux / L


CASES = [(c, e, L, "tanh", 1) for c in (False, True) for e in ("LB", "LA") for L in (1, 3)]
CASES += [(False, "LB", 1, "relu", 1), (True, "LA", 2, "relu", 1), (False, "LA", 1, "tanh", 2), (True, "LB", 2, "tanh", 2)]


@pytest.mark.parametrize("kl", [0.0, 0.3, 2.5])
@pytest.mark.parametrize("continuous,est,L,act,depth", CASES)
def test_weighted_gradient_matches_autograd(kl, continuous, est, L, act, depth):
    M, D, H, Z = 7, 11, 9, 4
    rng = np.random.RandomState(5 + L + depth)
    names = O.param_names(continuous, depth)
    shapes = O.param_shapes(D, H, Z, continuous, depth)
    params = [rng.normal(0, 0.3, s) for s in shapes]
    x, eps = rng.uniform(size=(M, D)), rng.normal(size=(L, M, Z))
    out = K.elbo_and_grads(params, x, eps, continuous, est, act=act, kl_weight=kl)
    tp = [torch.tensor(q, requires_grad=True) for q in params]
    loglik, aux = _torch_terms(tp, names, x, eps, continuous, est, act, depth)
    crit = (loglik + kl * aux).sum() - 0.5 * sum((q ** 2).sum() for q in tp)
    crit.backward()
    assert out.sgvb == pytest.approx((loglik + aux).sum().item(), rel=1e-12)      # the bound stays unweighted
    for g, q, n in zip(out.grads, tp, names):
        ref = q.grad.numpy()
        assert np.abs(g - ref).max() <= 1e-10 * max(np.abs(ref).max(), 1e-3), (n, np.abs(g - ref).max())


@pytest.mark.parametrize("continuous,est,L", [(False, "LB", 1), (True, "LA", 2)])
def test_weight_one_is_the_oracle_bit_for_bit(continuous, est, L):
    rng = np.random.RandomState(9)
    params = [rng.normal(0, 0.3, s) for s in O.param_shapes(10, 8, 3, continuous)]
    x, eps = rng.uniform(size=(6, 10)), rng.normal(size=(L, 6, 3))
    a = K.elbo_and_grads(params, x, eps, continuous, est, kl_weight=1.0)
    b = O.elbo_and_grads(params, x, eps, continuous, est)
    assert a.sgvb == b.sgvb
    for g, h in zip(a.grads, b.grads):
        np.testing.assert_array_equal(g, h)
    o1 = K.OracleKLVAEB(x, continuous, 8, 3, 6, L=L, estimator=est, params=params, kl_weight=1.0)
    o2 = O.OracleVAEB(x, continuous, 8, 3, 6, L=L, estimator=est, params=params)
    assert o1.update(0, eps) == o2.update(0, eps)
    for p, q in zip(o1.params, o2.params):
        np.testing.assert_array_equal(p, q)


def test_fullbayes_variant_weights_the_mean_objective():
    """VAEBfullbayes.py: the gradient of mean(loglik + beta aux) with no weight prior."""
    rng = np.random.RandomState(4)
    names = O.param_names(True)
    params = [rng.normal(0, 0.3, s) for s in O.param_shapes(10, 8, 3, True)]
    x, eps = rng.uniform(size=(6, 10)), rng.normal(size=(1, 6, 3))
    o = K.OracleKLVAEB(x, True, 8, 3, 6, params=params, variant="fullbayes", kl_weight=0.4)
    _, _, g = o.grads(x, eps)
    tp = [torch.tensor(q, requires_grad=True) for q in params]
    loglik, aux = _torch_terms(tp, names, x, eps, True, "LB", "tanh", 1)
    ((loglik + 0.4 * aux).mean()).backward()
    for a, q, n in zip(g, tp, names):
        np.testing.assert_allclose(a, q.grad.numpy(), rtol=1e-10, atol=1e-13, err_msg=n)


def test_oracle_rejects_full_vb():
    rng = np.random.RandomState(1)
    params = [rng.normal(0, 0.3, s) for s in O.param_shapes(10, 8, 3, False)]
    with pytest.raises(ValueError):
        K.OracleKLVAEB(rng.uniform(size=(6, 10)), False, 8, 3, 6, estimator="FVB", params=params)


@pytest.mark.parametrize("beta,warmup", [(1.0, 0), (0.25, 0), (3.0, 4), (1.0, 7), (0.3, 1000)])
def test_schedule_mirror_equals_the_documented_formula(beta, warmup):
    from vaeb_b200.model import kl_weight_at
    for n in list(range(1, 12)) + [warmup - 1, warmup, warmup + 1, 5 * warmup + 3]:
        if n < 1:
            continue
        got = kl_weight_at(beta, warmup, n)
        assert got.dtype == np.float32
        ref = np.float32(float(np.float32(beta)) * (1.0 if warmup == 0 else min(1.0, n / warmup)))
        assert got == ref, (beta, warmup, n, got, ref)
        assert float(got) == pytest.approx(K.kl_weight_at(beta, warmup, n), rel=1e-7)
    if warmup:
        assert kl_weight_at(beta, warmup, warmup + 5) == np.float32(beta)   # constant after the ramp


def test_cli_parses_the_kl_options_and_counts_warmup_in_updates():
    from vaeb_b200 import cli
    a = cli.parse_args(["--kl_weight", "0.5", "--kl_warmup", "3", "--batch_size", "100"])
    assert a["kl_weight"] == 0.5 and a["kl_warmup"] == 3
    d = cli.parse_args([])
    assert d["kl_weight"] == 1.0 and d["kl_warmup"] == 0          # the reference's bound
    # an epoch is N // batch_size updates (VAEB.py:571): the remainder rows are never visited
    assert cli.kl_warmup_updates(3, 1965, 100) == 3 * 19
    assert cli.kl_warmup_updates(0, 50000, 100) == 0
    assert cli.kl_warmup_updates(2, 50000, 100) == 1000


def test_data_parallel_refuses_ranks_with_different_kl_weights():
    from vaeb_b200 import distributed as vd
    vd.check_same_kl_weight([(0.5, 10, 3), (0.5, 10, 3)])
    for other in [(0.5, 10, 4), (1.0, 10, 3), (0.5, 0, 3)]:
        with pytest.raises(ValueError):
            vd.check_same_kl_weight([(0.5, 10, 3), other])
