"""CPU checks of the Adam rule (tests/adam_oracle.py) that the GPU tests compare the library with: the update against
torch.optim.Adam(maximize=True), and a whole training step of the oracle against torch autograd."""
import numpy as np
import pytest

from oracle import vaeb_oracle as O
from tests import adam_oracle as A

torch = pytest.importorskip("torch")


def _shapes():
    return [(7, 5), (5,), (3, 4)]


def test_adam_update_matches_torch_maximize():
    """Five steps in fp64, weight prior included: torch's weight_decay with maximize=True is g - prior * p."""
    rng = np.random.RandomState(1)
    lr, b1, b2, eps, prior = 0.003, 0.8, 0.99, 1e-8, 0.7
    p0 = [rng.normal(size=s) for s in _shapes()]
    params = [q.copy() for q in p0]
    m = [np.zeros_like(q) for q in p0]
    v = [np.zeros_like(q) for q in p0]
    tp = [torch.tensor(q, dtype=torch.float64, requires_grad=True) for q in p0]
    opt = torch.optim.Adam(tp, lr=lr, betas=(b1, b2), eps=eps, weight_decay=prior, maximize=True)
    for t in range(1, 6):
        grads = [rng.normal(size=s) * 10.0 ** rng.randint(-6, 2) for s in _shapes()]
        A.adam_update(params, m, v, grads, t, lr, b1, b2, eps, prior=prior)
        for q, g in zip(tp, grads):
            q.grad = torch.tensor(g, dtype=torch.float64)
        opt.step()
        for q, r in zip(params, tp):
            np.testing.assert_allclose(q, r.detach().numpy(), rtol=0, atol=1e-12)
    for q, mm, vv, r in zip(params, m, v, tp):
        st = opt.state[r]
        np.testing.assert_allclose(mm, st["exp_avg"].numpy() * -1.0, rtol=0, atol=1e-12)   # maximize: torch keeps -m
        np.testing.assert_allclose(vv, st["exp_avg_sq"].numpy(), rtol=0, atol=1e-12)


def _torch_sgvb(tp, names, x, eps, continuous):
    """The LB bound of VAEB.py:332-346 summed over the rows (oracle/vaeb_oracle.py's elbo_and_grads), in torch."""
    p = dict(zip(names, tp))
    h_e = torch.tanh(x @ p["W3"] + p["b3"])
    mu, ls = h_e @ p["W4"] + p["b4"], h_e @ p["W5"] + p["b5"]
    kl = 0.5 * (1.0 + ls - mu ** 2 - torch.exp(ls)).sum(1)
    ll = 0.0
    for l in range(eps.shape[0]):
        z = mu + torch.exp(0.5 * ls) * eps[l]
        h_d = torch.tanh(z @ p["W1"] + p["b1"])
        a = h_d @ p["W2"] + p["b2"]
        if continuous:
            lv = h_d @ p["W6"] + p["b6"]
            ll = ll + (-0.5 * np.log(2 * np.pi) - 0.5 * lv - 0.5 * (x - torch.sigmoid(a)) ** 2 / torch.exp(lv)).sum(1)
        else:
            ll = ll + (x * a - torch.nn.functional.softplus(a)).sum(1)
    return (ll / eps.shape[0] + kl).sum()


@pytest.mark.parametrize("continuous", [False, True])
def test_oracle_adam_training_step_matches_torch_autograd(continuous):
    """Three updates of OracleAdamVAEB against torch autograd of the same bound with torch.optim.Adam(maximize=True,
    weight_decay=prior_scale): the returned bounds, the parameters and the moments."""
    D, H, Z, M, L = 12, 9, 3, 6, 2
    rng = np.random.RandomState(3)
    x = rng.uniform(size=(3 * M, D))
    if not continuous:
        x = (x > 0.5).astype(np.float64)
    params = [rng.normal(0, 0.3, s) for s in O.param_shapes(D, H, Z, continuous)]
    lr, betas, eps_a = 0.01, (0.9, 0.999), 1e-8
    o = A.OracleAdamVAEB(x, continuous, H, Z, M, L=L, lr=lr, params=params, adam_betas=betas, adam_eps=eps_a)
    names = O.param_names(continuous)
    tp = [torch.tensor(q, dtype=torch.float64, requires_grad=True) for q in params]
    opt = torch.optim.Adam(tp, lr=lr, betas=betas, eps=eps_a, weight_decay=1.0, maximize=True)
    for step in range(3):
        e = rng.normal(size=(L, M, Z))
        got = o.update(step, e)
        xb = torch.tensor(x[step * M:(step + 1) * M])
        opt.zero_grad()
        sgvb = _torch_sgvb(tp, names, xb, torch.tensor(e), continuous)
        sgvb.backward()
        opt.step()
        assert abs(got - sgvb.item() / M) <= 1e-12 * max(1.0, abs(got))
        assert o.adam_t == step + 1
    for q, mm, vv, r in zip(o.params, o.ada, o.adam_v, tp):
        np.testing.assert_allclose(q, r.detach().numpy(), rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(mm, -opt.state[r]["exp_avg"].numpy(), rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(vv, opt.state[r]["exp_avg_sq"].numpy(), rtol=1e-9, atol=1e-14)


def test_oracle_adam_rejects_full_vb():
    D, H, Z = 6, 4, 2
    params = O.init_params(D, H, Z, False)
    with pytest.raises(ValueError):
        A.OracleAdamVAEB(np.zeros((4, D)), False, H, Z, 2, params=params, estimator="FVB")


def test_cli_optimizer_option():
    from vaeb_b200 import cli
    assert cli.parse_args([])["optimizer"] == "adagrad"
    assert cli.parse_args(["--optimizer", "adam"])["optimizer"] == "adam"


def test_peer_memory_needs_one_optimizer_on_every_rank():
    from vaeb_b200 import distributed as vd
    vd.check_same_optimizer(["adam", "adam"])
    with pytest.raises(ValueError):
        vd.check_same_optimizer(["adam", "adagrad"])
