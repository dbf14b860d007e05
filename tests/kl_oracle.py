"""CPU restatement of the KL weight of vaeb_set_kl_weight (test infrastructure, beside oracle/vaeb_oracle.py, whose
gradients and model object it builds on).  The n-th weighted update ascends loglik + beta_n * aux; its gradient is the
oracle's gradient of loglik + aux plus (beta_n - 1) times the gradient of the latent term aux alone."""
import numpy as np

from oracle import vaeb_oracle as O


def latent_term_grads(params, x, eps, continuous, estimator="LB", row_weight=None, act="tanh"):
    """Gradient of w * aux (summed over the rows, mean over the L samples) in reference order, no weight prior: the three
    latent-term lines of elbo_and_grads (-mu and 0.5 (1 - exp(ls)) for L^B; d prior / dz and the 0.5 of -log q for L^A)
    carried back through the encoder."""
    p = O.as_dict(params, continuous)
    dt = x.dtype
    L = eps.shape[0]
    w = dt.type(1.0 if row_weight is None else row_weight)
    hs = O.encoder_hiddens(p, x, act)
    h_e = hs[-1]
    mu, ls = h_e @ p["W4"] + p["b4"], h_e @ p["W5"] + p["b5"]
    sd = np.exp(0.5 * ls)
    if estimator == "LA":
        d_mu, d_ls = np.zeros_like(mu), np.zeros_like(ls)
        s = w * dt.type(1.0 / L)
        for l in range(L):
            z = mu + sd * eps[l]
            d_z = -s * z
            d_ls += s * 0.5
            d_mu += d_z
            d_ls += d_z * (0.5 * sd * eps[l])
    else:
        d_mu = w * (-mu)
        d_ls = w * 0.5 * (1.0 - np.exp(ls))
    g = {n: np.zeros_like(q) for n, q in p.items()}
    g["W4"], g["b4"] = h_e.T @ d_mu, d_mu.sum(axis=0)
    g["W5"], g["b5"] = h_e.T @ d_ls, d_ls.sum(axis=0)
    d_a3 = (d_mu @ p["W4"].T + d_ls @ p["W5"].T) * O.hidden_act_grad(h_e, act)
    for k in range(len(hs), 1, -1):
        g["W3_%d" % k] = hs[k - 2].T @ d_a3
        g["b3_%d" % k] = d_a3.sum(axis=0)
        d_a3 = (d_a3 @ p["W3_%d" % k].T) * O.hidden_act_grad(hs[k - 2], act)
    g["W3"], g["b3"] = x.T @ d_a3, d_a3.sum(axis=0)
    return [g[n] for n in O.param_names(continuous, len(hs))]


def elbo_and_grads(params, x, eps, continuous, estimator="LB", want_grads=True, prior_scale=1.0, row_weight=None,
                   act="tanh", kl_weight=1.0):
    """O.elbo_and_grads with the latent term weighted by kl_weight in the gradient; the bound stays unweighted.
    kl_weight = 1 returns the oracle's result itself."""
    out = O.elbo_and_grads(params, x, eps, continuous, estimator, want_grads, prior_scale, row_weight, act)
    if kl_weight == 1.0 or not want_grads:
        return out
    k = x.dtype.type(kl_weight - 1.0)
    ga = latent_term_grads(params, x, eps, continuous, estimator, row_weight, act)
    return O.StepOut(out.sgvb, out.per_row, [g + k * a for g, a in zip(out.grads, ga)])


def kl_weight_at(beta, warmup, n):
    """beta_n of the documented schedule, beta * min(1, n / warmup) (warmup = 0: beta), in float64."""
    return beta if warmup == 0 else beta * min(1.0, n / warmup)


class OracleKLVAEB(O.OracleVAEB):
    """OracleVAEB whose gradient weights the latent term by self.kl_weight (L^A / L^B, both variants)."""

    def __init__(self, *args, kl_weight=1.0, **kw):
        super().__init__(*args, **kw)
        if self.fvp is not None:
            raise ValueError("the KL weight is not wired to the full-VB estimators")
        self.kl_weight = kl_weight

    def _objective(self, x, eps, want_grads, zeta=None):
        sgvb, per_row, grads = super()._objective(x, eps, want_grads, zeta)
        if not want_grads or self.kl_weight == 1.0:
            return sgvb, per_row, grads
        fb = self.variant == "fullbayes"
        ga = latent_term_grads(self.params, x, eps, self.continuous, "LB" if fb else self.estimator,
                               1.0 / x.shape[0] if fb else None, "tanh" if fb else self.activation)
        k = x.dtype.type(self.kl_weight - 1.0)
        return sgvb, per_row, [g + k * a for g, a in zip(grads, ga)]
