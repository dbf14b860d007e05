"""CPU restatement of the Adam rule of vaeb_set_adam (test infrastructure, beside oracle/vaeb_oracle.py, whose
gradients and model object it builds on): the update itself and an OracleVAEB that applies it."""
import numpy as np

from oracle.vaeb_oracle import OracleVAEB, _zeros_like_list


def adam_coefficients(t, lr, b1, b2):
    """(alpha_t, s2_t) of Adam step t: lr / (1 - b1^t) and sqrt(1 - b2^t), in double as the library computes them."""
    return lr / (1.0 - b1 ** t), np.sqrt(1.0 - b2 ** t)


def adam_update(params, m, v, grads, t, lr, b1=0.9, b2=0.999, eps=1e-8, prior=0.0):
    """Adam step t (t = 1 for the first) in the ascent convention, in place:
    g = grad - prior*p; m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p += alpha_t m / (sqrt(v) / s2_t + eps).
    `grads` that already carry the weight prior (elbo_and_grads's) take prior = 0."""
    alpha, s2 = adam_coefficients(t, lr, b1, b2)
    for q, mm, vv, g in zip(params, m, v, grads):
        dt = q.dtype.type
        g = g - dt(prior) * q
        mm *= dt(b1)
        mm += dt(1.0 - b1) * g
        vv *= dt(b2)
        vv += dt(1.0 - b2) * g * g
        q += dt(alpha) * mm / (np.sqrt(vv) / dt(s2) + dt(eps))


class OracleAdamVAEB(OracleVAEB):
    """OracleVAEB whose update applies Adam: m in self.ada, v in self.adam_v, the step counter in self.adam_t.
    The gradients of the objective carry the weight prior (none for the VAEBfullbayes variant), as the library's do."""

    def __init__(self, *args, adam_betas=(0.9, 0.999), adam_eps=1e-8, **kw):
        kw.setdefault("optimizer", "adam")
        super().__init__(*args, **kw)
        if self.fvp is not None:
            raise ValueError("Adam is not wired to the full-VB estimators")
        self.b1, self.b2 = adam_betas
        self.adam_eps = adam_eps
        self.adam_v = _zeros_like_list(self.params)
        self.adam_t = 0

    def update(self, index, eps, zeta=None):
        xb = self.x[index * self.M:(index + 1) * self.M]
        sgvb, _, grads = self._objective(xb, np.asarray(eps, self.dtype), True, zeta)
        self.adam_t += 1
        adam_update(self.params, self.ada, self.adam_v, grads, self.adam_t, self.lr, self.b1, self.b2, self.adam_eps)
        return sgvb if self.variant == "fullbayes" else sgvb / self.M
