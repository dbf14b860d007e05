"""Host-side mirror of the reference's model class (VAEB.py:49-469) over the C-ABI.

`VAEB(x_train, continuous, hidden_units, latent_size, batch_size, L, learning_rate,
genericEstimator, fullVariational, params=None, prng=None, sigmaInit=None)` keeps the
reference's constructor signature, attribute names and the two callables the training loop
uses -- `model.update(index)` (VAEB.py:408-415) and `model.validate(x)` (VAEB.py:418-422) --
but every number is produced by the sm_100a kernels behind include/vaeb_b200.h.  There is
no CPU path in this module."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib, checkpoint, io
from .rng import RandomStreams

_NAMES_D = ["W3", "W4", "W5", "W1", "W2", "b3", "b4", "b5", "b1", "b2"]
_NAMES_C = ["W3", "W4", "W5", "W1", "W2", "W6", "b3", "b4", "b5", "b1", "b2", "b6"]


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class SharedParam(object):
    """Stands in for the Theano shared variables held in `self.params` (VAEB.py:60-115): a
    named view of one tensor of a device-resident flat buffer."""

    def __init__(self, model, which, index, name, shape):
        self._model, self._which, self._index = model, which, index
        self.name = name
        self.shape = shape

    def get_value(self, borrow=False):
        return self._model._get_buffer(self._which)[self._index]

    def eval(self):
        return self.get_value()

    def set_value(self, value, borrow=False):
        vals = self._model._get_buffer(self._which)
        vals[self._index] = _f32(value).reshape(self.shape)
        self._model._set_buffer(self._which, vals)

    def __array__(self, dtype=None, copy=None):
        v = self.get_value()
        return v.astype(dtype) if dtype is not None else v

    def __repr__(self):
        return "SharedParam(%s, shape=%s)" % (self.name, (self.shape,))


def _as_array(p):
    """ndarray from an ndarray, a SharedParam or anything with get_value()."""
    if hasattr(p, "get_value"):
        return _f32(p.get_value())
    return _f32(p)


class VAEB(object):
    # extension keywords (all keyword-only, defaults keep the reference behaviour):
    #   device         CUDA ordinal
    #   precision      'fp32' (FFMA tiles, 1e-4 tier) | 'bf16' (tcgen05, 1e-2 tier) |
    #                  'bf16x3' (tcgen05 with hi/lo operand split, 1e-4 tier)
    #   eps_mode       'philox' on-device noise | 'theano' host RandomStreams emulation
    #   sample_weights full-VB with sample_variational_params live (VAEB.py:127-129)
    #   variant        'vaeb' | 'fullbayes' (VAEBfullbayes.py objective/update scalars)
    #   optimizer      'adagrad' (getUpdates, VAEB.py:426-444) | 'adadelta' (getAdaDeltaUpdates, VAEB.py:449-469,
    #                  the alternative the reference keeps commented out at VAEB.py:404; rho = self.rho = 0.95) |
    #                  'adam' (Kingma & Ba 2015 with the weight prior, ascent; adam_betas, adam_eps; moments in
    #                  self.ADA (m) and self.ADAM_V (v), step counter in self.adam_step; L^A / L^B estimators)
    #   encoder_layers 1 (VAEB.py:245-251) | 2..4: the deeper encoders of Report/replication/replic.tex:46-57 -- extra H x H
    #                  hidden layers between the first one and the heads; their parameters W3_k, b3_k (k = 2..) follow the
    #                  reference's list, weights first; fp32 per-layer kernels, L^A / L^B estimators
    #   activation     'tanh' (the reference's hidden layers, VAEB.py:246,254) | 'sigmoid' | 'relu' (the alternatives of
    #                  Report/replication/replic.tex:73-82; fp32 per-layer kernels, L^A / L^B estimators)
    #   kl_weight      beta: weight of the latent term (-KL for L^B, log p(z) - log q(z|x) for L^A) in the gradient
    #   kl_warmup      updates over which that weight ramps linearly from beta/kl_warmup to beta (0: constant beta);
    #                  see set_kl_weight.  The defaults (1.0, 0) train on the reference's bound
    def __init__(self, x_train, continuous, hidden_units, latent_size, batch_size,
                 L, learning_rate, genericEstimator, fullVariational, params=None, prng=None, sigmaInit=None,
                 *, device=0, precision="fp32", eps_mode="philox", sample_weights=False, variant="vaeb", seed=10,
                 optimizer="adagrad", activation="tanh", encoder_layers=1, adam_betas=(0.9, 0.999), adam_eps=1e-8,
                 kl_weight=1.0, kl_warmup=0):
        x_train = np.asarray(x_train)
        [self.N, self.input_size] = x_train.shape       # VAEB.py:135
        self.n_hidden_units = hidden_units
        self.n_latent = latent_size
        self.continuous = bool(continuous)
        self.learning_rate = learning_rate
        self.batch_size = batch_size
        self.L = L
        self.eps = 1e-6                                 # VAEB.py:144
        self.rho = 0.95
        self.fullVBSigmaInit = 1e-3                     # VAEB.py:146
        self.prng = np.random.RandomState(10)           # forced, VAEB.py:148
        self.sigmaInit = 0.01                           # forced, VAEB.py:149
        self.genericEstimator = bool(genericEstimator)
        self.fullVariational = bool(fullVariational)
        self.variant = variant
        self.eps_mode = eps_mode
        self.seed = int(seed)
        self.sample_weights = bool(sample_weights)
        self.adam_betas = (float(adam_betas[0]), float(adam_betas[1]))
        self.adam_eps = float(adam_eps)
        self._rank, self._world = 0, 1
        if eps_mode not in ("philox", "theano"):
            raise ValueError("eps_mode must be 'philox' or 'theano'")
        if self.fullVariational:
            assert params is not None                   # VAEB.py:155

        # which bound getGradient builds (VAEB.py:378-383: LA wins over full-VB)
        if self.genericEstimator:
            est = _lib.EST_LA
        elif self.fullVariational:
            est = _lib.EST_FVB_SAMPLED if sample_weights else _lib.EST_FVB
        else:
            est = _lib.EST_LB
        self._estimator = est
        self._fvb = est in (_lib.EST_FVB, _lib.EST_FVB_SAMPLED)

        self._async_keep = []
        self.srng = RandomStreams(seed=10)              # VAEB.py:158
        self._eps_nodes = [self.srng.new_node() for _ in range(L)]

        self.precision = precision
        self._lib = _lib.load()
        cfg = _lib.Config(
            input_dim=self.input_size, hidden_units=hidden_units, latent_size=latent_size, batch_size=batch_size,
            L=L, continuous=int(self.continuous), estimator=est,
            variant=_lib.VARIANT_FULLBAYES if variant == "fullbayes" else _lib.VARIANT_VAEB,
            precision={"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16, "bf16x3": _lib.PREC_BF16X3}[precision], device=device,
            learning_rate=learning_rate, adagrad_eps=self.eps, prior_scale=1.0,
            sigma_vb_init=self.fullVBSigmaInit, seed=seed, encoder_hidden_layers=int(encoder_layers), reserved0=0)
        self.encoder_layers = int(encoder_layers)
        self._h = C.c_void_p()
        _lib.check(self._lib.vaeb_create(C.byref(cfg), C.byref(self._h)))
        self._names = list(_NAMES_C if self.continuous else _NAMES_D)
        self._names += ["W3_%d" % k for k in range(2, self.encoder_layers + 1)]
        self._names += ["b3_%d" % k for k in range(2, self.encoder_layers + 1)]
        n = C.c_int32()
        _lib.check(self._lib.vaeb_num_tensors(self._h, C.byref(n), None))
        self._shapes = []
        for i in range(n.value):
            r, c = C.c_int32(), C.c_int32()
            _lib.check(self._lib.vaeb_tensor_shape(self._h, i, C.byref(r), C.byref(c)))
            self._shapes.append((r.value, c.value) if self._names[i].startswith("W") else (c.value,))

        if params is None:
            values = self.initialize_params(None)
        else:
            params = list(params)
            if len(params) != len(self._shapes):      # VAEB.py:165-167 unpacks into a fixed-length list and fails loudly
                raise ValueError("expected %d parameter tensors, got %d" % (len(self._shapes), len(params)))
            values = [_as_array(p).reshape(s) for p, s in zip(params, self._shapes)]
        self._set_buffer(_lib.BUF_PARAMS, values)
        self.params = [SharedParam(self, _lib.BUF_PARAMS, i, nm, s)
                       for i, (nm, s) in enumerate(zip(self._names, self._shapes))]
        for p in self.params:
            setattr(self, p.name, p)                    # self.W3 ... self.b6 (VAEB.py:60-109)
        self.ADA = [SharedParam(self, _lib.BUF_ADA, i, "ada_" + nm, s)
                    for i, (nm, s) in enumerate(zip(self._names, self._shapes))]
        if self._fvb:
            # VAEB.py:117-125: interleaved [mu0, sigma0, mu1, sigma1, ...]
            self._set_buffer(_lib.BUF_VMU, values)
            self.full_variational_params = []
            for i, (nm, s) in enumerate(zip(self._names, self._shapes)):
                self.full_variational_params += [SharedParam(self, _lib.BUF_VMU, i, nm + "_mu_vb", s),
                                                 SharedParam(self, _lib.BUF_VSIG, i, nm + "_sigma_vb", s)]

        if optimizer not in ("adagrad", "adadelta", "adam"):
            raise ValueError("optimizer must be 'adagrad', 'adadelta' or 'adam'")
        self.optimizer = optimizer
        if optimizer == "adadelta":
            _lib.check(self._lib.vaeb_set_optimizer(self._h, _lib.OPT_ADADELTA, self.rho))
        if optimizer == "adam":
            b1, b2 = adam_betas
            _lib.check(self._lib.vaeb_set_adam(self._h, float(b1), float(b2), float(adam_eps)))
            self.ADAM_V = [SharedParam(self, _lib.BUF_ADAM_V, i, "adam_v_" + nm, s)
                           for i, (nm, s) in enumerate(zip(self._names, self._shapes))]
        if activation not in ("tanh", "sigmoid", "relu"):
            raise ValueError("activation must be 'tanh', 'sigmoid' or 'relu'")
        self.activation = activation
        if activation != "tanh":
            _lib.check(self._lib.vaeb_set_hidden_activation(self._h, {"sigmoid": 2, "relu": 3}[activation]))
        self.kl_weight, self.kl_warmup = 1.0, 0
        if kl_weight != 1.0 or kl_warmup != 0:
            self.set_kl_weight(kl_weight, kl_warmup)
        xf = _f32(x_train)
        _lib.check(self._lib.vaeb_upload_data(self._h, _ptr(xf), self.N))   # VAEB.py:184
        self._data_fp = checkpoint.data_fingerprint(xf)          # what a checkpoint of this model was trained on

    # ---- parameters -------------------------------------------------------------------
    def initialize_params(self, params):
        """VAEB.py:50-115: N(0, 0.01^2) weights from RandomState(10) in the reference's draw
        order (W3 and W4 are drawn twice: the first block, VAEB.py:58-67, is overwritten);
        zero biases."""
        D, H, Z = self.input_size, self.n_hidden_units, self.n_latent
        initW = lambda dimIn, dimOut: self.prng.normal(0, self.sigmaInit, (dimIn, dimOut)).astype(np.float32)
        initW(D, H)
        initW(H, Z)
        vals = {"W3": initW(D, H), "W4": initW(H, Z), "W5": initW(H, Z), "W1": initW(Z, H), "W2": initW(H, D)}
        if self.continuous:
            vals["W6"] = initW(H, D)
        for k in range(2, getattr(self, "encoder_layers", 1) + 1):      # deeper encoders: drawn after the reference's list
            vals["W3_%d" % k] = initW(H, H)
        return [vals[nm] if nm in vals else np.zeros(s, np.float32) for nm, s in zip(self._names, self._shapes)]

    def _get_buffer(self, which):
        out = [np.empty(s, np.float32) for s in self._shapes]
        ptrs = (C.c_void_p * len(out))(*[a.ctypes.data for a in out])
        _lib.check(self._lib.vaeb_get_tensors(self._h, which, ptrs))
        return out

    def _set_buffer(self, which, values):
        vals = [_f32(v).reshape(s) for v, s in zip(values, self._shapes)]
        ptrs = (C.c_void_p * len(vals))(*[a.ctypes.data for a in vals])
        _lib.check(self._lib.vaeb_set_tensors(self._h, which, ptrs))

    def get_params(self):
        return self._get_buffer(_lib.BUF_PARAMS)

    def set_params(self, values):
        self._set_buffer(_lib.BUF_PARAMS, values)

    def gradients(self, x=None, index=0, eps=None, zeta=None):
        """(SGVB, per-row bound, gradient list) of the training criterion (VAEB.py:386-399)
        without applying the update.  Full-VB: the list is interleaved [dmu0, dsigma0, ...]."""
        rows = self.batch_size if x is None else np.asarray(x).shape[0]
        xa = None if x is None else _f32(x)
        ea = None if eps is None else _f32(eps)
        za = None if zeta is None else np.concatenate([_f32(t).ravel() for t in zeta])
        sg = C.c_float()
        per_row = np.empty(rows, np.float32)
        _lib.check(self._lib.vaeb_gradients(self._h, _ptr(xa), rows, index, _ptr(ea), _ptr(za), C.byref(sg),
                                            _ptr(per_row)))
        if self._fvb:
            gm, gs = self._get_buffer(_lib.BUF_GMU), self._get_buffer(_lib.BUF_GSIG)
            grads = [t for pair in zip(gm, gs) for t in pair]
        else:
            grads = self._get_buffer(_lib.BUF_GRADS)
        return sg.value, per_row, grads

    # ---- noise ------------------------------------------------------------------------
    def _draw_eps(self, rows):
        if self.eps_mode != "theano":
            return None
        return np.stack([self.srng.normal(nd, (rows, self.n_latent)) for nd in self._eps_nodes])

    # ---- the two compiled functions ------------------------------------------------------
    def update(self, index, eps=None):
        """VAEB.py:408-415.  Returns SGVB / batch_size evaluated with the pre-update
        parameters (0-d float32 array, as Theano returns)."""
        ea = _f32(eps) if eps is not None else self._draw_eps(self.batch_size)
        out = C.c_float()
        _lib.check(self._lib.vaeb_update(self._h, int(index), _ptr(ea), C.byref(out)))
        return np.asarray(out.value, dtype=np.float32)

    def update_host(self, x_batch, eps=None):
        """One update on a minibatch that lives in HOST memory (end-to-end path)."""
        xa = _f32(x_batch)
        ea = _f32(eps) if eps is not None else self._draw_eps(xa.shape[0])
        out = C.c_float()
        _lib.check(self._lib.vaeb_update_host(self._h, _ptr(xa), xa.shape[0], _ptr(ea), C.byref(out)))
        return np.asarray(out.value, dtype=np.float32)

    def update_host_async(self, x_batch, scale=1.0 / 256.0):
        """Streaming form of update_host: enqueue one update on a minibatch in PINNED host memory and
        return at once (its H2D copy overlaps the previous update's kernel).  Collect the bounds with
        `collect()`; do not modify x_batch before that.  Philox noise only.

        A uint8 minibatch is sent as bytes (a quarter of the PCIe traffic) and expanded on the device to
        float32(x) * float32(scale) -- the form mnist.pkl.gz / freyfaces.pkl store their 8-bit pixels in."""
        if self.eps_mode == "theano":
            raise ValueError("update_host_async draws its noise on the device (eps_mode='philox')")
        if isinstance(x_batch, np.ndarray) and x_batch.dtype == np.uint8:
            if not x_batch.flags["C_CONTIGUOUS"] or x_batch.ndim != 2 or x_batch.shape[1] != self.input_size:
                raise ValueError("uint8 minibatch must be C-contiguous [rows, %d]" % self.input_size)
            self._async_keep.append(x_batch)
            _lib.check(self._lib.vaeb_update_host_async_u8(self._h, x_batch.ctypes.data, x_batch.shape[0], float(scale)))
            return
        xa = x_batch if (isinstance(x_batch, np.ndarray) and x_batch.dtype == np.float32 and
                         x_batch.flags["C_CONTIGUOUS"]) else _f32(x_batch)
        self._async_keep.append(xa)
        _lib.check(self._lib.vaeb_update_host_async(self._h, xa.ctypes.data, xa.shape[0]))

    def collect(self):
        """Bounds (SGVB / batch_size, pre-update parameters) of every update enqueued by
        update_host_async since the last collect, in submission order."""
        n = C.c_int32(8192)
        out = np.empty(8192, np.float32)
        _lib.check(self._lib.vaeb_collect(self._h, C.byref(n), _ptr(out)))
        self._async_keep = []
        return out[:n.value].copy()

    def update_many(self, batch_order):
        """The inner loop of train_model (VAEB.py:577-579) in one call; Philox noise only."""
        if self.eps_mode == "theano":
            return np.array([self.update(b) for b in batch_order], dtype=np.float32)
        order = np.ascontiguousarray(batch_order, dtype=np.int32)
        out = np.empty(len(order), np.float32)
        _lib.check(self._lib.vaeb_update_many(self._h, _ptr(order), len(order), _ptr(out)))
        return out

    def validate(self, x, eps=None, per_row=False):
        """VAEB.py:418-422: SGVB of x (a sum over rows; the caller divides)."""
        xa = _f32(x)                                    # allow_input_downcast=True
        ea = _f32(eps) if eps is not None else self._draw_eps(xa.shape[0])
        out = C.c_float()
        rows = np.empty(xa.shape[0], np.float32) if per_row else None
        _lib.check(self._lib.vaeb_validate(self._h, _ptr(xa), xa.shape[0], _ptr(ea), C.byref(out), _ptr(rows)))
        val = np.asarray(out.value, dtype=np.float32)
        return (val, rows) if per_row else val

    def log_px(self, x, L=5000, eps=None, row_offset=0, return_weights=False):
        """Importance-sampled log p(x_i) for every row of x (new; SURVEY.md 8a row a19)."""
        xa = _f32(x)
        ea = None if eps is None else _f32(eps)
        out = np.empty(xa.shape[0], np.float32)
        lw = np.empty((xa.shape[0], L), np.float32) if return_weights else None
        _lib.check(self._lib.vaeb_is_logpx(self._h, _ptr(xa), xa.shape[0], L, _ptr(ea), row_offset, _ptr(out),
                                           _ptr(lw)))
        return (out, lw) if return_weights else out

    def reconstruct(self, x, n_samples, eps=None, sample_output=True):
        """VAEB.py:267-300.  The decoder means (averaged over n_samples draws of z, or decoded
        from mu when n_samples <= 0) come from the device.  For the Gaussian decoder the
        reference then draws y ~ N(y_mu, diag(exp(y_log_sigma)**2)) through a dense DxD
        covariance on the host (VAEB.py:295-297, one row at a time); the diagonal draw below is
        the same distribution.  sample_output=False returns (y_mu, y_log_sigma) instead."""
        xa = _f32(x)
        single = xa.ndim == 1
        xa = xa.reshape(-1, self.input_size)
        ea = None if eps is None else _f32(eps)
        if ea is None and self.eps_mode == "theano" and n_samples > 0:
            ea = np.stack([self.srng.normal(self.srng.new_node(), (xa.shape[0], self.n_latent))
                           for _ in range(n_samples)])
        y = np.empty_like(xa)
        lv = np.empty_like(xa) if self.continuous else None
        _lib.check(self._lib.vaeb_reconstruct(self._h, _ptr(xa), xa.shape[0], int(n_samples), _ptr(ea), _ptr(y),
                                              _ptr(lv)))
        if self.continuous:
            if not sample_output:
                return (y[0], lv[0]) if single else (y, lv)
            y = y + np.exp(lv) * np.random.standard_normal(y.shape).astype(np.float32)
        return y[0] if single else y

    def decode(self, z):
        """The decoder alone (VAEB.py:253-265) on latent points z[n, Z]: y for the Bernoulli decoder,
        (mu, log_sigma) for the Gaussian one -- what the compiled `freyFace(z)` of freyFace.py:237-244 returns."""
        za = _f32(z).reshape(-1, self.n_latent)
        y = np.empty((za.shape[0], self.input_size), np.float32)
        lv = np.empty_like(y) if self.continuous else None
        _lib.check(self._lib.vaeb_decode(self._h, _ptr(za), za.shape[0], _ptr(y), _ptr(lv)))
        return (y, lv) if self.continuous else y

    freyFace = decode       # freyFace.py:137 names the compiled decoder function after its first use

    def encode(self, x):
        """The encoder alone (VAEB.py:245-251): (mu, log_var) of q(z|x) for every row of x.  The second head is a
        log-variance although the reference calls it log_sigma."""
        xa = _f32(x).reshape(-1, self.input_size)
        mu = np.empty((xa.shape[0], self.n_latent), np.float32)
        lv = np.empty_like(mu)
        _lib.check(self._lib.vaeb_encode(self._h, _ptr(xa), xa.shape[0], _ptr(mu), _ptr(lv)))
        return mu, lv

    def sample(self, n, step=0, row_offset=0, return_all=False):
        """n samples x ~ p(x|z), z ~ N(0, I) from the generative model (AEVB Fig. 5), drawn on the device from the
        Philox stream of (seed, step, row_offset + i).  return_all: (z, mean, lv, x), lv None for Bernoulli."""
        n = int(n)
        x = np.empty((n, self.input_size), np.float32)
        z = np.empty((n, self.n_latent), np.float32) if return_all else None
        mean = np.empty_like(x) if return_all else None
        lv = np.empty_like(x) if return_all and self.continuous else None
        _lib.check(self._lib.vaeb_sample(self._h, n, int(step), int(row_offset), _ptr(z), _ptr(mean), _ptr(lv), _ptr(x)))
        return (z, mean, lv, x) if return_all else x

    def validate_terms(self, x, eps=None):
        """The two terms of validate's per-row bound: (mean over L of log p(x|z), the term the estimator adds --
        -KL for L^B, the MC mean of log p(z) - log q(z|x) for L^A).  Same noise and step counter as validate."""
        xa = _f32(x)
        ea = _f32(eps) if eps is not None else self._draw_eps(xa.shape[0])
        loglik = np.empty(xa.shape[0], np.float32)
        aux = np.empty_like(loglik)
        _lib.check(self._lib.vaeb_validate_terms(self._h, _ptr(xa), xa.shape[0], _ptr(ea), _ptr(loglik), _ptr(aux)))
        return loglik, aux

    # ---- persistence ---------------------------------------------------------------------
    def save(self, file_name):
        """VAEB.py:189-203 (plus the `genericEstimator` entry `load` expects, VAEB.py:218)."""
        print('Saving model to: {0}'.format(file_name))
        header = dict(n_hidden_units=self.n_hidden_units, n_latent=self.n_latent, continuous=self.continuous,
                      learning_rate=self.learning_rate, batch_size=self.batch_size, prng=self.prng,
                      sigmaInit=self.sigmaInit, L=self.L, genericEstimator=self.genericEstimator)
        io.write_mdl(file_name, header, self.get_params())

    @staticmethod
    def load(file_name, data=None, **kwargs):
        """VAEB.py:206-242.  Like the reference it re-reads the dataset from the working
        directory unless `data=(x_train, x_valid)` is passed."""
        print('Loading model form : {0}'.format(file_name))
        header, params = io.read_mdl(file_name)
        if data is None:
            from .data import load_frey, load_mnist
            data = load_frey() if header["continuous"] else load_mnist()
        x_train = data[0]
        model = VAEB(x_train, header["continuous"], header["n_hidden_units"], header["n_latent"],
                     header["batch_size"], header["L"], header["learning_rate"], header["genericEstimator"], False,
                     params, header["prng"], header["sigmaInit"],
                     **dict({"encoder_layers": header.get("encoder_layers", 1)}, **kwargs))
        return model, data

    # ---- training state ------------------------------------------------------------------
    def _ctor_args(self):
        """The constructor arguments that shape the computation (everything but the data and the device)."""
        return dict(continuous=self.continuous, hidden_units=self.n_hidden_units, latent_size=self.n_latent,
                    batch_size=self.batch_size, L=self.L, learning_rate=self.learning_rate,
                    genericEstimator=self.genericEstimator, fullVariational=self.fullVariational,
                    precision=self.precision, eps_mode=self.eps_mode, sample_weights=self.sample_weights,
                    variant=self.variant, seed=self.seed, optimizer=self.optimizer, activation=self.activation,
                    encoder_layers=self.encoder_layers, adam_betas=list(self.adam_betas), adam_eps=self.adam_eps,
                    kl_weight=self.kl_weight, kl_warmup=self.kl_warmup)

    def _state_buffers(self):
        """(file name, which) of the buffers of the training state (include/vaeb_b200.h), in restore order: theta and
        zeta of sampled full VB (the draw of the current step) are restored after the counters."""
        bufs = [("params", _lib.BUF_PARAMS), ("ada", _lib.BUF_ADA)]
        if self.optimizer in ("adadelta", "adam"):
            bufs.append(("ada2", _lib.BUF_ADA2))
        if self._fvb:
            bufs += [("vmu", _lib.BUF_VMU), ("vsig", _lib.BUF_VSIG), ("ada_mu", _lib.BUF_ADA_MU),
                     ("ada_sig", _lib.BUF_ADA_SIG)]
        if self._estimator == _lib.EST_FVB_SAMPLED:
            bufs += [("theta", _lib.BUF_THETA), ("zeta", _lib.BUF_ZETA)]
        return bufs

    @property
    def step_counter(self):
        """The Philox step counter: every update, validate and reconstruct draws its noise from (seed, step)."""
        t = C.c_uint32()
        _lib.check(self._lib.vaeb_step_counter(self._h, C.byref(t)))
        return t.value

    @step_counter.setter
    def step_counter(self, t):
        _lib.check(self._lib.vaeb_set_step_counter(self._h, int(t)))

    def training_state(self):
        """(header, arrays) of a checkpoint: what `resume` needs to continue bit for bit."""
        if self._async_keep:
            raise ValueError("collect() the streaming updates before saving the training state")
        arrays = {}
        for name, which in self._state_buffers():
            for nm, a in zip(self._names, self._get_buffer(which)):
                arrays["%s.%s" % (name, nm)] = a
        arrays["counter.step"] = np.array(self.step_counter, dtype=np.uint32)
        arrays["counter.adam_step"] = np.array(self.adam_step, dtype=np.int64)
        arrays["counter.kl_step"] = np.array(self.kl_step, dtype=np.int64)
        if self.eps_mode == "theano":
            checkpoint.pack_random_state(arrays, "seedgen", self.srng.gen_seedgen.get_state())
            for k, node in enumerate(self.srng.nodes):
                checkpoint.pack_random_state(arrays, "node%d" % k, node.get_state())
        header = dict(vaeb_version=int(self._lib.vaeb_version()), args=self._ctor_args(),
                      tensors=[[n, list(s)] for n, s in zip(self._names, self._shapes)],
                      buffers=[name for name, _ in self._state_buffers()], world_size=self._world,
                      data=[self._data_fp], theano_nodes=len(self.srng.nodes) if self.eps_mode == "theano" else 0)
        return header, arrays

    def save_checkpoint(self, path, driver_state=None):
        """Write the complete training state to one .npz (vaeb_b200/checkpoint.py), atomically: parameters, optimizer
        state, full-VB state, the step, Adam and KL counters, the host noise streams and `driver_state` (a dict of
        arrays and scalars for the training loop).  `VAEB.resume` continues from it with the same bits as an
        uninterrupted run.  Data parallel: vaeb_b200.distributed.save_checkpoint."""
        if self._world > 1:
            raise ValueError("a data-parallel model saves with vaeb_b200.distributed.save_checkpoint")
        header, arrays = self.training_state()
        checkpoint.write(path, header, arrays, driver_state)

    @staticmethod
    def resume(path, x_train, device=0, rank=0, world_size=1, return_driver_state=False):
        """The model of a checkpoint, in exactly its saved state, on `device` with the rows `x_train` (this rank's
        shard in data-parallel runs; attach_data_parallel afterwards).  Built with the constructor (which selects the
        optimizer, the activation and the KL weight), then the buffers, then the counters.  ValueError naming the
        field on an unknown format version, another data set, world size or tensor shape, or a missing array."""
        header, arrays, driver = checkpoint.read(path)
        a = dict(header["args"])
        checkpoint.check_compatible(header, data=checkpoint.data_fingerprint(x_train), rank=rank, world_size=world_size)
        need = lambda name: checkpoint.require(arrays, name)
        params = [need("params.%s" % n) for n, _ in header["tensors"]]
        model = VAEB(x_train, a["continuous"], a["hidden_units"], a["latent_size"], a["batch_size"], a["L"],
                     a["learning_rate"], a["genericEstimator"], a["fullVariational"], params, device=device,
                     precision=a["precision"], eps_mode=a["eps_mode"], sample_weights=a["sample_weights"],
                     variant=a["variant"], seed=a["seed"], optimizer=a["optimizer"], activation=a["activation"],
                     encoder_layers=a["encoder_layers"], adam_betas=tuple(a["adam_betas"]), adam_eps=a["adam_eps"],
                     kl_weight=a["kl_weight"], kl_warmup=a["kl_warmup"])
        try:
            checkpoint.check_tensors(header, list(zip(model._names, model._shapes)))

            def restore(buffers):
                for name, which in buffers:
                    model._set_buffer(which, [checkpoint.require(arrays, "%s.%s" % (name, n), shape)
                                              for n, shape in zip(model._names, model._shapes)])

            draws = (_lib.BUF_THETA, _lib.BUF_ZETA)
            restore([b for b in model._state_buffers() if b[1] not in draws])
            if model.optimizer == "adam":
                model.adam_step = int(need("counter.adam_step"))
            model.kl_step = int(need("counter.kl_step"))
            model.step_counter = int(need("counter.step"))
            restore([b for b in model._state_buffers() if b[1] in draws])     # the draw of the restored step
            if model.eps_mode == "theano":
                model.srng.gen_seedgen.set_state(checkpoint.unpack_random_state(arrays, "seedgen"))
                model.srng.nodes = []
                for k in range(int(header["theano_nodes"])):
                    node = np.random.RandomState()
                    node.set_state(checkpoint.unpack_random_state(arrays, "node%d" % k))
                    model.srng.nodes.append(node)
        except BaseException:
            model.close()
            raise
        return (model, driver) if return_driver_state else model

    # ---- plumbing ------------------------------------------------------------------------
    def set_stream(self, cuda_stream):
        _lib.check(self._lib.vaeb_set_stream(self._h, C.c_void_p(cuda_stream)))

    def synchronize(self):
        _lib.check(self._lib.vaeb_synchronize(self._h))

    def profile_update(self, index=0, iters=20):
        """[(phase name, ms per launch, algorithmic flops, algorithmic bytes)] of one update."""
        cap = 32
        n = C.c_int32()
        t = np.zeros(cap, np.float32); fl = np.zeros(cap, np.float64); by = np.zeros(cap, np.float64)
        names = C.create_string_buffer(48 * cap)
        _lib.check(self._lib.vaeb_profile_update(self._h, int(index), int(iters), cap, C.byref(n), _ptr(t), _ptr(fl),
                                                 _ptr(by), C.cast(names, C.c_void_p)))
        return [(names.raw[48 * i:48 * i + 48].split(b"\0")[0].decode(), float(t[i]), float(fl[i]), float(by[i]))
                for i in range(n.value)]

    def apply_update(self):
        """Adagrad step (VAEB.py:426-444) with the gradients left in the buffer by `gradients()` (or written
        there by the caller): the second half of `update()` on its own."""
        _lib.check(self._lib.vaeb_apply_update(self._h))

    @property
    def adam_step(self):
        """Adam's step counter t: updates applied since Adam was selected.  With the moments (self.ADA and
        self.ADAM_V) it is the optimizer state a checkpoint saves and restores."""
        t = C.c_int64()
        _lib.check(self._lib.vaeb_adam_step(self._h, C.byref(t)))
        return t.value

    @adam_step.setter
    def adam_step(self, t):
        _lib.check(self._lib.vaeb_set_adam_step(self._h, int(t)))

    def set_kl_weight(self, beta, warmup=0):
        """Weight the latent term of the bound in the gradient: the n-th update applied after this call ascends
        loglik + beta_n * aux with beta_n = kl_weight_at(beta, warmup, n) -- a linear KL warm-up over `warmup` updates,
        or beta-VAE's constant beta when warmup = 0.  Resets kl_step to 0.  The bounds update() and friends return stay
        the unweighted SGVB / batch_size.  Not available for the full-VB estimators."""
        _lib.check(self._lib.vaeb_set_kl_weight(self._h, float(beta), int(warmup)))
        self.kl_weight, self.kl_warmup = float(beta), int(warmup)

    @property
    def kl_step(self):
        """Updates applied since set_kl_weight (the position in the warm-up): save and restore it to resume a run."""
        t = C.c_int64()
        _lib.check(self._lib.vaeb_kl_step(self._h, C.byref(t)))
        return t.value

    @kl_step.setter
    def kl_step(self, t):
        _lib.check(self._lib.vaeb_set_kl_step(self._h, int(t)))

    def profile_optimizer(self, iters=20):
        """(ms per launch, algorithmic bytes per launch) of the flat Adagrad pass over this model's buffers."""
        ms, by = C.c_float(), C.c_double()
        _lib.check(self._lib.vaeb_profile_optimizer(self._h, int(iters), C.byref(ms), C.byref(by)))
        return ms.value, by.value

    def step_kernel_name(self, rows=None):
        """The kernel update() runs for `rows` rows (default: the batch size)."""
        w = C.c_int32()
        _lib.check(self._lib.vaeb_step_kernel(self._h, int(rows or self.batch_size), C.byref(w)))
        return {2: "step_tc_kernel (tcgen05, one launch per update)", 1: "fused_step_kernel (fp32 FFMA, one launch per update)",
                0: "per-layer kernels"}[w.value]

    def launch_count(self):
        n = C.c_int64()
        _lib.check(self._lib.vaeb_launch_count(self._h, C.byref(n)))
        return n.value

    def attach_comm(self, unique_id, rank, world_size, nccl_library=None):
        path = (nccl_library or _lib.nccl_library_path()).encode()
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id))
        _lib.check(self._lib.vaeb_comm_attach(self._h, path, buf, rank, world_size))
        self._rank, self._world = int(rank), int(world_size)

    def p2p_export(self):
        """CUDA IPC handles (192 bytes) of this rank's gradient staging buffer, parameters and accumulators."""
        buf = (C.c_uint8 * 192)()
        _lib.check(self._lib.vaeb_comm_p2p_export(self._h, buf))
        return bytes(buf)

    def p2p_attach(self, all_handles):
        """`all_handles`: the p2p_export() bytes of every rank, in rank order."""
        blob = b"".join(all_handles)
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        _lib.check(self._lib.vaeb_comm_p2p_attach(self._h, buf, len(all_handles)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.vaeb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _PinnedBlock(object):
    """Owner of one cudaMallocHost block; freed when the last array viewing it goes away."""

    def __init__(self, nbytes):
        self._lib = _lib.load()
        self.ptr = C.c_void_p()
        _lib.check(self._lib.vaeb_host_alloc(int(nbytes), C.byref(self.ptr)))
        self.buf = (C.c_uint8 * int(nbytes)).from_address(self.ptr.value)

    def __del__(self):
        try:
            if self.ptr:
                self._lib.vaeb_host_free(self.ptr)
                self.ptr = C.c_void_p()
        except Exception:
            pass


def pinned_empty(shape, dtype=np.float32):
    """numpy array in page-locked host memory (what `update_host_async` requires)."""
    dt = np.dtype(dtype)
    n = int(np.prod(shape)) * dt.itemsize
    blk = _PinnedBlock(max(n, 1))
    buf = blk.buf
    blk.buf = None
    buf._owner = blk      # arr.base chain -> buf -> blk: the block is freed when the last view of it goes away
    return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)


def kl_weight_at(beta, warmup, n):
    """beta_n of set_kl_weight(beta, warmup) for the n-th update applied after the call (n >= 1), as the library
    computes it: beta * min(1, n / warmup) in double from the float32 beta, rounded to float32 once."""
    beta = float(np.float32(beta))
    if warmup == 0 or n >= warmup:
        return np.float32(beta)
    return np.float32(beta * (float(n) / float(warmup)))


def comm_unique_id(nccl_library=None):
    lib = _lib.load()
    buf = (C.c_uint8 * 128)()
    _lib.check(lib.vaeb_comm_unique_id((nccl_library or _lib.nccl_library_path()).encode(), buf))
    return bytes(buf)


def mlp_forward(x, Ws, bs, act_last="tanh", device=0):
    """degenerate-vae/mlp.py:66-74 `ConstructMLP` (tanh on every layer) / logpdf.py OutToReal,
    OutToProbs as the last layer, evaluated by the dense-layer kernels."""
    lib = _lib.load()
    xa = _f32(x)
    dims = [xa.shape[1]] + [int(W.shape[1]) for W in Ws]
    cfg = _lib.Config(input_dim=dims[0], hidden_units=max(dims), latent_size=1, batch_size=1, L=1, continuous=0,
                      estimator=0, variant=0, precision=0, device=device, learning_rate=0.0, adagrad_eps=1e-6,
                      prior_scale=1.0, sigma_vb_init=1e-3, seed=0)
    h = C.c_void_p()
    _lib.check(lib.vaeb_create(C.byref(cfg), C.byref(h)))
    try:
        Wa = [_f32(W) for W in Ws]
        ba = [_f32(b) for b in bs]
        out = np.empty((xa.shape[0], dims[-1]), np.float32)
        _lib.check(lib.vaeb_mlp_forward(
            h, _ptr(xa), xa.shape[0], len(Wa), (C.c_int32 * len(dims))(*dims),
            (C.c_void_p * len(Wa))(*[a.ctypes.data for a in Wa]), (C.c_void_p * len(ba))(*[a.ctypes.data for a in ba]),
            {"identity": 0, "tanh": 1, "sigmoid": 2}[act_last], _ptr(out)))
        return out
    finally:
        lib.vaeb_destroy(h)
