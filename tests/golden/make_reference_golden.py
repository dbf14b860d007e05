"""Golden vectors produced by THE REFERENCE'S OWN SOURCE, executed in this container.

    python tests/golden/make_reference_golden.py        (needs /root/reference; CPU only)

The reference is Python 2 + Theano and cannot run as is (SURVEY.md F7).  This script loads the
reference's files *where they lie* (/root/reference/VAEB.py, VAEBfullbayes.py, degenerate-vae/
{logpdf,mlp,infalg}.py -- nothing is copied into the repo), applies three py2->py3 token fixes in
memory (`print` statement, `.iteritems()`, `cPickle`) and executes them against
tests/golden/theano_shim.py, a lazy-graph stand-in for the handful of Theano calls the hot path
makes (dot/tanh/sigmoid/exp/log/sum/grad/function/shared/RandomStreams), evaluated by torch on
the CPU in float64.  So the model code that runs -- initialize_params, encoder, decoder,
reparam_trick, posterior_log_prob, getLA/getLB/getFVBL, the prior, T.grad targets, getUpdates,
the update/validate function signatures incl. `givens` slicing and pre-update outputs -- is the
reference's, line for line; only the tensor library underneath is substituted.

Outputs (tests/golden/ref_*.npz) hold the inputs (x, initial parameters, the noise each call
drew, in call order) and the outputs (returned bounds, parameters / Adagrad accumulators after
the updates).  tests/test_reference_golden.py checks the numpy oracle against them (CPU) and
tests/test_gpu_reference_golden.py checks the CUDA path against them (B200).
"""
import os
import re
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import theano_shim  # noqa: E402

REF = "/root/reference"


def load_reference_module(rel_path, name):
    """exec the reference file under a private module name (so its `__main__` block stays inert)."""
    path = os.path.join(REF, rel_path)
    src = open(path).read()
    src = re.sub(r"^(\s*)print\s+(?!\()(.+)$", r"\1print(\2)", src, flags=re.M)   # py2 print statement
    src = src.replace(".iteritems()", ".items()")
    src = re.sub(r"^import cPickle$", "import pickle as cPickle", src, flags=re.M)
    mod = types.ModuleType(name)
    mod.__file__ = path
    sys.modules[name] = mod
    exec(compile(src, path, "exec"), mod.__dict__)
    return mod


def shared_list(th, arrays, names):
    return [th.shared(value=np.array(a, dtype=th.config.floatX), name=n) for a, n in zip(arrays, names)]


def eps_of_calls(srng, start, L):
    """The draws logged since `start`, grouped per function call -> [L, rows, Z] (node l = sample l)."""
    d = srng.draws[start:]
    assert len(d) % L == 0
    calls = []
    for c in range(len(d) // L):
        grp = d[c * L:(c + 1) * L]
        assert [n for n, _ in grp] == list(range(L)), [n for n, _ in grp]
        calls.append(np.stack([a for _, a in grp]))
    return calls


NAMES_D = ["W3", "W4", "W5", "W1", "W2", "b3", "b4", "b5", "b1", "b2"]
NAMES_C = ["W3", "W4", "W5", "W1", "W2", "W6", "b3", "b4", "b5", "b1", "b2", "b6"]


def run_vaeb_case(V, th, x, continuous, H, Z, M, L, lr, generic, order, n_valid, params0=None, scale=None):
    """Build the reference model, run update(order[i]) and a validate(); return the fixture dict."""
    names = NAMES_C if continuous else NAMES_D
    if params0 is not None:
        params = shared_list(th, params0, names)
    else:
        params = None
    model = V.VAEB(x, continuous, H, Z, M, L, lr, generic, False, params)
    if params0 is None and scale is not None:
        # the 0.01-sigma initialisation keeps tanh linear; scale the weights up so every
        # nonlinearity is exercised (still the reference's own draws)
        for p in model.params:
            p.set_value(p.get_value() * scale if p.get_value().ndim == 2 else p.get_value())
    out = {"x": x.astype(np.float32), "continuous": continuous, "H": H, "Z": Z, "M": M, "L": L, "lr": lr, "generic": generic,
           "order": np.array(order)}
    for n, p in zip(names, model.params):
        out["init_" + n] = p.get_value().copy()
    rets, mark = [], 0
    for i in order:
        rets.append(float(model.update(i)))
    xv = x[:n_valid]
    val = float(model.validate(xv))
    calls = eps_of_calls(model.srng, 0, L)
    assert len(calls) == len(order) + 1
    for k, e in enumerate(calls[:-1]):
        out["eps_update_%d" % k] = e
    out["eps_validate"] = calls[-1]
    out["update_returns"] = np.array(rets)
    out["validate_return"] = np.float64(val)
    out["n_valid"] = n_valid
    for n, p, a in zip(names, model.params, model.ADA):
        out["final_" + n] = p.get_value().copy()
        out["ada_" + n] = a.get_value().copy()
    return out


def run_fvb_case(V, th, x, H, Z, M, lr, order, params0):
    """fullVariational=True (getFVBL, VAEB.py:349-367): gradients w.r.t. the (mu, sigma) pairs only."""
    params = shared_list(th, params0, NAMES_D)
    model = V.VAEB(x, False, H, Z, M, 1, lr, False, True, params)
    out = {"x": x.astype(np.float32), "H": H, "Z": Z, "M": M, "lr": lr, "order": np.array(order)}
    for n, p in zip(NAMES_D, params0):
        out["init_" + n] = np.array(p, dtype=np.float64)
    rets = [float(model.update(i)) for i in order]
    val = float(model.validate(x[:2 * M]))
    calls = eps_of_calls(model.srng, 0, 1)
    for k, e in enumerate(calls[:-1]):
        out["eps_update_%d" % k] = e
    out["eps_validate"] = calls[-1]
    out["update_returns"], out["validate_return"] = np.array(rets), np.float64(val)
    for i, n in enumerate(NAMES_D):
        out["final_mu_" + n] = model.full_variational_params[2 * i].get_value().copy()
        out["final_sigma_" + n] = model.full_variational_params[2 * i + 1].get_value().copy()
        out["final_map_" + n] = model.params[i].get_value().copy()
    return out


def run_fullbayes_case(F, th, x, continuous, H, Z, M, lr, order, scale):
    model = F.VAE(x, continuous, H, Z, M, 1, lr)
    names = NAMES_C if continuous else NAMES_D
    for p in model.params:
        if p.get_value().ndim == 2:
            p.set_value(p.get_value() * scale)
    out = {"x": x.astype(np.float32), "continuous": continuous, "H": H, "Z": Z, "M": M, "lr": lr, "order": np.array(order)}
    for n, p in zip(names, model.params):
        out["init_" + n] = p.get_value().copy()
    # VAEBfullbayes creates its RandomStreams inside getGradient: re-derive the draws it makes
    rs = np.random.RandomState(int(np.random.RandomState(10).randint(2 ** 30)))
    rets, eps = [], []
    for i in order:
        eps.append(rs.normal(0.0, 1.0, size=(M, Z)))
        rets.append(float(model.update(i)))
    eps.append(rs.normal(0.0, 1.0, size=(2 * M, Z)))
    val = float(model.validate(x[:2 * M]))
    for k, e in enumerate(eps[:-1]):
        out["eps_update_%d" % k] = e[None]
    out["eps_validate"] = eps[-1][None]
    out["update_returns"], out["validate_return"] = np.array(rets), np.float64(val)
    for n, p, a in zip(names, model.params, model.ADA):
        out["final_" + n] = p.get_value().copy()
        out["ada_" + n] = a.get_value().copy()
    return out


def fingerprint(t):
    f = np.asarray(t, np.float64).ravel()
    idx = np.linspace(0, f.size - 1, 16).astype(int)
    return np.concatenate([[f.sum(), (f * f).sum(), np.abs(f).max()], f[idx]])


def main():
    th = theano_shim.install("float64")
    V = load_reference_module("VAEB.py", "ref_VAEB")
    F = load_reference_module("VAEBfullbayes.py", "ref_VAEBfullbayes")
    rng = np.random.RandomState(20261018)

    def f32(a):          # data exactly representable in float32: the GPU path sees the same numbers
        return a.astype(np.float32).astype(np.float64)

    def bern_x(n, D):
        return f32(rng.uniform(size=(n, D)) * (rng.uniform(size=(n, D)) < 0.3))

    def cont_x(n, D):
        return f32(np.clip(0.5 + 0.2 * rng.normal(size=(n, D)), 0.0, 1.0))

    # ---- small models, every estimator x decoder, the reference's own initialisation ----------
    cases = {
        "disc_LB_L1": dict(x=bern_x(24, 40), continuous=False, H=24, Z=3, M=8, L=1, generic=False),
        "disc_LA_L2": dict(x=bern_x(24, 40), continuous=False, H=24, Z=3, M=8, L=2, generic=True),
        "cont_LB_L2": dict(x=cont_x(30, 36), continuous=True, H=20, Z=2, M=10, L=2, generic=False),
        "cont_LA_L1": dict(x=cont_x(30, 36), continuous=True, H=20, Z=2, M=10, L=1, generic=True),
    }
    g = {}
    for name, c in cases.items():
        r = run_vaeb_case(V, th, c["x"], c["continuous"], c["H"], c["Z"], c["M"], c["L"], 0.01, c["generic"],
                          order=[0, 2, 1, 0], n_valid=2 * c["M"] + 3, scale=40.0)
        for k, v in r.items():
            g["%s__%s" % (name, k)] = v
    np.savez_compressed(os.path.join(HERE, "ref_vaeb_small.npz"), **g)

    # ---- AdaDelta: the reference keeps `updates = self.getAdaDeltaUpdates(gradients)` commented out at
    # VAEB.py:404; swapping the method in is what un-commenting that line does -------------------------------
    g = {}
    keep = V.VAEB.getUpdates
    V.VAEB.getUpdates = V.VAEB.getAdaDeltaUpdates
    try:
        for name in ("disc_LB_L1", "cont_LA_L1"):
            c = cases[name]
            r = run_vaeb_case(V, th, c["x"], c["continuous"], c["H"], c["Z"], c["M"], c["L"], 0.01, c["generic"],
                              order=[0, 2, 1, 0, 1, 2], n_valid=2 * c["M"], scale=40.0)
            for k, v in r.items():
                if not k.startswith("ada_"):            # getAdaDeltaUpdates keeps its accumulators in local shared variables
                    g["%s__%s" % (name, k)] = v
    finally:
        V.VAEB.getUpdates = keep
    np.savez_compressed(os.path.join(HERE, "ref_adadelta_small.npz"), **g)

    # ---- the reference's initialisation at the real shapes (draw order, VAEB.py:50-125) -------
    g = {}
    for tag, (D, H, Z, cont) in {"mnist": (784, 500, 20, False), "frey": (560, 200, 2, True)}.items():
        theano_shim.config.floatX = "float32"       # the reference runs floatX=float32 (run_on_gpu.sh)
        m = V.VAEB(np.zeros((4, D)), cont, H, Z, 2, 1, 0.01, False, False)
        theano_shim.config.floatX = "float64"
        for n, p in zip(NAMES_C if cont else NAMES_D, m.params):
            assert p.get_value().dtype == np.float32
            g["%s__fp_%s" % (tag, n)] = fingerprint(p.get_value())
    np.savez_compressed(os.path.join(HERE, "ref_init_fingerprints.npz"), **g)

    # ---- Frey shape with the trained weights the reference ships (realistic magnitudes) --------
    from vaeb_b200 import io
    _, trained = io.read_mdl(os.path.join(REF, "reconstruction_res", "continuous_2.mdl"))
    x = cont_x(300, 560)
    g = {"x": x.astype(np.float32)}                 # the rows of both estimators, stored once (keeps the file < 1 MB)
    for est, generic in (("LB", False), ("LA", True)):
        r = run_vaeb_case(V, th, x, True, 200, 2, 100, 1, 0.01, generic, order=[1, 0], n_valid=300,
                          params0=[np.asarray(p, np.float64) for p in trained])
        for k, v in r.items():
            if k.startswith("init_") or k == "x":
                continue                            # init_ = tests/golden/frey_z2_trained_{encoder,decoder}.npz
            if k.startswith(("final_W", "ada_W")) and v.size > 2000:
                v = fingerprint(v)
                k = "fp_" + k
            g["%s__%s" % (est, k)] = v
    np.savez_compressed(os.path.join(HERE, "ref_vaeb_frey_trained.npz"), **g)

    # ---- MNIST shape, one update + validate at the reference's own initialisation --------------
    x = bern_x(200, 784)
    r = run_vaeb_case(V, th, x, False, 500, 20, 100, 1, 0.01, False, order=[1], n_valid=200)
    g = {}
    for k, v in r.items():
        if k.startswith("init_"):
            continue                                # = oracle.init_params (checked by fingerprints above)
        if k.startswith(("final_W", "ada_W")) and v.size > 2000:
            v, k = fingerprint(v), "fp_" + k
        g[k] = v
    np.savez_compressed(os.path.join(HERE, "ref_vaeb_mnist_init.npz"), **g)

    # ---- full-variational path (getFVBL) ---------------------------------------------------------
    D, H, Z, M = 40, 24, 3, 8
    x = bern_x(24, D)
    shapes = [(D, H), (H, Z), (H, Z), (Z, H), (H, D), (H,), (Z,), (Z,), (H,), (D,)]
    p0 = [rng.normal(0, 0.3, s) for s in shapes]
    r = run_fvb_case(V, th, x, H, Z, M, 0.01, [0, 1, 2], p0)
    np.savez_compressed(os.path.join(HERE, "ref_fvb_small.npz"), **r)

    # ---- VAEBfullbayes.py variant ----------------------------------------------------------------
    g = {}
    for tag, cont in (("disc", False), ("cont", True)):
        x = cont_x(24, 36) if cont else bern_x(24, 36)
        r = run_fullbayes_case(F, th, x, cont, 20, 3, 8, 0.01, [0, 2, 1], 40.0)
        for k, v in r.items():
            g["%s__%s" % (tag, k)] = v
    np.savez_compressed(os.path.join(HERE, "ref_fullbayes_small.npz"), **g)

    # ---- AE-side primitives: logpdf / mlp / infalg (degenerate-vae/) -----------------------------
    for stub in ("theano.printing", "theano.sandbox", "theano.sandbox.rng_mrg", "data"):
        m = types.ModuleType(stub)
        m.pydotprint = lambda *a, **k: None
        m.MRG_RandomStreams = theano_shim.RandomStreams
        sys.modules[stub] = m
    T = th.tensor
    T.dmatrix = T.matrix
    lp = load_reference_module("degenerate-vae/logpdf.py", "logpdf")
    ia = load_reference_module("degenerate-vae/infalg.py", "infalg")
    mlp = load_reference_module("degenerate-vae/mlp.py", "mlp")
    g = {}
    xs, ps = T.matrix("x"), T.matrix("p")
    f = th.function([xs, ps], lp.bernoulli(xs, ps))
    g["bernoulli_kat"] = f([[0, 0, 1], [0, 0, 1]], [[0.01, 0.01, 0.99], [0.01, 0.01, 0.99]])   # logpdf.py:119-123
    Y, P = bern_x(6, 9), rng.uniform(0.02, 0.98, size=(6, 9))
    MU, LS2 = rng.normal(size=(6, 9)), rng.normal(size=(6, 9))
    g["Y"], g["P"], g["MU"], g["LS2"] = Y, P, MU, LS2
    g["bernoulli"] = f(Y, P)
    ms, ls = T.matrix("m"), T.matrix("l")
    g["indep_normal"] = th.function([xs, ms, ls], lp.indep_normal(xs, ms, ls))(Y, MU, LS2)
    Ws = [rng.normal(0, 0.5, s) for s in ((9, 7), (7, 5), (5, 4))]
    bs = [rng.normal(0, 0.5, (s,)) for s in (7, 5, 4)]
    Wsh = [th.shared(w) for w in Ws]
    bsh = [th.shared(b) for b in bs]
    g["mlp_out"] = th.function([xs], mlp.ConstructMLP(xs, Wsh, bsh, T.tanh))(Y)
    for i, (w, b) in enumerate(zip(Ws, bs)):
        g["mlp_W%d" % i], g["mlp_b%d" % i] = w, b
    g["normal_prior"] = th.function([], mlp.ConstructNormalPrior(Wsh + bsh, 0.7))()
    s20, s21 = np.exp(LS2), np.exp(rng.normal(size=(6, 9)))
    g["s21"] = s21
    a, b_, c, d = T.matrix(), T.matrix(), T.matrix(), T.matrix()
    g["gauss_dkl"] = th.function([a, b_, c, d], mlp.GaussDKL(a, b_, c, d))(MU, s20, P, s21)
    g["out_to_probs"] = th.function([xs], lp.OutToProbs(xs, Wsh[0], bsh[0]))(Y)
    g["out_to_real"] = th.function([xs], lp.OutToReal(xs, Wsh[0], bsh[0]))(Y)
    # infalg.AdaGrad.construct: two steps on f = -sum((theta - c)^2) * scale
    theta = [th.shared(rng.normal(size=(4, 3))), th.shared(rng.normal(size=(5,)))]
    g["ag_theta0_0"], g["ag_theta0_1"] = theta[0].get_value().copy(), theta[1].get_value().copy()
    obj = -3.0 * T.sum(T.sqr(theta[0] - 0.5)) - 0.25 * T.sum(T.sqr(theta[1] + 1.0) * theta[1])
    opt = ia.AdaGrad(0.05) if _takes_eta(ia.AdaGrad) else ia.AdaGrad()
    if not hasattr(opt, "eta"):
        opt.eta = 0.05
    g["ag_eta"] = np.float64(opt.eta)
    step = th.function([], obj, updates=opt.construct(obj, theta))
    g["ag_obj"] = np.array([float(step()), float(step())])
    g["ag_theta2_0"], g["ag_theta2_1"] = theta[0].get_value().copy(), theta[1].get_value().copy()
    np.savez_compressed(os.path.join(HERE, "ref_ae_primitives.npz"), **g)

    # ---- AE baselines: ConstructAE of degenerate-vae/ae.py (binary + cont) and vanilla-ae/ae.py ------------------
    # theta order of the reference: Wenc + benc + [Wz, bz] + Wdec + bdec + [Wout, bout] | [Wmu, Wlogs2, bmu, blogs2];
    # stored under the VAEB names (W3=Wenc0, b3, W4=Wz, b4, W1=Wdec0, b1, W2=Wout|Wmu, b2, W6=Wlogs2, b6).
    ae_deg = load_reference_module("degenerate-vae/ae.py", "ae_degenerate")
    ae_van = load_reference_module("vanilla-ae/ae.py", "ae_vanilla")
    g = {}
    D, Hh, Dz, Ntr = 36, 20, 3, 40
    for tag, mod, otype, xs in (("deg_binary", ae_deg, "binary", bern_x(Ntr, D)), ("deg_cont", ae_deg, "cont", cont_x(Ntr, D)),
                                ("vanilla", ae_van, None, bern_x(Ntr, D))):
        np.random.seed(1234)                              # mlp.WeightMatrix / BiasVector draw from the global numpy RNG
        Xtr = th.shared(xs, "Xtr")
        kw = dict(Denc=[Hh], Dz=Dz, Ddec=[Hh], inf=ia.AdaGrad(0.01))
        if otype:
            kw["otype"] = otype
        train, reconstruct, encode, decode, theta = mod.ConstructAE(Xtr, **kw)
        if otype == "cont":
            names = ["W3", "b3", "W4", "b4", "W1", "b1", "W2", "W6", "b2", "b6"]
        else:
            names = ["W3", "b3", "W4", "b4", "W1", "b1", "W2", "b2"]
        assert len(theta) == len(names)
        for t_, n in zip(theta, names):
            if n.startswith("W"):                         # 0.01-sigma initialisation keeps every tanh linear: scale up
                t_.set_value(t_.get_value() * 40.0)
            g["%s__init_%s" % (tag, n)] = t_.get_value().copy()
        g["%s__x" % tag] = xs.astype(np.float32)
        idx_rng = np.random.RandomState(77)
        idxs = [idx_rng.permutation(Ntr)[:10].astype(np.int32) for _ in range(4)] + [np.arange(7, dtype=np.int32)]
        g["%s__idx" % tag] = np.stack([np.pad(i, (0, 10 - len(i)), constant_values=-1) for i in idxs])
        g["%s__train_returns" % tag] = np.array([float(train(i)) for i in idxs])
        for t_, n in zip(theta, names):
            g["%s__final_%s" % (tag, n)] = t_.get_value().copy()
        g["%s__reconstruct" % tag] = reconstruct(xs[:6])
        zz = encode(xs[:6])
        g["%s__encode" % tag] = zz
        g["%s__decode" % tag] = decode(zz)
    np.savez_compressed(os.path.join(HERE, "ref_ae_baselines.npz"), **g)
    print("wrote", sorted(f for f in os.listdir(HERE) if f.startswith("ref_")))


def _takes_eta(cls):
    import inspect
    try:
        return len(inspect.signature(cls.__init__).parameters) > 1
    except (TypeError, ValueError):
        return False


if __name__ == "__main__":
    main()
