"""The args/flags-dictionary CLI and the training driver of the reference (VAEB.py:25-38,
471-612), Python 3, over the B200 model class.  Same argument names (including the
`full_varational` spelling), defaults, printed blocks, `.trc` layout and `.mdl` layout."""
from __future__ import annotations

import os
import sys
import time

import numpy as np

from . import checkpoint, io
from .data import load_frey, load_mnist
from .model import VAEB

# name -> (default, type): the dictionary-driven CLI of VAEB.py:22-38; a new option is one more entry here
command_line_args = {'seed': (15485863, int),
                     'n_latent': (10, int),
                     'n_epochs': (2000, int),
                     'batch_size': (100, int),
                     'L': (1, int),
                     'hidden_unit': (-1, int),
                     'learning_rate': (0.01, float),
                     'trace_file': ('', str),
                     'save_file': ('', str),
                     'load_file': ('', str),
                     'vb_param_file': ('', str),
                     # --- extensions (defaults keep the reference behaviour) ---
                     'device': (0, int),
                     'precision': ('fp32', str),      # fp32 | bf16
                     'eps_mode': ('philox', str),     # philox | theano
                     'manifold_file': ('', str),      # PGM of the learned 2-d manifold (freyFace.py:346-369)
                     # PGM of 10 x 10 random samples (AEVB Fig. 5); a Bernoulli model shows its decoder means,
                     # since binary draws make a poor image
                     'sample_file': ('', str),
                     'optimizer': ('adagrad', str),  # adagrad (VAEB.py:426-444) | adadelta (VAEB.py:449-469) | adam
                     # weight of the latent term (-KL / log p(z) - log q(z|x)) in the gradient, and the epochs over
                     # which it ramps up linearly (KL warm-up); 1.0 and 0 train on the reference's bound
                     'kl_weight': (1.0, float),
                     'kl_warmup': (0, int),
                     # the complete training state (vaeb_b200/checkpoint.py), written every checkpoint_every epochs and
                     # after the last one; resume_file continues a run from such a file up to --n_epochs
                     'checkpoint_file': ('', str),
                     'checkpoint_every': (100, int),
                     'resume_file': ('', str)}
command_line_flags = ['continuous', 'generic_estimator', 'full_varational',
                      # --- extensions ---
                      'synthetic',        # synthetic data of the dataset's shape if the files are absent
                      'sample_weights']   # full-VB with sampled weights (VAEB.py:127-129 live)


def _pop_option(tokens, name, n_values):
    """Removes the first `--name` from `tokens` together with its `n_values` values; returns the values (a list)
    or None when the option is absent.  The reference's parser (VAEB.py:471-489) behaves the same way: first
    occurrence wins, later duplicates stay behind and end up in the 'unused' report."""
    key = "--" + name
    try:
        at = tokens.index(key)
    except ValueError:
        return None
    values = tokens[at + 1:at + 1 + n_values]
    if len(values) < n_values:                       # `--key` as the last token: the reference raises IndexError here
        raise IndexError("missing value for %s" % key)
    tokens[at:at + 1 + n_values] = []
    return values


def get_arg(arg, args, default, type_):
    """`--arg value` cast with the dictionary's type, else the default (VAEB.py:471-480)."""
    found = _pop_option(args, arg, 1)
    return default if found is None else type_(found[0])


def get_flag(flag, args):
    """True iff `--flag` was given (VAEB.py:483-489)."""
    return _pop_option(args, flag, 0) is not None


def parse_args(argv=None):
    """VAEB.py:491-504: every key of the two dictionaries ends up in the result; what is left over is reported."""
    tokens = list(sys.argv[1:] if argv is None else argv)
    parsed = {name: get_arg(name, tokens, default, cast) for name, (default, cast) in command_line_args.items()}
    parsed.update((name, get_flag(name, tokens)) for name in command_line_flags)
    if tokens:
        print('Have unused args: {0}'.format(tokens))
    return parsed


def print_args(args):
    """VAEB.py:507-512."""
    rule = '-' * 38
    body = ['\t{0}: {1}'.format(key, args[key]) for key in args]
    print('\n'.join(['Parameters used:', rule] + body + [rule]))


def _default_hidden(continuous, hidden_unit):
    # VAEB.py:542-543,551-552: 200 units for Frey Face, 500 for MNIST unless --hidden_unit says otherwise
    return hidden_unit if hidden_unit >= 0 else (200 if continuous else 500)


def kl_warmup_updates(epochs, n_rows, batch_size):
    """--kl_warmup is given in epochs; the model counts updates, N // batch_size of them per epoch (VAEB.py:571), so
    the weight grows with every update inside an epoch's update_many."""
    return int(epochs) * (int(n_rows) // int(batch_size))


def model_args(args, n_rows):
    """The constructor arguments of the model the command line describes (those a checkpoint records)."""
    continuous = bool(args['continuous'])
    return dict(continuous=continuous, hidden_units=_default_hidden(continuous, args['hidden_unit']),
                latent_size=args['n_latent'], batch_size=args['batch_size'], L=args['L'],
                learning_rate=args['learning_rate'], genericEstimator=bool(args['generic_estimator']),
                fullVariational=bool(args['full_varational']), precision=args.get('precision', 'fp32'),
                eps_mode=args.get('eps_mode', 'philox'), sample_weights=bool(args.get('sample_weights', False)),
                optimizer=args.get('optimizer', 'adagrad'), kl_weight=float(args.get('kl_weight', 1.0)),
                kl_warmup=kl_warmup_updates(args.get('kl_warmup', 0), n_rows, args['batch_size']))


def check_resume_args(saved, wanted):
    """A resumed run continues the saved model: a model-shaping option that differs from the checkpoint is an error,
    not a silent override.  `saved`: the checkpoint's constructor arguments; `wanted`: model_args of the command line."""
    diff = ["%s (checkpoint %r, command line %r)" % (k, saved[k], v) for k, v in wanted.items() if saved[k] != v]
    if diff:
        raise ValueError("--resume_file: the command line differs from the checkpoint in " + ", ".join(diff))


def loop_state(epochs_done, batch_order, trace_file=''):
    """What the training loop adds to a checkpoint: the completed epochs, numpy's global RNG, the minibatch order
    (each epoch shuffles the previous epoch's order in place) and the length of the trace file (-1: no trace)."""
    keys, aux = checkpoint.random_state_arrays(np.random.get_state())
    return {'epoch': int(epochs_done), 'np_random_keys': keys, 'np_random_aux': aux,
            'batch_order': np.asarray(batch_order, dtype=np.int64),
            'trace_bytes': os.path.getsize(trace_file) if trace_file else -1}


def rewind_trace(trace_file, trace_bytes):
    """A resumed run continues the trace file of the checkpoint: the lines that epochs after the checkpoint wrote
    before the run stopped are cut off (they are written again), so the file ends as an uninterrupted run's does.
    Without a trace at the checkpoint the file starts afresh."""
    if trace_bytes < 0:
        io.trace_header(trace_file)
        return
    if not os.path.exists(trace_file) or os.path.getsize(trace_file) < trace_bytes:
        raise ValueError("--resume_file: the trace file %s is shorter than the %d bytes it had at the checkpoint"
                         % (trace_file, trace_bytes))
    with open(trace_file, "r+b") as f:
        f.truncate(trace_bytes)


def train_model(args, data=None):
    """The training driver of VAEB.py:524-598: seed numpy's global RNG (it only drives the shuffle), load the
    dataset of the chosen mode, build the model (on top of --vb_param_file for full VB), then per epoch: shuffle
    the minibatch order, update on every minibatch, validate, write the trace line (twice, as the reference does)
    and print the two progress lines; finally save.  --checkpoint_file saves the training state every
    --checkpoint_every epochs and after the last one; --resume_file rebuilds model, epoch and shuffle RNG from such
    a file and continues to --n_epochs, appending to the trace file as the checkpoint left it."""
    np.random.seed(args['seed'])
    continuous = args['continuous']
    synthetic = args.get('synthetic', False)
    ext = dict(device=args.get('device', 0), precision=args.get('precision', 'fp32'),
               eps_mode=args.get('eps_mode', 'philox'))
    trace_file, save_file = args['trace_file'], args['save_file']
    resume_file, checkpoint_file = args.get('resume_file', ''), args.get('checkpoint_file', '')
    every = args.get('checkpoint_every', 100)

    print("loading data")
    if data is None:
        data = load_frey(synthetic=synthetic) if continuous else load_mnist(synthetic=synthetic)
    x_train, x_valid = data[0], data[1]

    start, driver = 0, None
    if resume_file:
        print("resuming from %s" % resume_file)
        model, driver = VAEB.resume(resume_file, x_train, device=ext['device'], return_driver_state=True)
        try:
            check_resume_args(model._ctor_args(), model_args(args, len(x_train)))
        except ValueError:
            model.close()
            raise
        np.random.set_state(checkpoint.random_state_tuple(driver['np_random_keys'], driver['np_random_aux']))
        start = int(driver['epoch'])
    else:
        print("creating the model")
        params = None
        if args['full_varational']:                    # VAEB.py:559-561: the MAP solution seeds the variational means
            seed_model, _ = VAEB.load(args['vb_param_file'], data=data, **ext)
            params = seed_model.get_params()
            seed_model.close()
        model = VAEB(x_train, continuous, _default_hidden(continuous, args['hidden_unit']), args['n_latent'],
                     args['batch_size'], args['L'], args['learning_rate'], args['generic_estimator'],
                     args['full_varational'], params, sample_weights=args.get('sample_weights', False),
                     optimizer=args.get('optimizer', 'adagrad'), kl_weight=args.get('kl_weight', 1.0),
                     kl_warmup=kl_warmup_updates(args.get('kl_warmup', 0), len(x_train), args['batch_size']), **ext)

    print("learning")
    tracing = len(trace_file) > 0
    if tracing and resume_file:
        rewind_trace(trace_file, int(driver['trace_bytes']))
    elif tracing:
        io.trace_header(trace_file)
    batch_order = np.arange(model.N // model.batch_size)           # the remainder rows are never visited (:571)
    if driver is not None:
        batch_order = np.asarray(driver['batch_order'], dtype=batch_order.dtype)
    for epoch in range(start, args['n_epochs']):
        t_epoch = time.time()
        np.random.shuffle(batch_order)
        # the reference accumulates `model.update(batch)` over the order (VAEB.py:577-579); update_many performs
        # the same updates in the same order without a host round trip per minibatch
        LB = float(np.sum(model.update_many(batch_order), dtype=np.float64)) / len(batch_order)
        LBvalidation = float(model.validate(x_valid)) / x_valid.shape[0]
        seen = model.N * (epoch + 1)
        if tracing:
            io.trace_line(trace_file, seen, LB, LBvalidation)
        print("Epoch %s : [Lower bound: %s, time: %s]" % (epoch, io.py2_float(LB), time.time() - t_epoch))
        print("          [Lower bound on validation set: %s]" % io.py2_float(LBvalidation))
        if tracing:                                                # every line appears twice (VAEB.py:591-593)
            io.trace_line(trace_file, seen, LB, LBvalidation)
        done = epoch + 1
        if checkpoint_file and (done == args['n_epochs'] or (every > 0 and done % every == 0)):
            model.save_checkpoint(checkpoint_file, driver_state=loop_state(done, batch_order, trace_file))

    if len(save_file) > 0:
        model.save(save_file)

    # freyFace.py:346-369 renders the learned manifold after training: the decoder on a 10 x 10 grid of Gaussian
    # quantiles, tiled into one image (VAEBImage.multipleImages)
    if len(args.get('manifold_file', '')) > 0:
        from . import manifold
        _, tiled = manifold.render(model)
        manifold.save_pgm(tiled, args['manifold_file'])
    if len(args.get('sample_file', '')) > 0:
        from . import manifold
        _, tiled = manifold.render_samples(model)
        manifold.save_pgm(tiled, args['sample_file'])

    return model, data


def main(argv=None):
    args = parse_args(argv)
    print_args(args)
    if len(args['load_file']) == 0:
        model, data = train_model(args)
    else:
        data = None
        if args.get('synthetic', False):
            data = load_frey(synthetic=True) if args['continuous'] else load_mnist(synthetic=True)
        model, data = VAEB.load(args['load_file'], data=data, device=args['device'], precision=args['precision'],
                                eps_mode=args['eps_mode'])
    return model, data
