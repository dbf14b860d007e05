"""The training-state file of `VAEB.save_checkpoint` / `VAEB.resume`: one `.npz` written with `np.savez` and read with
`np.load(allow_pickle=False)` -- no pickle, unlike the reference's `.mdl`.

Entries:
  header                 a JSON string: format version, vaeb_version(), the constructor arguments, the tensor names and
                         shapes, the world size, the data fingerprint of every rank and the names of every array below;
  <buffer>.<tensor>      the state buffers of include/vaeb_b200.h "The training state of a handle", float32
                         (buffer: params, ada, ada2, vmu, vsig, ada_mu, ada_sig);
  counter.<name>         the Philox step counter (uint32), adam_step and kl_step (int64), 0-d;
  rng.<name>.keys/.aux   host RandomState states (eps_mode='theano': the seed generator and every node of RandomStreams);
  driver.<name>          the arrays of an optional driver_state dict (its scalars go into the header).

A file is written to a temporary name in its directory and moved over the target with os.replace, so a job killed
mid-write leaves the previous checkpoint intact.  This module is numpy only; the model side is in model.py."""
from __future__ import annotations

import hashlib
import json
import os
import tempfile

import numpy as np

FORMAT_VERSION = 1


def data_fingerprint(x):
    """{'N', 'D', 'sha256'} of the float32 rows a model trains on."""
    xa = np.ascontiguousarray(x, dtype=np.float32)
    return {"N": int(xa.shape[0]), "D": int(xa.shape[1]), "sha256": hashlib.sha256(xa.data).hexdigest()}


def random_state_arrays(state):
    """(keys, aux) arrays of a RandomState.get_state() tuple: the 624 MT19937 words, and [pos, has_gauss,
    cached_gaussian] as float64 (all three exact there)."""
    name, keys, pos, has_gauss, cached = state
    if name != "MT19937":
        raise ValueError("unsupported bit generator %r" % (name,))
    return np.asarray(keys, dtype=np.uint32).copy(), np.array([pos, has_gauss, cached], dtype=np.float64)


def random_state_tuple(keys, aux):
    """Inverse of random_state_arrays: a tuple RandomState.set_state() accepts."""
    return ("MT19937", np.asarray(keys, dtype=np.uint32), int(aux[0]), int(aux[1]), float(aux[2]))


def pack_random_state(arrays, name, state):
    keys, aux = random_state_arrays(state)
    arrays["rng.%s.keys" % name] = keys
    arrays["rng.%s.aux" % name] = aux


def unpack_random_state(arrays, name):
    return random_state_tuple(require(arrays, "rng.%s.keys" % name), require(arrays, "rng.%s.aux" % name))


def _json_scalar(v):
    if isinstance(v, (bool, np.bool_)):
        return bool(v)
    if isinstance(v, (int, np.integer)):
        return int(v)
    if isinstance(v, (float, np.floating)):
        return float(v)
    if isinstance(v, str):
        return v
    raise TypeError("driver_state scalar %r is not a bool, int, float or str" % (v,))


def _file_mode(path):
    """The permission bits of the file being replaced, else those a new file gets under the process umask."""
    try:
        return os.stat(path).st_mode & 0o777
    except FileNotFoundError:
        umask = os.umask(0)
        os.umask(umask)
        return 0o666 & ~umask


def write(path, header, arrays, driver_state=None):
    """Write `header` (a JSON-able dict), `arrays` (name -> ndarray) and `driver_state` (name -> ndarray or scalar)
    to `path` atomically.  The header gains 'format_version', 'arrays' (name -> shape of every array stored) and
    'driver_scalars'."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    scalars = {}
    for k, v in (driver_state or {}).items():
        if isinstance(v, np.ndarray):
            arrays["driver." + k] = v
        else:
            scalars[k] = _json_scalar(v)
    for k, v in arrays.items():
        if v.dtype == object:
            raise TypeError("array %r has dtype object: it would need pickle" % k)
    header = dict(header, format_version=FORMAT_VERSION, driver_scalars=scalars,
                  arrays={k: list(v.shape) for k, v in arrays.items()})
    directory = os.path.dirname(os.path.abspath(path))
    fd, tmp = tempfile.mkstemp(prefix="." + os.path.basename(path) + ".", suffix=".tmp", dir=directory)
    try:
        with os.fdopen(fd, "wb") as f:
            np.savez(f, header=np.array(json.dumps(header, sort_keys=True)), **arrays)
            f.flush()
            os.fsync(f.fileno())
        os.chmod(tmp, _file_mode(path))               # mkstemp creates 0600; keep what a plain open() would give
        os.replace(tmp, path)
    except BaseException:
        try:
            os.unlink(tmp)
        except OSError:
            pass
        raise


def read(path):
    """(header, arrays, driver_state) of a checkpoint file.  ValueError on an unknown format version or on an array
    the header lists that is missing or has another shape."""
    with np.load(path, allow_pickle=False) as z:
        if "header" not in z.files:
            raise ValueError("%s: no header: not a checkpoint file" % path)
        header = json.loads(str(z["header"][()]))
        version = header.get("format_version")
        if version != FORMAT_VERSION:
            raise ValueError("%s: format_version %r, this library reads %d" % (path, version, FORMAT_VERSION))
        arrays = {}
        for name, shape in header["arrays"].items():
            if name not in z.files:
                raise ValueError("%s: array %r is missing" % (path, name))
            a = z[name]
            if list(a.shape) != list(shape):
                raise ValueError("%s: array %r has shape %s, the header says %s" % (path, name, list(a.shape), shape))
            arrays[name] = a
    driver = {k[len("driver."):]: v for k, v in arrays.items() if k.startswith("driver.")}
    driver.update(header.get("driver_scalars", {}))
    arrays = {k: v for k, v in arrays.items() if not k.startswith("driver.")}
    return header, arrays, driver


def require(arrays, name, shape=None):
    """arrays[name], or ValueError naming the array when it is missing or its shape is not `shape`."""
    if name not in arrays:
        raise ValueError("checkpoint array %r is missing" % name)
    a = arrays[name]
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("checkpoint array %r has shape %s, the model needs %s" % (name, tuple(a.shape), tuple(shape)))
    return a


def check_compatible(header, *, data, rank, world_size):
    """ValueError naming the field when the resuming side differs from the saved run: another world size, or rows
    (`data`, the fingerprint of this rank's rows) other than the saved run's."""
    if int(header["world_size"]) != int(world_size):
        raise ValueError("checkpoint world_size: saved with %d ranks, resuming with %d" % (header["world_size"], world_size))
    saved = header["data"][rank]
    for key in ("N", "D", "sha256"):
        if saved[key] != data[key]:
            raise ValueError("checkpoint data fingerprint (rank %d): %s is %r in the file, %r here"
                             % (rank, key, saved[key], data[key]))


def check_tensors(header, tensors):
    """ValueError naming the tensor when `tensors` [(name, shape)] of the model built from the saved constructor
    arguments differ from the saved ones."""
    saved_t = [(n, tuple(s)) for n, s in header["tensors"]]
    here_t = [(n, tuple(s)) for n, s in tensors]
    if len(saved_t) != len(here_t):
        raise ValueError("checkpoint tensors: %d in the file, %d in the model" % (len(saved_t), len(here_t)))
    for (n0, s0), (n1, s1) in zip(saved_t, here_t):
        if n0 != n1 or s0 != s1:
            raise ValueError("checkpoint tensor shape: %s%s in the file, %s%s in the model" % (n0, s0, n1, s1))
