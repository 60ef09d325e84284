"""Stored outputs of the reference's own code, so that the tests that compare against it run on any machine.

`reference(name, inputs, run)` returns run()'s result where the reference can be run here (`run` is not None: the
binaries built from the reference tree into oracle/_ref, or the tree itself); with SNIPER_RECORD_GOLDEN=1 it also stores
that result under tests/golden/ref_calls/.  Elsewhere (`run` is None) it returns the stored result.  A result is keyed
by `name` and a digest of `inputs` (every array, scalar and string the reference is given), so a test whose inputs
drift from the recorded ones finds nothing stored and fails instead of comparing against the wrong vectors.

Results are arrays, scalars, or lists / tuples / dicts of them.  Regenerate after changing a test's inputs, where the
reference is built:
    SNIPER_RECORD_GOLDEN=1 python -m pytest tests/test_host_cpu.py tests/test_iterator_cpu.py"""
import atexit
import hashlib
import os

import numpy as np
import pytest

DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_calls")
RECORD = os.environ.get("SNIPER_RECORD_GOLDEN") == "1"
_loaded = {}
_new = {}


def _digest(h, x):
    if isinstance(x, dict):
        for k in sorted(x):
            h.update(repr(k).encode())
            _digest(h, x[k])
    elif isinstance(x, (list, tuple)):
        h.update(b"[%d" % len(x))
        for v in x:
            _digest(h, v)
    elif hasattr(x, "detach"):                                          # torch tensor
        _digest(h, x.detach().cpu().numpy())
    elif isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x)
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    else:
        h.update(repr(x).encode())


def _encode(prefix, x, out):
    if isinstance(x, dict):
        out[prefix + "#dict"] = np.array(sorted(x), dtype=str)
        for k in x:
            _encode(prefix + "/" + k, x[k], out)
    elif isinstance(x, (list, tuple)):
        out[prefix + ("#list" if isinstance(x, list) else "#tuple")] = np.int64(len(x))
        for i, v in enumerate(x):
            _encode(prefix + "/%d" % i, v, out)
    else:
        out[prefix] = np.asarray(x.detach().cpu().numpy() if hasattr(x, "detach") else x)


def _decode(prefix, z):
    if prefix + "#dict" in z:
        return {str(k): _decode(prefix + "/" + str(k), z) for k in z[prefix + "#dict"]}
    for kind, ctor in (("#list", list), ("#tuple", tuple)):
        if prefix + kind in z:
            return ctor(_decode(prefix + "/%d" % i, z) for i in range(int(z[prefix + kind])))
    a = z[prefix]
    return a[()] if a.ndim == 0 else a


def _file(name):
    return os.path.join(DIR, name.split(".")[0] + ".npz")


def _stored(name):
    f = _file(name)
    if f not in _loaded:
        _loaded[f] = dict(np.load(f)) if os.path.exists(f) else {}
    return _loaded[f]


def _save():
    for f, entries in _new.items():
        old = dict(np.load(f)) if os.path.exists(f) else {}
        old.update(entries)
        os.makedirs(DIR, exist_ok=True)
        np.savez_compressed(f, **old)


atexit.register(_save)


def reference(name, inputs, run=None):
    h = hashlib.sha256()
    _digest(h, inputs)
    key = "%s-%s" % (name, h.hexdigest()[:20])
    if run is not None:
        res = run()
        if RECORD:
            _encode(key, res, _new.setdefault(_file(name), {}))
        return res
    z = _stored(name)
    if not any(k == key or k.startswith(key + "#") for k in z):
        pytest.fail("no stored reference output for %s (%s): record it where the reference is built" % (key, _file(name)))
    return _decode(key, z)
