"""Stored answers of the reference's own code (oracle/_ref/), so that the tests that pin the oracle and the
kernels to it run on any checkout.

The oracle/_ref/ libraries can only be compiled where the reference tree is present.  Every call the tests make
into them goes through `install()`: the call's inputs are hashed, and the answer recorded for exactly those inputs
is returned from tests/golden/ref_calls_*.npz (sharded to keep each file small).  A call whose inputs were never
recorded fails -- the comparison is never skipped.  Objects that keep state between calls (InterfaceAgglomeration) hash their whole call history.

Regenerate the store where oracle/_ref/ is built: `python tests/golden/make_ref_calls.py`.  It runs the tests that
use the reference with B200LDU_RECORD_REF=1, which calls the libraries and records every answer."""
import atexit
import hashlib
import json
import os

import numpy as np

SHARDS = 6
STORE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_calls_{}.npz")
RECORD = os.environ.get("B200LDU_RECORD_REF") == "1"

_index, _arrays = None, None        # replay: digest -> encoded answer, array name -> array
_rec_index, _rec_arrays = {}, {}    # record
_depth = [0]                        # calls made by a wrapped function itself are not recorded


def _feed(h, x):
    if x is None:
        h.update(b"N")
    elif isinstance(x, (bool, np.bool_)):
        h.update(b"b%d" % int(x))
    elif isinstance(x, (int, np.integer)):
        h.update(b"i%d" % int(x))
    elif isinstance(x, (float, np.floating)):
        h.update(b"f" + np.float64(x).tobytes())
    elif isinstance(x, str):
        h.update(b"s" + x.encode() + b"\0")
    elif isinstance(x, np.ndarray):
        a = np.ascontiguousarray(x)
        h.update(b"a" + a.dtype.str.encode() + repr(a.shape).encode())
        h.update(a.tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(b"l%d" % len(x))
        for v in x:
            _feed(h, v)
    elif isinstance(x, dict):
        h.update(b"d%d" % len(x))
        for k in sorted(x):
            _feed(h, k)
            _feed(h, x[k])
    else:
        raise TypeError(f"cannot hash an argument of type {type(x).__name__}")


def _digest(*parts):
    h = hashlib.sha256()
    _feed(h, parts)
    return h.hexdigest()[:32]


def _encode(x):
    if x is None or isinstance(x, (bool, str)):
        return {"v": x}
    if isinstance(x, int):
        return {"int": x}
    if isinstance(x, float):
        return {"float": x.hex()}
    if isinstance(x, np.generic):
        return {"np": x.dtype.str, "hex": x.tobytes().hex()}
    if isinstance(x, np.ndarray):
        name = "a_" + hashlib.sha256(x.dtype.str.encode() + repr(x.shape).encode() + np.ascontiguousarray(x).tobytes()).hexdigest()[:24]
        _rec_arrays[name] = x
        return {"array": name}
    if isinstance(x, (list, tuple)):
        return {"list" if isinstance(x, list) else "tuple": [_encode(v) for v in x]}
    if isinstance(x, dict):
        return {"dict": [[k, _encode(v)] for k, v in x.items()]}
    raise TypeError(f"cannot store a result of type {type(x).__name__}")


def _decode(e):
    if "v" in e:
        return e["v"]
    if "int" in e:
        return e["int"]
    if "float" in e:
        return float.fromhex(e["float"])
    if "np" in e:
        return np.frombuffer(bytes.fromhex(e["hex"]), dtype=e["np"])[0]
    if "array" in e:
        return _arrays[e["array"]].copy()
    if "list" in e:
        return [_decode(v) for v in e["list"]]
    if "tuple" in e:
        return tuple(_decode(v) for v in e["tuple"])
    return {k: _decode(v) for k, v in e["dict"]}


_ERRORS = {c.__name__: c for c in (RuntimeError, ValueError, NotImplementedError, AssertionError, TypeError)}


def _shard(key):
    return int(key[:2], 16) % SHARDS


def _load():
    global _index, _arrays
    if _index is None:
        index, arrays = {}, {}
        for s in range(SHARDS):
            with np.load(STORE.format(s)) as z:
                index.update(json.loads(str(z["index"])))
                arrays.update({k: z[k] for k in z.files if k != "index"})
        _index, _arrays = index, arrays
    return _index


def _call(name, key, live):
    """the answer of the reference for inputs `key`: live (and recorded) or replayed"""
    if not RECORD:
        e = _load().get(key)
        if e is None:
            raise AssertionError(f"{name}: no recorded answer of the reference for these inputs (digest {key}); "
                                 "regenerate tests/golden/ref_calls_*.npz with tests/golden/make_ref_calls.py")
        if "raise" in e:
            raise _ERRORS[e["raise"]](e["msg"])
        return _decode(e["ret"])
    if _depth[0]:
        return live()
    _depth[0] += 1
    try:
        out = live()
    except tuple(_ERRORS.values()) as ex:
        _rec_index[key] = {"fn": name, "raise": type(ex).__name__, "msg": str(ex)}
        raise
    finally:
        _depth[0] -= 1
    _rec_index[key] = {"fn": name, "ret": _encode(out)}
    return out


def _wrap_function(name, fn, live_when=None):
    def wrapped(*args, **kw):
        if live_when is not None and live_when(kw):
            return fn(*args, **kw)
        key = _digest(name, args, kw)
        out = _call(name, key, lambda: fn(*args, **kw))
        if RECORD:
            assert _digest(name, args, kw) == key, f"{name} changed its arguments: a replay would not see that"
        return out
    wrapped.__wrapped__ = fn
    wrapped.__doc__ = fn.__doc__
    return wrapped


def _wrap_class(name, cls, methods):
    """instances hash their constructor arguments and every call made on them so far"""
    class Replayed:
        def __init__(self, *args, **kw):
            self._state = _digest(name, args, kw)
            self._obj = cls(*args, **kw) if RECORD else None

    def method(m):
        def call(self, *args, **kw):
            self._state = _digest(self._state, m, args, kw)
            return _call(f"{name}.{m}", self._state, lambda: getattr(self._obj, m)(*args, **kw))
        return call
    for m in methods:
        setattr(Replayed, m, method(m))
    Replayed.__name__ = Replayed.__qualname__ = name
    Replayed.__doc__ = cls.__doc__
    return Replayed


REF_LDU_FUNCTIONS = ("interface_update", "pair_agglomerate", "solve", "gamg_solve_levels", "coarse_levels", "ldu_addressing",
                     "surface_integrate", "surface_integrate_vec", "gauss_gradf", "gauss_gradf_vec", "fvm",
                     "processor_interface_update", "fvm_fill", "euler_ddt", "interpolate_linear", "ldu_combine",
                     "fvm_assemble")


def install():
    """Route every entry point into the reference's compiled code through the store (idempotent)."""
    from oracle import limiters_oracle, mules_oracle, ref_ldu
    if getattr(ref_ldu, "_replay_installed", False):
        return
    for fn in REF_LDU_FUNCTIONS:
        # solve(binding=True) runs the product's own solvers behind the reference's tables: always live
        live_when = (lambda kw: kw.get("binding", False)) if fn == "solve" else None
        setattr(ref_ldu, fn, _wrap_function(f"ref_ldu.{fn}", getattr(ref_ldu, fn), live_when))
    ref_ldu.RefMatrix = _wrap_class("RefMatrix", ref_ldu.RefMatrix, ("op", "ainv", "jacobi"))
    ref_ldu.InterfaceAgglomeration = _wrap_class("InterfaceAgglomeration", ref_ldu.InterfaceAgglomeration,
                                                 ("agglomerate", "combine", "agglomerate_coeffs"))
    limiters_oracle.reference_limiter = _wrap_function("limiters_oracle.reference_limiter", limiters_oracle.reference_limiter)
    mules_oracle.reference = _wrap_function("mules_oracle.reference", mules_oracle.reference)
    ref_ldu._replay_installed = True
    if RECORD:
        atexit.register(_save)


def _arrays_of(e, out):
    if isinstance(e, dict):
        if "array" in e:
            out.add(e["array"])
        for v in e.values():
            _arrays_of(v, out)
    elif isinstance(e, list):
        for v in e:
            _arrays_of(v, out)
    return out


def _save():
    if not _rec_index:
        return
    for s in range(SHARDS):
        index = {k: e for k, e in _rec_index.items() if _shard(k) == s}
        names = set()
        for e in index.values():
            _arrays_of(e, names)
        np.savez_compressed(STORE.format(s), index=np.array(json.dumps(index, sort_keys=True, separators=(",", ":"))),
                            **{n: _rec_arrays[n] for n in sorted(names)})
    print(f"\nref_replay: {len(_rec_index)} calls, {len(_rec_arrays)} arrays -> {STORE.format('*')}")
