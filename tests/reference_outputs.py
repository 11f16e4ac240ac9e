"""The reference's own outputs for the exact inputs the tests give it, replayed from
tests/golden/reference_outputs.jsonl.  TEST INFRASTRUCTURE.

The reference (the original library's headers compiled on the Eigen-API shim into oracle/_ref) is not part of
this repository, so every call the tests make to it was run once and recorded.  A record is keyed by a digest of
the function's name and every argument, so a test whose inputs change finds no record and fails instead of
comparing against stale data.  A result of at most SMALL_BYTES is stored whole (tests may inspect it); a larger
one as the digest of each output array, which is all a bit-for-bit comparison needs: compare with `equal`.

The functions mirror oracle_binding's: with impl="oracle" they call the CPU oracle, with impl="ref" (or for the
ref_* functions) they return the recorded reference outputs.  To record them again where oracle/_ref is built:

    CNO_RECORD_REFERENCE=/tmp/ref.jsonl python -m pytest tests/test_oracle_pins.py tests/test_hz_oracle.py \\
        tests/test_al_oracle.py tests/test_lbfgsb.py tests/test_expressions_gpu.py      # (gpu-marked tests: on a GPU)
    sort -u /tmp/ref.jsonl > tests/golden/reference_outputs.jsonl

Recording runs each comparison against the live reference as well.
"""
import ctypes as C
import hashlib
import json
import os

import numpy as np

from oracle import oracle_binding as ob

STORE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.jsonl")
SMALL_BYTES = 256
RECORD = os.environ.get("CNO_RECORD_REFERENCE")
_records = None


class Digest(str):
    """SHA-256 (first 64 bits, hex) of an array's shape and bytes."""


def digest(a) -> Digest:
    if isinstance(a, Digest):
        return a
    a = np.ascontiguousarray(a)
    return Digest(hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()[:16])


def equal(a, b) -> bool:
    """Bit for bit: same shape, same bytes (of two arrays, or through the digest where one is stored as a digest)."""
    if isinstance(a, Digest) or isinstance(b, Digest):
        return digest(a) == digest(b)
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _canon(v):
    if isinstance(v, np.ndarray):
        return ["array", v.dtype.str, list(v.shape), hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest()]
    if isinstance(v, C.Structure):
        return [type(v).__name__] + [_canon(getattr(v, f)) for f, _ in v._fields_]
    if isinstance(v, (list, tuple)):
        return [_canon(e) for e in v]
    if isinstance(v, dict):
        return {k: _canon(e) for k, e in sorted(v.items())}
    if isinstance(v, (float, np.floating)):
        return float(v).hex()
    if isinstance(v, (bool, int, np.integer)):
        return int(v)
    if v is None or isinstance(v, str):
        return v
    raise TypeError(f"cannot key an argument of type {type(v).__name__}")


def _key(name, args, kwargs) -> str:
    text = json.dumps([name, _canon(list(args)), _canon(kwargs)])
    return hashlib.sha256(text.encode()).hexdigest()[:16]


# each function's result as named arrays, and back
def _as_arrays(name, r) -> dict:
    if name == "cstep":
        return {"io": np.array(r[0], np.float64), "flags": np.array(r[1:], np.int64)}
    if name == "hz_search_poly":
        return {"step": np.array(r[:3], np.float64), "nfev": np.array(r[3], np.int64)}
    if name == "condition_hessian":
        return {"value": r}
    if name == "ref_evaluate_expr":
        return {"value": r[0], "gradient": r[1]}
    return {k: v for k, v in r.items() if k != "seconds"}


def _from_arrays(name, r):
    if name == "cstep" and not isinstance(r["io"], Digest):
        return [float(v) for v in r["io"]], *(int(v) for v in r["flags"])
    if name == "hz_search_poly" and not isinstance(r["step"], Digest):
        return *(float(v) for v in r["step"]), int(r["nfev"])
    if name == "condition_hessian":
        return r["value"]
    if name == "ref_evaluate_expr":
        return r["value"], r["gradient"]
    return r


def stacked(name, results) -> dict:
    """The results of many calls of one function as arrays stacked along a new first axis (see `sweep`)."""
    arrays = [_as_arrays(name, r) for r in results]
    return {k: np.stack([a[k] for a in arrays]) for k in arrays[0]}


def _stored(arrays: dict) -> dict:
    if sum(a.nbytes for a in arrays.values()) <= SMALL_BYTES:
        return {k: [a.dtype.str, list(a.shape), a.tobytes().hex()] for k, a in arrays.items()}
    return {k: digest(a) for k, a in arrays.items()}


def _loaded(stored: dict) -> dict:
    return {k: Digest(v) if isinstance(v, str) else np.frombuffer(bytes.fromhex(v[2]), np.dtype(v[0])).reshape(v[1])
            for k, v in stored.items()}


def _lookup(key: str, name: str, run) -> dict:
    global _records
    if RECORD:
        if not ob.ref_available():
            raise RuntimeError("CNO_RECORD_REFERENCE is set but oracle/_ref is not built")
        out = _stored(run())
        with open(RECORD, "a") as f:
            f.write(json.dumps({"key": key, "fn": name, "out": out}, sort_keys=True) + "\n")
        return _loaded(out)
    if _records is None:
        with open(STORE) as f:
            _records = {r["key"]: r["out"] for r in map(json.loads, f)}
    if key not in _records:
        raise KeyError(f"no recorded reference output of {name} for these inputs (key {key}); "
                       "record it again as this module's docstring says")
    return _loaded(_records[key])


def _reference(name, *args, **kwargs):
    key = _key(name, args, kwargs)
    fn = getattr(ob, name)
    run = (lambda: _as_arrays(name, fn(*args, **kwargs))) if name.startswith("ref_") else \
        (lambda: _as_arrays(name, fn(*args, impl="ref", **kwargs)))
    return _from_arrays(name, _lookup(key, name, run))


def sweep(name, calls) -> dict:
    """The reference's results of many small calls of one function, `calls` = [(args, kwargs), ...], stacked as
    `stacked` stacks them: one record for the whole sweep."""
    key = _key(name + "/sweep", calls, {})
    fn = getattr(ob, name)
    return _lookup(key, name, lambda: stacked(name, [fn(*a, impl="ref", **k) for a, k in calls]))


def _oracle_or_reference(name):
    def call(*args, impl="oracle", **kwargs):
        if impl == "oracle":
            return getattr(ob, name)(*args, **kwargs)
        assert impl == "ref", impl
        return _reference(name, *args, **kwargs)
    call.__name__ = name
    call.__doc__ = f"oracle_binding.{name} (impl='oracle') or the recorded reference outputs (impl='ref')."
    return call


minimize = _oracle_or_reference("minimize")
al_minimize = _oracle_or_reference("al_minimize")
condition_hessian = _oracle_or_reference("condition_hessian")
cstep = _oracle_or_reference("cstep")


def hz_search_poly(coef, x0, alpha_init, impl="oracle"):
    return _oracle_or_reference("hz_search_poly")(coef, x0, alpha_init, impl=impl)


def ref_minimize_expr(*args, **kwargs):
    return _reference("ref_minimize_expr", *args, **kwargs)


def ref_evaluate_expr(*args, **kwargs):
    return _reference("ref_evaluate_expr", *args, **kwargs)


def ref_lbfgsb_minimize(*args, **kwargs):
    return _reference("ref_lbfgsb_minimize", *args, **kwargs)
