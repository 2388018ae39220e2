"""TEST INFRASTRUCTURE ONLY -- stored results of the reference's own code.

Tests that compare this project with the reference (its compiled operators, its Python front-end,
its headers and sources) read what the reference returned from tests/golden/reference_records.json,
so they run on any machine. An entry maps a test's key to a JSON value: plain numbers and strings,
and arrays as ``digest(a)`` (SHA-256 of dtype, shape and bytes), so the comparison stays bit for bit
while the file stays small (a digest is the first 128 bits of the SHA-256 hex string).

    B200KV_RECORD_REFERENCE=1 python -m pytest tests -m "not gpu"

re-runs the reference (oracle/_ref/libmxref.so built by `make -C oracle ref`, and the source tree it
was built from, or B200KV_REFERENCE_TREE) for every key the tests ask for and rewrites the file when
the session ends.
"""
import atexit
import hashlib
import json
import os

import numpy as np

import kvoracle as K

PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                    "reference_records.json")
_store = None


def recording():
    return os.environ.get("B200KV_RECORD_REFERENCE") == "1"


def digest(a):
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.view(np.uint8).tobytes())
    return h.hexdigest()[:32]


def digest_json(v):
    """SHA-256 of a JSON-able value (nested lists of ints, strings, ...)"""
    return hashlib.sha256(json.dumps(v, sort_keys=True).encode()).hexdigest()[:32]


def _load():
    global _store
    if _store is None:
        _store = {}
        if os.path.exists(PATH):
            with open(PATH) as f:
                _store = json.load(f)
        if recording():
            atexit.register(_save)
    return _store


def _save():
    with open(PATH, "w") as f:
        json.dump(_store, f, indent=0, sort_keys=True)
        f.write("\n")


def tree():
    """the reference's source tree (kvoracle.reference_tree), for records read from its sources"""
    t = K.reference_tree()
    assert t, "recording needs the reference tree: the one oracle/_ref was built from " \
        "(make -C oracle ref REF=<reference checkout>) or B200KV_REFERENCE_TREE=<reference checkout>"
    return t


class _Ops(object):
    """oracle/_ref/libmxref.so, checked when a record first uses it"""

    def __getattr__(self, name):
        r = K.ref()
        assert r is not None and r.has_ops(), "recording needs oracle/_ref/libmxref.so (make -C oracle ref)"
        return getattr(r, name)


def reference(key, compute):
    """What the reference returned for `key`. Recording: compute(ops) runs the reference's own code
    (ops: its compiled operators, oracle/_ref) and its JSON-able result is stored; otherwise the
    stored result is returned."""
    store = _load()
    if recording():
        store[key] = json.loads(json.dumps(compute(_Ops())))
    assert key in store, "no stored reference result for %r (see oracle/refrecord.py)" % key
    return store[key]
