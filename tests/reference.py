"""What the unmodified reference (oracle/_ref) answered, kept as SHA-256 digests in tests/golden/reference_digests.json.

The compiled reference exists only where its sources do, so the tests that compare with it compare with these digests
instead.  ``expect(got, call)``: ``call(lib)`` runs the operator on any qnnpack.h implementation and returns its output;
``got`` must be byte for byte what the reference returned for the same call.  An entry is keyed by a digest of the whole
call (operation names, create / setup arguments, every input byte), so an input that drifts fails as a missing entry
instead of comparing against the wrong answer.  ``tests/golden/make_golden.py`` records the table from oracle/_ref.
"""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")

# make_golden.py sets this to the compiled reference to record new digests instead of checking them
RECORD_WITH = None
_table = None


class _CallKey:
    """Stands in for a library: hashes every call and argument it receives instead of running anything."""

    def __init__(self):
        self.h = hashlib.sha256()

    def _feed(self, v):
        if isinstance(v, np.ndarray):
            self.h.update(f"nd{v.dtype.str}{v.shape}".encode())
            self.h.update(np.ascontiguousarray(v).tobytes())
        elif isinstance(v, (tuple, list)):
            self.h.update(f"seq{len(v)}".encode())
            for e in v:
                self._feed(e)
        elif isinstance(v, dict):
            self._feed(sorted(v.items()))
        elif isinstance(v, (bool, np.bool_)):
            self.h.update(f"b{bool(v)}".encode())
        elif isinstance(v, (int, np.integer)):
            self.h.update(f"i{int(v)}".encode())
        elif isinstance(v, (float, np.floating)):
            self.h.update(f"f{float(v)!r}".encode())
        elif v is None or isinstance(v, str):
            self.h.update(f"s{v}".encode())
        else:
            raise TypeError(f"cannot key an argument of type {type(v).__name__}")

    def __getattr__(self, name):
        def call(*args, **kw):
            self._feed((name, args, kw))
            return (0, None) if name.startswith("create") else 0
        return call


def _digest(out) -> str:
    h = hashlib.sha256()
    for a in (out if isinstance(out, (tuple, list)) else [out]):
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def _load():
    global _table
    if _table is None:
        with open(PATH) as f:
            _table = json.load(f)
    return _table


def expect(got, call, what: str = ""):
    """got: uint8 array (or a list of them); call(lib) -> the same from the library ``lib``."""
    k = _CallKey()
    call(k)
    key = k.h.hexdigest()[:32]
    if RECORD_WITH is not None:
        want = call(RECORD_WITH)
        _load()[key] = _digest(want)
        assert _digest(got) == _table[key], f"{what}: differs from the compiled reference"
        return
    table = _load()
    assert key in table, f"{what}: no reference output recorded for this call (inputs or arguments changed?)"
    assert _digest(got) == table[key], f"{what}: differs from the reference output recorded for this call"


def save():
    with open(PATH, "w") as f:
        json.dump(dict(sorted(_load().items())), f, indent=0)
        f.write("\n")
