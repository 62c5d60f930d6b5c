"""What the reference computed, kept with the tests so that the parity checks run without it.

A parity test hands `Golden.check` the arrays it computed and a callable that asks the reference for the same thing.
With oracle/_ref present the reference runs, the arrays are compared with its result directly and the stored result
(if any) must equal it; with CFHD_RECORD_REF=1 the digest of the reference's result is written to
tests/golden/ref_digests.json instead.  Without oracle/_ref the arrays are compared with that stored digest, so a
checkout that only has the repository still checks every restated function bit for bit against what the reference
produced for the same seeded input.
"""
import atexit
import hashlib
import json
import os

import numpy as np

import oracle_lib as ol

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_digests.json")
RECORD = os.environ.get("CFHD_RECORD_REF") == "1"
_stored = None
_recorded = {}


def digest(arrays):
    """SHA-256 (first 16 hex digits) over dtype, shape and bytes of every array, in order."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape};".encode())
        h.update(a.tobytes())
    return h.hexdigest()[:16]


def _load():
    global _stored
    if _stored is None:
        _stored = json.load(open(PATH)) if os.path.exists(PATH) else {}
    return _stored


def _save():
    data = dict(_load())
    data.update(_recorded)
    with open(PATH, "w") as f:
        json.dump(dict(sorted(data.items())), f, indent=0)
        f.write("\n")


class Golden:
    """One test's checks against the reference; `request` is the pytest fixture of the test."""

    def __init__(self, request):
        self.id = request.node.nodeid.split("::", 1)[1]
        self.module = os.path.splitext(os.path.basename(request.node.fspath))[0]
        self.n = 0

    def _key(self):
        self.n += 1
        return f"{self.module}::{self.id}#{self.n - 1}"

    def _record(self, key, value):
        if not _recorded:
            atexit.register(_save)
        _recorded[key] = value

    def check_values(self, got, want_fn, msg=""):
        """Small exact results (lists of ints): stored as they are rather than as a digest."""
        key = self._key()
        got = json.loads(json.dumps(got))
        if ol.ref_available():
            want = json.loads(json.dumps(want_fn()))
            assert got == want, msg
            if RECORD:
                self._record(key, want)
            elif key in _load():
                assert _load()[key] == want, f"stored reference result {key} is stale: record it again"
            return
        stored = _load()
        assert key in stored, f"no stored reference result for {key} (record with CFHD_RECORD_REF=1 where oracle/_ref exists)"
        assert got == stored[key], f"{msg}: differs from the reference's stored result {key}"

    def check(self, got, want_fn, msg=""):
        """got: list of arrays; want_fn() -> the reference's list of arrays for the same input."""
        key = self._key()
        got = [np.asarray(g) for g in got]
        if ol.ref_available():
            want = [np.asarray(w) for w in want_fn()]
            assert len(got) == len(want)
            for k, (g, w) in enumerate(zip(got, want)):
                bad = np.argwhere(g != w) if g.shape == w.shape else None
                assert g.shape == w.shape and bad.size == 0, \
                    f"{msg} array {k}: " + (f"first mismatches {bad[:8].tolist()}" if bad is not None else f"shape {g.shape} vs {w.shape}")
            if RECORD:
                self._record(key, digest(want))
            elif key in _load():
                assert _load()[key] == digest(want), f"stored reference result {key} is stale: record it again"
            return
        stored = _load()
        assert key in stored, f"no stored reference result for {key} (record with CFHD_RECORD_REF=1 where oracle/_ref exists)"
        assert digest(got) == stored[key], f"{msg}: differs from the reference's stored result {key}"
