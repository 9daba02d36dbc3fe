"""Recorded outputs of the reference's own CPU code, for the tests that pin the C restatement on it.

The reference (oracle/_ref/libtfluids_ref.so, compiled from the reference's sources by oracle/Makefile) is not
part of this repository, so those tests compare the oracle with what the reference computed for the same seeded
inputs, stored under tests/golden/:

  reference_outputs.json  bit-exact comparisons: a SHA-256 of each output's dtype, shape and bytes
  reference_outputs.npz   comparisons within a float tolerance: the outputs themselves

With the reference built, `TFL_RECORD_REFERENCE=1 python -m pytest tests/<module>.py` computes the outputs of
the tests it runs with oracle.Reference as well, checks the oracle against them and rewrites their records.
"""
import hashlib
import json
import os

import numpy as np

import oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DIGESTS = os.path.join(GOLD, "reference_outputs.json")
ARRAYS = os.path.join(GOLD, "reference_outputs.npz")
RECORD = os.environ.get("TFL_RECORD_REFERENCE") == "1"


def digest(a):
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()[:32]


class _Store:
    def __init__(self):
        self.digests = json.load(open(DIGESTS)) if os.path.exists(DIGESTS) else {}
        self.arrays = dict(np.load(ARRAYS)) if os.path.exists(ARRAYS) else {}

    def save(self):
        with open(DIGESTS, "w") as f:
            json.dump(self.digests, f, indent=0, sort_keys=True)
            f.write("\n")
        np.savez_compressed(ARRAYS, **self.arrays)


_store = None
_reference = None


class RecordedReference:
    """The reference's side of one test: `check(orc, run)` compares run(orc) with the recorded run(reference)."""

    def __init__(self, test_id):
        global _store
        if _store is None:
            _store = _Store()
        self.test_id = test_id

    def check(self, orc, run, tol=None):
        """run(be) -> {name: array}, the outputs of the operators under test on backend `be`.  Each output of
        the oracle must equal the reference's bit for bit, or, for a name in `tol`, lie within
        tol[name] * max|reference output| of it."""
        global _reference
        tol = tol or {}
        got = run(orc)
        if RECORD:
            if _reference is None:
                _reference = oracle.Reference()
            for name, want in run(_reference).items():
                key = "%s::%s" % (self.test_id, name)
                if name in tol:
                    _store.arrays[key] = np.ascontiguousarray(want)
                else:
                    _store.digests[key] = digest(want)
            _store.save()
        for name, a in got.items():
            key = "%s::%s" % (self.test_id, name)
            if name in tol:
                assert key in _store.arrays, "no recorded reference output for " + key
                want = _store.arrays[key]
                assert a.shape == want.shape, key
                err = np.abs(a.astype(np.float64) - want).max()
                assert err <= tol[name] * np.abs(want).max(), "%s: max|diff| = %g" % (key, err)
            else:
                assert key in _store.digests, "no recorded reference output for " + key
                assert digest(a) == _store.digests[key], "%s differs from the reference's output" % key
