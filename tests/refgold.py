"""Outputs of the reference's own routines (translated Fortran -> C, oracle/_ref) for the tests that compare with them.

The translated library can only be built where the reference's source lies.  So that the comparisons hold on every
checkout, the SHA-256 digest of every reference array a test compares with is recorded in
tests/golden/reference_digests.json, keyed by the test and the order of its comparisons:

  * where the library is present, the tests run it as before, and each reference array must also match its digest;
  * where it is absent, the reference calls are not made and the project's own value must match the digest, i.e. be
    the reference's value bit for bit.  Tests that then compare with a tolerance (the CUDA path) use that value.

Digests are taken of the float64 values in C order with -0.0 folded into 0.0 (np.array_equal does not tell them
apart).  To record them, run the tests where the library is present with ADFB_RECORD_REFERENCE=<path of the json>,
in one process (the entries of the tests run are merged into that file when it exits).  The CUDA tests record theirs
where a GPU is present.
"""
import atexit
import hashlib
import json
import os

import numpy as np

from oracle import refblockette as rb

AVAILABLE = rb.available()
PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
RECORD = os.environ.get("ADFB_RECORD_REFERENCE")

_digests = json.load(open(PATH)) if os.path.exists(PATH) else {}
_recorded = {}
_seen = {"test": None, "n": 0}


def digest(a):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64)) + 0.0
    return "%s:%s" % ("x".join(map(str, a.shape)), hashlib.sha256(a.tobytes()).hexdigest()[:32])


def _key():
    """test id without its directory, and the index of this comparison inside the test"""
    test = os.environ["PYTEST_CURRENT_TEST"].rsplit(" (", 1)[0].rsplit("/", 1)[-1]
    if _seen["test"] != test:
        _seen["test"], _seen["n"] = test, 0
    _seen["n"] += 1
    return test, _seen["n"] - 1


def run(fn):
    """fn() -- calls into the translated reference -- where the library is present; else None"""
    return fn() if AVAILABLE else None


def value(what, ref, pick, mine):
    """The reference's array `pick(ref)` (`ref`: what run() returned).  Where the reference is absent, the project's
    value `mine` (an array or a callable returning one) once its digest equals the one recorded for this comparison."""
    test, n = _key()
    if AVAILABLE:
        v = np.asarray(pick(ref))
        if RECORD:
            _recorded.setdefault(test, []).append([what, digest(v)])
            return v
    else:
        v = np.asarray(mine() if callable(mine) else mine)
    rec = _digests.get(test)
    assert rec is not None and n < len(rec), "no recorded reference output for %s #%d (%s)" % (test, n, what)
    assert rec[n][0] == what, "recorded reference output %s #%d is %r, not %r" % (test, n, rec[n][0], what)
    assert digest(v) == rec[n][1], "%s: %s differs from the reference's output (recorded digest)" % (test, what)
    return v


def same(what, ref, pick, mine):
    """assert that `mine` equals the reference's array `pick(ref)` bit for bit"""
    v = value(what, ref, pick, mine)
    mine = np.asarray(mine)
    assert np.array_equal(v, mine), "%s differs: max abs %.3e" % (what, np.abs(v - mine).max())


@atexit.register
def _write():
    if RECORD and _recorded:
        out = json.load(open(RECORD)) if os.path.exists(RECORD) else {}
        out.update(_recorded)
        with open(RECORD, "w") as f:   # one test per line
            f.write("{\n%s\n}\n" % ",\n".join("%s: %s" % (json.dumps(k), json.dumps(out[k], separators=(",", ":")))
                                             for k in sorted(out)))
