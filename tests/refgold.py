"""The reference's own outputs (oracle/_ref), kept as digests in tests/golden/ref_digests.json.

oracle/_ref is built from the reference's sources and exists only where those sources are at hand.  The tests that
compare with it take a `ref` fixture instead of calling it directly:

    ref.check(got, lambda: pyref.RefImage.from_array(a).resize(0.5).numpy())

Where oracle/_ref is built, check() runs the reference, requires `got` to equal its output (same shape and format,
equal values, NaN equal to NaN) and requires the stored digest of that output to be current.  Elsewhere `got` must
hash to the stored digest, which holds the same comparison.  Digests are kept per test in call order.

    VB200_RECORD_REF=1 python -m pytest tests/...     (with oracle/_ref built)

rewrites the stored digests of the tests that run.
"""
import atexit
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import pyref

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_digests.json")
LIVE = pyref.available()
RECORD = os.environ.get("VB200_RECORD_REF") == "1"
with open(PATH) as f:
    STORED = json.load(f)
_RECORDED = {}


def digest(a):
    """16 hex digits of SHA-256 over format, shape and values; -0.0 hashes as 0.0 and every NaN alike, as
    np.array_equal(equal_nan=True) compares them"""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)
        a[np.isnan(a)] = np.nan
    h = hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()[:16]


def _save():
    stored = dict(STORED)
    stored.update(_RECORDED)
    with open(PATH, "w") as f:
        json.dump(stored, f, indent=0, sort_keys=True)
        f.write("\n")


class Reference:
    def __init__(self, key):
        self.key = key
        self.n = 0

    def check(self, got, run_reference, msg=None):
        got = np.asarray(got)
        i = self.n
        self.n += 1
        if LIVE:
            want = np.asarray(run_reference())
            assert got.shape == want.shape and got.dtype == want.dtype, (msg, got.shape, want.shape, got.dtype, want.dtype)
            assert np.array_equal(got, want, equal_nan=got.dtype.kind == "f"), \
                (msg, "max diff %g" % np.nanmax(np.abs(got.astype(np.float64) - want.astype(np.float64))))
            if RECORD:
                if not _RECORDED:
                    atexit.register(_save)
                _RECORDED.setdefault(self.key, []).append(digest(want))
                return
            stored = STORED.get(self.key, [])
            assert i < len(stored) and stored[i] == digest(want), \
                "%s: stored digest #%d of the reference's output is stale (re-record with VB200_RECORD_REF=1)" % (self.key, i)
            return
        stored = STORED.get(self.key, [])
        assert i < len(stored), "%s: no stored digest #%d of the reference's output" % (self.key, i)
        assert digest(got) == stored[i], (msg, "differs from the reference's output (stored digest #%d, %s %s)"
                                          % (i, got.dtype, got.shape))


@pytest.fixture
def ref(request):
    """Reference outputs of the running test, live or from the stored digests."""
    return Reference("%s::%s" % (request.node.path.stem, request.node.name))
