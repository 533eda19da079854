"""Committed digests of what the reference library computed, so that the parity tests also run where
oracle/_ref/libsvtav1_ref.so cannot be built (the reference sources are not part of this repository).

A test takes the `golden` fixture and passes every output it compares with the reference through
`golden.check(got, want)`.  Where the reference library is loaded, `want` is its live result and the two
are asserted equal; everywhere, `got` is folded into one SHA-256 per test.  At the end of the test that
digest (and the number of checks) must equal the entry of tests/golden/reference_digests.json, so where
the library is absent `got` is still compared with what the reference computed, through its digest.
Values are folded by value (integers as int64), not by container type.

Inputs a test takes from the reference library (small, JSON) go through `golden.value(compute)`.

To record: build the reference library (`python __graft_entry__.py --oracle` with the reference tree at
oracle/Makefile's REF) and run the tests with SVT_B200_RECORD_GOLDEN=<file>; each passing test writes
its entry there, to be merged into tests/golden/reference_digests.json."""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
RECORD_ENV = "SVT_B200_RECORD_GOLDEN"
_stored = None


def _load():
    global _stored
    if _stored is None:
        with open(PATH) as f:
            _stored = json.load(f)
    return _stored


def _canonical(x):
    if hasattr(x, "cpu"):  # torch tensor
        x = x.cpu().numpy()
    a = np.asarray(x)
    if a.dtype.kind in "biu":
        return a.astype(np.int64)
    if a.dtype.kind == "f":
        return a.astype(np.float64)
    return a


def _fold(h, x):
    if isinstance(x, (tuple, list)):
        h.update(b"[%d]" % len(x))
        for e in x:
            _fold(h, e)
        return
    a = np.ascontiguousarray(_canonical(x))
    h.update(repr(a.shape).encode())
    h.update(a.tobytes())


def equal(a, b):
    if isinstance(a, (tuple, list)) or isinstance(b, (tuple, list)):
        return len(a) == len(b) and all(equal(x, y) for x, y in zip(a, b))
    return np.array_equal(_canonical(a), _canonical(b))


class Golden:
    def __init__(self, key, live):
        self.key, self.live = key, live
        self.h, self.n, self.values = hashlib.sha256(), 0, []

    def check(self, got, want=None, *context):
        """got == want (want: the reference's result, None where the library is absent)"""
        if self.live:
            assert want is not None and equal(got, want), context
        _fold(self.h, got)
        self.n += 1

    def value(self, compute):
        """an input the test takes from the reference library: compute() where it is loaded, else the recorded value"""
        if self.live:
            v = json.loads(json.dumps(compute()))
        else:
            stored = _load().get(self.key, {}).get("values", [])
            assert len(self.values) < len(stored), "%s: no recorded reference value #%d in %s" % (self.key, len(self.values), PATH)
            v = stored[len(self.values)]
        self.values.append(v)
        return v

    def result(self):
        r = {"checks": self.n, "sha256": self.h.hexdigest()}
        if self.values:
            r["values"] = self.values
        return r

    def verify(self):
        r = self.result()
        out = os.environ.get(RECORD_ENV)
        if out and self.live:
            rec = json.load(open(out)) if os.path.exists(out) else {}
            rec[self.key] = r
            with open(out, "w") as f:
                json.dump(rec, f, indent=1, sort_keys=True)
            return
        want = _load().get(self.key)
        assert want is not None, "%s: no digest recorded in %s" % (self.key, PATH)
        assert r == want, ("%s: outputs differ from what the reference computed (%d checks folded, %d recorded); run the test where "
                           "oracle/_ref/libsvtav1_ref.so is built to see the first differing output" % (self.key, r["checks"], want["checks"]))
