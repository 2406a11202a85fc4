"""Pinned outputs of the reference (the original project's own code) for the tests that compare against it.

Those tests run the reference where it can be built: its shaders compiled for the host (oracle/refshader), its vendored
meshoptimizer and glm (oracle/refscene).  Every reference output such a test compares against is reduced to an
order-independent array and pinned as a SHA-256 digest, in the order the test produces them, under the test's name in
tests/golden/reference_pins.json.  Where the reference cannot run, the test digests the project-side value it asserts equal
to the reference's and that digest must match the pin: the comparison stays bit for bit without the reference.

With the reference present the pins are checked against its live outputs.  To re-record them run the tests with
NIAGARA_RECORD_PINS=<json file> (tests/golden/reference_pins.json to update the committed file); entries of the tests that
ran are replaced, the others are kept.

A mismatch names the test, the output and its index in the test's sequence, but a digest carries no values.  To see what
differs, run the failing test where the reference is present: it then compares against the reference's live outputs and
reports the values.  With NIAGARA_RECORD_PINS pointing at a scratch file there, the digests it records show which outputs
changed against the committed ones."""
import contextlib
import hashlib
import json
import os

import numpy as np

PINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.json")
_loaded = None
current = None


def digest(*arrays):
    """SHA-256 (first 64 bits) of dtypes, shapes and bytes; every NaN counts as the same NaN."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        if a.dtype.kind == "f":
            a = np.where(np.isnan(a), np.array(np.nan, a.dtype), a)
        h.update(repr((a.dtype.descr, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()[:16]


def _pins():
    global _loaded
    if _loaded is None:
        _loaded = json.load(open(PINS)) if os.path.exists(PINS) else {}
    return _loaded


class Pins:
    def __init__(self, test, live):
        self.test, self.live = test, live
        self.record_to = os.environ.get("NIAGARA_RECORD_PINS") if live else None
        self.want = _pins().get(test)
        self.got = []
        if not self.record_to:
            assert self.want is not None, "no reference outputs pinned for %s (record them where the reference is present)" % test

    def check(self, what, *arrays):
        """Pins (recording) or checks the digest of the next compared output; `what` names it in a failure."""
        d = digest(*arrays)
        i = len(self.got)
        self.got.append(d)
        if not self.record_to:
            assert i < len(self.want), ("more outputs than the reference produced", self.test, i, what)
            assert d == self.want[i], ("differs from the reference's output", self.test, i, what)

    def close(self):
        if self.record_to:
            pins = json.load(open(self.record_to)) if os.path.exists(self.record_to) else {}
            pins[self.test] = self.got
            with open(self.record_to, "w") as f:
                json.dump(pins, f, indent=0, sort_keys=True)
                f.write("\n")
        else:
            assert len(self.got) == len(self.want), ("fewer outputs than the reference produced", self.test, len(self.got), len(self.want))


@contextlib.contextmanager
def pinned(request, live):
    """Pins of the running test (pytest's `request`); live: the reference itself runs in this test."""
    global current
    failed = request.session.testsfailed
    current = Pins("%s::%s" % (request.node.module.__name__, request.node.name), live)
    try:
        yield current
        if request.session.testsfailed == failed:  # (a failed test never produced the rest of its outputs)
            current.close()
    finally:
        current = None


def check(what, *arrays):
    """Pins or checks an output of the running test; outside a pinned test (the reference itself runs) there is nothing to do."""
    if current is not None:
        current.check(what, *arrays)
