"""What the unmodified reference computed, for the tests that compare against it.

The reference is not part of this repository, so its outputs on each such test's seeded inputs are kept as md5
digests in tests/golden/reference_md5.json, keyed by test and check.  A test hashes what it computed and compares
that with the stored digest; equal digests mean bit-identical outputs.

To regenerate the digests, build the reference under oracle/_ref (`make -C oracle ref`) and run the tests with
SPM_RECORD_REFERENCE=<file.json>: each check then runs the reference on the same input, asserts that the test's
output equals it, and writes the reference's digest to that file, to be merged into tests/golden/reference_md5.json.
"""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_md5.json")
RECORD = os.environ.get("SPM_RECORD_REFERENCE")
_golden = None


def md5(*arrays):
    """Digest of a sequence of arrays (or bytes) by value: integer arrays hash alike whatever their width."""
    h = hashlib.md5()
    for a in arrays:
        a = np.frombuffer(a, np.uint8) if isinstance(a, (bytes, bytearray)) else np.asarray(a)
        if a.dtype.kind in "iu":
            a = a.astype(np.int64)
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


class Reference:
    def __init__(self, request):
        self.test = f"{request.module.__name__}::{request.node.name}"

    def check(self, what, ours, reference):
        """Asserts that `ours` (a tuple of arrays) is what the reference computed for check `what` of this test.
        `reference` computes the reference's own tuple; it is called only when recording."""
        key = f"{self.test}::{what}"
        got = md5(*ours)
        if RECORD:
            want = md5(*reference())
            rec = json.load(open(RECORD)) if os.path.exists(RECORD) else {}
            rec[key] = want
            with open(RECORD, "w") as f:
                json.dump(rec, f, indent=0, sort_keys=True)
        else:
            global _golden
            if _golden is None:
                with open(GOLDEN) as f:
                    _golden = json.load(f)
            assert key in _golden, f"{key}: no recorded output of the reference"
            want = _golden[key]
        assert got == want, f"{key}: differs from the reference's output"
