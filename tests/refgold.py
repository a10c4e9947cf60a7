"""What the reference's own code returned, for the tests that pin the oracle to it.

The reference library (oracle/_ref/libref.so: the reference's sources compiled unmodified against the cv:: shim, recipe oracle/Makefile)
can only be built where the reference tree is present. So every test that compares the oracle with it keeps what the reference returned
on the test's own seeded inputs in tests/golden/ref_<module>.npz, and compares the oracle with that file. Where libref.so is built,
  CSLAM_RECORD_REF=1 python -m pytest tests/test_oracle_ref.py tests/test_oracle_projection.py ...
runs the reference again, checks the oracle against the live result and rewrites the files.

`value` stores the reference's result itself (small results, and results the test feeds back into the oracle); `same` stores only a
SHA-256 digest of the result's shape, dtype and bytes (large bit-exact results), so that each file stays small."""
import hashlib
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RECORD = os.environ.get("CSLAM_RECORD_REF") == "1"


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(("%s%s|" % (a.dtype.str if a.dtype.names is None else a.dtype.descr, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


class RefGolden:
    def __init__(self, name):
        self.path = os.path.join(GOLD, "ref_%s.npz" % name)
        self.data = {}
        if RECORD:
            from oracle import ref
            if not ref.available():
                pytest.fail("CSLAM_RECORD_REF=1 needs oracle/_ref/libref.so")
        if os.path.exists(self.path):
            with np.load(self.path) as z:
                self.data = {k: z[k] for k in z.files}

    def value(self, key, fn):
        """The reference's result fn() (an array, a number or a tuple of them): computed and stored when recording, else read back."""
        if RECORD:
            v = fn()
            for i, a in enumerate(v if isinstance(v, tuple) else (v,)):
                self.data["%s#%d" % (key, i)] = np.asarray(a)
            return v
        parts = sorted((k for k in self.data if k.rsplit("#", 1)[0] == key), key=lambda k: int(k.rsplit("#", 1)[1]))
        if not parts:
            raise KeyError("%s has no reference result %r" % (self.path, key))
        v = tuple(self.data[k] for k in parts)
        return v if len(v) > 1 else v[0]

    def same(self, key, actual, fn):
        """True if `actual` (an array or a tuple of arrays) is bit-identical to the reference's result fn()."""
        actual = actual if isinstance(actual, tuple) else (actual,)
        if RECORD:
            v = fn()
            self.data[key] = np.array(digest(*(v if isinstance(v, tuple) else (v,))))
        if key not in self.data:
            raise KeyError("%s has no reference result %r" % (self.path, key))
        return digest(*actual) == str(self.data[key])

    def save(self):
        if RECORD:
            np.savez_compressed(self.path, **self.data)


@pytest.fixture(scope="module")
def gold(request):
    g = RefGolden(request.module.__name__.rsplit(".", 1)[-1].replace("test_", "", 1))
    yield g
    g.save()
