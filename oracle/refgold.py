"""TEST INFRASTRUCTURE ONLY: stored results the parity tests and __graft_entry__.smoke() compare with
(tests/golden/reference/<test file>.npz), so that neither needs the reference sources or a build of them.

The files are fixed data; nothing in the repository writes them.  They hold two kinds of entries:

* 'digests': for every result a test compares bit for bit, its dtype, shape and the first 128 bits of the SHA-256 of
  its bytes.  These are the reference's own results on the test's seeded inputs: they were taken from this project's
  code as of commit bbc7083, whose test suite found these results byte-identical to the unmodified reference's.
* one array per result a test compares with a tolerance (poses, F, RANSAC counts, sub-pixel coordinates, triangulated and
  reconstructed points, SVD factors): this project's result at that commit, which was within the test's tolerance of
  the reference's.  It is not the reference's value, so it bounds drift from the tested behaviour, not the distance to
  the reference.  Three large sets are a fixed seeded sample of the entries (see the tests).
"""
import hashlib
import os

import numpy as np

DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden', 'reference')
_stored = {}


def digest(a):
    a = np.ascontiguousarray(a)
    return '%s %s %s' % (a.dtype.str, 'x'.join(map(str, a.shape)), hashlib.sha256(a.tobytes()).hexdigest()[:32])


def _read(path):
    out = dict(np.load(path))
    for line in out.pop('digests', []):
        k, d = str(line).split(' ', 1)
        out[k] = d
    return out


class Reference:
    """The stored results for one test case; `group` names the file, `case` the test (parameters included)."""

    def __init__(self, group, case):
        self.group, self.case = group, case

    def _key(self, key):
        return '%s::%s' % (self.case, key)

    def _load(self, key):
        if self.group not in _stored:
            _stored[self.group] = _read(os.path.join(DIR, self.group + '.npz'))
        k = self._key(key)
        if k not in _stored[self.group]:
            raise KeyError('no stored result %s in tests/golden/reference/%s.npz' % (k, self.group))
        return _stored[self.group][k]

    def same(self, key, got):
        """Assert that `got` equals the reference's result `key` bit for bit: dtype, shape and bytes."""
        d = digest(got)
        want = str(self._load(key))
        assert d == want, '%s: %s differs from the reference result %s' % (self._key(key), d, want)

    def value(self, key):
        """The stored result `key`, for a comparison with a tolerance."""
        return self._load(key)
