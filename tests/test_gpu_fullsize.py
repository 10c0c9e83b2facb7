"""GPU tests at BASELINE.json's full sizes: config 4 (3840x2160, tens of thousands of maxima) against the reference's
outputs (stored under tests/golden/reference, see oracle/refgold.py), plus size-independent properties of the match lists."""
import numpy as np
import pytest

import synth
import visocu_py as V
import host_py as H

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def pair4k():
    return synth.blob_pair(3840, 2160, seed=404, n_blobs=60000)


def test_flow_4k_matches_reference(reference, pair4k):
    a, b = pair4k
    hm = H.Matcher(V.Params())
    hm.push(a); hm.push(b); hm.match_features(0)
    reference.same('counts', np.array(list(hm.counts().values()), np.int64))
    assert hm.counts()['1c2'] > 40000
    got = hm.matches(2)
    assert len(got) > 30000
    reference.same('matches1', hm.matches(1))
    reference.same('matches2', got)


def test_match_list_properties(pair4k):
    a, b = pair4k
    hm = H.Matcher(V.Params())
    hm.push(a); hm.push(b); hm.match_features(0)
    m = hm.matches(2)
    c = hm.counts()
    assert np.all(np.diff(m['i1c']) > 0)                              # ascending current-feature index, no duplicates
    assert m['i1c'].max() < c['1c2'] and m['i1p'].max() < c['1p2'] and m['i1p'].min() >= 0
    assert len(np.unique(m['i1p'])) == len(m)                          # circle matching is one-to-one
    pix = m['u1c'].astype(np.int64) * 10000 + m['v1c'].astype(np.int64)
    assert len(np.unique(pix)) == len(m)                               # one match per pixel (matcher.cpp:1036-1039)
    assert np.all(m['u2p'] == -1) and np.all(m['i2c'] == -1)           # unused fields of a flow match
    flow = np.abs(m['u1c'] - m['u1p'] - 3) + np.abs(m['v1c'] - m['v1p'] - 1)
    assert np.mean(flow <= 2) > 0.98                                    # the synthetic pair is a (3,1) pixel shift
    # idempotence: replacing the current frame by itself and matching again gives the same list
    hm.push(b, replace=True); hm.match_features(0)
    assert hm.matches(2).tobytes() == m.tobytes()
    # matching a frame against itself: every surviving match is the identity
    hm.push(b); hm.match_features(0)
    s = hm.matches(2)
    same = (s['u1c'] == s['u1p']) & (s['v1c'] == s['v1p'])            # pixel refinement may slide along flat structure
    assert len(s) > 0.4 * c['1c2'] and same.mean() > 0.99
