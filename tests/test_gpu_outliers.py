"""Device-side Matcher::removeOutliers (csrc/outliers.cu) against the outputs of the unmodified reference (Triangle
"zQB" + support vote, matcher.cpp:1207-1377; stored under tests/golden/reference, see oracle/refgold.py): bit-exact
survivor lists, order included, also with several matches on one pixel.  Lists the device declines (non-zero status:
too long for shared memory, degenerate) must come back unchanged."""
import numpy as np
import pytest

import pyref
import visocu_py as V

pytestmark = pytest.mark.gpu


def _random_matches(rng, n, w, h, grid, dup):
    m = np.zeros(n, pyref.P_MATCH)
    for name in ('i1p', 'i2p', 'i1c', 'i2c'):
        m[name] = -1
    if dup:
        u = rng.integers(0, w // grid + 1, n) * grid; v = rng.integers(0, h // grid + 1, n) * grid
    else:
        cells = rng.choice((w // grid + 1) * (h // grid + 1), size=min(n, (w // grid + 1) * (h // grid + 1)), replace=False)
        u = (cells % (w // grid + 1)) * grid; v = (cells // (w // grid + 1)) * grid
        m = m[:len(cells)]
    m['u1c'] = u; m['v1c'] = v
    flow = rng.integers(-3, 4, (len(m), 2)) + (rng.random((len(m), 2)) < 0.1) * rng.integers(-20, 20, (len(m), 2))
    m['u1p'] = m['u1c'] - flow[:, 0]; m['v1p'] = m['v1c'] - flow[:, 1]
    disp = rng.integers(0, 30, len(m))
    m['u2c'] = m['u1c'] - disp; m['v2c'] = m['v1c']
    m['u2p'] = m['u1p'] - disp - rng.integers(-1, 2, len(m)); m['v2p'] = m['v1p']
    return m


@pytest.fixture(scope='module')
def rctx():
    c = V.Context(0)
    c.configure(V.Params(half_resolution=0), 1241, 376, 4)
    yield c
    c.close()


def test_device_outlier_removal_equals_reference(reference, rctx):
    rng = np.random.default_rng(7)
    lists, methods = [], []
    for trial in range(96):
        n = int(rng.integers(4, 4700)) if trial % 3 else int(rng.integers(4, 200))
        grid = int(rng.choice([1, 1, 2, 4, 8, 16]))
        w = int(rng.integers(60, 1300)); h = int(rng.integers(60, 400))
        # every other list has several matches per pixel: Triangle's choice among them (its randomised quicksort)
        # is replayed on the device
        lists.append(_random_matches(rng, n, w, h, grid, dup=trial % 2 == 1)); methods.append(int(rng.choice([0, 1, 2])))
    handled = 0
    for method in (0, 1, 2):
        sel = [(k, l) for k, (l, mth) in enumerate(zip(lists, methods)) if mth == method]
        got, status = rctx.remove_outliers([l for _, l in sel], method)
        for (k, l), g, st in zip(sel, got, status):
            if st == 0:
                handled += 1
                reference.same('list%d' % k, g)
            else:
                assert g.tobytes() == l.tobytes()
    assert handled >= 90                                  # only over-long lists may be declined here


def test_device_outlier_removal_declines_what_it_cannot_do(reference, rctx):
    rng = np.random.default_rng(8)
    dup = _random_matches(rng, 30, 8, 4, 4, dup=True)                   # only a handful of distinct positions
    dup['u1c'] = (dup['u1c'] // 8) * 8; dup['v1c'] = 0                  # ... in fact two: nothing to triangulate
    big = _random_matches(rng, 9000, 1240, 370, 1, dup=False)           # does not fit in shared memory
    tiny = _random_matches(rng, 3, 100, 100, 1, dup=False)              # <= 3: returned untouched (matcher.cpp:1210)
    line = np.zeros(40, pyref.P_MATCH); line['u1c'] = np.arange(40) * 3; line['v1c'] = 7; line['u1p'] = line['u1c']; line['v1p'] = 7
    got, status = rctx.remove_outliers([dup, big, tiny, line], 0)
    assert status[0] != 0 and status[1] == 1 and status[2] == 0
    assert got[0].tobytes() == dup.tobytes() and got[1].tobytes() == big.tobytes() and got[2].tobytes() == tiny.tobytes()
    if status[3] == 0:                                                   # all collinear: no triangle, nobody survives
        reference.same('collinear', got[3])


def test_device_nodes_of_large_triangulations(rctx, monkeypatch):
    """visocu_delaunay_subtrees through host/delaunay.cpp: a triangulation of more points than the device kernel holds is cut
    into nodes that the device builds; the edge list (hence every vote of removeOutliers) equals the all-host one.  The
    nodes are built under every kernel shape (VISOCU_RO_THREADS x VISOCU_RO_WARP, read when the context is configured),
    then under the default one, which the context keeps for the tests after this one."""
    import host_py as H
    rng = np.random.default_rng(41)
    norm = lambda e: np.unique(np.concatenate([np.sort(e[:, :2], 1), e[:, 2:]], 1), axis=0)
    sets = []
    for n, w, h, grid in ((6500, 1241, 376, 1), (20000, 3840, 2160, 2), (87000, 3840, 2160, 2), (60000, 3840, 2160, 1), (9000, 8000, 200, 1)):
        cells = rng.choice((w // grid) * (h // grid), size=n, replace=False)
        x = ((cells % (w // grid)) * grid + 2).astype(np.int32); y = ((cells // (w // grid)) * grid + 3).astype(np.int32)
        e_host, nodes0 = H.delaunay_edges(x, y)
        assert nodes0 == 0
        sets.append((x, y, norm(e_host), (n, w, h, grid)))
    for variant in [(t, wm) for t in (1024, 512, 256) for wm in ('1', '0')] + [None]:
        if variant is None:
            monkeypatch.delenv('VISOCU_RO_THREADS', raising=False); monkeypatch.delenv('VISOCU_RO_WARP', raising=False)
        else:
            monkeypatch.setenv('VISOCU_RO_THREADS', str(variant[0])); monkeypatch.setenv('VISOCU_RO_WARP', variant[1])
        rctx.configure(V.Params(half_resolution=0), 1241, 376, 4)
        for x, y, want, what in sets:
            e_dev, nodes = H.delaunay_edges(x, y, rctx)
            assert nodes >= 2, (variant, what, nodes)
            assert len(e_dev) == len(want) and np.array_equal(want, norm(e_dev)), (variant, what)


def test_large_lists_vote_with_device_nodes(reference):
    """Matcher::removeOutliers on lists of 3840x2160 size (the device declines them as a whole): survivors equal the reference's."""
    import host_py as H
    rng = np.random.default_rng(43)
    hm = H.Matcher(V.Params())
    img = np.zeros((480, 640), np.uint8)
    hm.push(img)                                            # gives the matcher its context
    for n, grid in ((20000, 2), (87000, 2)):
        m = _random_matches(rng, n, 3800, 2100, grid, False)
        reference.same('n%d' % n, hm.remove_outliers(m, 0))
