"""Device outlier removal (csrc/outliers.cu: k_remove_outliers) against the host Matcher::removeOutliers at every CTA size,
merge mode, batch shape and coordinate edge.

The oracle is an H.Matcher that was never pushed: it has no context, so host/delaunay.cpp triangulates and votes on the
CPU alone (test_host_cpu.py::test_remove_outliers_matches_reference pins that path to the unmodified reference).  The
device context is configured with the same V.Params, so both sides vote with the same tolerances.

Every case states the status it expects (0 handled; 1 too long for shared memory or a position outside 0..8191; 3 three
or fewer distinct positions), and the status is asserted: a declined list must come back unchanged, so a case cannot
pass by being declined.  Handled lists must equal the host survivors byte for byte, order included.

Each case runs under six kernel shapes, VISOCU_RO_THREADS in {1024, 512, 256} times VISOCU_RO_WARP in {1, 0} (a warp or
one thread per top-level merge).  The context reads both when it is configured.  The batch test also runs the unset
default, which picks 1024 threads for one or two lists and 512 for more.

Not covered: the kernel's internal guard (status 3 from the loop budget or the edge capacity), and the vote's branch for
lists whose compared quantities do not fit in shared memory (vote_in_smem == false).  Since the edge capacity is at
least 3.04 n + 64, 8 n + 2 n_vertices <= 4 ecap always holds, so that branch looks unreachable."""
import collections

import numpy as np
import pytest

import synth
import visocu_py as V
import host_py as H

VARIANTS = [(t, w) for t in (1024, 512, 256) for w in (1, 0)]
VARIANT_IDS = ['t%d-%s' % (t, 'warp' if w else 'thread') for t, w in VARIANTS]
SMEM_MAX = 227 * 1024 - 256          # dynamic shared memory of one CTA (visocu_launch_remove_outliers)
COORD_MAX = 8191                     # positions the 32-bit predicates take exactly
TOLS = (0, 1, 5, 20)

# lists per (variant, family) and status, printed at the end of the module (pytest -s)
STATS = collections.defaultdict(collections.Counter)


def _ro_smem_bytes(n):
    """Shared memory the kernel needs for a list of n records: ro_smem_bytes in csrc/outliers.cu."""
    e = int(V.lib().visocu_delaunay_edge_capacity(int(n)))
    return ((12 * e + 15) & ~15) + 4 * n + 16


def _largest_list():
    n = 4
    while _ro_smem_bytes(n + 1) <= SMEM_MAX:
        n += 1
    return n


# ------------------------------------------------------------------------------------------------------------ generators
def _records(rng, x, y, flow=3, disp=30):
    """Match records at current-left positions (x, y), in the style of test_gpu_outliers._random_matches: small random
    flows with a few large ones, random disparities.  i1c numbers the records so that every record is distinct."""
    n = len(x)
    m = np.zeros(n, V.P_MATCH)
    for name in ('i1p', 'i2p', 'i2c'):
        m[name] = -1
    m['i1c'] = np.arange(n)
    m['u1c'] = x; m['v1c'] = y
    fl = rng.integers(-flow, flow + 1, (n, 2)) + (rng.random((n, 2)) < 0.1) * rng.integers(-20, 20, (n, 2))
    m['u1p'] = m['u1c'] - fl[:, 0]; m['v1p'] = m['v1c'] - fl[:, 1]
    d = rng.integers(0, disp, n)
    m['u2c'] = m['u1c'] - d; m['v2c'] = m['v1c']
    m['u2p'] = m['u1p'] - d - rng.integers(-1, 2, n); m['v2p'] = m['v1p']
    return m


def _distinct(rng, n, w, h, grid=1, x0=0, y0=0):
    """n distinct positions on the multiples of `grid` inside [0, w] x [0, h], shifted by (x0, y0)."""
    nx, ny = w // grid + 1, h // grid + 1
    cells = rng.choice(nx * ny, size=n, replace=False)
    return (cells % nx) * grid + x0, (cells // nx) * grid + y0


def _lattice(k, s=1, x0=0, y0=0, kx=None):
    """Full kx x k lattice of spacing s: every unit cell is co-circular."""
    y, x = np.mgrid[0:k, 0:(kx or k)]
    return x.ravel() * s + x0, y.ravel() * s + y0


def _circle(r, cx, cy):
    """All integer points on the circle of radius r around (cx, cy)."""
    xs = np.arange(-r, r + 1)
    ys = np.rint(np.sqrt(r * r - xs * xs)).astype(np.int64)
    ok = ys * ys + xs * xs == r * r
    pts = {(int(a), int(s * b)) for a, b in zip(xs[ok], ys[ok]) for s in (1, -1)}
    p = np.array(sorted(pts))
    return p[:, 0] + cx, p[:, 1] + cy


def _shuffled(rng, m):
    return m[rng.permutation(len(m))]


def _point_sets(seed):
    """family -> [(list, expected status)]"""
    rng = np.random.default_rng(seed)
    R = lambda x, y, **kw: _shuffled(rng, _records(rng, np.asarray(x), np.asarray(y), **kw))
    fam = collections.defaultdict(list)
    # leaves of two and three points and the first merges
    for n in range(4, 41):
        fam['small'].append((R(*_distinct(rng, n, 60, 40, 1 + n % 3)), 0))
    # partition boundaries
    for k in range(2, 13):
        for n in (2 ** k - 1, 2 ** k, 2 ** k + 1):
            fam['pow2'].append((R(*_distinct(rng, n, 1240, 375)), 0))
    # uniform distinct points and grid-snapped sets full of co-circular ties
    for n in (50, 700, 3000):
        fam['uniform'].append((R(*_distinct(rng, n, 1240, 375)), 0))
    for g in range(1, 17):
        n = int(rng.integers(100, 1500))
        side = int(np.sqrt(3 * n)) + 1
        fam['grid'].append((R(*_distinct(rng, n, side * g, side * g // 2 + g, g, int(rng.integers(0, 50)))), 0))
    for k, s in ((2, 1), (3, 7), (4, 1), (5, 2), (7, 1), (8, 3), (16, 1), (31, 5), (32, 1), (33, 2), (64, 1), (75, 109)):
        fam['lattice'].append((R(*_lattice(k, s, int(rng.integers(0, 9)), int(rng.integers(0, 9)))), 0))
    fam['lattice'].append((R(*_lattice(3, 4, 5, 5, kx=200)), 0))              # three long rows
    # integer points on large circles, alone, concentric, and with points inside
    for r, c in ((5, (10, 10)), (25, (30, 40)), (65, (100, 70)), (325, (400, 400)), (1105, (4096, 4096)),
                 (2465, (4096, 4096)), (4095, (4095, 4096))):
        fam['circles'].append((R(*_circle(r, *c)), 0))
    x1, y1 = _circle(1105, 4096, 4096); x2, y2 = _circle(2465, 4096, 4096); x3, y3 = _circle(3315, 4096, 4096)
    fam['circles'].append((R(np.concatenate([x1, x2, x3]), np.concatenate([y1, y2, y3])), 0))
    xi, yi = _distinct(rng, 300, 1400, 1400, 1, 3400, 3400)
    keep = (xi - 4096) ** 2 + (yi - 4096) ** 2 < 1100 ** 2
    fam['circles'].append((R(np.concatenate([x1, xi[keep]]), np.concatenate([y1, yi[keep]])), 0))
    # collinear leaves and merges across both cut axes: rows, columns, diagonals, two parallel rows or columns
    for n in (4, 5, 7, 33, 100, 1000):
        a = np.arange(n)
        fam['lines'].append((R(a * 3 + 1, np.full(n, 7)), 0))
        fam['lines'].append((R(np.full(n, 9), a * 2), 0))
        fam['lines'].append((R(a + 2, a + 5), 0))
        fam['lines'].append((R(a * 2, 2 * n - a * 2), 0))
        fam['lines'].append((R(np.concatenate([a, a]) * 4, np.repeat([3, 4 + n % 5], n)), 0))
        fam['lines'].append((R(np.repeat([0, 1 + n], n), np.concatenate([a, a + 1])), 0))
    return fam


def _coordinate_sets(seed):
    """(list, expected status, what) at the edges of the positions: fractions, truncation toward zero, 0 and 8191."""
    rng = np.random.default_rng(seed)
    R = lambda x, y: _shuffled(rng, _records(rng, np.asarray(x, np.float32), np.asarray(y, np.float32)))
    out = []
    x, y = _distinct(rng, 400, 300, 200)
    frac = rng.choice(np.array([0.0, 0.25, 0.5, 0.999], np.float32), (2, len(x)))
    out.append((R(x + frac[0], y + frac[1]), 0, 'fractional positions'))
    xn, yn = x.astype(np.float32), y.astype(np.float32)
    xn[:20] = rng.choice(np.array([-0.5, -0.999], np.float32), 20); yn[20:40] = rng.choice(np.array([-0.5, -0.999], np.float32), 20)
    out.append((R(xn, yn), 0, 'positions in (-1, 0) truncate to 0'))
    xs, ys = _distinct(rng, 300, COORD_MAX, COORD_MAX)
    border = np.array([0, COORD_MAX, 0, COORD_MAX, 0, 4000, COORD_MAX, 4000]), np.array([0, 0, COORD_MAX, COORD_MAX, 4000, 0, 4000, COORD_MAX])
    out.append((R(np.concatenate([xs, border[0]]), np.concatenate([ys, border[1]])), 0, 'corners and edges of 0..8191'))
    edge = R(np.concatenate([xs, border[0]]), np.concatenate([ys, border[1]]))
    edge['u1c'][edge['u1c'] == COORD_MAX] = np.float32(8191.999)
    out.append((edge, 0, '8191.999 truncates to 8191'))
    # co-circular lattice over the whole square: every axis-aligned rectangle of it is co-circular
    gx = np.unique(np.concatenate([[0, COORD_MAX], rng.integers(1, COORD_MAX, 38)]))
    gy = np.unique(np.concatenate([[0, COORD_MAX], rng.integers(1, COORD_MAX, 38)]))
    X, Y = np.meshgrid(gx, gy)
    out.append((R(X.ravel(), Y.ravel()), 0, 'lattice spanning 0..8191'))
    out.append((R(*_lattice(40, 210, 0, 0)), 0, 'regular lattice 0..8190'))
    for axis in ('u1c', 'v1c'):
        m = R(*_distinct(rng, 200, 500, 300))
        m[axis][7] = 8192
        out.append((m, 1, '8192 in %s' % axis))
    return out


def _negative_lists(seed):
    """A record at a negative position in a list whose flows all agree (the host keeps it), without and with two other
    records on one pixel.  The device must decline both: its predicates do not take negative coordinates."""
    rng = np.random.default_rng(seed)
    x, y = _lattice(10, 3, 0, 0)
    m = _records(rng, np.concatenate([x, [-3]]), np.concatenate([y, [13]]), flow=0, disp=1)
    m['u1p'] = m['u1c'] - 2; m['v1p'] = m['v1c'] + 1                     # one flow for all: every edge agrees
    dup = np.concatenate([m, m[44:45]])
    dup['i1c'][-1] = len(m); dup['u1c'][-1] += np.float32(0.5)           # a second record on the pixel (12, 12)
    return [(m, 'negative x'), (dup, 'negative x and a duplicate elsewhere')]


def _duplicate_sets(seed):
    rng = np.random.default_rng(seed)
    out = []
    for d in list(range(2, 11)) + [17, 31, 50]:
        x, y = _distinct(rng, 40, 60, 40)
        px = np.concatenate([x, np.full(d - 1, x[0])]); py = np.concatenate([y, np.full(d - 1, y[0])])
        m = _records(rng, px.astype(np.float32) + rng.choice([0, 0.25, 0.75], len(px)).astype(np.float32), py)
        out.append((_shuffled(rng, m), 0, '%d records on one pixel' % d))
    for n in (4, 10, 100):
        out.append((_records(rng, np.full(n, 17), np.full(n, 5)), 3, 'all %d records on one pixel' % n))
    for k, n in ((2, 10), (3, 8), (3, 60)):
        x, y = _distinct(rng, k, 20, 20)
        out.append((_shuffled(rng, _records(rng, np.resize(x, n), np.resize(y, n))), 3, '%d distinct positions' % k))
    x, y = _distinct(rng, 4, 20, 20)
    out.append((_shuffled(rng, _records(rng, np.resize(x, 9), np.resize(y, 9))), 0, '4 distinct positions'))
    out.append((_records(rng, rng.integers(0, 20, 500), rng.integers(0, 15, 500)), 0, '500 records on 300 pixels'))
    x, y = _distinct(rng, 2000, 1240, 375, 8)
    out.append((_shuffled(rng, _records(rng, np.resize(x, 4000), np.resize(y, 4000))), 0, 'every position twice'))
    return out


def _boundary_list(rng, ft, dt):
    """A list whose triangle edges compare flows and disparities equal to the tolerances and one float32 step either side.

    A column at x = 0 alternates records of flow D (u1p = -D) and of disparity E (u2c = u2p = -E): at u1c = 0 both
    subtractions are exact.  D and E cycle through prev(tol), tol, next(tol) and 0.  The other records have integer flows
    and disparities from a few values, so that integer sums land on the tolerances too."""
    def near(t):
        t = np.float32(t)
        return [np.nextafter(t, np.float32(-1)), t, np.nextafter(t, np.float32(1e9))] if t > 0 else [t, np.float32(1)]
    Ds, Es = near(ft), near(dt)
    ny = 24
    cy = np.arange(ny) * 2
    ox, oy = _distinct(rng, 150, 40, 2 * ny, 1, 1, 0)
    n = ny + len(ox)
    m = np.zeros(n, V.P_MATCH)
    for name in ('i1p', 'i2p', 'i2c'):
        m[name] = -1
    m['i1c'] = np.arange(n)
    m['u1c'] = np.concatenate([np.zeros(ny), ox]); m['v1c'] = np.concatenate([cy, oy])
    vals = np.array([0, 1, 2, 3, 5, 10, 20])
    fu = rng.choice(vals, n) * rng.choice([-1, 1], n); fv = rng.choice(vals, n) * (rng.random(n) < 0.3)
    d = rng.choice(vals, n)
    m['u1p'] = m['u1c'] - fu; m['v1p'] = m['v1c'] - fv
    m['u2c'] = m['u1c'] - d; m['v2c'] = m['v1c']
    m['u2p'] = m['u1p'] - d; m['v2p'] = m['v1p']
    for k in range(ny):
        if k % 2 == 0:
            D = -Ds[(k // 2) % len(Ds)] if k % 4 == 0 else Ds[(k // 2) % len(Ds)]
            m['u1p'][k] = -D; m['v1p'][k] = m['v1c'][k]; m['u2c'][k] = 0; m['u2p'][k] = -D
        else:
            E = Es[(k // 2) % len(Es)]
            m['u1p'][k] = 0; m['v1p'][k] = m['v1c'][k]; m['u2c'][k] = -E; m['u2p'][k] = -E
    return _shuffled(rng, m)


def _edge_quantities(m, method):
    """Per triangle edge of the host triangulation: the flow sum and the disparity difference the vote compares, in
    float32 operation by operation as matcher.cpp does."""
    e, _ = H.delaunay_edges(m['u1c'].astype(np.int32), m['v1c'].astype(np.int32))
    e = e[e[:, 2] > 0]
    f32 = np.float32
    fu = (m['u1c'] - m['u1p']).astype(f32); fv = (m['v1c'] - m['v1p']).astype(f32)
    fd = (m['u1c'] - m['u2c'] if method == 1 else m['u1p'] - m['u2p']).astype(f32)
    a, b = e[:, 0], e[:, 1]
    flow = (np.abs(fu[a] - fu[b]) + np.abs(fv[a] - fv[b])).astype(f32)
    disp = np.abs(fd[a] - fd[b]).astype(f32)
    return flow, disp


# --------------------------------------------------------------------------------------------------------------- harness
@pytest.fixture(scope='module')
def octx():
    c = V.Context(0)
    yield c
    c.close()
    if STATS:
        print('\ndevice outlier removal, lists per status:')
        for (variant, family), cnt in sorted(STATS.items()):
            print('  %-14s %-12s %s' % (variant, family, ' '.join('status %d: %d' % kv for kv in sorted(cnt.items()))))


def _use(monkeypatch, variant):
    for k in ('VISOCU_RO_THREADS', 'VISOCU_RO_WARP'):
        monkeypatch.delenv(k, raising=False)
    if variant is not None:
        monkeypatch.setenv('VISOCU_RO_THREADS', str(variant[0]))
        monkeypatch.setenv('VISOCU_RO_WARP', str(variant[1]))
    return 'default' if variant is None else VARIANT_IDS[VARIANTS.index(variant)]


def _configure(octx, params):
    octx.configure(params, 1241, 376, 1)
    return H.Matcher(params)


def _run(octx, hm, lists, method, expect, tag, family, what=None):
    """One device call on `lists`; every status as expected, handled lists equal to the host's survivors, declined ones
    unchanged.  Returns the device lists."""
    got, status = octx.remove_outliers(lists, method)
    for k, (l, g, st, ex) in enumerate(zip(lists, got, status, expect)):
        where = '%s %s method %d list %d (%s, %d records)' % (tag, family, method, k, what[k] if what else '', len(l))
        assert st == ex, '%s: status %d, expected %d' % (where, st, ex)
        if st == 0:
            want = hm.remove_outliers(l, method)
            assert g.tobytes() == want.tobytes(), '%s: %d survivors, host %d' % (where, len(g), len(want))
        else:
            assert g.tobytes() == l.tobytes(), '%s: a declined list changed' % where
        STATS[(tag, family)][int(st)] += 1
    return got


# ----------------------------------------------------------------------------------------------------------------- tests
def test_vote_lists_put_edges_on_the_tolerance():
    """The vote lists do what _boundary_list claims: for every method and tolerance, triangle edges compare flows (method
    0, 2) and disparities (1, 2) equal to the tolerance and one float32 step below and above it."""
    rng = np.random.default_rng(71)
    for ft in TOLS[1:]:
        for dt in TOLS[1:]:
            m = _boundary_list(rng, ft, dt)
            for method in (0, 1, 2):
                flow, disp = _edge_quantities(m, method)
                for q, t in ((flow, ft), (disp, dt)):
                    t = np.float32(t)
                    for v in (np.nextafter(t, np.float32(-1)), t, np.nextafter(t, np.float32(1e9))):
                        assert (q == v).any(), (ft, dt, method, v)


def test_largest_list_is_near_the_shared_memory_limit():
    n = _largest_list()
    assert 5600 < n < 5800 and _ro_smem_bytes(n) <= SMEM_MAX < _ro_smem_bytes(n + 1)


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS, ids=VARIANT_IDS)
def test_point_sets_equal_host(octx, monkeypatch, variant):
    """n = 4..40, n = 2^k - 1, 2^k, 2^k + 1 up to 4097, uniform and grid-snapped sets, lattices, points on circles, lines."""
    tag = _use(monkeypatch, variant)
    hm = _configure(octx, V.Params())
    for family, cases in sorted(_point_sets(11).items()):
        for method in (0, 1, 2):
            sel = [c for k, c in enumerate(cases) if k % 3 == method]
            if sel:
                _run(octx, hm, [l for l, _ in sel], method, [s for _, s in sel], tag, family)
        assert STATS[(tag, family)][0] >= len(cases)


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS, ids=VARIANT_IDS)
def test_shared_memory_capacity(octx, monkeypatch, variant):
    """The longest list that fits the 227 KB of a CTA is handled and one record more is declined, alone and in one
    launch with small lists (which clamps the launch's shared memory to the limit)."""
    tag = _use(monkeypatch, variant)
    hm = _configure(octx, V.Params())
    rng = np.random.default_rng(13)
    n = _largest_list()
    big = _records(rng, *_distinct(rng, n + 1, 1240, 375))
    fit, over = big[:n], big
    small = [_records(rng, *_distinct(rng, k, 300, 200)) for k in (4, 100, 1000)]
    for method in (0, 1, 2):
        _run(octx, hm, [fit], method, [0], tag, 'capacity')
        _run(octx, hm, [over], method, [1], tag, 'capacity')
        _run(octx, hm, [small[0], fit, small[1], over, small[2]], method, [0, 0, 0, 1, 0], tag, 'capacity')
    assert STATS[(tag, 'capacity')][0] == 3 * 5


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS, ids=VARIANT_IDS)
def test_coordinate_edges(octx, monkeypatch, variant):
    """Fractional and slightly negative positions (truncated toward zero), 0 and 8191 on both axes and co-circular sets
    over the whole square (the 32-bit predicates at their limit), and 8192 (declined)."""
    tag = _use(monkeypatch, variant)
    hm = _configure(octx, V.Params())
    cases = _coordinate_sets(17)
    for method in (0, 1, 2):
        _run(octx, hm, [c[0] for c in cases], method, [c[1] for c in cases], tag, 'coordinates', [c[2] for c in cases])


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS, ids=VARIANT_IDS)
def test_negative_position_is_declined(octx, monkeypatch, variant):
    """A negative position goes to the host whether or not the list also has two records on one pixel (the duplicate
    replay must not hide the record from the kernel's range check)."""
    tag = _use(monkeypatch, variant)
    hm = _configure(octx, V.Params())
    cases = _negative_lists(19)
    for method in (0, 1, 2):
        for m, what in cases:
            kept = hm.remove_outliers(m, method)
            assert len(kept) > len(m) // 2 and (kept['u1c'] < 0).any()     # the host keeps the record
            _run(octx, hm, [m], method, [1], tag, 'negative', [what])


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS, ids=VARIANT_IDS)
def test_duplicate_positions(octx, monkeypatch, variant):
    """2 to 50 records on one pixel, every record on one pixel, and lists of three or fewer distinct positions."""
    tag = _use(monkeypatch, variant)
    hm = _configure(octx, V.Params())
    cases = _duplicate_sets(23)
    for method in (0, 1, 2):
        _run(octx, hm, [c[0] for c in cases], method, [c[1] for c in cases], tag, 'duplicates', [c[2] for c in cases])


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS, ids=VARIANT_IDS)
def test_vote_tolerances(octx, monkeypatch, variant):
    """Every method at flow and disparity tolerances 0, 1, 5 and 20, on lists whose edges compare exactly the tolerance
    and one float32 step either side of it (the vote's strict '<' decides them) and on random lists."""
    tag = _use(monkeypatch, variant)
    rng = np.random.default_rng(29)
    for ft in TOLS:
        for dt in TOLS:
            hm = _configure(octx, V.Params(outlier_flow_tolerance=ft, outlier_disp_tolerance=dt))
            lists = [_boundary_list(rng, ft, dt), _records(rng, *_distinct(rng, 600, 200, 100), flow=4, disp=8),
                     _records(rng, *_distinct(rng, 300, 200, 100, 4), flow=12, disp=25)]
            for method in (0, 1, 2):
                got = _run(octx, hm, lists, method, [0, 0, 0], tag, 'vote')
                if ft == 0 and method != 1 or dt == 0 and method != 0:
                    assert all(len(g) == 0 for g in got)          # nothing is below a tolerance of 0
    assert STATS[(tag, 'vote')][0] == 16 * 3 * 3


def _batch_lists(rng, n_jobs, n_max):
    """Ragged jobs of every kind with their expected status."""
    out = []
    for j in range(n_jobs):
        kind = j % 7
        if kind == 0:
            m, s = _records(rng, *_distinct(rng, int(rng.integers(4, 2500)), 1240, 375)), 0
        elif kind == 1:
            n, (x, y) = int(rng.integers(20, 1500)), _distinct(rng, 1500, 400, 200, 2)
            pick = rng.integers(0, n, n)                  # about a third of the records share a pixel
            m, s = _records(rng, x[pick], y[pick]), 0
        elif kind == 2:
            k = int(rng.integers(2, 30))
            m, s = _shuffled(rng, _records(rng, *_lattice(k, int(rng.integers(1, 5))))), 0
        elif kind == 3:
            m, s = _records(rng, *_distinct(rng, int(rng.integers(0, 4)), 100, 100)), 0
        elif kind == 4:
            n = int(rng.integers(4, 300))
            m, s = _records(rng, np.arange(n) * 2, np.full(n, j % 50)), 0
        elif kind == 5:
            x, y = _distinct(rng, int(rng.integers(1, 4)), 30, 30)
            m, s = _records(rng, np.resize(x, 12), np.resize(y, 12)), 3
        else:
            m, s = _records(rng, *_distinct(rng, int(rng.integers(4, 400)), 100, 60)), 0
        out.append((m, s))
    if n_jobs >= 64:
        out[n_jobs // 2] = (_records(rng, *_distinct(rng, n_max + 1, 1240, 375)), 1)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('n_jobs', [1, 2, 3, 64, 300])
@pytest.mark.parametrize('variant', VARIANTS + [None], ids=VARIANT_IDS + ['default'])
def test_batches(octx, monkeypatch, variant, n_jobs):
    """Ragged batches in one call: every list equals the host's, a repeated call returns the same bytes, and a list's
    survivors do not depend on its position in the batch or on its neighbours."""
    tag = _use(monkeypatch, variant)
    hm = _configure(octx, V.Params())
    rng = np.random.default_rng(31 + n_jobs)
    cases = _batch_lists(rng, n_jobs, _largest_list())
    lists, expect = [c[0] for c in cases], [c[1] for c in cases]
    for method in (0, 1, 2):
        first = _run(octx, hm, lists, method, expect, tag, 'batch%d' % n_jobs)
        again, status = octx.remove_outliers(lists, method)
        assert status.tolist() == expect and all(a.tobytes() == b.tobytes() for a, b in zip(first, again))
        perm = np.roll(np.arange(n_jobs)[::-1], 1)
        moved, status = octx.remove_outliers([lists[k] for k in perm], method)
        assert status.tolist() == [expect[k] for k in perm]
        assert all(moved[i].tobytes() == first[k].tobytes() for i, k in enumerate(perm))


@pytest.fixture(scope='module')
def scenes():
    """Eight frames: two blob stereo quads (0-3, 4-7) of different fields, disparities and motions."""
    return list(synth.blob_quad(1241, 376, seed=61, shift=(3, 1), disparity=12)) + \
        list(synth.blob_quad(1241, 376, seed=63, shift=(-2, 2), disparity=7))


QUADS = {0: [(0, -1, 2, -1), (4, -1, 6, -1)], 1: [(-1, -1, 2, 3), (-1, -1, 6, 7)], 2: [(0, 1, 2, 3), (4, 5, 6, 7)]}


@pytest.mark.gpu
@pytest.mark.parametrize('variant', VARIANTS, ids=VARIANT_IDS)
def test_matching_path(octx, monkeypatch, scenes, variant):
    """visocu_match with outlier removal behind the matching kernels, every method and refinement, batches of 1 and 5:
    where the device handled a list it equals the host's removeOutliers of what the same call returns without outlier
    removal; a declined list comes back whole.  Stereo and quad lists with several matches on one pixel go through the
    duplicate replay (k_outlier_keys, ro_resolve_duplicates, the rep flags), sub-pixel refinement through the keep flags."""
    tag = _use(monkeypatch, variant)
    vp = V.Params()
    vp.match_radius //= 2                                  # the Matcher constructor's halving for half resolution
    octx.configure(vp, 1241, 376, 8)
    octx.push_frames(list(range(8)), scenes)
    hm = H.Matcher(V.Params())
    dup_handled = keep_handled = 0
    for method in (0, 1, 2):
        for refine in (0, 1, 2):
            for nb in (1, 5):
                quads = [QUADS[method][k % 2] for k in range(nb)]
                raw = octx.match(quads, method, 1, refine=refine)
                got, done = octx.match(quads, method, 1, refine=refine, outliers=True)
                for j in range(nb):
                    where = '%s method %d refine %d batch %d job %d (%d matches)' % (tag, method, refine, nb, j, len(raw[j]))
                    assert len(raw[j]) > 100, where
                    if done[j]:
                        want = hm.remove_outliers(raw[j], method)
                        assert got[j].tobytes() == want.tobytes(), '%s: %d survivors, host %d' % (where, len(got[j]), len(want))
                        pos = np.stack([raw[j]['u1c'].astype(np.int32), raw[j]['v1c'].astype(np.int32)], 1)
                        dup_handled += method != 0 and len(np.unique(pos, axis=0)) < len(pos)
                        keep_handled += refine == 2
                    else:
                        assert got[j].tobytes() == raw[j].tobytes(), where
                    STATS[(tag, 'match')][0 if done[j] else 1] += 1
    assert dup_handled > 0 and keep_handled > 0, (dup_handled, keep_handled)
