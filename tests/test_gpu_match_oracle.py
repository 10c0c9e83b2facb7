"""The matcher (csrc/match.cu: k_match, k_match_count / k_match_emit, k_refine, the fused flow call) against the plain-C
restatement oracle/viso_oracle.c, at every method, search window, refinement mode and batch shape.

match.cu rests on equivalence arguments that fixed cases can pass by luck, so every run here compares what they claim:

  * the match lists byte for byte, order included (flow, stereo, quad, quad with Tr_delta; pass 0 and 1; refinement 0
    and 1).  The packed key (SAD, u_bin, v_bin, index) must pick the candidate the reference's ordered loop keeps first:
    saturated checkerboards, stripes and a constant image at nms_tau = 0 (four identical features per NMS cell, every SAD
    0) make the tie order the whole result, and exercise the three-record look-back of the "pixel already matched" rule;
  * the work counters of visocu_match_stats (entries of the scanned bins, candidates inside the window) against the
    oracle's counts, exactly: they check the integer window bounds even where a wrong bound would not change a winner.
    Synthetic per-bin prior ranges put window bounds on x.5, one ulp either side of an integer, zero-width and inverted
    spans, and beyond the image and beyond [-1, 65534];
  * sub-pixel refinement (refinement 2, a constant pseudo-inverse on the device, a least-squares solve per match in the
    oracle): integer fields and the kept set equal except for matches whose decision sits within 1e-6 of a threshold
    (counted, few), coordinates within SUBPIXEL_ULPS float32 steps;
  * pixel and sub-pixel refinement through visocu_refine on hand-built lists whose points sit on every coordinate around
    the early-return limits and whose minima land on the border of the 7x7 search;
  * batches of 1, 3, 128, 129 and 300 ragged jobs with per-job ranges and per-job Tr_delta (some null), the per-list copy
    path of lists over 64 MB, and VISOCU_ECAPACITY one match short;
  * the fused flow call (visocu_match_fused) in all three delivery layouts, against the oracle chain of the Matcher.

Out of scope: a prior bound whose bin (bound / match_binsize) does not fit an int.  The reference converts it with a
plain float -> int cast, which is undefined behaviour (x86 gives INT_MIN, clamped to bin 0); the device saturates.
Every synthetic bound here keeps |bound / binsize| < 2^31.

The oracle runs once per distinct (images, parameters, matching inputs), cached for the module; dense contents use small
match radii to keep its quadratic scan short."""
import ctypes as C

import numpy as np
import pytest

import synth
import pyoracle as O
import visocu_py as V
import host_py as H

MARGIN = 6                         # VISO_MARGIN
ECAPACITY = -4                     # VISOCU_ECAPACITY
NEAR = 1e-6                        # sub-pixel decisions closer than this to their threshold may go either way
# device (constant pseudo-inverse) vs oracle (least-squares solve per match): coordinates at most this many float32 steps
# apart.  On a B200 (sm_100a) the largest difference over about 67,000 kept matches was 0; one step at u = 1241 is 1.2e-4
SUBPIXEL_ULPS = 1
TR_MOVE = np.array([[1, 0, 0.01, 0.02], [0, 1, 0, 0], [-0.01, 0, 1, -0.3], [0, 0, 0, 1]], np.float64)
INTRINSICS = dict(f=645.2, cu=635.9, cv=194.1, base=0.54)
# degenerate predictions: x2c = y2c = 1 and z2c = 1e-12 (every predicted cost ~1e15) or 0 (+inf): no candidate of the
# predicted hop beats the initial cost 1e7, so it returns feature 0
TR_ZTINY = np.array([[0, 0, 0, 1 + INTRINSICS['base']], [0, 0, 0, 1], [0, 0, 0, 1e-12], [0, 0, 0, 1]], np.float64)
TR_ZERO = np.array([[0, 0, 0, 1 + INTRINSICS['base']], [0, 0, 0, 1], [0, 0, 0, 0], [0, 0, 0, 1]], np.float64)
TRS = {None: None, 'move': TR_MOVE, 'ztiny': TR_ZTINY, 'zzero': TR_ZERO}


# ---------------------------------------------------------------------------------------------------------------- inputs
def _checker(w, h, p, ox=0, oy=0):
    y, x = np.mgrid[0:h, 0:w]
    return ((((x + ox) // p + (y + oy) // p) % 2) * 255).astype(np.uint8)


def _images(kind, w, h):
    """(1p, 2p, 1c, 2c): two stereo pairs of one content; the right image sees the scene moved left (positive
    disparity) and the current pair sees it moved."""
    if kind in ('blob', 'empty'):
        a, b, c, d = synth.blob_quad(w, h, seed=61, shift=(3, 1), disparity=12)
        if kind == 'empty':                # no feature in the current right image: stereo and quad match nothing
            d = np.full((h, w), 128, np.uint8)
    elif kind == 'noise':
        big = np.random.default_rng(62).integers(0, 256, (h + 16, w + 16), dtype=np.uint8)
        crop = lambda dx, dy: big[8 + dy:8 + dy + h, 8 + dx:8 + dx + w]
        a, b, c, d = crop(0, 0), crop(4, 0), crop(-3, -1), crop(1, -1)
    elif kind == 'checker':                # saturated squares: every response repeats one period away
        a, b, c, d = _checker(w, h, 4), _checker(w, h, 4, 2, 0), _checker(w, h, 4, 1, 1), _checker(w, h, 4, 3, 1)
    elif kind == 'stripes':
        y, x = np.mgrid[0:h, 0:w]
        st = lambda o: (((x + o) // 3 + (y // 9)) % 2 * 255).astype(np.uint8)
        a, b, c, d = st(0), st(2), st(1), st(3)
    elif kind == 'const':                  # at nms_tau = 0: four features per cell, all descriptors alike
        a = b = c = d = np.full((h, w), 128, np.uint8)
    else:
        raise ValueError(kind)
    return [np.ascontiguousarray(i, np.uint8) for i in (a, b, c, d)]


def _quad(method):
    return {0: (0, -1, 2, -1), 1: (-1, -1, 2, 3), 2: (0, 1, 2, 3)}[method]


# ---------------------------------------------------------------------------------------------------------------- cases
def _case(kind, w, h, method, pass_=1, prior=None, tr=None, refine=0, expect='some', **kw):
    kw.setdefault('half_resolution', 1)
    if kind in ('noise', 'checker', 'stripes', 'const'):
        kw.setdefault('match_radius', 20)
    if kind == 'const':
        kw.setdefault('nms_tau', 0)
    if kind in ('checker', 'stripes', 'const') and expect == 'some':
        expect = 'ties'                    # ties everywhere: few circles close, but some do (checked per method)
    if tr is not None:
        for k, v in INTRINSICS.items():
            kw.setdefault(k, v)
    scene = '%dx%d-%s-%s' % (w, h, kind, '-'.join('%s%s' % (k.replace('_', '')[:6], v) for k, v in sorted(kw.items())))
    name = '%s-m%d-p%d-%s-%s-r%d' % (scene, method, pass_, prior, tr, refine)
    return dict(name=name, scene=scene, kind=kind, w=w, h=h, kw=kw, method=method, pass_=pass_, prior=prior, tr=tr,
                refine=refine, expect=expect)


def _cases():
    cs = []
    for m in (0, 1, 2):
        for k, bs in enumerate((1, 7, 16, 50, 127, 1300)):          # 1300: one bin wider than the image
            cs.append(_case('blob', 1241, 376, m, k % 2, match_binsize=bs, half_resolution=k // 3))
        for k, r in enumerate((0, 1, 3, 200, 5000)):                # 5000: larger than the image
            cs.append(_case('blob', 1241, 376, m, k % 2, match_radius=r, half_resolution=(k + 1) % 2,
                            expect='some' if r >= 200 else 'any'))
        for k, n in enumerate((1, 2, 5)):
            cs.append(_case('blob', 1242, 375, m, k % 2, nms_n=n, half_resolution=k % 2))
        cs.append(_case('blob', 1241, 376, m, 1, multi_stage=0))
        cs.append(_case('blob', 1241, 376, m, 1, multi_stage=0, half_resolution=0, match_binsize=16))
        for k, (w, h) in enumerate(((1241, 376), (1242, 375), (337, 211), (130, 70), (64, 1000), (2000, 40))):
            cs.append(_case('blob', w, h, m, k % 2, half_resolution=(k + m) % 2,
                            expect='some' if min(w, h) >= 200 else 'any'))
        for kind in ('noise', 'checker', 'stripes'):
            cs.append(_case(kind, 337, 211, m, 1, half_resolution=0, match_binsize=16))
            cs.append(_case(kind, 337, 211, m, 0, half_resolution=1, match_radius=10))
        cs.append(_case('noise', 1241, 376, m, 1, half_resolution=0, match_radius=6, match_binsize=7))
        cs.append(_case('const', 337, 211, m, 1, half_resolution=0))
        cs.append(_case('const', 130, 70, m, 0, half_resolution=1, match_binsize=7))
        cs.append(_case('empty', 337, 211, m, 1, half_resolution=0, expect='some' if m == 0 else 'none'))
        # priors: the oracle's own (from its pass-0 list) and synthetic per-bin ranges
        cs.append(_case('blob', 1241, 376, m, 1, 'oracle'))
        cs.append(_case('blob', 1241, 376, m, 1, 'oracle', half_resolution=0, match_binsize=16))
        for k, bs in enumerate((7, 16, 50)):
            cs.append(_case('blob', 1241, 376, m, k % 2, 'synthetic', match_binsize=bs, half_resolution=k % 2, expect='any'))
        cs.append(_case('checker', 337, 211, m, 1, 'synthetic', half_resolution=0, match_binsize=7, expect='any'))
        # refinement inside visocu_match
        for rf in (1, 2):
            cs.append(_case('blob', 1241, 376, m, 1, refine=rf, half_resolution=0))
            cs.append(_case('blob', 1242, 375, m, 1, 'oracle', refine=rf))
        cs.append(_case('noise', 337, 211, m, 1, refine=2, half_resolution=0, match_binsize=16))
        for dt in (0, 1, 2, 10):
            if m:
                cs.append(_case('blob', 1241, 376, m, dt % 2, match_disp_tolerance=dt, half_resolution=dt // 2 % 2))
    # quad matching with a motion prediction
    for tr in ('move', 'ztiny', 'zzero'):
        for prior in (None, 'oracle', 'synthetic'):
            cs.append(_case('blob', 1242, 376, 2, 1, prior, tr, nms_n=2, half_resolution=0,
                            expect='any' if prior == 'synthetic' or tr != 'move' else 'some'))
        cs.append(_case('blob', 1241, 376, 2, 0, None, tr, expect='any'))
    cs.append(_case('blob', 1242, 376, 2, 1, None, 'move', refine=1, nms_n=2, half_resolution=0))
    cs.append(_case('blob', 1242, 376, 2, 1, None, 'move', refine=2, nms_n=2, half_resolution=0))
    cs.append(_case('noise', 337, 211, 2, 1, None, 'move', half_resolution=0, match_binsize=16, expect='any'))
    c = _case('blob', 1242, 376, 2, 1, None, 'move', nms_n=2, half_resolution=0, f=0.0)      # f = 0: up = cu, vp = cv
    c['name'] += '-f0'
    cs.append(c)
    names = [c['name'] for c in cs]
    assert len(set(names)) == len(names), 'duplicate case'
    return cs


CASES = _cases()


def _synthetic_ranges(nbin, seed):
    """Per-bin ranges whose bounds sit on x.5, one ulp either side of an integer, give zero-width and inverted spans, and
    reach beyond the image and beyond [-1, 65534] (|bound| < 2^31 bins at every bin size)."""
    f = np.float32
    up, dn = lambda x: np.nextafter(f(x), f(np.inf)), lambda x: np.nextafter(f(x), f(-np.inf))
    pairs = [(-20.5, 20.5), (-10, 10), (dn(-7), up(7)), (up(-7), dn(7)), (0, 0), (3, 3), (5, -5), (-2.5, 30.25),
             (-5000, 5000), (-70000, 70000), (-1e6, -9e5), (dn(-1.5), up(2.5)), (-40, 12)]
    rng = np.random.default_rng(seed)
    pick = rng.integers(0, len(pairs), (nbin, 2, 4))
    out = np.zeros((nbin, 16), np.float32)
    lo = np.array([p[0] for p in pairs], np.float32); hi = np.array([p[1] for p in pairs], np.float32)
    out[:, 0:4], out[:, 4:8] = lo[pick[:, 0]], hi[pick[:, 0]]
    out[:, 8:12], out[:, 12:16] = lo[pick[:, 1]], hi[pick[:, 1]]
    return out


def _nbin(w, h, bs):
    return int(np.ceil(np.float32(w) / np.float32(bs))) * int(np.ceil(np.float32(h) / np.float32(bs)))


# ---------------------------------------------------------------------------------------------------------------- oracle
class Oracle:
    """One oracle run per distinct input, kept for the module."""

    def __init__(self):
        self.imgs, self.feats, self.runs = {}, {}, {}

    def images(self, kind, w, h):
        key = (kind, w, h)
        if key not in self.imgs:
            self.imgs[key] = _images(kind, w, h)
        return self.imgs[key]

    def features(self, case):
        if case['scene'] not in self.feats:
            op = O.Params(**case['kw'])
            self.feats[case['scene']] = [O.compute_features(i, op) for i in self.images(case['kind'], case['w'], case['h'])]
        return self.feats[case['scene']]

    def planes(self, case):
        f, half = self.features(case), case['kw']['half_resolution']
        out = {}
        for name, x in zip(('1p', '2p', '1c', '2c'), f):
            out['du' + name] = x['du_full'] if half else x['du']
            out['dv' + name] = x['dv_full'] if half else x['dv']
        return out

    def ranges(self, case):
        """The prior ranges of the case's pass (None: no prior)."""
        if case['prior'] is None:
            return None
        if case['prior'] == 'synthetic':
            return _synthetic_ranges(_nbin(case['w'], case['h'], O.Params(**case['kw']).match_binsize), len(case['scene']))
        first, _ = self.match(dict(case, pass_=0, prior=None, refine=0))
        eff = O.Params(**case['kw']).effective()
        return O.prior_statistics(first, case['method'], self.features(case)[0]['dims'], eff)

    def match(self, case):
        """(raw match list of the case's pass, (scanned entries, window candidates))"""
        key = (case['scene'], case['method'], case['pass_'], case['prior'], case['tr'])
        if key not in self.runs:
            f = self.features(case)
            rec = 'rec1' if case['pass_'] == 0 else 'rec2'
            used = [k in _quad(case['method']) for k in range(4)]
            recs = [f[k][rec] if used[k] else None for k in range(4)]
            self.runs[key] = O.matching(case['method'], *recs, f[0]['dims'], O.Params(**case['kw']).effective(),
                                        ranges=self.ranges(case), tr_delta=TRS[case['tr']], counts=True)
        return self.runs[key]


@pytest.fixture(scope='module')
def oracle():
    return Oracle()


def _device_params(kw):
    vp = V.Params(**kw)
    if vp.half_resolution:
        vp.match_radius = vp.match_radius // 2       # the Matcher constructor's halving (matcher.cpp:59-60)
    return vp


def _match(ctx, quads, method, pass_, ranges=None, trs=None, refine=0, caps=None):
    """visocu_match with a capacity per job, per-job ranges and per-job Tr_delta (None entries allowed).
    Returns (rc, lists)."""
    nj = len(quads)
    q = np.zeros(nj, V.QUAD)
    for k, t in enumerate(quads):
        q[k] = tuple(t)
    caps = np.ascontiguousarray(caps, np.int32)
    outs = [np.zeros(max(int(c), 1), V.P_MATCH) for c in caps]
    optr = (C.c_void_p * nj)(*[o.ctypes.data for o in outs])
    nout = np.zeros(nj, np.int32)
    keep = []
    rptr = tptr = None
    if ranges is not None:
        keep += [np.ascontiguousarray(r, np.float32) for r in ranges]
        rptr = (C.c_void_p * nj)(*[r.ctypes.data for r in keep[-nj:]])
    if trs is not None:
        ts = [None if t is None else np.ascontiguousarray(np.asarray(t, np.float64)[:3, :4]) for t in trs]
        keep += [t for t in ts if t is not None]
        tptr = (C.c_void_p * nj)(*[None if t is None else t.ctypes.data for t in ts])
    rc = V.lib().visocu_match(ctx.h, nj, V._p(q), method, pass_, int(ranges is not None), rptr, tptr, int(refine), optr,
                              V._p(caps), V._p(nout), None)
    return rc, [outs[k][:nout[k]].copy() for k in range(nj)]


def _first_difference(got, want, what):
    if len(got) != len(want):
        return '%s: %d matches, oracle %d' % (what, len(got), len(want))
    g, w = got.view(np.int32).reshape(-1, 12), want.view(np.int32).reshape(-1, 12)
    rows = np.unique(np.argwhere(g != w)[:, 0])
    if not len(rows):
        return '%s: equal' % what
    i = rows[0]
    return '%s: %d differing matches, first #%d: device %s, oracle %s' % (what, len(rows), i, got[i], want[i])


def _push(ctx, case, oracle, n_frames=4):
    ctx.configure(_device_params(case['kw']), case['w'], case['h'], n_frames)
    ctx.push_frames([0, 1, 2, 3], oracle.images(case['kind'], case['w'], case['h']))


def _key_fields(m, method):
    return {0: ('i1p', 'i1c'), 1: ('i1c', 'i2c'), 2: ('i1p', 'i2p', 'i1c', 'i2c')}[method]


def _compare_subpixel(got, want, keep, margin, method, what):
    """Kept sets and integer fields equal except for near-threshold decisions; coordinates within SUBPIXEL_ULPS steps.
    Returns (number of near-threshold exceptions, largest coordinate difference)."""
    kf = _key_fields(got, method)
    key = lambda r: tuple(int(r[f]) for f in kf)
    dev = {key(r): r for r in got}
    ora = {key(r): (r, k, mg) for r, k, mg in zip(want, keep, margin)}
    assert len(dev) == len(got), what + ': duplicate matches'
    near, dmax = 0, 0.0
    for k, (r, kept, mg) in ora.items():
        if (k in dev) != bool(kept):
            assert mg < NEAR, '%s: match %s kept %s on the device, %s by the oracle (decision margin %g)' % (
                what, r, k in dev, bool(kept), mg)
            near += 1
            continue
        if not kept:
            continue
        g = dev[k]
        for f in ('u1c', 'v1c', 'i1p', 'i2p', 'i1c', 'i2c'):
            assert g[f] == r[f], '%s: field %s of %s: device %s' % (what, f, r, g)
        for f in ('u1p', 'v1p', 'u2p', 'v2p', 'u2c', 'v2c'):
            d = abs(float(g[f]) - float(r[f]))
            dmax = max(dmax, d)
            assert d <= SUBPIXEL_ULPS * np.spacing(np.float32(abs(r[f]))), '%s: %s of %s: device %r, oracle %r' % (
                what, f, r, g[f], r[f])
    assert set(dev) <= set(ora), what + ': the device kept a match the oracle never had'
    # the device list keeps the oracle's order
    order = [key(r) for r, kept in zip(want, keep) if key(r) in dev]
    assert order == [key(r) for r in got], what + ': order'
    assert near <= 1 + len(want) // 1000, '%s: %d near-threshold decisions differ' % (what, near)
    return near, dmax


# ---------------------------------------------------------------------------------------------------------------- tests
def test_oracle_side_of_every_case(oracle):
    """The case table is meaningful: cases with structure give matches, a frame without features in a needed set gives
    none, every method meets every value of every axis, and the window test rejects candidates somewhere (the
    counters differ)."""
    assert len(CASES) > 150
    bad = []
    for case in CASES:
        got, (scanned, cand) = oracle.match(case)
        if case['expect'] == 'some' and len(got) < 10:
            bad.append((case['name'], len(got)))
        if case['expect'] == 'none' and (len(got) or scanned):
            bad.append((case['name'], len(got)))
        assert cand <= scanned, case['name']
    assert not bad, 'unexpected match counts: %s' % bad
    for m in (0, 1, 2):
        for kind in ('checker', 'stripes', 'const'):
            assert sum(len(oracle.match(c)[0]) for c in CASES if c['method'] == m and c['kind'] == kind) > 0, (m, kind)
    for m in (0, 1, 2):
        mine = [c for c in CASES if c['method'] == m]
        for axis, values in (('match_binsize', (1, 7, 16, 50, 127)), ('match_radius', (0, 1, 3, 200, 5000)),
                             ('half_resolution', (0, 1)), ('multi_stage', (0,))):
            assert {c['kw'].get(axis) for c in mine} >= set(values), (m, axis)
        assert {c['pass_'] for c in mine} == {0, 1} and {c['refine'] for c in mine} == {0, 1, 2}
        assert {c['prior'] for c in mine} == {None, 'oracle', 'synthetic'}
        assert {c['kind'] for c in mine} >= {'blob', 'noise', 'checker', 'stripes', 'const', 'empty'}
        if m:
            assert {c['kw'].get('match_disp_tolerance') for c in mine} >= {0, 1, 2, 10}
    # degenerate predictions really leave every predicted hop at feature 0: the result differs from the plain search
    c = next(c for c in CASES if c['tr'] == 'ztiny' and c['prior'] is None)
    assert oracle.match(c)[0].tobytes() != oracle.match(dict(c, tr=None))[0].tobytes()


def test_refine_lists_reach_every_limit():
    """The hand-built refinement lists cover both sides of every early-return limit."""
    for w, h in ((337, 211), (1241, 376)):
        us, vs = _edge_coords(w), _edge_coords(h)
        for lim in (MARGIN + 2, MARGIN + 3):
            assert {lim - 1, lim} <= set(us) and {w - 1 - lim, w - lim} <= set(us)
            assert {lim - 1, lim} <= set(vs) and {h - 1 - lim, h - lim} <= set(vs)


@pytest.mark.gpu
@pytest.mark.parametrize('case', CASES, ids=[c['name'] for c in CASES])
def test_match_equals_oracle(ctx, oracle, case):
    method, pass_, refine = case['method'], case['pass_'], case['refine']
    raw, (scanned, cand) = oracle.match(case)
    _push(ctx, case, oracle)
    ranges = oracle.ranges(case)
    ctx.match_stats()
    rc, got = _match(ctx, [_quad(method)], method, pass_, None if ranges is None else [ranges],
                     None if case['tr'] is None else [TRS[case['tr']]], refine, [len(raw) + 1])
    assert rc == 0, V.lib().visocu_last_error(ctx.h)
    got = got[0]
    assert ctx.match_stats() == (cand, scanned), 'counters (window candidates, scanned entries)'
    if refine == 0:
        want = raw
    elif refine == 1:
        want = O.refine_pixel(raw, method, oracle.features(case)[0]['dims'], oracle.planes(case))
    else:
        want, keep, margin = O.refine_subpixel(raw, method, oracle.features(case)[0]['dims'], oracle.planes(case))
        near, dmax = _compare_subpixel(got, want, keep, margin, method, case['name'])
        print('sub-pixel %s: %d kept, %d near-threshold, max coordinate difference %.3g' % (case['name'], keep.sum(), near, dmax))
        return
    assert got.tobytes() == want.tobytes(), _first_difference(got, want, case['name'])


def _edge_coords(n):
    """Integer coordinates on both sides of the early-return limits of relocateMinimum (MARGIN + 2) and
    parabolicFitting (MARGIN + 3), at both ends of an axis of length n, plus a few inside."""
    near = [c for lim in (MARGIN + 2, MARGIN + 3) for c in range(lim - 3, lim + 4)]
    return sorted(set(near + [n - 1 - c for c in near] + [n // 3, n // 2]))


@pytest.mark.gpu
@pytest.mark.parametrize('w,h,half', [(337, 211, 0), (1241, 376, 1)])
@pytest.mark.parametrize('method', [0, 1, 2])
def test_refine_hand_built_lists(ctx, oracle, w, h, half, method):
    """visocu_refine (pixel and sub-pixel) on lists whose points lie on every coordinate around the early-return limits,
    and on true matches displaced by up to 3 pixels (minima on the border of the 7x7 search)."""
    case = _case('blob', w, h, method, 1, half_resolution=half)
    _push(ctx, case, oracle)
    f = oracle.features(case)
    dims = f[0]['dims']
    rng = np.random.default_rng(7 + method)
    anchors = f[2]['rec2'][rng.choice(len(f[2]['rec2']), 64)]
    us, vs = _edge_coords(w), _edge_coords(h)
    rows = []
    for k, (u2, v2) in enumerate([(u, v) for u in us for v in (vs[0], vs[len(vs) // 2], vs[-1])] +
                                 [(u, v) for v in vs for u in (us[0], us[len(us) // 2], us[-1])]):
        a = anchors[k % len(anchors)]
        rows.append((u2, v2, a[0], a[1]))
    raw = oracle.match(dict(case, pass_=1, prior=None, tr=None, refine=0))[0]
    for k, r in enumerate(raw[:300]):
        dx, dy = k % 7 - 3, k // 7 % 7 - 3
        src = {0: ('u1p', 'v1p'), 1: ('u2c', 'v2c'), 2: ('u2c', 'v2c')}[method]
        rows.append((r[src[0]] + dx, r[src[1]] + dy, r['u1c'], r['v1c']))
    m = np.zeros(len(rows), V.P_MATCH)
    for k, (u2, v2, u1, v1) in enumerate(rows):
        m[k] = (u2, v2, k, u2, v2, k, u1, v1, k, u2, v2, k)
    want = O.refine_pixel(m, method, dims, oracle.planes(case))
    got = ctx.refine(_quad(method), method, m, 1)
    assert got.tobytes() == want.tobytes(), _first_difference(got, want, 'pixel refinement')
    assert (want['u1p'] != m['u1p']).any() or (want['u2c'] != m['u2c']).any()
    want, keep, margin = O.refine_subpixel(m, method, dims, oracle.planes(case))
    got = ctx.refine(_quad(method), method, m, 2)
    assert 0 < keep.sum() < len(keep)
    near, dmax = _compare_subpixel(got, want, keep, margin, method, 'sub-pixel refinement')
    print('hand-built sub-pixel m%d %dx%d: %d kept, %d near-threshold, max coordinate difference %.3g' % (
        method, w, h, keep.sum(), near, dmax))


# ---------------------------------------------------------------------------------------------------------------- batches
def _batch_frames(oracle):
    """Nine frames: two different blob quads (0-3, 4-7) and a constant image without features (8)."""
    return oracle.images('blob', 1241, 376) + list(synth.blob_quad(1241, 376, seed=63, shift=(-2, 2), disparity=7)) + \
        [np.full((376, 1241), 128, np.uint8)]


@pytest.mark.gpu
@pytest.mark.parametrize('method', [0, 1, 2])
@pytest.mark.parametrize('n_jobs', [1, 3, 128, 129, 300])
def test_batches_equal_single_jobs(ctx, oracle, method, n_jobs):
    """Ragged batches: jobs over two different quads, mixed quads that share frames, jobs with an empty needed set, per-job
    ranges (none, the oracle's, synthetic) and for quad matching per-job Tr_delta with null entries.  Every list equals the
    oracle's and the counters sum over the jobs."""
    imgs = _batch_frames(oracle)
    kw = dict(half_resolution=1)
    ctx.configure(_device_params(kw), 1241, 376, 9)
    ctx.push_frames(list(range(9)), imgs)
    op = O.Params(**kw)
    feats = [O.compute_features(i, op) for i in imgs] if 'batch_feats' not in oracle.feats else oracle.feats['batch_feats']
    oracle.feats['batch_feats'] = feats
    dims = feats[0]['dims']
    nbin = _nbin(1241, 376, op.match_binsize)
    quads = [(0, 1, 2, 3), (4, 5, 6, 7), (0, 1, 6, 7), (4, 5, 2, 3), (8, 1, 2, 3), (0, 1, 2, 8), (2, 3, 6, 7)]
    rsets = [None, 'oracle', 'synthetic']
    jobs = [(quads[(3 * j + j // 7) % len(quads)], rsets[j % 3], [None, 'move', None, 'ztiny'][j % 4] if method == 2 else None)
            for j in range(n_jobs)]
    cache = oracle.runs.setdefault('batch', {})

    def run(q, prior, tr):
        key = (method, q, prior, tr)
        if key not in cache:
            need = [k in [i for i, f in enumerate(_quad(method)) if f >= 0] for k in range(4)]
            recs = [feats[q[k]]['rec2'] if need[k] else None for k in range(4)]
            rng = None
            if prior == 'synthetic':
                rng = _synthetic_ranges(nbin, sum(q))
            elif prior == 'oracle':
                first = O.matching(method, *[feats[q[k]]['rec1'] if need[k] else None for k in range(4)], dims, op.effective())
                rng = O.prior_statistics(first, method, dims, op.effective())
            raw, cnt = O.matching(method, *recs, dims, op.effective(), ranges=rng, tr_delta=TRS[tr], counts=True)
            cache[key] = (raw, cnt, rng if rng is not None else np.zeros((nbin, 16), np.float32))
        return cache[key]

    want = [run(q, p, t) for q, p, t in jobs]
    dq = [tuple(f if f >= 0 and _quad(method)[k] >= 0 else -1 for k, f in enumerate(q)) for q, _, _ in jobs]
    ctx.match_stats()
    # a job without a prior gets ranges it does not read only if the call passes ranges at all: one call with, one without
    for with_prior in (False, True):
        sel = [j for j in range(n_jobs) if (jobs[j][1] is not None) == with_prior]
        if not sel:
            continue
        rc, got = _match(ctx, [dq[j] for j in sel], method, 1, [want[j][2] for j in sel] if with_prior else None,
                         [TRS[jobs[j][2]] for j in sel] if method == 2 else None, 0, [len(want[j][0]) + 1 for j in sel])
        assert rc == 0, V.lib().visocu_last_error(ctx.h)
        for k, j in enumerate(sel):
            assert got[k].tobytes() == want[j][0].tobytes(), _first_difference(got[k], want[j][0], 'job %d %s' % (j, jobs[j]))
    scanned = sum(w[1][0] for w in want); cand = sum(w[1][1] for w in want)
    assert ctx.match_stats() == (cand, scanned)
    assert any(len(w[0]) for w in want)
    if n_jobs > len(quads):
        assert any(len(w[0]) == 0 for w in want)         # the jobs with an empty needed set


@pytest.mark.gpu
def test_capacity_and_per_list_copy(ctx, oracle):
    """128 jobs over two full-resolution noise frames: the staging buffer would exceed 64 MB, so the lists are copied one
    by one; and a call with room for one match less than the oracle finds returns VISOCU_ECAPACITY."""
    case = _case('noise', 1241, 376, 0, 1, half_resolution=0, match_radius=3, match_binsize=16)
    raw, (scanned, cand) = oracle.match(case)
    nq = len(oracle.features(case)[2]['rec2'])
    assert len(raw) > 100 and (nq + 1) * 48 * 128 > 64 << 20
    _push(ctx, case, oracle)
    ctx.match_stats()
    rc, got = _match(ctx, [_quad(0)] * 128, 0, 1, caps=[len(raw)] * 128)
    assert rc == 0, V.lib().visocu_last_error(ctx.h)
    for j in range(128):
        assert got[j].tobytes() == raw.tobytes(), _first_difference(got[j], raw, 'job %d' % j)
    assert ctx.match_stats() == (128 * cand, 128 * scanned)
    rc, _ = _match(ctx, [_quad(0)], 0, 1, caps=[len(raw) - 1])
    assert rc == ECAPACITY


# ---------------------------------------------------------------------------------------------------------------- fused
def _cell_count(length, n):
    s = length - 2 * n - 12
    return (s + n) // (n + 1) if s > 0 else 0


def _expected_layout(w, h, kw):
    """What fused_layout / k_deliver pick: 2 = 12 bytes per match, 1 = 24 bytes, 0 = lists copied after the header."""
    p = V.Params(**kw)
    wm, hm = (w // 2, h // 2) if p.half_resolution else (w, h)
    ns = p.nms_n * 3
    if ns > 10:
        ns = max(p.nms_n, 10)
    cap = [4 * _cell_count(wm, n) * _cell_count(hm, n) + 32 for n in (ns, p.nms_n)]
    al = lambda x: (x + 255) // 256 * 256
    full = 256 + al((cap[0] + 1) * 48) + al((cap[1] + 1) * 48)
    if full > 8 << 20:
        return 0
    return 2 if max(cap) <= 0xFFFF else 1


FUSED = [(1241, 376, dict(), 1), (1241, 376, dict(), 128), (1241, 376, dict(half_resolution=0), 3),
         (1241, 376, dict(half_resolution=0, nms_n=1), 2), (1241, 376, dict(half_resolution=0, nms_n=1), 128)]


@pytest.mark.gpu
@pytest.mark.parametrize('refine', [0, 1])
@pytest.mark.parametrize('w,h,kw,n_jobs', FUSED, ids=['%dx%d-%s-j%d' % (w, h, '-'.join('%s%s' % i for i in kw.items()), n)
                                                      for w, h, kw, n in FUSED])
def test_fused_flow_equals_oracle_chain(ctx, oracle, w, h, kw, n_jobs, refine):
    """visocu_match_fused: both survivor lists and the prior ranges equal the Matcher chain on the oracle (pass 0,
    removeOutliers, prior statistics, pass 1, pixel refinement, removeOutliers) in every delivery layout.

    The outlier kernel may decline a list (for example one too long for a CTA): it is then delivered whole and the Matcher
    finishes the job on the host (Matcher::takeFused).  A declined first list stops the fused second pass (no queries, and
    the ranges of an empty list); the Matcher removes the outliers of the first list, computes the ranges and repeats
    pass 1.  A declined second list gets its outliers removed on the host.  Both branches are followed here."""
    kw = dict(kw, refinement=refine)
    case = _case('blob', w, h, 0, 0, **kw)
    f = oracle.features(case)
    op = O.Params(**case['kw'])
    eff = op.effective()
    dims = f[0]['dims']
    hm = H.Matcher(V.Params(**case['kw']))
    key = ('fused', case['scene'])
    if key not in oracle.runs:
        raw1 = O.matching(0, f[0]['rec1'], None, f[2]['rec1'], None, dims, eff)
        l1 = hm.remove_outliers(raw1, 0)
        rng = O.prior_statistics(l1, 0, dims, eff)
        raw2 = O.matching(0, f[0]['rec2'], None, f[2]['rec2'], None, dims, eff, ranges=rng)
        if refine:
            raw2 = O.refine_pixel(raw2, 0, dims, oracle.planes(case))
        oracle.runs[key] = (raw1, l1, rng, len(raw2), hm.remove_outliers(raw2, 0),
                            O.prior_statistics(np.zeros(0, O.P_MATCH), 0, dims, eff))
    raw1, l1, rng, n_raw2, l2, rng_empty = oracle.runs[key]
    assert len(l1) > 20 and len(l2) > 100
    _push(ctx, case, oracle)
    nbin = len(rng)
    q = np.zeros(n_jobs, V.QUAD)
    q[:] = (0, -1, 2, -1)
    p1 = (C.c_void_p * n_jobs)(); p2 = (C.c_void_p * n_jobs)()
    n1, d1, n2, d2 = (np.zeros(n_jobs, np.int32) for _ in range(4))
    rout = [np.zeros((nbin, 16), np.float32) for _ in range(n_jobs)]
    rptr = (C.c_void_p * n_jobs)(*[r.ctypes.data for r in rout])
    counts = np.zeros(4 * n_jobs, np.int32); compact = C.c_int32(-1)
    rc = V.lib().visocu_match_fused(ctx.h, n_jobs, V._p(q), refine, p1, V._p(n1), V._p(d1), p2, V._p(n2), V._p(d2), rptr,
                                    V._p(counts), C.byref(compact))
    assert rc == 0, V.lib().visocu_last_error(ctx.h)
    assert compact.value == _expected_layout(w, h, case['kw']), 'delivery layout'
    words = {2: 3, 1: 6, 0: 12}[compact.value]
    lists = []
    for j in range(n_jobs):
        got1 = np.frombuffer((C.c_uint8 * (48 * int(n1[j]))).from_address(p1[j]), V.P_MATCH).copy() if n1[j] else np.zeros(0, V.P_MATCH)
        raw = np.frombuffer((C.c_uint32 * (words * int(n2[j]))).from_address(p2[j]), np.uint32).reshape(-1, words).copy() \
            if n2[j] else np.zeros((0, words), np.uint32)
        got2 = np.zeros(len(raw), V.P_MATCH)
        for fld in ('u2p', 'v2p', 'i2p', 'u2c', 'v2c', 'i2c'):
            got2[fld] = -1
        if words == 12:
            got2 = raw.view(V.P_MATCH).reshape(-1).copy()
        elif words == 6:
            for k, fld in enumerate(('u1p', 'v1p', 'i1p', 'u1c', 'v1c', 'i1c')):
                got2[fld] = raw[:, k].copy().view(np.float32 if fld[0] != 'i' else np.int32)
        else:
            got2['u1p'], got2['v1p'] = raw[:, 0] & 0xFFFF, raw[:, 0] >> 16
            got2['u1c'], got2['v1c'] = raw[:, 1] & 0xFFFF, raw[:, 1] >> 16
            got2['i1p'], got2['i1c'] = raw[:, 2] & 0xFFFF, raw[:, 2] >> 16
        lists.append((got1, got2))
    redo = None
    for j in range(n_jobs):
        got1, got2 = lists[j]
        assert counts[4 * j:4 * j + 4].tolist() == [len(f[0]['rec1']), len(f[0]['rec2']), len(f[2]['rec1']), len(f[2]['rec2'])]
        if d1[j]:
            assert got1.tobytes() == l1.tobytes(), _first_difference(got1, l1, 'job %d list 1' % j)
            assert rout[j].tobytes() == rng.tobytes(), 'job %d: prior ranges' % j
            if not d2[j]:
                got2 = hm.remove_outliers(got2, 0)
        else:
            assert got1.tobytes() == raw1.tobytes(), _first_difference(got1, raw1, 'job %d declined list 1' % j)
            assert hm.remove_outliers(got1, 0).tobytes() == l1.tobytes(), 'job %d: list 1 after removeOutliers' % j
            assert len(got2) == 0, 'job %d: the second pass ran on a declined first list' % j
            assert rout[j].tobytes() == rng_empty.tobytes(), 'job %d: prior ranges of the stopped second pass' % j
            if redo is None:                 # the Matcher's repeat of pass 1 with the host's ranges
                rc, got = _match(ctx, [(0, -1, 2, -1)], 0, 1, [rng], None, refine, [n_raw2 + 1])
                assert rc == 0, V.lib().visocu_last_error(ctx.h)
                redo = hm.remove_outliers(got[0], 0)
            got2 = redo
        assert got2.tobytes() == l2.tobytes(), _first_difference(got2, l2, 'job %d list 2' % j)
    print('fused %dx%d %s j%d r%d: layout %d, first lists declined %d, second lists declined %d' % (
        w, h, kw, n_jobs, refine, compact.value, n_jobs - int(d1.sum()), int((d1 & (1 - d2)).sum())))
