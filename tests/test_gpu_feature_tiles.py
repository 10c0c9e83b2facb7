"""The feature front end (fused filter + NMS kernel, ordered compaction, bin index) against the plain-C restatement
oracle/viso_oracle.c, bit for bit, at every tile configuration, load path and launch size.

k_filter_nms cuts each image into tiles, and the cut is not fixed: visocu_configure builds up to three tile levels and a
push launch runs the largest one that still gives about one CTA per SM, so the tiles that run depend on how many frames
one launch carries.  VISOCU_TILE pins one tile shape, VISOCU_TMA=0 stages tiles with plain loads and
VISOCU_FUSED_HALF=0 runs half-resolution mode with separate half-image and Sobel kernels.  Every execution variant of a
case must give the oracle's results for the same image and parameters:

  * the record counts of the push, and the sparse / dense records (order included);
  * the whole du / dv planes (the oracle defines every byte: zero padding behind each row, 128 on the two-pixel border),
    in half-resolution mode also the full-resolution planes and the half image;
  * one flow matching pass on frames (0, 1), which checks the bins the push built: pass 0 (sparse) with multi_stage,
    else pass 1 without priors.

Nothing is masked: the oracle pads every row with zeros as the device does, so descriptor word 11 of maxima at
u = w-7, which test_gpu_parity masks against the reference (that one reads uninitialised pad bytes there), is compared
too.  The oracle runs once per distinct (image, parameters), cached for the module."""
import numpy as np
import pytest

import synth
import pyoracle as O
import visocu_py as V

MAX_BATCH = 128                    # VISO_MAX_BATCH: a push of more frames is split into launches of at most this many
TAU_ABOVE_ALL = 4081               # |blob| <= 16 * 255 = 4080, |checkerboard| <= 8 * 255: no response reaches this


# ---------------------------------------------------------------------------------------------------------------- inputs
def _shift(img, dx, dy):
    return np.ascontiguousarray(np.roll(np.roll(img, dy, axis=0), dx, axis=1))


def _checker(w, h, p, ox=0, oy=0):
    y, x = np.mgrid[0:h, 0:w]
    return ((((x + ox) // p + (y + oy) // p) % 2) * 255).astype(np.uint8)


def _images(kind, w, h):
    """Four distinct images (a, b, c, d) of one content; (a, b) is the pair the matching pass runs on, b is a moved."""
    if kind == 'blob':
        a, b = synth.blob_pair(w, h, seed=41)
        c, d = synth.blob_pair(w, h, seed=42)
    elif kind == 'noise':            # uniform noise: a maximum in nearly every cell
        rng = np.random.default_rng(43)
        big = rng.integers(0, 256, (h + 8, w + 8), dtype=np.uint8)
        a, b = big[4:4 + h, 4:4 + w], big[3:3 + h, 1:1 + w]
        c, d = rng.integers(0, 256, (2, h, w), dtype=np.uint8)
    elif kind == 'checker':          # saturated 0/255 squares: equal responses one period apart (NMS ties)
        a = _checker(w, h, 3)
        b, c, d = _checker(w, h, 3, 1, 2), _checker(w, h, 2), _checker(w, h, 5, 2, 0)
    elif kind == 'stripes':          # saturated stripes: equal responses all along a stripe
        y, x = np.mgrid[0:h, 0:w]
        a = ((x // 3) % 2 * 255).astype(np.uint8)
        b = _shift(a, 2, 0)
        c = ((y // 3) % 2 * 255).astype(np.uint8)
        d = (((x + y) // 4) % 2 * 255).astype(np.uint8)
    elif kind == 'const':            # no response anywhere
        a, b, c, d = (np.full((h, w), v, np.uint8) for v in (128, 0, 255, 77))
    else:
        raise ValueError(kind)
    return [np.ascontiguousarray(i, np.uint8) for i in (a, b, c, d)]


# ---------------------------------------------------------------------------------------------------------------- cases
# execution variants: (environment, frame slots, launches); a launch is the list of image indices of one push call, the
# frames of a push fill the slots in order.  Frames 0 and 1 always hold images 0 and 1.
VARIANTS = {
    'single': ({}, 2, [[0], [1]]),                                     # one frame per launch
    'b128': ({}, 128, [[k % 4 for k in range(128)]]),                  # one full launch
    'b129': ({}, 129, [[k % 4 for k in range(129)]]),                  # one push, split 128 + 1
    'tile1x1t32': ({'VISOCU_TILE': '1,1,32'}, 2, [[0, 1]]),
    'tilewide': ({'VISOCU_TILE': '200,3,256'}, 2, [[0, 1]]),          # wider than any image here: the shrink loop runs
    'tile3x2t64': ({'VISOCU_TILE': '3,2,64'}, 2, [[0, 1]]),
    'tile7x5t128': ({'VISOCU_TILE': '7,5,128'}, 2, [[0, 1]]),
    'tile40x1': ({'VISOCU_TILE': '40,1,256'}, 2, [[0, 1]]),
    'tile1x40': ({'VISOCU_TILE': '1,40,256'}, 2, [[0, 1]]),
    'tile4x3t512': ({'VISOCU_TILE': '4,3,512'}, 2, [[0, 1]]),
    # the other load paths, each at launches of 1, 9 and 20 frames (three different levels at 1241x376)
    'tma0': ({'VISOCU_TMA': '0'}, 30, [[0], [1] + [k % 4 for k in range(2, 10)], [k % 4 for k in range(20)]]),
    'fused0': ({'VISOCU_FUSED_HALF': '0'}, 30, [[0], [1] + [k % 4 for k in range(2, 10)], [k % 4 for k in range(20)]]),
}
ALL = list(VARIANTS)


def _case(w, h, kind='blob', variants=ALL, **kw):
    kw.setdefault('half_resolution', 1)
    if kind != 'blob':
        kw.setdefault('match_radius', 20)      # dense contents: keeps the oracle's matching pass short
    vs = [v for v in variants if v != 'fused0' or kw['half_resolution']]
    name = '%dx%d-%s-%s' % (w, h, kind, '-'.join('%s%d' % (k.replace('_', '')[:5], v) for k, v in sorted(kw.items())))
    return dict(name=name, w=w, h=h, kind=kind, kw=kw, variants=vs)


def _cases():
    cs = []
    sizes = [(1241, 376), (1242, 375),
             (1248, 376), (1249, 376), (1247, 376),             # w % 16 = 0, 1, 15; 1249: bpl > 2 bplm at half resolution
             (337, 211), (130, 70), (64, 1000), (2000, 40)]
    for half in (1, 0):
        for w, h in sizes:
            cs.append(_case(w, h, half_resolution=half))
        # the smallest image with cells in both passes (sparse n = 9: 31 samples at matching resolution)
        m = 62 if half else 31
        cs.append(_case(m, m, 'noise', ['single', 'b128', 'b129', 'tile1x1t32', 'tilewide', 'tma0', 'fused0'], half_resolution=half))
        # every NMS size (sparse n = min(3 n, max(10, n)))
        for n in range(1, 15):
            if n != 3:
                cs.append(_case(1241, 376, variants=['single', 'b128', 'tile3x2t64', 'tma0', 'fused0'], nms_n=n, half_resolution=half))
        # thresholds: 0 (every cell extreme is a candidate, clamped windows take the plain scan), 1, above every response
        for tau in (0, 1, TAU_ABOVE_ALL):
            for kind in ('blob', 'noise', 'const'):
                cs.append(_case(1241, 376, kind, ['single', 'b128', 'tma0', 'fused0'], nms_tau=tau, half_resolution=half))
        for kind in ('noise', 'checker', 'stripes', 'const'):
            cs.append(_case(1241, 376, kind, half_resolution=half))
            cs.append(_case(337, 211, kind, ['single', 'b128', 'tile7x5t128'], half_resolution=half))
        # dense pass only: the tiles align to the dense cells
        cs.append(_case(1241, 376, multi_stage=0, half_resolution=half))
        for kind in ('noise', 'checker'):
            cs.append(_case(1241, 376, kind, ['single', 'b128', 'tile3x2t64', 'tma0', 'fused0'], multi_stage=0, half_resolution=half))
        m = 38 if half else 19
        cs.append(_case(130, 70, variants=['single', 'b128', 'b129', 'tile1x1t32', 'tilewide'], multi_stage=0, half_resolution=half))
        cs.append(_case(m, m, 'noise', ['single', 'b128', 'b129', 'tile1x1t32', 'tilewide'], multi_stage=0, half_resolution=half))
    cs.append(_case(1249, 376, 'checker', half_resolution=1))
    cs.append(_case(655, 200, 'noise', ['single', 'b128', 'tile7x5t128', 'tma0', 'fused0'], half_resolution=1))
    names = [c['name'] for c in cs]
    assert len(set(names)) == len(names), 'duplicate case'
    return cs


CASES = _cases()
RUNS = [(c, v) for c in CASES for v in c['variants']]


# ---------------------------------------------------------------------------------------------------------------- oracle
class Oracle:
    """One oracle run per distinct (content, size, parameters, image)."""

    def __init__(self):
        self.imgs, self.feats, self.matches = {}, {}, {}

    def images(self, case):
        key = (case['kind'], case['w'], case['h'])
        if key not in self.imgs:
            self.imgs[key] = _images(*key)
        return self.imgs[key]

    def features(self, case, k):
        key = (case['name'], k)
        if key not in self.feats:
            f = O.compute_features(self.images(case)[k], O.Params(**case['kw']))
            if case['kw']['half_resolution']:
                f['half'] = O.half_image(O.pad(self.images(case)[k]), case['w'])[0]
            self.feats[key] = f
        return self.feats[key]

    def flow(self, case):
        if case['name'] not in self.matches:
            op = O.Params(**case['kw'])
            fa, fb = self.features(case, 0), self.features(case, 1)
            r = 'rec1' if op.multi_stage else 'rec2'
            self.matches[case['name']] = O.matching(0, fa[r], None, fb[r], None, fa['dims'], op.effective())
        return self.matches[case['name']]


@pytest.fixture(scope='module')
def oracle():
    return Oracle()


def _cell_count(length, n):
    """NMS cells along one axis (viso_cell_count: origins n + margin, n + margin + n + 1, ... below length - n - margin)"""
    s = length - 2 * n - 12
    return (s + n) // (n + 1) if s > 0 else 0


def _device_params(kw):
    vp = V.Params(**kw)
    if vp.half_resolution:
        vp.match_radius = vp.match_radius // 2       # the Matcher constructor's halving (matcher.cpp:59-60)
    return vp


def _first_difference(got, want, what):
    if got.shape != want.shape:
        return '%s: shape %s, oracle %s' % (what, got.shape, want.shape)
    idx = np.argwhere(got != want)
    return '%s: %d differing entries, first at %s: device %s, oracle %s' % (
        what, len(idx), tuple(idx[0]), got[tuple(idx[0])], want[tuple(idx[0])])


def _records_difference(got, want, wm, scale):
    msg = _first_difference(got, want, 'records')
    if got.shape == want.shape:
        rows = np.unique(np.argwhere(got != want)[:, 0])
        msg += '; first differing record: device %s, oracle %s' % (got[rows[0]].tolist(), want[rows[0]].tolist())
        # the parity tests mask descriptor word 11 of maxima at u = w-7 (the reference reads pad bytes there)
        g, o = got.copy(), want.copy()
        g[(g[:, 0] // scale) >= wm - 7, 11] = 0
        o[(o[:, 0] // scale) >= wm - 7, 11] = 0
        if np.array_equal(g, o):
            msg += ' (only descriptor word 11 at u = w-7 differs)'
    return msg


# ---------------------------------------------------------------------------------------------------------------- tests
def test_oracle_side_of_every_case(oracle):
    """The case table is meaningful: a content with structure gives features in every pass that has cells (over the
    case's four images), a constant image gives none unless tau = 0 (then all four classes in every cell), tau above every
    response gives none, and the blob pairs give matches."""
    assert len(RUNS) > 400
    empty = []
    for case in CASES:
        op = O.Params(**case['kw'])
        wm, hm = (case['w'] // 2, case['h'] // 2) if op.half_resolution else (case['w'], case['h'])
        for p, rec in ((0, 'rec1'), (1, 'rec2')):
            n = min(3 * op.nms_n, max(10, op.nms_n)) if p == 0 else op.nms_n
            cells = _cell_count(wm, n) * _cell_count(hm, n) if p == 1 or op.multi_stage else 0
            assert p == 0 or cells > 0, case['name']
            nf = [len(oracle.features(case, k)[rec]) for k in range(4)]
            if op.nms_tau >= TAU_ABOVE_ALL or cells == 0:
                assert nf == [0] * 4, (case['name'], p)
            elif case['kind'] == 'const':
                assert nf == [4 * cells if op.nms_tau == 0 else 0] * 4, (case['name'], p)
            elif sum(nf) == 0:
                empty.append((case['name'], p))
        if case['kind'] == 'blob' and op.nms_tau < TAU_ABOVE_ALL and min(case['w'], case['h']) >= 200:
            assert len(oracle.flow(case)) > 20, case['name']
    assert not empty, 'no features: %s' % empty


@pytest.mark.gpu
@pytest.mark.parametrize('half', [1, 0])
def test_launch_size_picks_tile_level(ctx, half):
    """Which tiles run at 1241x376: the levels visocu_configure builds and, for every launch size, the level a push launch
    runs on (the largest whose tiles give the launch at least one CTA per SM).  On a 148-SM B200 the parity tests' launches
    of at most 6 frames all run the smallest level."""
    ctx.configure(_device_params(dict(half_resolution=half)), 1241, 376, 2)
    levels, _ = ctx.tile_levels(1)
    tiles = [lv['ntx'] * lv['nty'] for lv in levels]
    assert len(levels) == 3 and tiles == sorted(tiles)
    assert tiles == ([8, 18, 36] if half else [36, 78, 156])
    sm = ctx.device_info()['sm_count']
    for n in range(1, MAX_BATCH + 1):
        want = next((k for k, t in enumerate(tiles) if t * n >= sm), len(tiles) - 1)
        assert ctx.tile_levels(n)[1] == want, n
    if sm == 148:
        first = [min(n for n in range(1, MAX_BATCH + 1) if ctx.tile_levels(n)[1] <= k) for k in range(3)]
        assert first == ([19, 9, 1] if half else [5, 2, 1])
        assert all(ctx.tile_levels(n)[1] == 2 for n in range(1, 7)) if half else ctx.tile_levels(1)[1] == 2


@pytest.mark.gpu
@pytest.mark.parametrize('case,variant', RUNS, ids=['%s-%s' % (c['name'], v) for c, v in RUNS])
def test_features_match_oracle(ctx, oracle, monkeypatch, case, variant):
    env, n_slots, launches = VARIANTS[variant]
    for k in ('VISOCU_TILE', 'VISOCU_TMA', 'VISOCU_FUSED_HALF'):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    w, h, kw = case['w'], case['h'], case['kw']
    vp = _device_params(kw)
    half, multi = bool(kw['half_resolution']), bool(vp.multi_stage)
    scale = 2 if half else 1
    imgs = oracle.images(case)
    ctx.configure(vp, w, h, n_slots)
    slot_img, counts, picks, slot = [], [], [], 0
    for ids in launches:
        frames = list(range(slot, slot + len(ids)))
        ns, nd = ctx.push_frames(frames, [imgs[i] for i in ids])
        picks.append(ctx.tile_levels(min(len(ids), MAX_BATCH))[1])
        slot_img += ids; counts += list(zip(ns.tolist(), nd.tolist())); slot += len(ids)
    assert slot == n_slots
    where = 'launch levels %s of %s' % (picks, ctx.tile_levels(1)[0])
    for f, k in enumerate(slot_img):
        want = oracle.features(case, k)
        at = 'frame %d (image %d), %s' % (f, k, where)
        assert counts[f] == (len(want['rec1']), len(want['rec2'])), 'counts, ' + at
        for p, rec in ((0, 'rec1'), (1, 'rec2')):
            if p == 0 and not multi:
                continue
            got = ctx.features(f, p)
            assert np.array_equal(got, want[rec]), 'pass %d %s, %s' % (p, _records_difference(got, want[rec], w // scale, scale), at)
        planes = [(0, 'du'), (1, 'dv')] + ([(2, 'du_full'), (3, 'dv_full'), (5, 'half')] if half else [])
        for which, name in planes:
            got, (gw, gh, gb) = ctx.plane(f, which)
            assert (gh, gb) == want[name].shape, '%s dims, %s' % (name, at)
            assert np.array_equal(got, want[name]), '%s, %s' % (_first_difference(got, want[name], name), at)
    got = ctx.match([(0, -1, 1, -1)], 0, 0 if multi else 1)[0]
    want = oracle.flow(case)
    assert got.tobytes() == want.tobytes(), 'flow matching on frames (0, 1): %d matches, oracle %d, %s' % (len(got), len(want), where)
