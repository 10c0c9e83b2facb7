"""Post-filters of dense disparity (masked 3x3 median and speckle removal, include/visocu.h): the plain-C oracle against an
independent numpy / scipy restatement on crafted maps and on the corridor's ground truth (CPU); visocu_disparity_filter
and visocu_disparity with filters bit for bit against the oracle over sizes, contents, parameters and batch shapes,
argument checks, the runner and the host layer (GPU)."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse
from scipy.sparse.csgraph import connected_components

import disp_filter_oracle
import synth
import sgm_oracle
import visocu_py as V
from test_gpu_disparity import (CONTENTS, SIZES as SGM_SIZES, _stereo_params, content, new_ctx, oracle, sgm_params,
                                size_ctx)  # noqa: F401  (size_ctx is a fixture)

SIZES = [(1, 1), (1, 1000), (1000, 1), (31, 17), (33, 33), (1241, 376), (2000, 40), (64, 1000)]   # (w, h)
KINDS = ('blocky', 'noise', 'invalid', 'const', 'checker', 'serpentine', 'steps', 'edge0', 'exact')
MAX_RANGE = 256                          # largest speckle_range of visocu_disparity_filter
TILE = 32                                # borders of 32 are borders of every power-of-two tile up to 32
# (median, speckle_size, speckle_range); 'wh' = w * h, 'max' = MAX_RANGE
PARAMS = [(0, 0, 0), (1, 0, 0), (0, 1, 0), (1, 50, 1), (0, 50, 2), (1, 200, 'max'), (0, 200, 1), (1, 'wh', 2),
          (0, 'wh', 0), (1, 1, 'max'), (0, 50, 'max'), (1, 200, 0)]


def resolve(prm, w, h):
    m, s, r = prm
    return m, w * h if s == 'wh' else s, MAX_RANGE if r == 'max' else r


def crafted(kind, w, h, size=50, r=2, seed=0):
    """An (h, w) int16 map in 1/16 pixel, -1 = invalid."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    if kind == 'blocky':                 # 6 x 6 regions, jitter of +-12, 5 % holes
        cells = rng.integers(0, 16 * 80, (h // 6 + 1, w // 6 + 1))
        m = cells[y // 6, x // 6] + rng.integers(-12, 13, (h, w))
        m[rng.random((h, w)) < 0.05] = -1
    elif kind == 'noise':
        m = rng.integers(0, 16 * 64, (h, w))
        m[rng.random((h, w)) < 0.1] = -1
    elif kind == 'invalid':
        m = np.full((h, w), -1)
    elif kind == 'const':
        m = np.full((h, w), 300)
    elif kind == 'checker':              # valid / invalid checkerboard: every valid pixel is a component of its own
        m = np.where((x + y) % 2 == 0, rng.integers(0, 2000, (h, w)), -1)
    elif kind == 'serpentine':           # one-pixel-wide serpentine through every tile: all valid pixels are one component
        turn = np.where((y // 4) % 2 == 0, w - 1, 0)
        m = np.where((y % 4 == 0) | (x == turn), 100, -1)
    elif kind == 'steps':                # neighbours exactly 16 r apart on the left, 16 r + 1 on the right
        m = np.where(x < w // 2, ((x + y) % 2) * 16 * r, ((x + y) % 2) * (16 * r + 1))
    elif kind == 'edge0':                # -1 beside values 0 .. 16 r: invalid pixels must connect nothing
        m = rng.integers(0, 16 * r + 1, (h, w))
        m[rng.random((h, w)) < 0.3] = -1
    elif kind == 'exact':                # components of exactly size and size + 1 pixels across tile borders
        m = np.full((h, w), -1)
        busy = np.zeros((h + 2, w + 2), bool)
        base = size if 1 <= size <= 4096 else 50
        j = 0
        for cy in [TILE * k for k in range(1, h // TILE + 1)] or [h // 2]:
            for cx in [TILE * k for k in range(1, w // TILE + 1)] or [w // 2]:
                n = base + (j % 2)
                cw = n if h < 3 else (1 if w < 3 else min(n, 12))
                rows = -(-n // cw)
                x0, y0 = max(cx - cw // 2, 0), max(cy - rows // 2, 0)
                if x0 + cw > w or y0 + rows > h or busy[y0:y0 + rows + 2, x0:x0 + cw + 2].any():
                    continue
                cells = np.zeros(rows * cw, bool)
                cells[:n] = True
                blk = m[y0:y0 + rows, x0:x0 + cw]
                blk[cells.reshape(rows, cw)] = 16 * (5 + j % 7)
                busy[y0 + 1:y0 + rows + 1, x0 + 1:x0 + cw + 1] = True
                j += 1
    else:
        raise ValueError(kind)
    return np.asarray(m).astype(np.int16)


# ----------------------------------------------------------------------------- numpy / scipy restatement
def np_filter(m, median, size, r):
    h, w = m.shape
    m = m.astype(np.int64)
    if median:
        BIG = 1 << 20                    # clipped and invalid samples sort last
        pad = np.pad(np.where(m >= 0, m, BIG), 1, constant_values=BIG)
        stack = np.sort(np.stack([pad[1 + dy:1 + dy + h, 1 + dx:1 + dx + w] for dy in (-1, 0, 1) for dx in (-1, 0, 1)], -1), -1)
        n = (stack < BIG).sum(-1)
        med = np.take_along_axis(stack, np.maximum((n - 1) // 2, 0)[..., None], -1)[..., 0]
        m = np.where(m >= 0, med, m)
    if size > 0:
        idx = np.arange(h * w).reshape(h, w)
        a_all, b_all = [], []
        for a, b, va, vb in ((idx[:, :-1], idx[:, 1:], m[:, :-1], m[:, 1:]), (idx[:-1], idx[1:], m[:-1], m[1:])):
            e = (va >= 0) & (vb >= 0) & (np.abs(va - vb) <= 16 * r)
            a_all.append(a[e]); b_all.append(b[e])
        a, b = np.concatenate(a_all), np.concatenate(b_all)
        g = scipy.sparse.coo_matrix((np.ones(len(a)), (a, b)), shape=(h * w, h * w))
        _, lab = connected_components(g, directed=False)
        small = (np.bincount(lab)[lab] <= size).reshape(h, w)
        m = np.where((m >= 0) & small, -1, m)
    return m.astype(np.int16)


CPU_CASES = [(w, h, kind, PARAMS[(3 * i + j + off) % len(PARAMS)]) for i, (w, h) in enumerate(SIZES)
             for j, kind in enumerate(KINDS) for off in (0, 5)]


@pytest.mark.parametrize('w,h,kind,prm', CPU_CASES, ids=['%dx%d-%s-m%s-s%s-r%s' % ((w, h, k) + p) for w, h, k, p in CPU_CASES])
def test_oracle_equals_numpy(w, h, kind, prm):
    med, size, r = resolve(prm, w, h)
    m = crafted(kind, w, h, size, r, seed=w + h)
    got = disp_filter_oracle.filter(m, med, size, r)
    np.testing.assert_array_equal(got, np_filter(m, med, size, r))


def component_sizes(m, r=0):
    """Per valid pixel the size of its speckle component (connected at |difference| <= 16 r); 0 for invalid pixels."""
    h, w = m.shape
    idx = np.arange(h * w).reshape(h, w)
    a_all, b_all = [], []
    for a, b, va, vb in ((idx[:, :-1], idx[:, 1:], m[:, :-1], m[:, 1:]), (idx[:-1], idx[1:], m[:-1], m[1:])):
        e = (va >= 0) & (vb >= 0) & (np.abs(va.astype(np.int64) - vb) <= 16 * r)
        a_all.append(a[e]); b_all.append(b[e])
    a, b = np.concatenate(a_all), np.concatenate(b_all)
    _, lab = connected_components(scipy.sparse.coo_matrix((np.ones(len(a)), (a, b)), shape=(h * w, h * w)), directed=False)
    return np.where(m >= 0, np.bincount(lab)[lab].reshape(h, w), 0)


def test_crafted_contents_do_what_they_say():
    """What the cases rely on: the serpentine is one component across tiles, the exact sizes are there and straddle tile
    borders, the 16 r steps join and the 16 r + 1 ones do not, and -1 beside 0 connects nothing."""
    w, h = 200, 70
    s = crafted('serpentine', w, h)
    n = int((s >= 0).sum())
    assert np.all(component_sizes(s)[s >= 0] == n)
    assert np.array_equal(disp_filter_oracle.filter(s, 0, n - 1, 0), s) and np.all(disp_filter_oracle.filter(s, 0, n, 0) == -1)
    for size in (1, 50, 200):
        e = crafted('exact', w, h, size)
        sz = component_sizes(e)
        assert {size, size + 1} == set(np.unique(sz[e >= 0]).tolist())
        ys, xs = np.nonzero(e >= 0)
        assert (xs % TILE == 0).any() and (xs % TILE == TILE - 1).any()
        assert np.array_equal(disp_filter_oracle.filter(e, 0, size, 0), np.where(sz == size, -1, e))
    st = crafted('steps', 64, 8, r=2)
    sz = component_sizes(st, 2)
    assert np.all(sz[:, :32] >= 8 * 32) and np.all(sz[:, 33:] == 1)
    z = np.array([[-1, 0, -1, 0], [0, -1, 0, -1]], np.int16)
    assert np.all(disp_filter_oracle.filter(z, 0, 1, 1) == -1)


def test_oracle_corridor_ground_truth():
    """Frame 0 of the corridor at the SGM defaults, median then speckle removal (100, 2), inside the mask of
    test_gpu_disparity's ground-truth test.  Measured with the oracle: valid fraction 0.9979 / 0.9979 / 0.9977 / 0.9978
    and 29 / 9 / 6 / 0 pixels more than 3 px from the truth for unfiltered / median / speckle / both."""
    L, R = synth.corridor_stereo_frame(0)
    raw = sgm_oracle.sgm(L, R, sgm_params())
    out = disp_filter_oracle.filter(raw, 1, 100, 2)
    Z = synth.corridor_depth(0)
    truth = 16.0 * synth.KITTI_F * 0.54 / Z
    mask = (Z < 400.0) & (np.arange(L.shape[1])[None, :] >= 128)
    valid = out >= 0
    bad = valid & (np.abs(out.astype(np.float64) - truth) > 48.0)
    print('corridor filtered: valid %.4f, %d pixels off by more than 3 px' % (valid[mask].mean(), bad[mask].sum()))
    assert bad[mask].sum() == 0
    assert valid[mask].mean() >= 0.997


# ----------------------------------------------------------------------------- visocu_disparity_filter against the oracle
_filter_ctx = []


@pytest.fixture(scope='module')
def fctx():
    """One unconfigured context: the filter does not depend on a frame geometry."""
    if not _filter_ctx:
        _filter_ctx.append(V.Context(0))
    yield _filter_ctx[0]
    _filter_ctx.pop().close()


def run_filter(c, maps, prm, device):
    """The maps filtered by visocu_disparity_filter on host maps or on one device tensor; returns numpy copies."""
    import torch
    if device:
        t = torch.as_tensor(np.stack(maps)).cuda()
        c.disparity_filter(t, *prm)
        return list(t.cpu().numpy())
    out = [m.copy() for m in maps]
    c.disparity_filter(out, *prm)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('w,h', SIZES, ids=['%dx%d' % s for s in SIZES])
def test_filter_equals_oracle(fctx, w, h):
    """Every crafted content at every parameter set, in one call per parameter set: host maps, then a device tensor three
    times over (the same bytes each time: the order of the atomics does not show)."""
    for prm in PARAMS:
        med, size, r = resolve(prm, w, h)
        maps = [crafted(kind, w, h, size, r, seed=w + h + j) for j, kind in enumerate(KINDS)]
        want = [disp_filter_oracle.filter(m, med, size, r) for m in maps]
        got = run_filter(fctx, maps, (med, size, r), False)
        for kind, g, wnt in zip(KINDS, got, want):
            assert np.array_equal(g, wnt), (prm, kind, int(np.sum(g != wnt)))
        for _ in range(3):
            got = run_filter(fctx, maps, (med, size, r), True)
            for kind, g, wnt in zip(KINDS, got, want):
                assert np.array_equal(g, wnt), (prm, kind, 'device', int(np.sum(g != wnt)))


@pytest.mark.gpu
@pytest.mark.parametrize('n', [1, 7, 128, 129])
@pytest.mark.parametrize('w,h', [(31, 17), (1241, 376), (64, 1000)], ids=['31x17', '1241x376', '64x1000'])
def test_filter_batches(fctx, n, w, h):
    """n maps of every kind in one call (two launch groups at 129), host and device, with the median and speckle removal;
    the launch count per group is the header's."""
    prm = (1, 50, 2)
    maps = [crafted(KINDS[k % len(KINDS)], w, h, 50, 2, seed=k) for k in range(n)]
    want = [disp_filter_oracle.filter(m, *prm) for m in maps]
    for device in (False, True):
        l0 = fctx.launch_count()
        got = run_filter(fctx, maps, prm, device)
        assert fctx.launch_count() - l0 == 5 * ((n + 127) // 128)
        for k in range(n):
            assert np.array_equal(got[k], want[k]), (device, k)


@pytest.mark.gpu
def test_filter_launches_and_noop(fctx):
    """2 launches for the median alone, 4 for speckle removal alone, none with both off (maps unchanged)."""
    maps = [crafted('blocky', 100, 60, seed=s) for s in range(3)]
    for prm, launches in (((1, 0, 0), 2), ((0, 10, 1), 4), ((1, 10, 1), 5), ((0, 0, 5), 0)):
        l0 = fctx.launch_count()
        got = run_filter(fctx, maps, prm, True)
        assert fctx.launch_count() - l0 == launches, prm
        assert all(np.array_equal(g, disp_filter_oracle.filter(m, *prm)) for g, m in zip(got, maps)), prm


@pytest.mark.gpu
def test_maps_never_join(fctx):
    """Map 0's last row and map 1's first row are one run of equal values that would be one component of 2 w pixels if the
    maps lay one after the other: in one call each row is a component of w pixels and goes at speckle_size = w."""
    w, h = 70, 40
    a = np.full((h, w), -1, np.int16); a[-1] = 160
    b = np.full((h, w), -1, np.int16); b[0] = 160
    side_a = np.full((h, w), -1, np.int16); side_a[:, -1] = 160    # the same across the right / left columns
    side_b = np.full((h, w), -1, np.int16); side_b[:, 0] = 160
    for maps, size in (([a, b], w), ([side_a, side_b], h)):
        assert np.all(disp_filter_oracle.filter(np.concatenate(maps, 0 if size == w else 1), 0, size, 0) == np.concatenate(maps, 0 if size == w else 1))
        for device in (False, True):
            got = run_filter(fctx, maps, (0, size, 0), device)
            assert all(np.all(g == -1) for g in got), device


@pytest.mark.gpu
def test_filter_errors_leave_maps_untouched(fctx):
    w, h = 40, 30
    maps = [np.full((h, w), 0x5A5A, np.int16) for _ in range(2)]
    arr = (C.c_void_p * 2)(*[m.ctypes.data for m in maps])
    EINVAL = -1

    def call(n=2, mp=arr, ww=w, hh=h, on_dev=0, med=1, size=10, r=1):
        return V.lib().visocu_disparity_filter(fctx.h, n, mp, ww, hh, on_dev, med, size, r)
    assert call(size=w * h) == 0 and np.all(maps[0] == -1)             # the whole map is one component of w h pixels
    for m in maps:
        m[:] = 0x5A5A
    for bad in (dict(n=-1), dict(mp=None), dict(mp=(C.c_void_p * 2)(maps[0].ctypes.data, None)), dict(ww=0), dict(hh=0),
                dict(ww=-3), dict(ww=1 << 13, hh=(1 << 11) + 1), dict(on_dev=2), dict(med=2), dict(med=-1), dict(size=-1),
                dict(r=-1), dict(r=257)):
        assert call(**bad) == EINVAL, bad
    assert all(np.all(m == 0x5A5A) for m in maps)
    assert call(n=0, mp=None) == 0
    assert call(r=256) == 0 and call(size=0, med=0) == 0


# ----------------------------------------------------------------------------- visocu_disparity with the filters
FILTERS = [(1, 0, 0), (0, 100, 2), (1, 100, 2), (1, 1000, 0), (0, 10, 'D')]
SGM_FILTER_CASES = [(w, h, D, paths, FILTERS[(i + j) % len(FILTERS)], CONTENTS[(i + 2 * j) % len(CONTENTS)])
                    for i, (w, h) in enumerate(SGM_SIZES[:4] + SGM_SIZES[5:7]) for j, (D, paths) in enumerate(((64, 4), (128, 8), (256, 8)))]


@pytest.mark.gpu
@pytest.mark.parametrize('w,h,D,paths,flt,kind', SGM_FILTER_CASES,
                         ids=['%dx%d-D%d-p%d-m%s-s%s-r%s-%s' % ((w, h, D, p) + f + (k,)) for w, h, D, p, f, k in SGM_FILTER_CASES])
def test_disparity_with_filters_equals_oracle(size_ctx, w, h, D, paths, flt, kind):
    """visocu_disparity with the filters = oracle SGM, then the oracle filter; the launches per group are SGM's and the
    filters', and the filters off give SGM's launches."""
    c, pairs = size_ctx(w, h)
    i = CONTENTS.index(kind)
    med, size, r = flt[0], flt[1], D if flt[2] == 'D' else flt[2]
    p = sgm_params(max_disp=D, paths=paths, median=med, speckle_size=size, speckle_range=r)
    l0 = c.launch_count()
    got = c.disparity([2 * i], [2 * i + 1], p)[0]
    assert c.launch_count() - l0 == (4 if paths == 4 else 6) + {(1, 0): 2, (0, 1): 4, (1, 1): 5}[(med, int(size > 0))]
    raw = oracle(*pairs[i], sgm_params(max_disp=D, paths=paths))
    want = disp_filter_oracle.filter(raw, med, size, r)
    assert np.array_equal(got, want), int(np.sum(got != want))
    l0 = c.launch_count()
    assert np.array_equal(c.disparity([2 * i], [2 * i + 1], sgm_params(max_disp=D, paths=paths))[0], raw)
    assert c.launch_count() - l0 == (4 if paths == 4 else 6)


@pytest.mark.gpu
@pytest.mark.parametrize('n', [1, 129])
def test_disparity_filters_batches(n):
    """Host and device outputs of n pairs with the filters: every map equals the oracle; 6 + 5 launches per group."""
    import torch
    w, h = 337, 211
    rng = np.random.default_rng(n)
    imgs = [content('blob', w, h, seed=s)[s % 2] for s in range(4)] + list(synth.corridor_stereo_frame(0, w, h))
    c = new_ctx(w, h, 6)
    try:
        c.push_frames(np.arange(6), imgs=imgs)
        left = rng.integers(0, 6, n).astype(np.int32); right = rng.integers(0, 6, n).astype(np.int32)
        left[0], right[0] = 4, 5
        p = sgm_params(median=1, speckle_size=100, speckle_range=2)
        l0 = c.launch_count()
        host = c.disparity(left, right, p)
        assert c.launch_count() - l0 == 11 * ((n + 127) // 128)
        want = {}
        for k in range(n):
            key = (left[k], right[k])
            if key not in want:
                want[key] = disp_filter_oracle.filter(oracle(imgs[key[0]], imgs[key[1]], sgm_params()), 1, 100, 2)
            assert np.array_equal(host[k], want[key]), k
        t = c.disparity_tensor(left, right, p)
        assert np.array_equal(t.cpu().numpy(), np.stack(host))
        # re-filtering the unfiltered device maps with the stand-alone call gives the same maps
        raw = c.disparity_tensor(left, right, sgm_params())
        c.disparity_filter(raw, 1, 100, 2)
        torch.cuda.synchronize()
        assert np.array_equal(raw.cpu().numpy(), np.stack(host))
    finally:
        c.close()


@pytest.mark.gpu
def test_disparity_bad_filter_fields():
    w, h = 130, 70
    c = new_ctx(w, h, 2)
    try:
        c.push_frames([0, 1], imgs=list(content('blob', w, h)))
        out = np.full((h, w), 0x5A5A, np.int16)
        ptr = (C.c_void_p * 1)(out.ctypes.data)
        ok_l, ok_r = np.array([0], np.int32), np.array([1], np.int32)
        for b in (dict(median=2), dict(median=-1), dict(speckle_size=-1), dict(speckle_range=-1),
                  dict(speckle_range=65, max_disp=64), dict(speckle_range=129)):
            p = sgm_params(**b)
            assert V.lib().visocu_sgm_check(C.byref(p)) == -1, b
            assert V.lib().visocu_disparity(c.h, 1, ok_l.ctypes.data_as(C.c_void_p), ok_r.ctypes.data_as(C.c_void_p),
                                            C.byref(p), ptr, 0) == -1, b
        assert np.all(out == 0x5A5A)
        p = sgm_params(speckle_range=64, max_disp=64, speckle_size=5, median=1)
        assert V.lib().visocu_sgm_check(C.byref(p)) == 0
    finally:
        c.close()


# ----------------------------------------------------------------------------- runner and host layer
@pytest.mark.gpu
@pytest.mark.parametrize('mode', [2, 4])
def test_runner_filtered_disparity(mode):
    """A 12-frame corridor stereo drive of 3 sequences on 2 workers with filtered disparity and without disparity: the same
    matches, motions, inliers, ok flags (and points in mode 4); each sequence's last map equals the oracle; bad filter
    fields are refused."""
    import host_py as H
    S, T = 3, 12
    W, HT = 1241, 376
    dims = np.array([W, HT, W], np.int32)
    drives = [[tuple(np.ascontiguousarray(x) for x in synth.corridor_stereo_frame(k, seed=1234 + s)) for k in range(T)]
              for s in range(S)]
    make = H.Runner.stereo if mode == 2 else H.Runner.stereo_sfm
    on, off = make(0, S, 2, _stereo_params()), make(0, S, 2, _stereo_params())
    for b in (dict(median=2), dict(speckle_size=-1), dict(speckle_range=-1), dict(speckle_range=129)):
        assert not on.set_disparity(sgm_params(**b)), b
    p = sgm_params(median=1, speckle_size=100, speckle_range=2)
    assert on.set_disparity(p)
    for k in range(T):
        res = []
        for r in (on, off):
            secs, nm, ok = r.step([d[k][0].ctypes.data for d in drives], dims, ptrs2=[d[k][1].ctypes.data for d in drives])
            res.append((nm.copy(), ok.copy()))
        assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1]), k
        for s in range(S):
            assert on.matches(s).tobytes() == off.matches(s).tobytes(), (k, s)
            assert np.array_equal(on.motion(s), off.motion(s)) and np.array_equal(on.inliers(s), off.inliers(s)), (k, s)
            if mode == 4:
                assert on.points(s).tobytes() == off.points(s).tobytes(), (k, s)
    for s in range(S):
        got = on.disparity_tensor(s)
        want = disp_filter_oracle.filter(oracle(*drives[s][T - 1], sgm_params()), 1, 100, 2)
        assert got is not None and np.array_equal(got.cpu().numpy(), want), s


@pytest.mark.gpu
def test_facades_with_filters():
    """StereoSfm.disparity_tensor, Stereo.disparity and Matcher.disparity with filter params equal Context.disparity."""
    import host_py as H
    W, HT = 1241, 376
    frames = [synth.corridor_stereo_frame(k, W, HT) for k in range(3)]
    p = sgm_params(max_disp=64, paths=4, median=1, speckle_size=200, speckle_range=1)
    sfm, vo = H.StereoSfm(_stereo_params(), W, HT), H.Stereo(_stereo_params())
    for L, R in frames:
        sfm.update(L, R)
        vo.process(L, R)
    c = new_ctx(W, HT, 2)
    try:
        c.push_frames([0, 1], imgs=list(frames[-1]))
        want = c.disparity([0], [1], p)[0]
        assert not np.array_equal(want, c.disparity([0], [1], sgm_params(max_disp=64, paths=4))[0])
    finally:
        c.close()
    assert np.array_equal(sfm.disparity_tensor(p).cpu().numpy(), want)
    assert np.array_equal(vo.disparity(p), want)
    m = H.Matcher(V.Params())
    m.push(*frames[-1])
    assert np.array_equal(m.disparity(p), want)
