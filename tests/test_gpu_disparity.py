"""Dense stereo disparity (visocu_disparity, semi-global matching): the plain-C oracle against an independent numpy
restatement and against the corridor's ground-truth depth (CPU), the device bit for bit against the oracle over sizes,
disparity ranges, paths, parameters and contents, batching, outputs, lane ordering, rectification, argument checks, the
host layer and the runner (GPU)."""
import ctypes as C

import numpy as np
import pytest

import synth
import sgm_oracle
import visocu_py as V

DEFAULTS = dict(max_disp=128, paths=8, p1=10, p2=120, uniqueness=95, lr_max_diff=1, subpixel=1)
PARAM_SETS = [dict(), dict(uniqueness=100, lr_max_diff=-1, subpixel=0), dict(uniqueness=90, lr_max_diff=0, p1=1, p2=2),
              dict(uniqueness=0, lr_max_diff=1, p1=63, p2=150), dict(uniqueness=100, lr_max_diff=0, subpixel=0, p1=63, p2=150),
              dict(uniqueness=90, lr_max_diff=-1, p1=1, p2=2)]


def sgm_params(**kw):
    d = dict(DEFAULTS); d.update(kw)
    return V.SgmParams(**d)


def content(kind, w, h, seed=0, disp=7):
    """A left / right pair of (h, w) uint8 images."""
    rng = np.random.default_rng(seed)
    if kind == 'noise':
        base = rng.integers(0, 256, (h, w + disp), dtype=np.uint8)
        return base[:, disp:].copy(), np.ascontiguousarray(base[:, :w])
    if kind == 'blob':
        lp, rp, _, _ = synth.blob_quad(w, h, seed=seed + 1, disparity=disp)
        return lp, rp
    if kind == 'corridor':
        return synth.corridor_stereo_frame(0, w, h)
    if kind == 'const':
        return np.full((h, w), 77, np.uint8), np.full((h, w), 77, np.uint8)
    if kind == 'stripes':                      # saturated vertical stripes: ties everywhere
        x = np.arange(w)
        L = np.where((x // 3) % 2 == 0, 255, 0).astype(np.uint8)[None, :].repeat(h, 0)
        return L, np.roll(L, -2, axis=1)
    raise ValueError(kind)


# ----------------------------------------------------------------------------- numpy restatement
def _census(I):
    h, w = I.shape
    I = I.astype(np.int32)
    pad = np.pad(I, ((3, 3), (4, 4)), mode='edge')
    bits = np.zeros((h, w), np.uint64)
    b = 0
    for dy in range(-3, 4):
        for dx in range(-4, 5):
            if dx == 0 and dy == 0:
                continue
            bits |= (pad[3 + dy:3 + dy + h, 4 + dx:4 + dx + w] < I).astype(np.uint64) << np.uint64(b)
            b += 1
    return bits


def np_sgm(L, R, p):
    """The algorithm of include/visocu.h in numpy: returns (out int16 (h, w), S int64 (h, w, D))."""
    h, w = L.shape
    D = p.max_disp
    cl, cr = _census(L), _census(R)
    Cv = np.full((h, w, D), 62, np.int64)
    for d in range(min(D, w)):
        Cv[:, d:, d] = np.bitwise_count(cl[:, d:] ^ cr[:, :w - d])

    def step(Lp, c):
        M = Lp.min(-1, keepdims=True)
        best = np.minimum(Lp, M + p.p2)
        best[..., 1:] = np.minimum(best[..., 1:], Lp[..., :-1] + p.p1)
        best[..., :-1] = np.minimum(best[..., :-1], Lp[..., 1:] + p.p1)
        return c + best - M

    dirs = [(1, 0), (-1, 0), (0, 1), (0, -1), (1, 1), (-1, 1), (1, -1), (-1, -1)][:p.paths]
    S = np.zeros((h, w, D), np.int64)
    xs = np.arange(w)
    for rx, ry in dirs:
        Lr = np.zeros((h, w, D), np.int64)
        if ry == 0:
            order = range(w) if rx > 0 else range(w - 1, -1, -1)
            for i, x in enumerate(order):
                Lr[:, x] = Cv[:, x] if i == 0 else step(Lr[:, x - rx], Cv[:, x])
        else:
            order = range(h) if ry > 0 else range(h - 1, -1, -1)
            for i, y in enumerate(order):
                row = Cv[y].copy()
                if i > 0:
                    src = xs - rx
                    ok = (src >= 0) & (src < w)
                    row[ok] = step(Lr[y - ry][src[ok]], Cv[y][ok])
                Lr[y] = row
        S += Lr
    ds = S.argmin(-1)
    smin = np.take_along_axis(S, ds[..., None], -1)[..., 0]
    far = np.abs(np.arange(D)[None, None, :] - ds[..., None]) > 1
    m2 = np.where(far, S, 1 << 30).min(-1)
    valid = ~(100 * smin > p.uniqueness * m2)
    if p.lr_max_diff >= 0:
        T = np.full((h, w, D), 1 << 30, np.int64)
        for d in range(min(D, w)):
            T[:, :w - d, d] = S[:, d:, d]
        dR = T.argmin(-1)
        xr = xs[None, :] - ds
        valid &= xr >= 0
        dRx = np.take_along_axis(dR, np.clip(xr, 0, w - 1), 1)
        valid &= np.abs(dRx - ds) <= p.lr_max_diff
    v = 16 * ds
    if p.subpixel:
        inner = (ds > 0) & (ds < D - 1)
        a = np.take_along_axis(S, np.clip(ds - 1, 0, D - 1)[..., None], -1)[..., 0]
        c = np.take_along_axis(S, np.clip(ds + 1, 0, D - 1)[..., None], -1)[..., 0]
        den = a + c - 2 * smin
        off = np.where(den > 0, np.floor_divide(16 * (a - c) + den, np.where(den > 0, 2 * den, 1)), 0)
        v = np.where(inner, v + off, v)
    return np.where(valid, v, -1).astype(np.int16), S


ORACLE_CASES = [(w, h, paths, k, kind) for (w, h) in ((48, 20), (37, 29), (100, 24)) for paths in (4, 8)
                for k in range(len(PARAM_SETS)) for kind in ('noise', 'blob', 'const', 'stripes')]


@pytest.mark.parametrize('w,h,paths,k,kind', ORACLE_CASES, ids=['%dx%d-p%d-s%d-%s' % c for c in ORACLE_CASES])
def test_oracle_equals_numpy(w, h, paths, k, kind):
    p = sgm_params(max_disp=64, paths=paths, **PARAM_SETS[k])
    L, R = content(kind, w, h, seed=k)
    out, S = sgm_oracle.sgm(L, R, p, want_S=True)
    ref, Sref = np_sgm(L, R, p)
    assert int(Sref.max()) <= 8 * (62 + p.p2)
    np.testing.assert_array_equal(S.astype(np.int64), Sref)
    np.testing.assert_array_equal(out, ref)


# The fraction of the corridor's pixels (ground truth closer than the 400 m cap, x >= D) that the oracle keeps valid and
# within one pixel of 16 f base / Z, measured with the default parameters at 1241x376.
CORRIDOR_GOOD = 0.9956


def test_oracle_corridor_ground_truth():
    L, R = synth.corridor_stereo_frame(0)
    out = sgm_oracle.sgm(L, R, sgm_params())
    Z = synth.corridor_depth(0)
    truth = 16.0 * synth.KITTI_F * 0.54 / Z
    mask = (Z < 400.0) & (np.arange(L.shape[1])[None, :] >= 128)
    good = (out >= 0) & (np.abs(out.astype(np.float64) - truth) <= 16.0)
    frac = good[mask].mean()
    print('corridor: %.4f of %d pixels valid and within one pixel' % (frac, mask.sum()))
    assert frac >= CORRIDOR_GOOD - 0.01


def test_oracle_blob_disparity():
    L, R, _, _ = synth.blob_quad(disparity=12)
    out = sgm_oracle.sgm(L, R, sgm_params(subpixel=0))
    sel = out[:, 128:]
    ok = sel[sel >= 0]
    assert ok.size > 0.5 * sel.size
    assert (ok // 16 == 12).mean() >= 0.99


# ----------------------------------------------------------------------------- device against the oracle
SIZES = [(1241, 376), (1242, 375), (1249, 376), (337, 211), (130, 70), (64, 1000), (2000, 40), (50, 40)]
CONTENTS = ('corridor', 'blob', 'noise', 'const', 'stripes')
GPU_CASES = [(w, h, D, paths, (i + j) % len(PARAM_SETS), CONTENTS[(i + 2 * j) % len(CONTENTS)])
             for i, (w, h) in enumerate(SIZES) for j, (D, paths) in enumerate((D, p) for D in (64, 128, 256) for p in (4, 8))]
_oracle_cache = {}


def oracle(L, R, p):
    key = (L.tobytes(), R.tobytes(), tuple(getattr(p, n) for n, _ in V.SgmParams._fields_))
    if key not in _oracle_cache:
        _oracle_cache[key] = sgm_oracle.sgm(L, R, p)
    return _oracle_cache[key]


def new_ctx(w, h, n_frames, half=0):
    c = V.Context(0)
    c.configure(V.Params(half_resolution=half, match_radius=100 if half else 200), w, h, n_frames)
    return c


_size_ctx = {}


@pytest.fixture(scope='module')
def size_ctx():
    """One context per size holding every content pair in frames (2 k, 2 k + 1)."""
    def get(w, h):
        if (w, h) not in _size_ctx:
            c = new_ctx(w, h, 2 * len(CONTENTS))
            pairs = [content(kind, w, h, seed=3) for kind in CONTENTS]
            c.push_frames(np.arange(2 * len(CONTENTS)), imgs=[im for pr in pairs for im in pr])
            _size_ctx[(w, h)] = (c, pairs)
        return _size_ctx[(w, h)]
    yield get
    for c, _ in _size_ctx.values():
        c.close()
    _size_ctx.clear()


@pytest.mark.gpu
@pytest.mark.parametrize('w,h,D,paths,k,kind', GPU_CASES, ids=['%dx%d-D%d-p%d-s%d-%s' % c for c in GPU_CASES])
def test_device_equals_oracle(size_ctx, w, h, D, paths, k, kind):
    c, pairs = size_ctx(w, h)
    i = CONTENTS.index(kind)
    p = sgm_params(max_disp=D, paths=paths, **PARAM_SETS[k])
    got = c.disparity([2 * i], [2 * i + 1], p)[0]
    want = oracle(*pairs[i], p)
    assert np.array_equal(got, want), int(np.sum(got != want))


@pytest.mark.gpu
@pytest.mark.parametrize('n', [1, 4, 17, 128, 129])
def test_batches_and_outputs(n):
    """Pairs drawn from 6 frames (shared frames, swapped pairs, a frame against itself), pushed at a wider pitch: every map
    equals the oracle, host and tensor outputs agree, three calls give the same bytes, and each group of at most 128 pairs
    is 6 launches."""
    import torch
    w, h = 337, 211
    rng = np.random.default_rng(n)
    imgs = [content('blob', w, h, seed=s)[s % 2] for s in range(4)] + list(synth.corridor_stereo_frame(0, w, h))
    c = new_ctx(w, h, 6)
    try:
        pitch = w + 19
        padded = [np.pad(im, ((0, 0), (0, pitch - w)), constant_values=200) for im in imgs]
        c.push_frames(np.arange(6), imgs=padded, bpl_in=pitch)
        left = rng.integers(0, 6, n).astype(np.int32); right = rng.integers(0, 6, n).astype(np.int32)
        left[0], right[0] = 4, 5
        if n > 1:
            left[1], right[1] = 5, 4
        p = sgm_params()
        l0 = c.launch_count()
        host = c.disparity(left, right, p)
        groups = (n + 127) // 128
        assert c.launch_count() - l0 == 6 * groups
        for k in range(n):
            assert np.array_equal(host[k], oracle(imgs[left[k]], imgs[right[k]], p)), k
        for _ in range(3):
            t = c.disparity_tensor(left, right, p)
            assert t.dtype == torch.int16 and tuple(t.shape) == (n, h, w)
            assert np.array_equal(t.cpu().numpy(), np.stack(host))
            again = c.disparity(left, right, p)
            assert all(np.array_equal(a, b) for a, b in zip(again, host))
    finally:
        c.close()


@pytest.mark.gpu
def test_lazy_push_on_another_lane():
    """A lazy push (no counts read back) on lane 0 followed directly by a disparity call on lane 4 sees the new images."""
    w, h = 1241, 376
    c = new_ctx(w, h, 2)
    try:
        c.push_frames([0, 1], imgs=list(content('noise', w, h)))
        c.disparity([0], [1])
        L, R = synth.corridor_stereo_frame(0, w, h)
        c.push_frames([0, 1], imgs=[L, R], want_counts=False)
        assert V.lib().visocu_set_lane(c.h, 4) == 0
        got = c.disparity([0], [1])[0]
        assert np.array_equal(got, oracle(L, R, sgm_params()))
    finally:
        c.close()


@pytest.mark.gpu
def test_half_resolution_same_map():
    w, h = 1241, 376
    L, R = synth.corridor_stereo_frame(2, w, h)
    maps = []
    for half in (0, 1):
        c = new_ctx(w, h, 2, half)
        try:
            c.push_frames([0, 1], imgs=[L, R])
            maps.append(c.disparity([0], [1])[0])
        finally:
            c.close()
    assert np.array_equal(maps[0], maps[1])
    assert np.array_equal(maps[0], oracle(L, R, sgm_params()))


@pytest.mark.gpu
def test_rectified_push():
    """After a rectifying push of a distorted pair, the map equals the oracle on the two rectified frame images."""
    import host_py as H
    src, out = (1392, 512), (1241, 376)
    cam0 = V.Camera(959.8, 957.5, 696.0, 224.0, -0.37, 0.20, 1.2e-3, -3.4e-4, -0.07)
    cam1 = V.Camera(955.1, 953.0, 690.3, 229.5, -0.365, 0.19, -6e-4, 8e-4, -0.06)
    a = np.radians(1.0)
    Rrel = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    cams = list(H.stereo_rectify(cam0, cam1, Rrel, np.array([-0.54, 0.01, 0.005]), *out)[:2])
    raw = [synth.blob_pair(*src, seed=s)[0] for s in (3, 4)]
    c = new_ctx(*out, 2)
    try:
        c.set_rectification(cams, *src)
        c.push_frames_rectified([0, 1], [0, 1], imgs=raw)
        L = np.ascontiguousarray(c.plane(0, 4)[0][:, :out[0]]); R = np.ascontiguousarray(c.plane(1, 4)[0][:, :out[0]])
        p = sgm_params(paths=4, max_disp=64)
        assert np.array_equal(c.disparity([0], [1], p)[0], oracle(L, R, p))
    finally:
        c.close()


@pytest.mark.gpu
def test_errors_leave_output_untouched():
    w, h = 130, 70
    c = new_ctx(w, h, 3)
    un = V.Context(0)
    try:
        c.push_frames([0, 1], imgs=list(content('blob', w, h)))
        out = np.full((h, w), 0x5A5A, np.int16)
        ptr = (C.c_void_p * 1)(out.ctypes.data)
        ok_l, ok_r = np.array([0], np.int32), np.array([1], np.int32)

        def call(ctx, n=1, left=ok_l, right=ok_r, p=None, outp=ptr, on_dev=0):
            p = sgm_params() if p is None else p
            return V.lib().visocu_disparity(ctx.h, n, None if left is None else left.ctypes.data_as(C.c_void_p),
                                            None if right is None else right.ctypes.data_as(C.c_void_p),
                                            None if p is False else C.byref(p), outp, on_dev)
        EINVAL, ESTATE = -1, -5
        bad = [dict(max_disp=96), dict(max_disp=32), dict(paths=2), dict(paths=16), dict(p1=0), dict(p1=120, p2=120),
               dict(p1=10, p2=151), dict(uniqueness=-1), dict(uniqueness=101), dict(lr_max_diff=-2), dict(lr_max_diff=129),
               dict(subpixel=2)]
        for b in bad:
            assert call(c, p=sgm_params(**b)) == EINVAL, b
        assert call(c, p=False) == EINVAL
        assert call(c, n=-1) == EINVAL
        assert call(c, left=None) == EINVAL and call(c, right=None) == EINVAL and call(c, outp=None) == EINVAL
        assert call(c, outp=(C.c_void_p * 1)(None)) == EINVAL
        assert call(c, on_dev=2) == EINVAL
        for l, r in ((3, 1), (0, -1), (-1, 0)):
            assert call(c, left=np.array([l], np.int32), right=np.array([r], np.int32)) == EINVAL
        assert call(c, left=np.array([2], np.int32)) == ESTATE            # frame 2 was never pushed
        assert call(un) == ESTATE                                           # not configured
        assert np.all(out == 0x5A5A)
        l0 = c.launch_count()
        assert call(c, n=0, left=None, right=None, outp=None) == 0 and c.launch_count() == l0
        assert call(c, p=sgm_params(lr_max_diff=128, paths=4, max_disp=128)) == 0 and not np.all(out == 0x5A5A)
    finally:
        c.close(); un.close()


# ----------------------------------------------------------------------------- host layer and runner
def _stereo_params():
    import host_py as H
    return H.StereoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, base=0.54,
                          bucket_max_features=2)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', [2, 4])
def test_runner_disparity_changes_nothing(mode):
    """A 30-frame corridor stereo drive of 3 sequences on 2 workers, with disparity on and off: the same matches, motions,
    inliers, ok flags (and points in mode 4); each sequence's map at the last step equals the oracle on that step's images."""
    import host_py as H
    S, T = 3, 30
    W, HT = 1241, 376
    dims = np.array([W, HT, W], np.int32)
    drives = [[tuple(np.ascontiguousarray(x) for x in synth.corridor_stereo_frame(k, seed=1234 + s)) for k in range(T)]
              for s in range(S)]
    make = H.Runner.stereo if mode == 2 else H.Runner.stereo_sfm
    on, off = make(0, S, 2, _stereo_params()), make(0, S, 2, _stereo_params())
    p = sgm_params()
    assert on.set_disparity(p)
    assert not on.set_disparity(sgm_params(p1=0))
    assert on.disparity_tensor(0) is None
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
        assert off.disparity_tensor(0) is None
    for s in range(S):
        got = on.disparity_tensor(s)
        assert got is not None and tuple(got.shape) == (HT, W)
        assert np.array_equal(got.cpu().numpy(), oracle(*drives[s][T - 1], p)), s
    assert on.set_disparity(None) and on.disparity_tensor(0) is None


@pytest.mark.gpu
def test_set_disparity_other_modes():
    import host_py as H
    mp = H.MonoParams(match=V.Params())
    for r in (H.Runner(0, 2, 1, 0, 0, mp), H.Runner(0, 2, 1, 1, 0, mp), H.Runner.sfm(0, 2, 1, mp)):
        assert not r.set_disparity(sgm_params())


@pytest.mark.gpu
def test_facades_against_context():
    """StereoSfm.disparity_tensor, Stereo.disparity and Matcher.disparity equal Context.disparity on the same frames; a mono
    push gives None."""
    import host_py as H
    W, HT = 1241, 376
    frames = [synth.corridor_stereo_frame(k, W, HT) for k in range(3)]
    p = sgm_params(max_disp=64, paths=4)
    sfm, vo = H.StereoSfm(_stereo_params(), W, HT), H.Stereo(_stereo_params())
    for L, R in frames:
        sfm.update(L, R)
        vo.process(L, R)
    c = new_ctx(W, HT, 2)
    try:
        c.push_frames([0, 1], imgs=list(frames[-1]))
        want = c.disparity([0], [1], p)[0]
    finally:
        c.close()
    assert np.array_equal(sfm.disparity_tensor(p).cpu().numpy(), want)
    assert np.array_equal(vo.disparity(p), want)
    m = H.Matcher(V.Params())
    m.push(*frames[-1])
    assert np.array_equal(m.disparity(p), want)
    m.push(frames[0][0])
    assert m.disparity(p) is None


@pytest.mark.parametrize('device', ['cpu', pytest.param('cuda', marks=pytest.mark.gpu)])
def test_disparity_to_points(device):
    import torch
    import host_py as H
    rng = np.random.default_rng(5)
    d = rng.integers(-1, 16 * 90, (37, 53)).astype(np.int16)
    d[3, :] = 0
    f, cu, cv, base = 645.2, 26.5, 18.0, 0.54
    got = H.disparity_to_points(torch.as_tensor(d, device=device), f, cu, cv, base)
    assert got.dtype == torch.float32 and got.device.type == device
    v, u = np.nonzero(d > 0)
    Z = (np.float32(16.0 * f * base) / d[v, u].astype(np.float32)).astype(np.float32)
    X = (u.astype(np.float32) - np.float32(cu)) * Z / np.float32(f)
    Y = (v.astype(np.float32) - np.float32(cv)) * Z / np.float32(f)
    np.testing.assert_allclose(got.cpu().numpy(), np.stack([X, Y, Z], 1), rtol=1e-6)
