"""Undistortion and stereo rectification of raw camera images: the host maps (host/rectify.cpp) against a numpy float64
restatement, Bouguet's stereo rectification on a synthetic rig, the argument checks, k_rectify byte-exact against numpy
applying the library's own map, and the rectifying push through the matcher, the odometry, the facades and the runner."""
import ctypes as C

import numpy as np
import pytest

import synth
import visocu_py as V
import host_py as H

KITTI_RAW = (1392, 512)
OUT = (1241, 376)


def _raw_cam(fx=959.8, fy=957.5, cx=696.0, cy=224.0, k1=-0.37, k2=0.20, p1=1.2e-3, p2=-3.4e-4, k3=-0.07, **kw):
    return V.Camera(fx, fy, cx, cy, k1, k2, p1, p2, k3, **kw)


def _rot(axis, deg):
    a = np.asarray(axis, np.float64); a = a / np.linalg.norm(a)
    t = np.radians(deg)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K


def _rig():
    """A KITTI-raw-like rig: two distorted cameras, a relative rotation of a few degrees, T = (-0.54, 0.01, 0.005) m."""
    cam0 = _raw_cam()
    cam1 = _raw_cam(fx=955.1, fy=953.0, cx=690.3, cy=229.5, k1=-0.365, k2=0.19, p1=-6e-4, p2=8e-4, k3=-0.06)
    return cam0, cam1, _rot((0.3, 1.0, -0.2), 3.0), np.array([-0.54, 0.01, 0.005])


def np_map(c, src_w, src_h, out_w, out_h):
    """The map of host/rectify.h restated in numpy float64."""
    R = c.rotation()
    v, u = np.mgrid[0:out_h, 0:out_w].astype(np.float64)
    a, b = (u - c.cu) / c.f, (v - c.cv) / c.f
    X = R[0, 0] * a + R[1, 0] * b + R[2, 0]
    Y = R[0, 1] * a + R[1, 1] * b + R[2, 1]
    Z = R[0, 2] * a + R[1, 2] * b + R[2, 2]
    x, y = X / Z, Y / Z
    r2 = x * x + y * y
    radial = 1.0 + r2 * (c.k1 + r2 * (c.k2 + r2 * c.k3))
    xd = x * radial + 2.0 * c.p1 * x * y + c.p2 * (r2 + 2.0 * x * x)
    yd = y * radial + c.p1 * (r2 + 2.0 * y * y) + 2.0 * c.p2 * x * y
    sx = np.clip(32.0 * (c.fx * xd + c.cx), 0, 32.0 * (src_w - 1))
    sy = np.clip(32.0 * (c.fy * yd + c.cy), 0, 32.0 * (src_h - 1))
    return np.stack([np.rint(sx), np.rint(sy)], -1).astype(np.int32)


def apply_map(raw, src_w, m, bpl):
    h, w = m.shape[:2]
    src_h = raw.shape[0]
    x32, y32 = m[..., 0].astype(np.int64), m[..., 1].astype(np.int64)
    ix, fx, iy, fy = x32 >> 5, x32 & 31, y32 >> 5, y32 & 31
    ix1, iy1 = np.minimum(ix + 1, src_w - 1), np.minimum(iy + 1, src_h - 1)
    r = raw.astype(np.int64)
    v = ((32 - fx) * (32 - fy) * r[iy, ix] + fx * (32 - fy) * r[iy, ix1] + (32 - fx) * fy * r[iy1, ix] + fx * fy * r[iy1, ix1]
         + 512) >> 10
    out = np.zeros((h, bpl), np.uint8)
    out[:, :w] = v
    return out


def _rectification(cams, src, out, base=0.0):
    return H.Rectification(cams, src[0], src[1], out[0], out[1], base)


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize('src,out', [(KITTI_RAW, OUT), ((333, 217), (301, 171)), ((1001, 97), (1007, 93))])
def test_map_against_numpy(src, out):
    """Every entry within one 1/32 unit of the float64 restatement, at least 99.99 % equal (the rest are rounding ties)."""
    cam0, cam1, R, T = _rig()
    s = src[0] / 1392.0
    for c in H.stereo_rectify(cam0, cam1, R, T, *out)[:2]:
        for name in ('fx', 'fy', 'cx', 'cy', 'f', 'cu', 'cv'):
            setattr(c, name, getattr(c, name) * s)
        got = H.rectify_map(c, src[0], src[1], out[0], out[1])
        want = np_map(c, src[0], src[1], out[0], out[1])
        d = np.abs(got.astype(np.int64) - want)
        assert d.max() <= 1, d.max()
        assert np.mean(d == 0) >= 0.9999, np.mean(d == 0)
        assert got[..., 0].max() <= 32 * (src[0] - 1) and got[..., 1].max() <= 32 * (src[1] - 1) and got.min() >= 0


def test_stereo_rectify_synthetic_rig():
    """Both rotations orthonormal, equal rows for random 3-D points seen by both rectified cameras, base = |T|."""
    cam0, cam1, R, T = _rig()
    r0, r1, base = H.stereo_rectify(cam0, cam1, R, T, *OUT)
    assert abs(base - np.linalg.norm(T)) <= 1e-12
    assert r0.f == r1.f == min(cam0.fy, cam1.fy) and r0.cu == r1.cu and r0.cv == r1.cv
    for r in (r0, r1):
        Q = r.rotation()
        assert np.abs(Q @ Q.T - np.eye(3)).max() < 1e-12 and abs(np.linalg.det(Q) - 1) < 1e-12
        assert (r.fx, r.k1) == ((cam0 if r is r0 else cam1).fx, (cam0 if r is r0 else cam1).k1)
    rng = np.random.default_rng(3)
    X0 = np.stack([rng.uniform(-10, 10, 500), rng.uniform(-3, 3, 500), rng.uniform(4, 80, 500)], 1)
    X1 = X0 @ R.T + T
    A, B = X0 @ r0.rotation().T, X1 @ r1.rotation().T
    v0, v1 = r0.f * A[:, 1] / A[:, 2] + r0.cv, r1.f * B[:, 1] / B[:, 2] + r1.cv
    assert np.abs(v0 - v1).max() <= 1e-9
    d = r0.f * A[:, 0] / A[:, 2] - r1.f * B[:, 0] / B[:, 2]            # disparity: positive, f b / z
    assert np.allclose(d, r0.f * base / A[:, 2], rtol=1e-9)
    assert abs(r0.cu - ((OUT[0] - 1) / 2 - r0.f * np.mean([r.rotation()[0, 2] / r.rotation()[2, 2] for r in (r0, r1)]))) < 1e-9


def test_identity_map():
    """No distortion, R = I, the same K and equal sizes: the integer identity (every fraction 0)."""
    c = V.Camera(700.0, 700.0, 600.0, 180.0)
    m = H.rectify_map(c, 1241, 376, 1241, 376)
    v, u = np.mgrid[0:376, 0:1241]
    assert np.array_equal(m[..., 0], 32 * u) and np.array_equal(m[..., 1], 32 * v)


@pytest.mark.parametrize('case', ['nan', 'inf_R', 'fx0', 'fy_neg', 'f0', 'src_w15', 'src_h8192', 'behind'])
def test_einval_host(case):
    """Each camera and size the library rejects, checked on the host before any device work."""
    c = _raw_cam(k1=0.0, k2=0.0, p1=0.0, p2=0.0, k3=0.0, f=900.0, cu=620.0, cv=187.0)
    src = list(KITTI_RAW)
    if case == 'nan': c.k2 = float('nan')
    if case == 'inf_R': c.R[4] = float('inf')
    if case == 'fx0': c.fx = 0.0
    if case == 'fy_neg': c.fy = -1.0
    if case == 'f0': c.f = 0.0
    if case == 'src_w15': src[0] = 15
    if case == 'src_h8192': src[1] = 8192
    if case == 'behind': c.R[:] = list(_rot((0, 1, 0), 120).reshape(9))
    with pytest.raises(V.VisocuError, match=': -1 '):
        H.rectify_map(c, src[0], src[1], *OUT)


# ---------------------------------------------------------------------------------------------------------------- GPU

def _images(kind, n, w, h, bpl, seed):
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        if kind == 'random':
            img = rng.integers(0, 256, (h, bpl), dtype=np.uint8)
        else:
            v, u = np.mgrid[0:h, 0:bpl]
            img = ((3 * u + 5 * v + 17 * i) % 256).astype(np.uint8)
        out.append(np.ascontiguousarray(img))
    return out


KERNEL_CASES = [
    # name, src (w, h), out (w, h), bpl_in extra, on_device, frames per push, contents, two cameras
    ('kitti-b4-host', KITTI_RAW, OUT, 0, 0, 4, 'random', False),
    ('kitti-b17-dev-pitch', KITTI_RAW, OUT, 13, 1, 17, 'gradient', True),
    ('kitti-b128-keep-mixed', KITTI_RAW, OUT, 0, 2, 128, 'random', True),
    ('320x200-b1', (320, 200), (322, 160), 0, 0, 1, 'random', False),
    ('odd-b17-dev', (333, 217), (301, 171), 7, 1, 17, 'random', True),
    ('odd-b4-keep', (1001, 97), (1007, 93), 3, 2, 4, 'gradient', True),
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', KERNEL_CASES, ids=[c[0] for c in KERNEL_CASES])
def test_k_rectify_bytes(case):
    """The rectified frame plane (pad columns included) equals numpy applying the library's own map, for every frame of
    the same push run three times with new images (plain launch, graph capture, graph replay)."""
    name, src, out, extra, on_device, n, kind, two = case
    cam0, cam1, R, T = _rig()
    s = src[0] / 1392.0
    cams = list(H.stereo_rectify(cam0, cam1, R, T, *out)[:2 if two else 1])
    for c in cams:
        for f in ('fx', 'fy', 'cx', 'cy', 'f', 'cu', 'cv'):
            setattr(c, f, getattr(c, f) * s)
    ctx = V.Context(0)
    try:
        ctx.configure(V.Params(), out[0], out[1], n)
        ctx.set_rectification(cams, src[0], src[1])
        maps = [ctx.rectify_map(k, *out) for k in range(len(cams))]
        assert np.array_equal(maps[0], H.rectify_map(cams[0], src[0], src[1], *out))
        frames = np.arange(n)[::-1].copy()
        cam_idx = np.random.default_rng(1).integers(0, len(cams), n)
        bpl_in = src[0] + extra
        # frame planes with nonzero pad columns (a plain push at the frame pitch lands in the planes as it is), so that a
        # rectifying push has to write the zero pads itself
        bpl = out[0] + 15 - (out[0] - 1) % 16
        ctx.push_frames(frames, imgs=[np.full((out[1], bpl), 0xAB, np.uint8)] * n, bpl_in=bpl)
        assert np.all(ctx.plane(int(frames[0]), 4)[0][:, out[0]:] == 0xAB) and bpl > out[0]
        for rep in range(3):
            imgs = [np.ascontiguousarray(i[:src[1]]) for i in _images(kind, n, src[0], src[1], bpl_in, 100 * rep + len(name))]
            if on_device == 1:
                ptrs = [ctx.device_alloc(i.nbytes) for i in imgs]
                for p, i in zip(ptrs, imgs):
                    ctx.memcpy_h2d(p, i)
                ctx.push_frames_rectified(frames, cam_idx, ptrs=ptrs, bpl_in=bpl_in, on_device=1)
                ctx.sync()
                for p in ptrs:
                    ctx.device_free(p)
            else:
                ctx.push_frames_rectified(frames, cam_idx, imgs=imgs, bpl_in=bpl_in, on_device=on_device)
            for i in range(n):
                got = ctx.plane(int(frames[i]), 4)[0]
                want = apply_map(imgs[i], src[0], maps[cam_idx[i]], got.shape[1])
                assert np.array_equal(got, want), (rep, i, int(np.sum(got != want)))
    finally:
        ctx.close()


def _identity_rect(w, h):
    c = V.Camera(645.2, 645.2, 635.9, 194.1)
    return _rectification([c, c], (w, h), (w, h), 0.54)


@pytest.mark.gpu
def test_identity_changes_nothing():
    """An identity rectification gives the plain push's feature records (both passes) and, through the Matcher, the same
    flow and quad match lists, byte for byte."""
    W, HT = OUT
    seq = [synth.corridor_stereo_frame(k) for k in range(3)]
    plain, rect = V.Context(0), V.Context(0)
    try:
        for c in (plain, rect):
            c.configure(V.Params(), W, HT, 6)
        rect.set_rectification([_identity_rect(W, HT).cams[0]], W, HT)
        imgs = [np.ascontiguousarray(x) for pair in seq for x in pair]
        plain.push_frames(np.arange(6), imgs=imgs)
        rect.push_frames_rectified(np.arange(6), np.zeros(6, np.int32), imgs=imgs)
        for f in range(6):
            for ps in (0, 1):
                assert plain.features(f, ps).tobytes() == rect.features(f, ps).tobytes(), (f, ps)
            assert np.array_equal(plain.plane(f, 4)[0], rect.plane(f, 4)[0])
    finally:
        plain.close(); rect.close()
    for method in (0, 2):
        a, b = H.Matcher(V.Params()), H.Matcher(V.Params())
        assert b.set_rectification(_identity_rect(W, HT))
        for left, right in seq:
            for m in (a, b):
                m.push(left, right if method == 2 else None)
                m.match_features(method)
        assert len(a.matches()) > 100
        assert a.matches().tobytes() == b.matches().tobytes()
        assert a.matches(1).tobytes() == b.matches(1).tobytes()


# ---- end to end: a corridor drive seen through a distorted, rotated rig
F_RAW = 700.0
RAW_CAMS = [dict(fx=F_RAW, fy=F_RAW + 2.0, cx=698.0, cy=258.0, k1=-0.37, k2=0.20, p1=6e-4, p2=-4e-4, k3=-0.05),
            dict(fx=F_RAW - 3.0, fy=F_RAW - 1.0, cx=693.0, cy=254.0, k1=-0.36, k2=0.19, p1=-5e-4, p2=7e-4, k3=-0.04)]
Q = [_rot((0.2, 1.0, 0.1), 0.5), _rot((-0.4, 1.0, 0.3), -0.5)]     # raw camera k = Q[k] x rectified camera k: about 1 deg apart


def _true_rectification():
    cams = [V.Camera(**c, R=Q[k].T, f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV) for k, c in enumerate(RAW_CAMS)]
    return _rectification(cams, KITTI_RAW, OUT, 0.54)


def _raw_sampling(k):
    """Where the 4x4 subsamples of every raw pixel of camera k look in the undistorted image: (16, h, w) u and v."""
    c = RAW_CAMS[k]
    sub = (np.arange(4) + 0.5) / 4 - 0.5
    v, u = np.mgrid[0:KITTI_RAW[1], 0:KITTI_RAW[0]].astype(np.float64)
    U = (u[None, None] + sub[None, :, None, None]).reshape(4, 1, *u.shape)
    U = np.broadcast_to(U, (4, 4) + u.shape).reshape(16, *u.shape)
    V_ = np.broadcast_to((v[None] + sub[:, None, None])[:, None], (4, 4) + v.shape).reshape(16, *v.shape)
    xd, yd = (U - c['cx']) / c['fx'], (V_ - c['cy']) / c['fy']
    x, y = xd.copy(), yd.copy()
    for _ in range(30):                               # the inverse of the distortion, by fixed-point iteration
        r2 = x * x + y * y
        radial = 1 + r2 * (c['k1'] + r2 * (c['k2'] + r2 * c['k3']))
        dx = 2 * c['p1'] * x * y + c['p2'] * (r2 + 2 * x * x)
        dy = c['p1'] * (r2 + 2 * y * y) + 2 * c['p2'] * x * y
        x, y = (xd - dx) / radial, (yd - dy) / radial
    ray = np.stack([x, y, np.ones_like(x)], -1) @ Q[k]              # Q^T (x, y, 1): into the rectified camera
    return (synth.KITTI_F * ray[..., 0] / ray[..., 2] + synth.KITTI_CU,
            synth.KITTI_F * ray[..., 1] / ray[..., 2] + synth.KITTI_CV)


def _distort(img, su, sv):
    h, w = img.shape
    su, sv = np.clip(su, 0, w - 1.001), np.clip(sv, 0, h - 1.001)
    u0, v0 = np.floor(su).astype(np.int64), np.floor(sv).astype(np.int64)
    a, b = su - u0, sv - v0
    I = img.astype(np.float64)
    val = (1 - a) * (1 - b) * I[v0, u0] + a * (1 - b) * I[v0, u0 + 1] + (1 - a) * b * I[v0 + 1, u0] + a * b * I[v0 + 1, u0 + 1]
    return np.ascontiguousarray(np.clip(np.rint(val.mean(0)), 0, 255).astype(np.uint8))


def _angle_deg(Ra, Rb):
    return np.degrees(np.arccos(np.clip((np.trace(Ra @ Rb.T) - 1) / 2, -1, 1)))


@pytest.fixture(scope='module')
def raw_drive():
    T = 6
    orig = [synth.corridor_stereo_frame(k) for k in range(T)]
    samp = [_raw_sampling(k) for k in range(2)]
    raw = [tuple(_distort(o[k], *samp[k]) for k in range(2)) for o in orig]
    return orig, raw


def _stereo_params(**kw):
    return H.StereoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, base=0.54, **kw)


def _mono_params():
    return H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08)


def _within(ref, got):
    t_ok = np.linalg.norm(got[:3, 3] - ref[:3, 3]) <= 0.02 * np.linalg.norm(ref[:3, 3])
    return t_ok and _angle_deg(got[:3, :3], ref[:3, :3]) < 0.1


@pytest.mark.gpu
def test_end_to_end_odometry(raw_drive):
    """Raw distorted pairs with the rig's rectification against the undistorted originals: stereo odometry ok on every
    frame, translation within 2 % and rotation within 0.1 deg; mono odometry ok on every frame on both inputs and rotation
    within 0.1 deg.  The mono runs use bucket 1000 and 20 000 RANSAC iterations: with the defaults (bucket 2, 2 000
    iterations) the 8-point estimate scatters by 0.1 - 0.2 deg per frame between two runs on slightly different images, so
    the comparison would measure RANSAC, not the rectification.  The same stereo run on the raw images without
    rectification misses the stereo bounds."""
    orig, raw = raw_drive
    ref, rec, bad = H.Stereo(_stereo_params()), H.Stereo(_stereo_params()), H.Stereo(_stereo_params())
    assert rec.set_rectification(_true_rectification())
    mp = lambda: H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08,
                              bucket_max_features=1000, ransac_iters=20000)
    mref, mrec = H.Mono(mp()), H.Mono(mp())
    assert mrec.set_rectification(_true_rectification())
    stereo, misses, mono = [], 0, []
    for k in range(len(orig)):
        ok_ref, ok_rec, ok_bad = ref.process(*orig[k]), rec.process(*raw[k]), bad.process(*raw[k])
        mo_ref, mo_rec = mref.process(orig[k][0]), mrec.process(raw[k][0])
        if k == 0:
            continue
        stereo.append((k, ok_ref, ok_rec, _within(ref.motion(), rec.motion())))
        misses += not (ok_bad and _within(ref.motion(), bad.motion()))
        mono.append((k, mo_ref, mo_rec, _angle_deg(mref.motion()[:3, :3], mrec.motion()[:3, :3])))
    assert len(stereo) == len(mono) == len(orig) - 1
    assert all(a and b and c for _, a, b, c in stereo), stereo
    assert misses > 0
    assert all(a and b and d < 0.1 for _, a, b, d in mono), mono


def _ptrs(frames):
    return [np.ascontiguousarray(f).ctypes.data for f in frames]


@pytest.mark.gpu
@pytest.mark.parametrize('mode', [1, 2, 4])
def test_runner_against_facades(raw_drive, mode):
    """Runner modes 1, 2 and 4 with rectification equal per-sequence facades with rectification: matches, motion and points
    byte for byte (mode 2's motion within 1e-9: its facade estimates on the host, the runner on the device)."""
    orig, raw = raw_drive
    S, T = 3, len(raw)
    drives = [[tuple(np.ascontiguousarray(np.roll(x, 3 * s, axis=1)) for x in raw[k]) for k in range(T)] for s in range(S)]
    rect = _true_rectification()
    dims = np.array([KITTI_RAW[0], KITTI_RAW[1], KITTI_RAW[0]], np.int32)
    if mode == 1:
        runner, facades = H.Runner(0, S, 2, 1, 0, _mono_params()), [H.Mono(_mono_params()) for _ in range(S)]
    elif mode == 2:
        runner, facades = H.Runner.stereo(0, S, 2, _stereo_params()), [H.Stereo(_stereo_params()) for _ in range(S)]
    else:
        runner = H.Runner.stereo_sfm(0, S, 2, _stereo_params())
        facades = [H.StereoSfm(_stereo_params(), *KITTI_RAW) for _ in range(S)]
    try:
        assert runner.set_rectification(rect)
        assert all(f.set_rectification(rect) for f in facades)
        for k in range(T):
            left = [drives[s][k][0].ctypes.data for s in range(S)]
            right = [drives[s][k][1].ctypes.data for s in range(S)] if mode != 1 else None
            secs, nm, ok = runner.step(left, dims, ptrs2=right)
            for s in range(S):
                if mode == 1:
                    oks = facades[s].process(drives[s][k][0])
                elif mode == 2:
                    oks = facades[s].process(*drives[s][k])
                else:
                    oks = facades[s].update(*drives[s][k])
                vo = facades[s].odometry() if mode == 4 else facades[s]
                assert bool(ok[s]) == oks, (k, s)
                assert runner.matches(s).tobytes() == vo.matches().tobytes(), (k, s)
                if mode == 2:       # the facade estimates on the host, the runner on the device: equal to rounding
                    assert np.abs(runner.motion(s) - vo.motion()).max() < 1e-9, (k, s)
                else:
                    assert runner.motion(s).tobytes() == vo.motion().tobytes(), (k, s)
                if mode == 4:
                    assert runner.points(s).tobytes() == facades[s].points().tobytes(), (k, s)
            assert k == 0 or all(ok), k
        assert not runner.set_rectification(rect)
    finally:
        runner.close()


@pytest.mark.gpu
def test_refusals_leave_state(ctx):
    """A rectifying push without maps (ESTATE), a bad camera index or pitch (EINVAL) changes no frame; setRectification
    after the first frame returns False and the objects go on as before."""
    W, HT = OUT
    ctx.configure(V.Params(), W, HT, 2)
    a, b = (np.ascontiguousarray(x) for x in synth.corridor_stereo_frame(0))
    ctx.push_frames([0, 1], imgs=[a, b])
    before = [ctx.plane(f, 4)[0] for f in (0, 1)], [ctx.features(f, 1).tobytes() for f in (0, 1)]
    raw = np.zeros((KITTI_RAW[1], KITTI_RAW[0]), np.uint8)
    with pytest.raises(V.VisocuError, match=': -5 '):
        ctx.push_frames_rectified([0], [0], imgs=[raw])
    ctx.set_rectification([_true_rectification().cams[0]], *KITTI_RAW)
    with pytest.raises(V.VisocuError, match=': -1 '):
        ctx.push_frames_rectified([0], [1], imgs=[raw])
    with pytest.raises(V.VisocuError, match=': -1 '):
        ctx.push_frames_rectified([1], [0], imgs=[raw[:, :1000]], bpl_in=1000)
    with pytest.raises(V.VisocuError, match=': -1 '):
        ctx.set_rectification([_raw_cam(f=900.0, cu=620.0, cv=187.0, R=_rot((0, 1, 0), 120))], *KITTI_RAW)
    after = [ctx.plane(f, 4)[0] for f in (0, 1)], [ctx.features(f, 1).tobytes() for f in (0, 1)]
    assert all(np.array_equal(x, y) for x, y in zip(before[0], after[0])) and before[1] == after[1]
    with pytest.raises(V.VisocuError, match=': -1 '):
        ctx.set_rectification([_true_rectification().cams[0]] * 3, *KITTI_RAW)
    ctx.configure(V.Params(), W, HT, 2)                       # configure drops the maps
    with pytest.raises(V.VisocuError, match=': -5 '):
        ctx.push_frames_rectified([0], [0], imgs=[raw])

    seq = [synth.corridor_stereo_frame(k) for k in range(3)]
    late, plain = H.Stereo(_stereo_params()), H.Stereo(_stereo_params())
    sfm = H.StereoSfm(_stereo_params(), W, HT)
    for k, (left, right) in enumerate(seq):
        assert late.process(left, right) == plain.process(left, right)
        sfm.update(left, right)
        assert not late.set_rectification(_true_rectification())
        assert not sfm.set_rectification(_true_rectification())
        assert late.matches().tobytes() == plain.matches().tobytes() and late.motion().tobytes() == plain.motion().tobytes()
    m = H.Matcher(V.Params())
    m.push(seq[0][0])
    assert not m.set_rectification(_true_rectification())
    assert not H.Stereo(_stereo_params()).set_rectification(_rectification(_true_rectification().cams[:1], KITTI_RAW, OUT))
