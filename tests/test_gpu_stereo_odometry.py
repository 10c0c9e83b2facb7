"""Stereo odometry on the device: visocu_stereo_motion (3-point RANSAC over Gauss-Newton fits and the final refinement,
batched over match lists) against the host estimate of VisualOdometryStereo, and the stereo mode of the sequence runner
against stand-alone VisualOdometryStereo objects.  The host code restates the reference (tests/test_host_cpu.py pins it);
here it is the reference for the device path."""
import ctypes as C

import numpy as np
import pytest

import synth
import visocu_py as V
import host_py as H

F, CU, CV, BASE = 645.2, 635.9, 194.1, 0.54


def _params(**kw):
    d = dict(f=F, cu=CU, cv=CV, base=BASE)
    d.update(kw)
    return H.StereoParams(match=V.Params(), **d)


def rig_matches(n, seed, noise=0.3, outliers=0.15):
    """The rig of test_host_cpu.py::test_stereo_odometry_from_matches: points 5-50 m ahead, 0.8 m forward with a slight yaw."""
    rng = np.random.RandomState(seed)
    P = np.stack([rng.uniform(-10, 10, n), rng.uniform(-3, 1.6, n), rng.uniform(5, 50, n)], 1)
    yaw = 0.01 * (1 + seed % 3)
    R = np.array([[np.cos(yaw), 0, np.sin(yaw)], [0, 1, 0], [-np.sin(yaw), 0, np.cos(yaw)]])
    Q = P @ R.T + np.array([0.02, -0.01, -0.8])

    def project(X, shift):
        return F * (X[:, 0] - shift) / X[:, 2] + CU, F * X[:, 1] / X[:, 2] + CV

    m = np.zeros(n, V.P_MATCH)
    for name in ('i1p', 'i2p', 'i1c', 'i2c'):
        m[name] = np.arange(n)
    m['u1p'], m['v1p'] = project(P, 0.0); m['u2p'], m['v2p'] = project(P, BASE)
    m['u1c'], m['v1c'] = project(Q, 0.0); m['u2c'], m['v2c'] = project(Q, BASE)
    for name in ('u1p', 'v1p', 'u2p', 'u1c', 'v1c', 'u2c'):
        m[name] += rng.normal(0, noise, n).astype(np.float32)
    m['v2p'] = m['v1p']; m['v2c'] = m['v1c']
    bad = rng.rand(n) < outliers
    m['u1c'][bad] += rng.uniform(-40, 40, bad.sum()).astype(np.float32)
    return m


def test_batch_prepare_draws_the_process_table():
    """batchPrepare draws the RANSAC table that process(matches) draws (one getRandomSample(N, 3) per iteration), frame
    after frame; with fewer than 6 matches it draws nothing, as estimateMotion returns before its first draw."""
    a, b = H.Stereo(_params()), H.Stereo(_params())
    first = None
    for seed in (5, 6):
        m = rig_matches(400, seed)
        assert a.process_matches(m)
        assert b.batch_prepare(m)
        assert a.samples().shape == (200, 3)
        assert np.array_equal(a.samples(), b.samples())
        assert a.samples().min() >= 0 and a.samples().max() < 400
        if first is None:
            first = a.samples()
    assert not np.array_equal(first, a.samples())
    before = b.samples()
    assert not b.batch_prepare(rig_matches(5, 7))
    assert np.array_equal(b.samples(), before)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _rotation(tr):
    sx, cx, sy, cy, sz, cz = np.sin(tr[0]), np.cos(tr[0]), np.sin(tr[1]), np.cos(tr[1]), np.sin(tr[2]), np.cos(tr[2])
    return np.array([[cy * cz, -cy * sz, sy],
                     [sx * sy * cz + cx * sz, -sx * sy * sz + cx * cz, -sx * cy],
                     [-cx * sy * cz + sx * sz, cx * sy * sz + sx * cz, cx * cy]])


def _errors(m, R, t, p):
    """getInlier's unweighted squared reprojection error of every match under (R, t) (numpy, float disparity as the host)."""
    d = np.maximum(m['u1p'] - m['u2p'], np.float32(0.0001)).astype(np.float64)
    u1p, v1p = m['u1p'].astype(np.float64), m['v1p'].astype(np.float64)
    P = np.stack([(u1p - p.cu) * p.base / d, (v1p - p.cv) * p.base / d, p.f * p.base / d], 1)
    Q = P @ R.T + t
    pred = np.stack([p.f * Q[:, 0] / Q[:, 2] + p.cu, p.f * Q[:, 1] / Q[:, 2] + p.cv,
                     p.f * (Q[:, 0] - p.base) / Q[:, 2] + p.cu, p.f * Q[:, 1] / Q[:, 2] + p.cv], 1)
    obs = np.stack([m['u1c'], m['v1c'], m['u2c'], m['v2c']], 1).astype(np.float64)
    return ((obs - pred) ** 2).sum(1)


def _device_and_host(ctx, m, p, want_all=False):
    """(device object after batchFinish, host object after process_matches, host ok, device ok, raw device result)"""
    dev, host = H.Stereo(p), H.Stereo(p)
    ok_h = host.process_matches(m)
    assert dev.batch_prepare(m)
    r = ctx.stereo_motion([m], [dev.samples()], p, want_all=want_all)[0]
    ok_d = dev.batch_finish(r['tr'], r['ok'], r['mask'])
    assert ok_d == r['ok']
    return dev, host, ok_h, ok_d, r


def _same_state(dev, host, ok_h, ok_d):
    assert ok_d == ok_h
    assert np.array_equal(dev.inliers(), host.inliers())
    Md, Mh = dev.motion(), host.motion()
    assert np.array_equal(np.isnan(Md), np.isnan(Mh))
    assert np.nan_to_num(np.abs(Md - Mh)).max() < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize('reweighting', [1, 0])
@pytest.mark.parametrize('n', [400, 1500, 4000, 20000])
def test_stereo_motion_against_host(ctx, n, reweighting):
    """Same sample table, same matches: the device gives the host's ok, the identical inlier set and the motion within
    1e-9.  Every scored hypothesis' count is recomputed from its tr_all row; counts may differ only by rounding at the
    threshold (at most 1 % of the hypotheses)."""
    p = _params(reweighting=reweighting)
    m = rig_matches(n, seed=n + reweighting)
    dev, host, ok_h, ok_d, r = _device_and_host(ctx, m, p, want_all=True)
    assert ok_h
    _same_state(dev, host, ok_h, ok_d)
    assert len(host.inliers()) > 0.7 * n
    assert r['n_inliers'] == len(host.inliers()) and np.array_equal(r['inliers'], host.inliers())
    assert abs(host.motion()[2, 3] + 0.8) < 0.05
    counts, tr_all = r['counts'], r['tr_all']
    assert counts.min() >= -1 and (counts > 0).sum() > 0.5 * len(counts)
    scored = np.nonzero(counts >= 0)[0]
    again = np.array([(_errors(m, _rotation(tr_all[k]), tr_all[k][3:], p) < p.inlier_threshold ** 2).sum() for k in scored])
    differ = np.nonzero(again != counts[scored])[0]
    assert len(differ) <= max(1, len(counts) // 100), (scored[differ], again[differ], counts[scored][differ])
    assert r['best_iter'] == int(np.argmax(counts)) and counts[r['best_iter']] == r['n_inliers']


def _raw_call(ctx, lists, N, samples, p, outs):
    """visocu_stereo_motion with caller-made pointer arrays (None entries stay null)."""
    nj = len(N)
    arr = lambda xs: (C.c_void_p * nj)(*[None if x is None else x.ctypes.data for x in xs])
    tr6, ok, masks, ninl, best = outs
    return V.lib().visocu_stereo_motion(ctx.h, nj, arr(lists), V._p(np.asarray(N, np.int32)), arr(samples), C.byref(p),
                                        V._p(tr6), V._p(ok), arr(masks), V._p(ninl), V._p(best), None, None)


@pytest.mark.gpu
def test_stereo_motion_failure_cases(ctx):
    """Degenerate inputs give what the host object gives: no calibration (f = 0: every prediction is NaN, every hypothesis
    'converges' to NaN and scores 0), all matches on one pixel (rank-deficient normal equations), fewer than 6 inliers.
    Malformed calls are refused with VISOCU_EINVAL and write nothing."""
    m = rig_matches(400, 3)
    # f = 0: the host fails with no inliers; the device scores every hypothesis 0 (not -1) and has no winner
    p0 = _params(f=0.0)
    dev, host, ok_h, ok_d, r = _device_and_host(ctx, m, p0, want_all=True)
    assert not ok_h and len(host.inliers()) == 0
    _same_state(dev, host, ok_h, ok_d)
    assert r['best_iter'] == -1 and r['n_inliers'] == 0 and np.all(r['counts'] == 0)
    # all matches on one pixel: every sample is three copies of one match and the normal equations are singular (rank 3).
    # The same ok and inliers; the minimiser is not unique (the step's null-space part is rounding noise over a pivot made
    # of rounding noise), so instead of the motion: both motions map the pixel within the threshold
    one = np.repeat(m[:1], 50)
    dev, host, ok_h, ok_d, r = _device_and_host(ctx, one, _params())
    assert ok_d == ok_h and np.array_equal(dev.inliers(), host.inliers())
    if ok_h:
        assert len(host.inliers()) == 50
        for T in (dev.motion(), host.motion()):
            assert np.all(_errors(one, T[:3, :3], T[:3, 3], _params()) < 2.0 ** 2)
    # 12 matches: 5 from one motion, 7 with independent offsets of 20-40 px
    rng = np.random.RandomState(9)
    few = rig_matches(12, 11, noise=0.0, outliers=0.0)
    few['u1c'][5:] += (rng.uniform(20, 40, 7) * rng.choice([-1, 1], 7)).astype(np.float32)
    few['v1c'][5:] += (rng.uniform(20, 40, 7) * rng.choice([-1, 1], 7)).astype(np.float32)
    dev, host, ok_h, ok_d, r = _device_and_host(ctx, few, _params())
    assert not ok_h and len(host.inliers()) < 6
    _same_state(dev, host, ok_h, ok_d)
    # malformed calls
    sp = V.StereoMotionParams(f=F, cu=CU, cv=CV, base=BASE, inlier_threshold=2.0, ransac_iters=200, reweighting=1)
    good = np.ascontiguousarray(m)
    smp = np.random.RandomState(1).randint(0, 400, (200, 3)).astype(np.int32)
    bad_smp = smp.copy(); bad_smp[17, 2] = 400
    for lists, N, samples in (([good], [5], [smp % 5]), ([good], [400], [bad_smp]), ([None], [400], [smp]),
                              ([good], [400], [None]), ([good, good], [400, 400], [smp, bad_smp])):
        nj = len(N)
        outs = (np.full((nj, 6), 7.0), np.full(nj, 7, np.int32), [np.full(400, 7, np.uint8) for _ in range(nj)],
                np.full(nj, 7, np.int32), np.full(nj, 7, np.int32))
        assert _raw_call(ctx, lists, N, samples, sp, outs) == -1
        assert np.all(outs[0] == 7.0) and np.all(outs[1] == 7) and all(np.all(x == 7) for x in outs[2])
        assert np.all(outs[3] == 7) and np.all(outs[4] == 7)


@pytest.mark.gpu
def test_stereo_motion_batching_and_determinism(ctx):
    """One call over jobs of different N gives, byte for byte, what the jobs give one at a time; a repeated call gives the
    same bytes (no floating-point atomics, a fixed reduction tree)."""
    p = _params()
    lists = [rig_matches(n, seed=40 + k) for k, n in enumerate((400, 20000, 1500, 6, 4000))]
    tables = []
    for ml in lists:
        h = H.Stereo(p)
        assert h.batch_prepare(ml)
        tables.append(h.samples())
    keys = ('tr', 'mask', 'counts', 'tr_all')
    both = [ctx.stereo_motion(lists, tables, p, want_all=True) for _ in range(2)]
    for a, b in zip(*both):
        for k in keys:
            assert a[k].tobytes() == b[k].tobytes(), k
    for j, (ml, t) in enumerate(zip(lists, tables)):
        one = ctx.stereo_motion([ml], [t], p, want_all=True)[0]
        for k in keys:
            assert one[k].tobytes() == both[0][j][k].tobytes(), (j, k)
        assert (one['ok'], one['n_inliers'], one['best_iter']) == (both[0][j]['ok'], both[0][j]['n_inliers'], both[0][j]['best_iter'])
    assert sum(r['ok'] for r in both[0]) >= 4


@pytest.mark.gpu
@pytest.mark.parametrize('bucket', [2, 1000])
def test_stereo_runner_against_objects(bucket):
    """Runner mode 2 (quad matching of all sequences in one MatcherBatch with each sequence's predicted motion, one
    visocu_stereo_motion per worker) against stand-alone VisualOdometryStereo objects on the same frames: per step the same
    ok, byte-identical match lists, the same inliers and the motion within 1e-9."""
    S, T = 5, 6
    frames = [[synth.corridor_stereo_frame(k, seed=1234 + s) for k in range(T)] for s in range(S)]
    p = H.StereoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, base=0.54,
                       bucket_max_features=bucket)
    objs = [H.Stereo(p) for _ in range(S)]
    runner = H.Runner.stereo(0, S, 2, p)
    dims = np.array([1241, 376, 1241], np.int32)
    try:
        for k in range(T):
            left = [np.ascontiguousarray(frames[s][k][0]) for s in range(S)]
            right = [np.ascontiguousarray(frames[s][k][1]) for s in range(S)]
            secs, nm, ok = runner.step([a.ctypes.data for a in left], dims, ptrs2=[a.ctypes.data for a in right])
            for s in range(S):
                ok_h = objs[s].process(left[s], right[s])
                assert bool(ok[s]) == ok_h, (k, s)
                if k == 0:
                    continue
                assert ok_h, (k, s)
                mh = objs[s].matches()
                assert nm[s] == len(mh) and len(mh) > (100 if bucket == 2 else 1000)
                assert runner.matches(s).tobytes() == mh.tobytes(), (k, s)
                assert np.array_equal(runner.inliers(s), objs[s].inliers()), (k, s)
                assert np.abs(runner.motion(s) - objs[s].motion()).max() < 1e-9, (k, s)
    finally:
        runner.close()
