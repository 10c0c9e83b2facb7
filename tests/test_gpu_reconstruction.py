"""Reconstruction on the device: visocu_recon_points (triangulation, point type, Gauss-Newton refinement, distance and
ray-angle tests of the finished tracks of many Reconstruction updates at once) against the host functions of
Reconstruction, and the structure-from-motion mode of the sequence runner against stand-alone StructureFromMotion objects.
The host code restates the reference (tests/test_host_cpu.py pins it); here it is the reference for the device path."""
import ctypes as C

import numpy as np
import pytest

import synth
import visocu_py as V
import host_py as H

PARAMS = [(0, 2, 3.0), (1, 2, 2.0), (2, 3, 1.0)]      # point_type, min_track_length, min_angle of the host-vs-reference test
MAX_DIST = 30.0


def _recon():
    return H.Recon(synth.KITTI_F, synth.KITTI_CU, synth.KITTI_CV)


def _close(a, b):
    return len(a) == len(b) and (len(a) == 0 or np.abs(a - b).max() <= 1e-5 * max(1.0, np.abs(a).max()))


@pytest.mark.parametrize('point_type,min_len,min_angle', PARAMS)
def test_batch_api_equals_update(point_type, min_len, min_angle):
    """The batch API through its C entries and Python binding (batch_prepare, batch_job, host_eval, batch_finish) leaves
    the points update() leaves, byte for byte, after every frame.  update() is these same three steps, so this pins the
    entries and the job they hand out; test_host_cpu.py::test_reconstruction_matches_reference pins update() itself."""
    a, b = _recon(), _recon()
    kept = 0
    for m, tr in synth.track_sequence(n_frames=14, n_points=700, seed=21):
        a.update(m, tr, point_type, min_len, MAX_DIST, min_angle)
        n = b.batch_prepare(m, tr, point_type, min_len, MAX_DIST, min_angle)
        job = b.batch_job()
        assert n == len(job['tracks'])
        status, xyz = b.host_eval()
        b.batch_finish(status, xyz)
        assert a.points().tobytes() == b.points().tobytes()
        kept += int((status == 0).sum())
    assert kept == len(a.points()) > 50


def test_window_holds_at_most_six_frames():
    """A track anchored at frame U ends by update U + 5, and the front frame is popped first: at most 6 frames."""
    r = _recon()
    sizes = []
    for m, tr in synth.track_sequence(n_frames=200, drop=0.05):
        r.batch_prepare(m, tr, 0, 2, MAX_DIST, 3.0)
        job = r.batch_job()
        sizes.append(len(job['frames']))
        t = job['tracks']
        assert np.all((t['n_obs'] >= 2) & (t['n_obs'] <= 6) & (t['first'] >= 0) & (t['first'] + t['n_obs'] <= sizes[-1]))
        r.batch_finish(*r.host_eval())
    assert max(sizes) == 6


# ---------------------------------------------------------------------------------------------------------------- GPU
def _numpy_tests(job, status, xyz):
    """pointDistance and rayAngle recomputed from xyz in float64; they must give the status (0, 4 or 5) the call gave."""
    fr = job['frames']
    n = len(fr)
    for k in np.nonzero(np.isin(status, (0, 4, 5)))[0]:
        t = job['tracks'][k]
        p = xyz[k].astype(np.float64)
        mid = n - 1 - (n - int(t['first'])) // 2
        dist = np.sqrt(((fr[mid]['center'] - p) ** 2).sum())
        v1, v2 = fr[t['first']]['center'] - p, fr[n - 1]['center'] - p
        n1, n2 = np.sqrt((v1 ** 2).sum()), np.sqrt((v2 ** 2).sum())
        angle = 1000.0 if n1 < 1e-10 or n2 < 1e-10 else np.degrees(np.arccos(abs(((v1 / n1) * (v2 / n2)).sum())))
        want = 4 if not dist < job['max_dist'] else (5 if not angle > job['min_angle'] else 0)
        assert status[k] == want, (k, status[k], dist, angle)


@pytest.mark.gpu
@pytest.mark.parametrize('point_type,min_len,min_angle', PARAMS)
@pytest.mark.parametrize('n_points', [600, 6000])
def test_recon_points_against_host(ctx, n_points, point_type, min_len, min_angle):
    """The prepared jobs of whole sequences: the device status equals the host's for every track, kept points agree to
    1e-5 x max(1, |p|), statuses 0, 2, 4 and 5 all occur, and distance and angle recomputed in numpy give the status."""
    r = _recon()
    seen = set()
    for m, tr in synth.track_sequence(n_frames=14, n_points=n_points, seed=21):
        r.batch_prepare(m, tr, point_type, min_len, MAX_DIST, min_angle)
        job = r.batch_job()
        hs, hx = r.host_eval()
        ds, dx = ctx.recon_points([job])[0]
        differ = np.nonzero(ds != hs)[0]
        assert len(differ) == 0, (differ, hs[differ], ds[differ])
        kept = hs == 0
        assert _close(hx[kept], dx[kept])
        assert np.all(dx[np.isin(ds, (1, 3))] == 0)
        _numpy_tests(job, ds, dx)
        seen |= set(ds.tolist())
        r.batch_finish(hs, hx)
    assert {0, 2, 4, 5} <= seen, seen


def _look_at_job(centers, obs, min_angle=3.0, zero_row=None):
    """A job of cameras with the newest camera's orientation at `centers` (newest last, in its coordinates) and one track
    per entry of obs: (first, [(u, v), ...])."""
    K = np.array([[synth.KITTI_F, 0, synth.KITTI_CU], [0, synth.KITTI_F, synth.KITTI_CV], [0, 0, 1]])
    fr = np.zeros(len(centers), V.RECON_FRAME)
    for k, c in enumerate(centers):
        inv = np.hstack([np.eye(3), -np.asarray(c, np.float64)[:, None]])
        proj = K @ inv
        if zero_row == k:
            proj[2] = 0
        fr[k]['proj'], fr[k]['inv'], fr[k]['center'] = proj.ravel(), inv.ravel(), c
    tr = np.zeros(len(obs), V.RECON_TRACK)
    for i, (first, uv) in enumerate(obs):
        tr[i]['first'], tr[i]['n_obs'] = first, len(uv)
        for k, (u, v) in enumerate(uv):
            tr[i]['u'][k], tr[i]['v'][k] = u, v
    road = np.zeros((3, 4))
    road[0, 0] = 1; road[1, 1] = road[2, 2] = np.cos(-0.08); road[1, 2] = -np.sin(-0.08); road[2, 1] = np.sin(-0.08); road[1, 3] = -1.6
    return dict(frames=fr, tracks=tr, cam_road=road.ravel(), max_dist=MAX_DIST, min_angle=min_angle, point_type=0)


def _project(P, c):
    X = np.asarray(P, np.float64) - c
    return synth.KITTI_F * X[0] / X[2] + synth.KITTI_CU, synth.KITTI_F * X[1] / X[2] + synth.KITTI_CV


@pytest.mark.gpu
def test_recon_points_rare_statuses(ctx):
    """Hand-built jobs: parallel rays (the camera moved sideways, the same pixel in both frames) fail initPoint (status 1);
    a middle frame whose third projection row is zero fails refinePoint (status 3); the same track with a sound middle
    frame is kept, at the point it was made from."""
    centers = [np.array([-2.0, 0, 0]), np.array([-1.0, 0, 0]), np.zeros(3)]
    P = np.array([0.5, 0.3, 10.0])
    track = (0, [_project(P, c) for c in centers])
    parallel = _look_at_job(centers[1:], [(0, [(700.0, 200.0), (700.0, 200.0)])])
    bad_middle = _look_at_job(centers, [track], zero_row=1)
    control = _look_at_job(centers, [track])
    (s1, x1), (s3, x3), (s0, x0) = ctx.recon_points([parallel, bad_middle, control])
    assert s1.tolist() == [1] and np.all(x1 == 0)
    assert s3.tolist() == [3] and np.all(x3 == 0)
    assert s0.tolist() == [0] and np.abs(x0[0] - P).max() < 1e-3


def _sequence_jobs(n_frames, n_points, seed):
    r = _recon()
    jobs = []
    for m, tr in synth.track_sequence(n_frames=n_frames, n_points=n_points, seed=seed):
        r.batch_prepare(m, tr, 0, 2, MAX_DIST, 3.0)
        jobs.append(r.batch_job())
        r.batch_finish(*r.host_eval())
    return jobs


@pytest.mark.gpu
def test_recon_points_batching_and_determinism(ctx):
    """One call over 20 jobs (the first one without tracks) gives the bytes of one call per job; a repeated call gives the
    same bytes; a call with tracks is one launch, a call without none."""
    jobs = _sequence_jobs(21, 3000, 5)
    assert len(jobs) == 20 and len(jobs[0]['tracks']) == 0 and sum(len(j['tracks']) for j in jobs[1:]) > 1000
    n0 = ctx.launch_count()
    both = [ctx.recon_points(jobs) for _ in range(2)]
    assert ctx.launch_count() == n0 + 2
    for (sa, xa), (sb, xb) in zip(*both):
        assert sa.tobytes() == sb.tobytes() and xa.tobytes() == xb.tobytes()
    for j, job in enumerate(jobs):
        n0 = ctx.launch_count()
        s, x = ctx.recon_points([job])[0]
        assert ctx.launch_count() == n0 + (1 if len(job['tracks']) else 0)
        assert s.tobytes() == both[0][j][0].tobytes() and x.tobytes() == both[0][j][1].tobytes(), j


def _raw_call(ctx, jobs, status, xyz, jobs_null=False, status_null=False, xyz_null=False):
    nj = len(jobs)
    arr = (V.ReconJob * nj)()
    keep = []
    for j, job in enumerate(jobs):
        fr, tr = job['frames'], job['tracks']
        keep += [fr, tr]
        a = arr[j]
        a.frames = None if fr is None else fr.ctypes.data
        a.n_frames = job['n_frames']
        a.tracks = None if tr is None else tr.ctypes.data
        a.n_tracks = job['n_tracks']
        a.cam_road[:] = list(job['cam_road'])
        a.max_dist, a.min_angle, a.point_type = job['max_dist'], job['min_angle'], job['point_type']
    sp = (C.c_void_p * nj)(*[None if s is None else s.ctypes.data for s in status])
    xp = (C.c_void_p * nj)(*[None if x is None else x.ctypes.data for x in xyz])
    return V.lib().visocu_recon_points(ctx.h, nj, None if jobs_null else arr, None if status_null else sp, None if xyz_null else xp)


@pytest.mark.gpu
def test_recon_points_malformed_calls(ctx):
    """Null pointers, a window outside [1, 8] frames, n_obs outside [2, 6], observations outside the window and a negative
    track count are refused with VISOCU_EINVAL, and nothing is written."""
    good = next(j for j in _sequence_jobs(8, 600, 3) if len(j['tracks']) > 3)
    good = dict(good, n_frames=len(good['frames']), n_tracks=len(good['tracks']))
    nt = good['n_tracks']

    def with_track(field, value):
        tr = good['tracks'].copy()
        tr[nt // 2][field] = value
        return dict(good, tracks=tr)

    frames9 = np.concatenate([good['frames']] * 3)[:9]
    cases = [dict(good, frames=None), dict(good, tracks=None), dict(good, n_frames=0), dict(good, frames=frames9, n_frames=9),
             dict(good, n_tracks=-1), with_track('n_obs', 1), with_track('n_obs', 7), with_track('first', -1),
             with_track('first', good['n_frames'] - 1)]
    calls = [([good, c], {}, None) for c in cases] + [([good], dict(jobs_null=True), None), ([good], dict(status_null=True), None),
                                                       ([good], dict(xyz_null=True), None), ([good, good], {}, 'status'),
                                                       ([good, good], {}, 'xyz')]
    for k, (jobs, kw, missing) in enumerate(calls):
        status = [np.full(nt, 7, np.int32) for _ in jobs]
        xyz = [np.full((nt, 3), 7.0, np.float32) for _ in jobs]
        if missing == 'status':
            status[1] = None                                   # a job with tracks but no status array
        if missing == 'xyz':
            xyz[1] = None                                      # ... or no point array
        assert _raw_call(ctx, jobs, status, xyz, **kw) == -1, k
        assert all(s is None or np.all(s == 7) for s in status) and all(x is None or np.all(x == 7) for x in xyz), k
    status, xyz = [np.full(nt, 7, np.int32)], [np.full((nt, 3), 7.0, np.float32)]
    assert _raw_call(ctx, [good], status, xyz) == 0 and np.all(status[0] <= 5)


@pytest.mark.gpu
@pytest.mark.parametrize('n_points', [600, 6000])
def test_device_reconstruction_of_whole_sequences(ctx, n_points):
    """batchPrepare, the device call and batchFinish over whole sequences against update() on the same stream: the same
    number of points after every frame, coordinates within 1e-5 x max(1, |p|)."""
    a, b = _recon(), _recon()
    for m, tr in synth.track_sequence(n_frames=30, n_points=n_points, seed=8, drop=0.1):
        a.update(m, tr, 0, 2, MAX_DIST, 3.0)
        b.batch_prepare(m, tr, 0, 2, MAX_DIST, 3.0)
        b.batch_finish(*ctx.recon_points([b.batch_job()])[0])
        assert _close(a.points(), b.points())
    assert len(a.points()) > (100 if n_points == 600 else 1000)


def _mono_params(bucket):
    return H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08,
                        bucket_max_features=bucket)


@pytest.mark.gpu
@pytest.mark.parametrize('bucket', [2, 1000])
def test_sfm_runner_against_facade(bucket):
    """Runner mode 3 against stand-alone StructureFromMotion objects on the same frames: per step the same ok, the pose
    within 1e-9, the same number of points and coordinates within 1e-5 x max(1, |p|); run() gives the bytes of stepping.
    Sequence 1 barely moves at step 3 (frame 3 is frame 2 shifted by one pixel: the odometry fails), so step 4 has to push
    with replace, i.e. match frame 2 against frame 4.  Its matches at step 4 are those of a stand-alone VisualOdometryMono
    that pushes with replace, and differ from the matches of one that does not."""
    S, T = 3, 7
    frames = [synth.corridor_sequence(T, seed=1234 + s) for s in range(S)]
    frames[1][3] = np.roll(frames[1][2], 1, axis=1)
    frames = [[np.ascontiguousarray(f) for f in seq] for seq in frames]
    p = _mono_params(bucket)
    objs = [H.Sfm(p, 1241, 376) for _ in range(S)]
    dims = np.array([1241, 376, 1241], np.int32)
    ptrs = [[frames[s][k].ctypes.data for s in range(S)] for k in range(T)]
    runner = H.Runner.sfm(0, S, 2, p)
    oks = []
    try:
        for k in range(T):
            secs, nm, ok = runner.step(ptrs[k], dims)
            oks.append(ok)
            for s in range(S):
                assert bool(ok[s]) == objs[s].update(frames[s][k]), (k, s)
                assert np.abs(runner.pose(s) - objs[s].pose()).max() < 1e-9, (k, s)
                assert _close(objs[s].points(), runner.points(s)), (k, s, len(objs[s].points()), len(runner.points(s)))
            if k == 4:
                step4 = runner.matches(1)
        assert not oks[3][1] and oks[4][1] and all(oks[k][s] for k in range(1, T) for s in (0, 2)), np.array(oks)
        assert min(len(runner.points(s)) for s in range(S)) > 20
        want = ([runner.points(s).tobytes() for s in range(S)], [runner.pose(s).tobytes() for s in range(S)])
    finally:
        runner.close()
    replaced, kept = H.Mono(p), H.Mono(p)
    for k in range(5):
        replaced.process(frames[1][k], replace=(k == 4))
        kept.process(frames[1][k])
    assert step4.tobytes() == replaced.matches().tobytes() and len(step4) > 20
    assert step4.tobytes() != kept.matches().tobytes()
    again = H.Runner.sfm(0, S, 2, p)
    try:
        secs, nm, ok = again.run(ptrs, dims)
        assert np.array_equal(ok, np.array(oks))
        assert [again.points(s).tobytes() for s in range(S)] == want[0]
        assert [again.pose(s).tobytes() for s in range(S)] == want[1]
    finally:
        again.close()
