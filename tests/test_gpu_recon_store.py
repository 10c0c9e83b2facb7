"""Device point stores: visocu_recon_update (the move of every stored point into the new camera frame, the evaluation of the
finished tracks and the append of the kept points, on the device) against the host Reconstruction, whose batch halves and
affineTransform are the reference; and the structure-from-motion runner modes, whose points now live in such stores."""
import ctypes as C
import functools

import numpy as np
import pytest

import synth
import visocu_py as V
import host_py as H

W, HT = 1241, 376
DIMS = np.array([W, HT, W], np.int32)
RECON = (0, 2, 30.0, 3.0)       # the facades' constants: point type, min track length, max distance, min angle


def _recon():
    return H.Recon(synth.KITTI_F, synth.KITTI_CU, synth.KITTI_CV)


def test_batch_prepare_tracks_equals_batch_prepare():
    """batchPrepareTracks hands out the job batchPrepare hands out (frames, tracks, parameters) on the same object history,
    and leaves the host points where they are."""
    a, b = _recon(), _recon()
    moved = 0
    for m, tr in synth.track_sequence(n_frames=20, n_points=700, seed=21):
        before = b.points()
        na, nb = a.batch_prepare(m, tr, *RECON), b.batch_prepare_tracks(m, tr, *RECON)
        assert b.points().tobytes() == before.tobytes()
        moved += int(len(before) > 0 and a.points().tobytes() != before.tobytes())
        ja, jb = a.batch_job(), b.batch_job()
        assert na == nb == len(jb['tracks'])
        assert ja['frames'].tobytes() == jb['frames'].tobytes() and ja['tracks'].tobytes() == jb['tracks'].tobytes()
        assert ja['cam_road'].tobytes() == jb['cam_road'].tobytes()
        assert (ja['max_dist'], ja['min_angle'], ja['point_type']) == (jb['max_dist'], jb['min_angle'], jb['point_type'])
        result = a.host_eval()
        a.batch_finish(*result)
        b.batch_finish(*result)
    assert moved > 10 and len(b.points()) > 50


# ---------------------------------------------------------------------------------------------------------------- GPU
def _random_points(rng, n):
    """Finite floats over the whole exponent range, with subnormals, +-1e30 and exact zeros mixed in."""
    mag = 10.0 ** rng.uniform(-44, 30, (n, 3))
    p = (np.where(rng.rand(n, 3) < 0.5, -1.0, 1.0) * mag).astype(np.float32)
    normal = (rng.standard_normal((n, 3)) * 20).astype(np.float32)
    p = np.where(rng.rand(n, 3) < 0.5, normal, p)
    special = np.array([0.0, -0.0, 1e-40, -3e-42, 1e30, -1e30, 1e-45], np.float32)
    k = rng.rand(n, 3) < 0.05
    p[k] = special[rng.randint(0, len(special), int(k.sum()))]
    assert np.all(np.isfinite(p))
    return np.ascontiguousarray(p)


def _rigid(rng):
    q, r = np.linalg.qr(rng.standard_normal((3, 3)))
    T = np.eye(4)
    T[:3, :3] = q * np.sign(np.diag(r))
    T[:3, 3] = rng.uniform(-1e4, 1e4, 3)
    return T


def _empty_job():
    r = _recon()
    r.batch_prepare(np.zeros(0, V.P_MATCH), np.eye(4), *RECON)
    job = r.batch_job()
    assert len(job['tracks']) == 0
    return job


@pytest.mark.gpu
def test_move_is_bit_exact(ctx):
    """Stores of 0, 1, 3, 4, 5, 1000 and 2^20 + 7 points (every tail length, the vector path) moved in one call by random
    rigid transforms with large translations: the bytes of the host's own affineTransform, twice in a row; one launch."""
    rng = np.random.RandomState(3)
    sizes = [0, 1, 3, 4, 5, 1000, 2 ** 20 + 7]
    stores = [ctx.recon_store() for _ in sizes]
    try:
        pts = [_random_points(rng, n) for n in sizes]
        for s, p in zip(stores, pts):
            s.append(p)
            assert s.count == len(p) and s.read().tobytes() == p.tobytes()
        job = _empty_job()
        for _ in range(2):
            trs = [_rigid(rng) for _ in sizes]
            n0 = ctx.launch_count()
            kept = ctx.recon_update(stores, trs, [job] * len(sizes))
            assert ctx.launch_count() == n0 + 1 and not kept.any()
            for k, (s, T) in enumerate(zip(stores, trs)):
                pts[k] = H.affine_points(T, pts[k])
                assert s.count == sizes[k] and s.read().tobytes() == pts[k].tobytes(), sizes[k]
    finally:
        for s in stores:
            s.close()


def _mono_params(bucket):
    return H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08,
                        bucket_max_features=bucket)


@functools.lru_cache(maxsize=None)
def _drive(bucket, T, seed=1234):
    """(matches, motion) of every successful frame pair of a corridor drive under the mono odometry runner (mode 1)."""
    frames = [np.ascontiguousarray(f) for f in synth.corridor_sequence(T, seed=seed)]
    r = H.Runner(0, 1, 1, 1, 0, _mono_params(bucket))
    out = []
    try:
        for k, f in enumerate(frames):
            secs, nm, ok = r.step([f.ctypes.data], DIMS)
            if k > 0 and ok[0]:
                out.append((r.matches(0), r.motion(0)))
    finally:
        r.close()
    return out


def _check_update(ctx, store, T, job):
    """One update of `store` against recon_points on the same job: kept count, status and point bytes, appended rows."""
    before = store.read()
    kept, [(status, xyz)] = ctx.recon_update([store], [T], [job], want_status=True)
    ds, dx = ctx.recon_points([job])[0]
    assert status.tobytes() == ds.tobytes() and xyz.tobytes() == dx.tobytes()
    assert kept[0] == int((status == 0).sum()) == store.count - len(before)
    assert store.read(len(before)).tobytes() == xyz[status == 0].tobytes()
    assert store.read(0, len(before)).tobytes() == H.affine_points(T, before).tobytes()
    return status, xyz


@pytest.mark.gpu
@pytest.mark.parametrize('source', ['corridor2', 'corridor1000', 'tracks'])
def test_evaluate_and_append(ctx, source):
    """Jobs of H.Recon's batch halves on corridor drives (bucket 2 and 1000) and on synthetic tracks: the kept count is the
    number of status-0 tracks, the optional status and points are recon_points' bytes, and the appended rows are the
    status-0 points in track order, behind the moved ones."""
    steps = (_drive(int(source[8:]), 12) if source.startswith('corridor')
             else synth.track_sequence(n_frames=14, n_points=3000, seed=21))
    r = _recon()
    store = ctx.recon_store()
    try:
        kept = 0
        for m, T in steps:
            r.batch_prepare_tracks(m, T, *RECON)
            status, _ = _check_update(ctx, store, T, r.batch_job())
            kept += int((status == 0).sum())
        assert kept > 20 and store.count == kept
    finally:
        store.close()


def _sequence_jobs(n_frames, n_points, seed):
    r = _recon()
    jobs = []
    for m, tr in synth.track_sequence(n_frames=n_frames, n_points=n_points, seed=seed):
        r.batch_prepare(m, tr, *RECON)
        jobs.append((r.batch_job(), tr))
        r.batch_finish(*r.host_eval())
    return jobs


@pytest.mark.gpu
def test_batching(ctx):
    """One call over 20 stores and jobs (the first job without tracks) leaves the bytes of one call per job, and returns
    the same kept counts, statuses and points."""
    rng = np.random.RandomState(9)
    jobs = _sequence_jobs(21, 3000, 5)
    assert len(jobs) == 20 and len(jobs[0][0]['tracks']) == 0
    init = [(rng.standard_normal((int(rng.randint(0, 3000)), 3)) * 10).astype(np.float32) for _ in jobs]
    together = [ctx.recon_store() for _ in jobs]
    alone = [ctx.recon_store() for _ in jobs]
    try:
        for s, t, p in zip(together, alone, init):
            s.append(p); t.append(p)
        kept, res = ctx.recon_update(together, [tr for _, tr in jobs], [j for j, _ in jobs], want_status=True)
        for k, (job, tr) in enumerate(jobs):
            kept1, [(s1, x1)] = ctx.recon_update([alone[k]], [tr], [job], want_status=True)
            assert kept1[0] == kept[k] and s1.tobytes() == res[k][0].tobytes() and x1.tobytes() == res[k][1].tobytes(), k
            assert alone[k].read().tobytes() == together[k].read().tobytes(), k
        assert kept[0] == 0 and kept.sum() > 500
    finally:
        for s in together + alone:
            s.close()


@pytest.mark.gpu
def test_whole_sequence_against_host(ctx):
    """A store that starts with room for 16 points, driven by batch_prepare_tracks + recon_update over a 40-frame drive at
    bucket 1000, holds the bytes of an H.Recon driven by batch_prepare + recon_points + batch_finish after every update."""
    steps = _drive(1000, 40)
    assert len(steps) >= 35
    host, dev = _recon(), _recon()
    store = ctx.recon_store(initial_capacity=16)
    try:
        for m, T in steps:
            host.batch_prepare(m, T, *RECON)
            host.batch_finish(*ctx.recon_points([host.batch_job()])[0])
            dev.batch_prepare_tracks(m, T, *RECON)
            ctx.recon_update([store], [T], [dev.batch_job()])
            assert store.read().tobytes() == host.points().tobytes()
        assert store.count > 5000
    finally:
        store.close()


def _stereo_params(bucket):
    return H.StereoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, base=0.54,
                          bucket_max_features=bucket)


def _stereo_drives(S, T, failed):
    """As tests/test_gpu_stereo_sfm.py makes them: the right image of frame k of drive s (failed = (s, k)) is shifted down
    by 40 rows, so that no motion explains its matches and the odometry fails."""
    drives = [[tuple(np.ascontiguousarray(x) for x in synth.corridor_stereo_frame(k, seed=1234 + s)) for k in range(T)]
              for s in range(S)]
    s, k = failed
    drives[s][k] = (drives[s][k][0], np.ascontiguousarray(np.roll(drives[s][k][1], 40, axis=0)))
    return drives


@pytest.mark.gpu
@pytest.mark.parametrize('mode', [3, 4])
def test_runner_against_host_composition(ctx, mode):
    """30 frames of 3 sequences on 2 workers (mode 3), or with frame 3 of sequence 1 failing (mode 4): after every step each
    sequence's points equal, byte for byte, those of H.Recon's batch halves and recon_points fed the runner's matches and
    motions, and its pose equals theirs accumulated in numpy within 1e-9.  points_tensor holds the same bytes on the
    device, and the device count is the host count."""
    import torch
    S, T = 3, 30
    if mode == 3:
        drives = [[np.ascontiguousarray(f) for f in synth.corridor_sequence(T, seed=1234 + s)] for s in range(S)]
        runner = H.Runner.sfm(0, S, 2, _mono_params(1000))
    else:
        drives = _stereo_drives(S, T, failed=(1, 3))
        runner = H.Runner.stereo_sfm(0, S, 2, _stereo_params(1000))
    hosts = [_recon() for _ in range(S)]
    poses = [np.eye(4) for _ in range(S)]
    oks = []
    try:
        for k in range(T):
            if mode == 3:
                secs, nm, ok = runner.step([drives[s][k].ctypes.data for s in range(S)], DIMS)
            else:
                secs, nm, ok = runner.step([d[k][0].ctypes.data for d in drives], DIMS, ptrs2=[d[k][1].ctypes.data for d in drives])
            oks.append(ok.copy())
            for s in range(S):
                if k > 0 and ok[s]:
                    Tm = runner.motion(s)
                    poses[s] = poses[s] @ np.linalg.inv(Tm)
                    hosts[s].batch_prepare(runner.matches(s), Tm, *RECON)
                    hosts[s].batch_finish(*ctx.recon_points([hosts[s].batch_job()])[0])
                pts = runner.points(s)
                assert pts.tobytes() == hosts[s].points().tobytes(), (k, s)
                assert np.abs(runner.pose(s) - poses[s]).max() < 1e-9, (k, s)
                assert runner.device_points(s)[1] == len(pts), (k, s)
        for s in range(S):
            t = runner.points_tensor(s)
            assert t.dtype == torch.float32 and t.is_cuda and tuple(t.shape) == (len(runner.points(s)), 3)
            assert t.cpu().numpy().tobytes() == runner.points(s).tobytes()
        assert min(len(runner.points(s)) for s in range(S)) > 1000
        if mode == 4:
            assert not oks[3][1] and oks[4][1], np.array(oks)
    finally:
        runner.close()


@pytest.mark.gpu
def test_stereo_facade_device_points():
    """The stereo facade's host points are a mirror of its device store: points_tensor and device_points agree with them.
    The first frame has no motion (update returns False) and reconstructs nothing."""
    sfm = H.StereoSfm(_stereo_params(2), W, HT)
    assert sfm.device_points() == (0, 0)
    for k in range(6):
        left, right = (np.ascontiguousarray(x) for x in synth.corridor_stereo_frame(k))
        assert sfm.update(left, right) == (k > 0), k
        pts = sfm.points()
        assert sfm.device_points()[1] == len(pts)
        assert sfm.points_tensor().cpu().numpy().tobytes() == pts.tobytes()
    assert len(sfm.points()) > 20


@pytest.mark.gpu
def test_launches(ctx):
    """A call with points and tracks is 3 launches (move, evaluation, append), with points only 1, with neither 0."""
    job = next(j for j, _ in _sequence_jobs(8, 600, 3) if len(j['tracks']) > 10)
    full, empty = ctx.recon_store(), ctx.recon_store()
    try:
        full.append(np.ones((100, 3), np.float32))
        for stores, jobs, want in (([full], [job], 3), ([full], [_empty_job()], 1), ([empty], [_empty_job()], 0)):
            n0 = ctx.launch_count()
            ctx.recon_update(stores, [np.eye(4)], jobs)
            assert ctx.launch_count() == n0 + want, want
    finally:
        full.close(); empty.close()


def _raw_update(ctx, stores, trs, jobs, status=None, arrays_null=()):
    nj = len(jobs)
    arr, keep = V.Context._job_array(jobs)
    t = [None if x is None else np.ascontiguousarray(np.asarray(x, np.float64)[:3, :4]) for x in trs]
    tp = (C.c_void_p * nj)(*[None if x is None else x.ctypes.data for x in t])
    sp = (C.c_void_p * nj)(*[None if s is None else s.h.value for s in stores])
    st = None if status is None else (C.c_void_p * nj)(*[None if x is None else x.ctypes.data for x in status])
    return V.lib().visocu_recon_update(ctx.h, nj, None if 'stores' in arrays_null else sp, None if 'tr' in arrays_null else tp,
                                       None if 'jobs' in arrays_null else arr, None, st, None)


@pytest.mark.gpu
def test_refusals(ctx):
    """Every malformed call is refused with VISOCU_EINVAL and changes no store: null arrays, a null store or transform, a
    store of another context, a store named twice, a bad job or track, a missing status array, and appends and reads
    outside the store."""
    job = next(j for j, _ in _sequence_jobs(8, 600, 3) if len(j['tracks']) > 3)
    nt = len(job['tracks'])
    other = V.Context(0)
    a, b, foreign = ctx.recon_store(), ctx.recon_store(), other.recon_store()
    try:
        a.append(np.arange(30, dtype=np.float32).reshape(10, 3)); b.append(np.ones((5, 3), np.float32))
        foreign.append(np.ones((2, 3), np.float32))
        snap = lambda: [(s.count, s.read().tobytes()) for s in (a, b, foreign)]
        want = snap()
        I = np.eye(4) * 2
        bad_track = job['tracks'].copy(); bad_track[0]['n_obs'] = 1
        cases = [dict(stores=[a, b], trs=[I, I], jobs=[job, job], arrays_null=('stores',)),
                 dict(stores=[a, b], trs=[I, I], jobs=[job, job], arrays_null=('tr',)),
                 dict(stores=[a, b], trs=[I, I], jobs=[job, job], arrays_null=('jobs',)),
                 dict(stores=[a, None], trs=[I, I], jobs=[job, job]),
                 dict(stores=[a, b], trs=[I, None], jobs=[job, job]),
                 dict(stores=[a, foreign], trs=[I, I], jobs=[job, job]),
                 dict(stores=[a, a], trs=[I, I], jobs=[job, job]),
                 dict(stores=[a, b], trs=[I, I], jobs=[job, dict(job, frames=job['frames'][:0])]),
                 dict(stores=[a, b], trs=[I, I], jobs=[job, dict(job, tracks=bad_track)]),
                 dict(stores=[a, b], trs=[I, I], jobs=[job, job], status=[np.zeros(nt, np.int32), None])]
        for k, kw in enumerate(cases):
            assert _raw_update(ctx, **kw) == -1, k
            assert snap() == want, k
        L = V.lib()
        x = np.ones((4, 3), np.float32)
        assert L.visocu_recon_store_append(ctx.h, a.h, H._p(x), C.c_int64(-1)) == -1
        assert L.visocu_recon_store_append(ctx.h, a.h, None, C.c_int64(4)) == -1
        assert L.visocu_recon_store_append(ctx.h, foreign.h, H._p(x), C.c_int64(4)) == -1
        out = np.full((20, 3), 7.0, np.float32)
        for first, count in ((-1, 1), (0, -1), (0, 11), (10, 1), (11, 0)):
            assert L.visocu_recon_store_read(ctx.h, a.h, C.c_int64(first), C.c_int64(count), H._p(out)) == -1, (first, count)
        assert L.visocu_recon_store_read(ctx.h, a.h, C.c_int64(0), C.c_int64(1), None) == -1
        assert L.visocu_recon_store_read(ctx.h, foreign.h, C.c_int64(0), C.c_int64(1), H._p(out)) == -1
        assert L.visocu_recon_store_destroy(ctx.h, foreign.h) == -1
        assert np.all(out == 7.0) and snap() == want
        assert _raw_update(ctx, [a, b], [I, I], [job, job]) == 0 and a.count >= 10
    finally:
        a.close(); b.close(); foreign.close()
        other.close()
