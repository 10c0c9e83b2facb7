"""Stereo structure from motion: the StructureFromMotionStereo facade (stereo odometry and reconstruction estimated on the
device) against the host composition of VisualOdometryStereo::process and Reconstruction::update, and the stereo
structure-from-motion mode of the sequence runner (mode 4) against stand-alone facades.  The host classes restate the
reference (tests/test_host_cpu.py pins them); here they are the reference for the device path."""
import ctypes as C

import numpy as np
import pytest

import synth
import visocu_py as V
import host_py as H

W, HT = 1241, 376
DIMS = np.array([W, HT, W], np.int32)
RECON = (0, 2, 30.0, 3.0)       # the facades' constants: point type, min track length, max distance, min angle


def _params(bucket):
    return H.StereoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, base=0.54,
                          bucket_max_features=bucket)


def _drives(S, T, failed=None):
    """S stereo corridor drives of T (left, right) frames.  failed = (s, k): the right image of frame k of drive s is shifted
    down by 40 rows, so that its features sit where the stereo geometry puts none: quad matching keeps a few chance matches
    that no motion explains, and the odometry fails.  (A uniform image would not do: without features the matcher keeps
    the previous frame's matches, as the reference's does, and the odometry succeeds on them.)"""
    drives = [[tuple(np.ascontiguousarray(x) for x in synth.corridor_stereo_frame(k, seed=1234 + s)) for k in range(T)]
              for s in range(S)]
    if failed is not None:
        s, k = failed
        drives[s][k] = (drives[s][k][0], np.ascontiguousarray(np.roll(drives[s][k][1], 40, axis=0)))
    return drives


def _close(a, b):
    return len(a) == len(b) and (len(a) == 0 or np.abs(a - b).max() <= 1e-5 * max(1.0, np.abs(a).max()))


@pytest.mark.gpu
@pytest.mark.parametrize('bucket', [2, 1000])
def test_facade_against_host_composition(bucket):
    """The facade against H.Stereo.process followed by H.Recon.update with the same replace flags, the pose accumulated in
    numpy: per frame the same ok, byte-identical matches, the same inliers, motion and pose within 1e-9, the same number
    of points and coordinates within 1e-5 x max(1, |p|)."""
    p = _params(bucket)
    for s, drive in enumerate(_drives(3, 8)):
        sfm = H.StereoSfm(p, W, HT)
        vo = sfm.odometry()
        host, recon = H.Stereo(p), H.Recon(synth.KITTI_F, synth.KITTI_CU, synth.KITTI_CV)
        pose, replace = np.eye(4), False
        for k, (left, right) in enumerate(drive):
            ok = sfm.update(left, right)
            ok_h = host.process(left, right, replace)
            assert ok == ok_h, (s, k)
            if k > 0 and ok_h:
                pose = pose @ np.linalg.inv(host.motion())
                recon.update(host.matches(), host.motion(), *RECON)
            replace = k > 0 and not ok_h
            assert vo.matches().tobytes() == host.matches().tobytes(), (s, k)
            assert np.array_equal(vo.inliers(), host.inliers()), (s, k)
            assert np.abs(vo.motion() - host.motion()).max() < 1e-9, (s, k)
            assert np.abs(sfm.pose() - pose).max() < 1e-9, (s, k)
            assert _close(recon.points(), sfm.points()), (s, k, len(recon.points()), len(sfm.points()))
            assert ok or k == 0, (s, k)
        assert len(sfm.points()) > 20, s


@pytest.mark.gpu
def test_failed_frame_is_replaced():
    """Frame 3 has a right image that does not fit the left one: the matcher produces a new match list for it (not the
    previous frame's) and the frame fails.  The next update pushes with replace, so step 4 matches frame 2 against frame 4:
    its matches are those of a stand-alone VisualOdometryStereo that pushes frame 4 with replace, and differ from those of
    one that does not."""
    p = _params(2)
    drive = _drives(2, 6, failed=(1, 3))[1]
    sfm = H.StereoSfm(p, W, HT)
    vo = sfm.odometry()
    oks, matches = [], []
    for left, right in drive:
        oks.append(sfm.update(left, right))
        matches.append(vo.matches())
    assert not oks[3] and matches[3].tobytes() != matches[2].tobytes(), len(matches[3])
    assert oks[1] and oks[2] and oks[4] and oks[5], oks
    replaced, kept = H.Stereo(p), H.Stereo(p)
    for k in range(5):
        replaced.process(*drive[k], replace=(k == 4))
        kept.process(*drive[k])
    assert matches[4].tobytes() == replaced.matches().tobytes() and len(matches[4]) > 20
    assert matches[4].tobytes() != kept.matches().tobytes()


def _left_right(drives, k):
    return [d[k][0].ctypes.data for d in drives], [d[k][1].ctypes.data for d in drives]


@pytest.mark.gpu
def test_stereo_sfm_runner_against_facades():
    """Runner mode 4 (5 sequences, 2 workers, 7 steps, frame 3 of sequence 1 failing) against stand-alone facades: both
    make the same device calls and both kernels batch byte-identically, so per step the same ok and byte-identical
    matches, inliers, motion, pose and points.  run() gives the bytes of stepping."""
    S, T = 5, 7
    drives = _drives(S, T, failed=(1, 3))
    p = _params(2)
    facades = [H.StereoSfm(p, W, HT) for _ in range(S)]
    runner = H.Runner.stereo_sfm(0, S, 2, p)
    oks = []
    try:
        for k in range(T):
            left, right = _left_right(drives, k)
            secs, nm, ok = runner.step(left, DIMS, ptrs2=right)
            oks.append(ok)
            for s in range(S):
                assert bool(ok[s]) == facades[s].update(*drives[s][k]), (k, s)
                vo = facades[s].odometry()
                assert runner.matches(s).tobytes() == vo.matches().tobytes(), (k, s)
                assert nm[s] == len(vo.matches()), (k, s)
                assert runner.inliers(s).tobytes() == vo.inliers().tobytes(), (k, s)
                assert runner.motion(s).tobytes() == vo.motion().tobytes(), (k, s)
                assert runner.pose(s).tobytes() == facades[s].pose().tobytes(), (k, s)
                assert runner.points(s).tobytes() == facades[s].points().tobytes(), (k, s)
        assert not oks[3][1] and oks[4][1] and all(oks[k][s] for k in range(1, T) for s in (0, 2, 3, 4)), np.array(oks)
        assert min(len(runner.points(s)) for s in range(S)) > 20
        want = ([runner.points(s).tobytes() for s in range(S)], [runner.pose(s).tobytes() for s in range(S)])
    finally:
        runner.close()
    again = H.Runner.stereo_sfm(0, S, 2, p)
    try:
        steps = [_left_right(drives, k) for k in range(T)]
        secs, nm, ok = again.run([a for a, b in steps], DIMS, ptr_steps2=[b for a, b in steps])
        assert np.array_equal(ok, np.array(oks))
        assert [again.points(s).tobytes() for s in range(S)] == want[0]
        assert [again.pose(s).tobytes() for s in range(S)] == want[1]
    finally:
        again.close()


@pytest.mark.gpu
def test_refusals():
    """A mode-4 step or run without right images returns -1, writes nothing and pushes nothing: the runner stays in step
    with facades that never saw those calls.  points() and pose() of a mode-2 runner still report that it has neither."""
    S, T = 2, 3
    drives = _drives(S, T)
    p = _params(2)
    facades = [H.StereoSfm(p, W, HT) for _ in range(S)]
    runner = H.Runner.stereo_sfm(0, S, 2, p)
    L = H.lib()
    try:
        for k in range(T):
            left, right = _left_right(drives, k)
            nm, ok = np.full(S, 7, np.int32), np.full(S, 7, np.int32)
            assert L.visob_runner_step(runner.h, (C.c_void_p * S)(*left), None, H._p(DIMS), 0, 0, H._p(nm), H._p(ok)) == -1.0
            assert L.visob_runner_run(runner.h, 1, (C.c_void_p * S)(*left), None, H._p(DIMS), 0, 0, H._p(nm), H._p(ok)) == -1.0
            assert np.all(nm == 7) and np.all(ok == 7)
            secs, nm, ok = runner.step(left, DIMS, ptrs2=right)
            assert secs >= 0
            for s in range(S):
                assert bool(ok[s]) == facades[s].update(*drives[s][k]), (k, s)
                assert runner.matches(s).tobytes() == facades[s].odometry().matches().tobytes(), (k, s)
                assert runner.pose(s).tobytes() == facades[s].pose().tobytes(), (k, s)
                assert runner.points(s).tobytes() == facades[s].points().tobytes(), (k, s)
        assert all(ok)
    finally:
        runner.close()
    stereo = H.Runner.stereo(0, S, 2, p)
    try:
        left, right = _left_right(drives, 0)
        stereo.step(left, DIMS, ptrs2=right)
        out = np.full((4, 4), 7.0)
        assert L.visob_runner_get_points(stereo.h, 0, None, 0) == -1
        L.visob_runner_get_pose(stereo.h, 0, H._p(out))
        assert np.all(out == 7.0)
    finally:
        stereo.close()
