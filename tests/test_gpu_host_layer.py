"""GPU parity of the drop-in C++ classes (libviso_b200.so) against the outputs of the reference classes (stored under
tests/golden/reference, see oracle/refgold.py): final getMatches() after outlier removal and bucketing (P7), and
VisualOdometryMono::process end to end (P8, toleranced)."""
import numpy as np
import pytest

import synth
import visocu_py as V
import host_py as H

pytestmark = pytest.mark.gpu


def pad_safe_width(w, nms_n, half):
    """True if no maximum can sit at u = w-7, where the reference's descriptor depends on uninitialised pad bytes
    (SURVEY.md 8c caveat 3): (w - 2n - 13) mod (n+1) != 0 for the sparse and the dense neighbourhood size."""
    wm = w // 2 if half else w
    ns = nms_n * 3
    if ns > 10:
        ns = max(nms_n, 10)
    return all((wm - 2 * n - 13) % (n + 1) != 0 for n in (ns, nms_n))


@pytest.mark.parametrize('kw', [dict(), dict(half_resolution=0), dict(multi_stage=0), dict(nms_n=4, half_resolution=0),
                                dict(refinement=0)],
                         ids=['defaults', 'fullres', 'singlestage', 'nms4', 'norefine'])
def test_matcher_flow_final_list(reference, kw):
    p = V.Params(**kw)
    width = 1241 if pad_safe_width(1241, p.nms_n, p.half_resolution) else 1242
    assert pad_safe_width(width, p.nms_n, p.half_resolution)
    a, b = synth.blob_pair(width, 376, seed=41)
    hm = H.Matcher(V.Params(**kw))
    hm.push(a); hm.push(b); hm.match_features(0)
    reference.same('counts', np.array(list(hm.counts().values()), np.int64))
    reference.same('matches1', hm.matches(1))
    got = hm.matches(2)
    assert len(got) > 1000
    reference.same('matches2', got)
    # prior statistics of the host layer against the reference's (P5), on the stages that are defined for flow
    if V.Params(**kw).multi_stage:
        reference.same('ranges', hm.prior(hm.matches(1), 0).reshape(-1, 4, 4)[:, :, :2])
    g = hm.gain(np.arange(50))
    assert abs(g - float(reference.value('gain'))) < 1e-6


def test_matcher_sequence_ring_buffer_and_replace(reference):
    """Three frames, the third pushed with replace=true, dims given with a caller stride larger than the width."""
    seq = synth.blob_sequence(3, 800, 300, seed=43)
    hm = H.Matcher(V.Params())
    hm.push(seq[0]); hm.push(seq[1]); hm.match_features(0)
    reference.same('first', hm.matches(2))
    hm.push(seq[2], replace=True); hm.match_features(0)
    assert len(hm.matches(2)) > 300
    reference.same('replaced', hm.matches(2))
    hm.push(seq[1]); hm.match_features(0)
    reference.same('third', hm.matches(2))


def test_matcher_quad_final_list_and_bucketing(reference):
    assert pad_safe_width(1242, 2, 0)
    lp, rpv, lc, rc = synth.blob_quad(1242, 376, seed=45)
    kw = dict(nms_n=2, half_resolution=0)
    hm = H.Matcher(V.Params(**kw))
    hm.push(lp, rpv); hm.push(lc, rc); hm.match_features(2)
    got = hm.matches(2)
    assert len(got) > 1000
    reference.same('matches2', got)
    # bucketing draws from the process-wide rand() stream: compare the kept SET per bucket size, not the order
    hm.bucket(1000, 50.0, 50.0)
    b = hm.matches(2)
    reference.same('bucketed_set', np.sort(b, order=list(b.dtype.names)))


def test_matcher_error_behaviour(capfd):
    hm = H.Matcher(V.Params())
    hm.match_features(0)                      # nothing pushed: silently no matches (matcher.cpp:190-212)
    assert len(hm.matches(2)) == 0
    img = synth.blob_pair(200, 100, seed=1)[0]
    hm.push(img)
    hm.match_features(0)                      # only one frame: still silent
    assert len(hm.matches(2)) == 0
    H.lib().visob_matcher_push(hm.h, None, None, np.array([200, 100, 100], np.int32).ctypes.data_as(__import__('ctypes').c_void_p), 0)
    assert 'ERROR: Image dimension mismatch!' in capfd.readouterr().err


def test_filter_namespace(reference):
    img = synth.blob_pair(256, 128, seed=9)[0]
    du, dv = H.filter_call(0, img)
    reference.same('sobel5x5_du', du[2:-2, 2:-2]); reference.same('sobel5x5_dv', dv[2:-2, 2:-2])
    reference.same('blob5x5', H.filter_call(2, img)[3:-2, 3:-2])


def _mono_params(bucket_max):
    return H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08,
                        bucket_max_features=bucket_max)


def test_mono_odometry_sequence(reference):
    """VisualOdometryMono::process over a short corridor drive.  Both the reference and this object draw the RANSAC
    samples from a fresh std::default_random_engine(71) and bucket with rand() after srand(0), so the sample tables
    coincide as long as the match lists do.  Tolerances (SURVEY.md 8d P8): rotation entries 1e-6 absolute, translation
    1e-6 relative."""
    seq = synth.corridor_sequence(4, seed=1234)
    hv = H.Mono(_mono_params(2))
    for k in range(len(seq)):
        ok_h = hv.process(seq[k])
        assert ok_h == bool(reference.value('ok%d' % k))
        if k == 0:
            continue
        assert ok_h
        b = hv.matches()
        assert len(b) > 100
        reference.same('matches%d' % k, b)                        # same bucketed list, same order
        reference.same('inliers%d' % k, hv.inliers())
        Th = hv.motion()
        Tr = reference.value('motion%d' % k)
        assert np.abs(Tr[:3, :3] - Th[:3, :3]).max() < 1e-6
        assert np.abs(Tr[:3, 3] - Th[:3, 3]).max() < 1e-6 * max(1.0, np.abs(Tr[:3, 3]).max())
        assert abs(Th[2, 3]) > 0.3                               # the drive moves 0.8 m forward per frame


def test_matcher_stereo_method1(reference):
    """Matcher method 1 (stereo, matcher.cpp:1045-1084): one stereo pair, left-right-left circle, positive disparity."""
    lp, rpv, lc, rc = synth.blob_quad(1244, 376, seed=47)
    for mode, kw in (('fullres', dict(half_resolution=0)), ('defaults', dict())):
        assert pad_safe_width(1244, 3, kw.get('half_resolution', 1))
        hm = H.Matcher(V.Params(**kw))
        hm.push(lc, rc); hm.match_features(1)
        got = hm.matches(2)
        assert len(got) > 1000
        assert np.all(got['u1c'] >= got['u2c']) and np.all(got['i1p'] == -1)
        reference.same(mode + '_matches1', hm.matches(1))
        reference.same(mode + '_matches2', got)


def _sample(n, k=512):
    return np.sort(np.random.default_rng(0).choice(n, min(n, k), replace=False))


def test_matcher_subpixel_refinement(reference):
    """refinement = 2 (parabolicFitting, matcher.cpp:1379-1454) with the flow demo's parameters
    (matlab/demo_matching_flow.m:12-21).  Integer stages identical; the sub-pixel coordinates come from a
    double-precision least-squares solve done differently here (constant pseudo-inverse instead of a Gauss-Jordan solve
    per match): tolerance 1e-4 pixel, on a fixed sample of 512 matches per list (coordinates stored
    for that sample)."""
    kw = dict(nms_n=4, refinement=2, half_resolution=0)
    assert pad_safe_width(1242, 4, 0)
    a, b = synth.blob_pair(1242, 376, seed=49)
    hm = H.Matcher(V.Params(**kw))
    hm.push(a); hm.push(b); hm.match_features(0)
    got = hm.matches(2)
    assert len(got) > 1000
    reference.same('flow_integer', np.stack([got[f] for f in ('i1p', 'i1c', 'u1c', 'v1c')], 1))
    rows = _sample(len(got))
    want_u, want_v = reference.value('flow_u1p'), reference.value('flow_v1p')
    assert np.abs(got['u1p'][rows] - want_u).max() < 1e-4 and np.abs(got['v1p'][rows] - want_v).max() < 1e-4
    frac = np.abs(want_u - np.round(want_u))
    assert (frac > 1e-3).mean() > 0.5                                   # it really is sub-pixel
    # quad matching with sub-pixel refinement: three relocations per match
    lp, rpv, lc, rc = synth.blob_quad(1242, 376, seed=51)
    kw = dict(nms_n=2, refinement=2, half_resolution=0)
    hm = H.Matcher(V.Params(**kw))
    hm.push(lp, rpv); hm.push(lc, rc); hm.match_features(2)
    got = hm.matches(2)
    assert len(got) > 500
    reference.same('quad_integer', np.stack([got[f] for f in ('i1p', 'i2p', 'i1c', 'i2c', 'u1c', 'v1c')], 1))
    rows = _sample(len(got))
    for f in ('u1p', 'v1p', 'u2p', 'v2p', 'u2c', 'v2c'):
        assert np.abs(got[f][rows] - reference.value('quad_' + f)).max() < 1e-4


def test_sequence_runner_equals_single_matchers(reference):
    """Sharded runner (MatcherBatch per worker: one batched launch per GPU stage for all of a worker's sequences) gives,
    for every sequence and frame, exactly the list the reference gives."""
    S, T = 5, 3
    seqs = [synth.blob_sequence(T, 500, 260, seed=60 + s) for s in range(S)]
    mp = H.MonoParams(match=V.Params())
    for threads in (1, 2):
        runner = H.Runner(0, S, threads, 0, 0, mp)
        dims = np.array([500, 260, 500], np.int32)
        for k in range(T):
            imgs = [np.ascontiguousarray(seqs[s][k]) for s in range(S)]
            secs, nm, ok = runner.step([i.ctypes.data for i in imgs], dims)
            if k == 0:
                assert nm.tolist() == [0] * S
        got = [runner.matches(s) for s in range(S)]
        runner.close()
        for s in range(S):
            assert len(got[s]) > 300, (threads, s)
            reference.same('seq%d' % s, got[s])


def test_mono_runner_equals_single_objects():
    """Mono odometry through the sharded runner (shared MatcherBatch + per-sequence odometry objects) equals stand-alone
    VisualOdometryMono objects: same matches, same inliers, same pose."""
    S, T = 3, 3
    seqs = [synth.corridor_sequence(T, seed=1234 + s) for s in range(S)]
    hp = _mono_params(2)
    runner = H.Runner(0, S, 2, 1, 0, hp)
    dims = np.array([1241, 376, 1241], np.int32)
    poses = []
    for k in range(T):
        imgs = [np.ascontiguousarray(seqs[s][k]) for s in range(S)]
        secs, nm, ok = runner.step([i.ctypes.data for i in imgs], dims)
        assert k == 0 or ok.tolist() == [1] * S
    got_m = [runner.matches(s) for s in range(S)]
    got_T = [runner.motion(s) for s in range(S)]
    runner.close()
    for s in range(S):
        hv = H.Mono(hp)
        for k in range(T):
            hv.process(seqs[s][k])
        assert hv.matches().tobytes() == got_m[s].tobytes()
        assert np.abs(hv.motion() - got_T[s]).max() < 1e-9


def test_quad_matching_with_motion_prediction(reference):
    """Tr_delta-guided quad matching (matcher.cpp:1112-1138): double-precision cost SAD + 4 * distance to the predicted
    position.  The GPU uses explicit IEEE operations without FMA contraction, so the list is compared bit-exactly against
    the reference built with -ffp-contract=off."""
    assert pad_safe_width(1242, 2, 0)
    lp, rpv, lc, rc = synth.blob_quad(1242, 376, seed=53, shift=(3, 1), disparity=12)
    kw = dict(nms_n=2, half_resolution=0)
    Tr = np.eye(4); Tr[0, 3] = 0.02; Tr[2, 3] = -0.3; Tr[0, 2] = 0.01; Tr[2, 0] = -0.01
    hm = H.Matcher(V.Params(**kw))
    hm.set_intrinsics(645.2, 635.9, 194.1, 0.54)
    hm.push(lp, rpv); hm.push(lc, rc); hm.match_features(2, tr_delta=Tr)
    got = hm.matches(2)
    assert len(got) > 500
    reference.same('matches2', got)


def test_stereo_odometry_sequence(reference):
    """VisualOdometryStereo::process over a short stereo corridor drive: quad matching with motion prediction from the
    second pair on, 3-point RANSAC + Gauss-Newton on the host.  Same sample stream as the reference (built with
    -ffp-contract=off; a fresh engine(71) on both sides), same matches -> same inliers; pose within 1e-6 (rotation
    entries absolute, translation relative)."""
    frames = [synth.corridor_stereo_frame(k, seed=1234) for k in range(4)]
    kw = dict(f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, base=0.54)
    hv = H.Stereo(H.StereoParams(match=V.Params(), **kw))
    for k, (l, r) in enumerate(frames):
        ok_h = hv.process(l, r)
        assert ok_h == bool(reference.value('ok%d' % k))
        if k == 0:
            continue
        assert ok_h and len(hv.matches()) > 100
        reference.same('matches%d' % k, hv.matches())
        reference.same('inliers%d' % k, hv.inliers())
        Th = hv.motion()
        Tr = reference.value('motion%d' % k)
        assert np.abs(Tr[:3, :3] - Th[:3, :3]).max() < 1e-6
        assert np.abs(Tr[:3, 3] - Th[:3, 3]).max() < 1e-6 * max(1.0, np.abs(Tr[:3, 3]).max())
        assert abs(abs(Th[2, 3]) - 0.8) < 0.05                      # 0.8 m forward per frame, metric thanks to the baseline


def test_structure_from_motion_facade(reference):
    """StructureFromMotion::update (sfm.hh:46-77): odometry, pose accumulation, replace-on-failure and track-based
    reconstruction.  The reference facade itself needs the OpenCL headers, so the reference side was its few lines
    restated on top of the reference's own VisualOdometryMono and Reconstruction objects (a fresh sample generator)."""
    seq = synth.corridor_sequence(7, seed=1234)
    sfm = H.Sfm(_mono_params(2), 1241, 376)
    for k in range(len(seq)):
        sfm.update(seq[k])
    got_pts = sfm.points()
    want_pts = reference.value('points')
    assert len(want_pts) > 20
    assert len(got_pts) == len(want_pts)
    assert np.abs(got_pts - want_pts).max() <= 1e-3 * max(1.0, np.abs(want_pts).max())
    assert np.abs(sfm.pose() - reference.value('pose')).max() < 1e-5


def test_pipelined_runner_equals_stepwise(reference):
    """runner.run keeps several steps of every sequence in flight (MatcherBatch::stepSubmit / stepCollect: consecutive steps
    on different lanes of the context, a ring of four frames per sequence, steps replayed as CUDA graphs once they repeat):
    per step and sequence the same match counts as stepping synchronously, the same final lists as the reference, and for
    the odometry mode the same poses.  Twelve steps, so that every lane runs plain, captured and replayed."""
    S, T = 5, 12
    dims = np.array([500, 260, 500], np.int32)
    seqs = [synth.blob_sequence(T, 500, 260, seed=80 + s) for s in range(S)]
    imgs = [[np.ascontiguousarray(seqs[s][k]) for s in range(S)] for k in range(T)]
    ptrs = [[i.ctypes.data for i in row] for row in imgs]
    mp = H.MonoParams(match=V.Params())
    a = H.Runner(0, S, 2, 0, 0, mp)
    counts_step = np.array([a.step(ptrs[k], dims)[1] for k in range(T)])
    want = [a.matches(s) for s in range(S)]
    a.close()
    for s in range(S):
        reference.same('seq%d' % s, want[s])
    for depth in (1, 2, 3):
        H.set_pipeline_depth(depth)
        b = H.Runner(0, S, 2, 0, 0, mp)
        secs, nm, ok = b.run(ptrs, dims)
        got = [b.matches(s) for s in range(S)]
        b.close()
        assert np.array_equal(nm, counts_step) and nm[1:].min() > 300, depth
        for s in range(S):
            assert got[s].tobytes() == want[s].tobytes(), (depth, s)
    H.set_pipeline_depth(3)
    # the same frames in pinned host memory: the runner copies them asynchronously (visocu_push_frames, on_device = 2)
    import torch
    pinned = torch.empty((T, S, 260, 500), dtype=torch.uint8).pin_memory()
    pinned.numpy()[:] = np.stack([np.stack(row) for row in imgs])
    pptrs = [[pinned[k, s].data_ptr() for s in range(S)] for k in range(T)]
    b = H.Runner(0, S, 2, 0, 0, mp)
    secs, nm, ok = b.run(pptrs, dims)
    got = [b.matches(s) for s in range(S)]
    b.close()
    assert np.array_equal(nm, counts_step)
    for s in range(S):
        assert got[s].tobytes() == want[s].tobytes(), ('pinned', s)
    # the drop-in pushBack consumes a pinned image before it returns: the caller may overwrite its buffer at once
    hm = H.Matcher(V.Params())
    buf = torch.empty((260, 500), dtype=torch.uint8).pin_memory()
    for k in (T - 2, T - 1):
        buf.numpy()[:] = seqs[0][k]
        hm.push(buf.numpy())                                 # a view of the pinned buffer: same address
        buf.numpy()[:] = 0
    hm.match_features(0)
    assert hm.matches(2).tobytes() == want[0].tobytes()
    # odometry mode
    S, T = 3, 7
    seqs = [synth.corridor_sequence(T, seed=1234 + s) for s in range(S)]
    imgs = [[np.ascontiguousarray(seqs[s][k]) for s in range(S)] for k in range(T)]
    ptrs = [[i.ctypes.data for i in row] for row in imgs]
    dims = np.array([1241, 376, 1241], np.int32)
    hp = _mono_params(2)
    a = H.Runner(0, S, 2, 1, 0, hp)
    oks = np.array([a.step(ptrs[k], dims)[2] for k in range(T)])
    want_T = [a.motion(s) for s in range(S)]; want_m = [a.matches(s) for s in range(S)]
    a.close()
    b = H.Runner(0, S, 2, 1, 0, hp)
    secs, nm, ok = b.run(ptrs, dims)
    assert np.array_equal(ok, oks) and ok[1:].min() == 1
    for s in range(S):
        assert b.matches(s).tobytes() == want_m[s].tobytes()
        assert np.abs(b.motion(s) - want_T[s]).max() < 1e-9
    b.close()


def test_device_prior_ranges_equal_reference(reference):
    """Multi-stage flow matching computes Matcher::computePriorStatistics (matcher.cpp:734-868) on the device between the
    two passes (k_prior_ranges): the ranges must be bit-identical to the reference's statistics of the same first-pass
    list, in half- and full-resolution mode."""
    a, b = synth.blob_pair(1244, 376, seed=91, shift=(4, -2))
    for mode, kw in (('defaults', dict()), ('fullres', dict(half_resolution=0))):
        assert pad_safe_width(1244, 3, kw.get('half_resolution', 1))
        hm = H.Matcher(V.Params(**kw))
        hm.push(a); hm.push(b); hm.match_features(0)
        first = hm.matches(1)
        assert len(first) > 200
        reference.same(mode + '_matches1', first)
        # flow matching uses stages 0 and 1 of the four a range holds (matcher.cpp:1020-1026); the others are never read
        reference.same(mode + '_ranges', hm.ranges().reshape(-1, 4, 4)[:, :, :2])
