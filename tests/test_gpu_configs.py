"""GPU parity on the configurations BASELINE.json names beyond the flow default: config 3b (mono odometry with the CLI's
bucket.max_features = 1000, reference main.cpp:71, N ~ 4 k matches into RANSAC), RANSAC alone at that size, the pose
kernels against the reference's own triangulateChieral / findBestPlane, and config 4 (3840x2160 at the stated density of
120 k blobs) in both half_resolution modes."""
import numpy as np
import pytest

import synth
import pyref
import pyoracle as O
import visocu_py as V
import host_py as H

pytestmark = pytest.mark.gpu


def _mono_params(bucket_max):
    return H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08,
                        bucket_max_features=bucket_max)


def _normalized_F(F):
    F = F / np.linalg.norm(F)
    k = np.argmax(np.abs(F))
    return F * np.sign(F.flat[k])


@pytest.fixture(scope='module')
def corridor():
    return synth.corridor_sequence(21, seed=1234)


def test_mono_odometry_bucket1000_sequence(reference, corridor):
    """Config 3b: VisualOdometryMono::process over 21 corridor frames with bucket.max_features = 1000 (main.cpp:71): every
    match survives the bucketing (shuffled per bucket), about 4 k matches enter RANSAC and the refit of the winning
    hypothesis runs on thousands of inliers (viso_mono.cpp:61-69).  Same rand() / sample streams as the reference (each
    object starts from srand(0) and a fresh std::default_random_engine), so: bucketed list bit-exact, inlier set exact,
    rotation entries 1e-6 absolute, translation 1e-6 relative."""
    hv = H.Mono(_mono_params(1000))
    sizes = []
    for k in range(len(corridor)):
        ok_h = hv.process(corridor[k])
        assert ok_h == bool(reference.value('ok%d' % k)), k
        if k == 0:
            continue
        assert ok_h, k
        b = hv.matches()
        sizes.append(len(b))
        reference.same('matches%d' % k, b)
        reference.same('inliers%d' % k, hv.inliers())
        Th = hv.motion()
        Tr = reference.value('motion%d' % k)
        assert np.abs(Tr[:3, :3] - Th[:3, :3]).max() < 1e-6, k
        assert np.abs(Tr[:3, 3] - Th[:3, 3]).max() < 1e-6 * max(1.0, np.abs(Tr[:3, 3]).max()), k
    assert min(sizes) > 2500                                    # the RANSAC problem really is thousands of matches


def test_ransac_4k_against_reference(ctx, reference, corridor):
    """visocu_ransac_F at N ~ 4 k (the refit's Householder QR over thousands of rows, the scoring grid over thousands of
    matches) against the reference's RANSAC (built with -ffp-contract=off) on the same sample table.  The matches are those
    of the first two frames above, normalised by the plain-C restatement (the reference's bytes, see test_oracle_vs_ref.py).
    Tolerances as in test_ransac_against_reference: winner, inlier count and inlier set exact; F (unit Frobenius norm,
    fixed sign) to 1e-8; at most 1 % of the per-hypothesis counts may differ (rank-deficient 8-point systems, matches
    within rounding of the threshold)."""
    hv = H.Mono(_mono_params(1000))
    hv.process(corridor[0]); hv.process(corridor[1])
    pm = hv.matches()
    assert len(pm) > 2500
    ok, pmn, Tp, Tc = O.normalize(pm)
    assert ok
    reference.same('normalized', pmn)
    rng = np.random.default_rng(6)
    iters = 400
    samples = np.stack([rng.choice(len(pmn), 8, replace=False) for _ in range(iters)]).astype(np.int32)
    uv = np.stack([pmn['u1p'], pmn['v1p'], pmn['u1c'], pmn['v1c']], axis=1)
    got = ctx.ransac([uv], [samples], 1e-5, want_all=True)[0]
    want_counts = reference.value('counts')
    diff = got['counts'] != want_counts
    assert diff.mean() <= 0.01, 'hypothesis counts differ for %d of %d (max |delta| %d)' % (
        diff.sum(), iters, np.abs(got['counts'] - want_counts).max())
    assert got['best_iter'] == int(reference.value('best_iter'))
    assert got['n_inliers'] > 1000 and got['n_inliers'] == int(reference.value('n_inliers'))
    reference.same('inliers', got['inliers'])
    assert np.abs(_normalized_F(got['F']) - _normalized_F(reference.value('F'))).max() < 1e-8


def test_pose_kernels_against_reference(ctx, reference):
    """k_triangulate / k_plane_sums against the reference's own triangulateChieral (viso_mono.cpp:394-431) and
    findBestPlane (viso_mono.cpp:74-98) on the same inputs.  The triangulated point is the null vector of a 4x4 system
    (sign and scale arbitrary): compared as unit vectors with fixed sign, 1e-7 absolute, on a fixed sample of the points
    (stored for that sample, see oracle/refgold.py); the chirality count and the winning plane candidate exactly."""
    rng = np.random.default_rng(17)
    n = 700
    K = np.array([[645.2, 0, 635.9], [0, 645.2, 194.1], [0, 0, 1.0]])
    Xw = np.stack([rng.uniform(-5, 5, n), rng.uniform(-2, 2, n), rng.uniform(4, 40, n), np.ones(n)])
    a = 0.02
    R = np.array([[np.cos(a), 0.0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    t = np.array([0.1, 0.02, -0.8])
    P1 = K @ np.hstack([np.eye(3), np.zeros((3, 1))])
    x1 = P1 @ Xw
    x2 = (K @ np.hstack([R, t[:, None]])) @ Xw
    pm = np.zeros(n, pyref.P_MATCH)
    pm['u1p'] = x1[0] / x1[2] + rng.normal(0, 0.2, n); pm['v1p'] = x1[1] / x1[2] + rng.normal(0, 0.2, n)
    pm['u1c'] = x2[0] / x2[2] + rng.normal(0, 0.2, n); pm['v1c'] = x2[1] / x2[2] + rng.normal(0, 0.2, n)
    uv = np.stack([pm['u1p'], pm['v1p'], pm['u1c'], pm['v1c']], 1)
    cands = [(R, t), (R, -t), (R.T, t), (R.T, -t)]
    P2 = np.stack([K @ np.hstack([Rc, tc[:, None]]) for Rc, tc in cands])
    Xg, nf = ctx.triangulate(uv, P1, P2)
    cols = np.sort(np.random.default_rng(0).choice(n, 100, replace=False))
    for s in range(len(cands)):
        assert nf[s] == int(reference.value('num%d' % s)), s
        A = Xg[s][:, cols] / np.linalg.norm(Xg[s][:, cols], axis=0)
        B = reference.value('X%d' % s)
        sgn = np.sign(np.sum(A * B, axis=0))
        assert np.abs(A * sgn - B).max() < 1e-7, s
    assert nf[0] > 0.95 * n
    # ground-plane vote: pitch 0 makes d = first row of x_plane exactly (n = (cos 0, sin 0))
    d = np.concatenate([rng.normal(1.6, 0.02, 300), rng.uniform(0.2, 5, 120)])
    rng.shuffle(d)
    thr, wgt = 0.5, 1.0 / (2 * 0.05 ** 2)
    got = ctx.best_plane(d, thr, wgt)
    assert d[got] == float(reference.value('best_d'))
    assert ctx.best_plane(np.full(10, 0.1), thr, wgt) == 0


@pytest.fixture(scope='module')
def pair4k_dense():
    return synth.blob_pair(3840, 2160, seed=405, n_blobs=120000)


@pytest.mark.parametrize('half', [1, 0], ids=['halfres', 'fullres'])
def test_flow_4k_stated_density(reference, pair4k_dense, half):
    """Config 4 at the density SURVEY 8(d) states (120 k blobs; half_resolution = 0: > 150 k maxima per frame and the
    SAD search over all of them): feature counts, both match lists and the final list bit-exact."""
    a, b = pair4k_dense
    hm = H.Matcher(V.Params(half_resolution=half))
    hm.push(a); hm.push(b); hm.match_features(0)
    reference.same('counts', np.array(list(hm.counts().values()), np.int64))
    assert hm.counts()['1c2'] > (120000 if half == 0 else 60000)
    got = hm.matches(2)
    assert len(got) > 40000
    reference.same('matches1', hm.matches(1))
    reference.same('matches2', got)
