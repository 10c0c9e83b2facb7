"""CPU tests: pin the plain-C restatement (oracle/viso_oracle.c) against the outputs of the unmodified reference on the
same seeded inputs (SURVEY.md 8c: the reference holds no golden vectors for this path; its outputs are stored under
tests/golden/reference, see oracle/refgold.py).  Integer stages bit-exact, FP64 stages to the stated tolerance.  Needs no GPU.
Stereo matching, motion-predicted quad matching and sub-pixel refinement are pinned against the results stored for
tests/test_gpu_host_layer.py (same inputs, the whole Matcher chain)."""
import numpy as np
import pytest

import synth
import pyref
import refgold
import pyoracle as O
import visocu_py as V
import host_py as H


def valid(p, w, m=2):
    return p[m:-m, m:w - m]


@pytest.fixture(scope='module')
def img():
    return synth.blob_pair(400, 240, seed=17)


def test_simd_known_answers(reference):
    """The reference's own unit test (test/simd.cpp:100-131) pins the 16- and 32-byte SAD: same check here."""
    rng = np.random.default_rng(0)
    s32, s16 = [], []
    for _ in range(50):
        a = rng.integers(0, 256, 32, dtype=np.uint8); b = rng.integers(0, 256, 32, dtype=np.uint8)
        s32.append(O.sad(a, b)); s16.append(O.sad(a[:16], b[:16]))
        assert s32[-1] == int(np.abs(a.astype(int) - b.astype(int)).sum())
    reference.same('sad32', np.array(s32, np.int64)); reference.same('sad16', np.array(s16, np.int64))
    assert O.sad(np.zeros(32, np.uint8), np.full(32, 255, np.uint8)) == 8160


def test_filters(reference, img):
    I = O.pad(img[0])
    w = img[0].shape[1]
    du, dv = O.sobel5x5(I)
    reference.same('sobel5x5_du', valid(du, w)); reference.same('sobel5x5_dv', valid(dv, w))
    du, dv = O.sobel3x3(I)
    reference.same('sobel3x3_du', valid(du, w, 1)); reference.same('sobel3x3_dv', valid(dv, w, 1))
    reference.same('blob5x5', O.blob5x5(I)[3:-2, 3:w - 2])
    reference.same('checkerboard5x5', valid(O.checkerboard5x5(I), w)[:-1])


def test_half_image_and_nms(reference, img):
    I = O.pad(img[0])
    w = img[0].shape[1]
    h1, d1 = O.half_image(I, w)
    reference.same('half_dims', np.array(d1, np.int64)); reference.same('half_image', h1[:, :d1[0]])
    f1 = O.blob5x5(I); f2 = O.checkerboard5x5(I)
    for n in (2, 3, 9, 10):
        reference.same('nms%d' % n, O.nms(f1, f2, w, n, 50))
    assert [O.lib().vo_sparse_nms_n(k) for k in (1, 2, 3, 4, 8, 12)] == [3, 6, 9, 10, 10, 12]


@pytest.mark.parametrize('kw', [dict(), dict(half_resolution=0), dict(half_resolution=0, nms_n=2), dict(multi_stage=0)],
                         ids=['defaults', 'fullres', 'nms2', 'singlestage'])
def test_features_matching_refinement(reference, img, kw):
    """computeFeatures records, flow matching pass 1, priors, pass 2 and pixel refinement, all bit-exact.  The first-pass
    survivors that feed the priors come from the host layer's removeOutliers, which tests/test_host_cpu.py pins."""
    op = O.Params(**kw)
    a, b = img
    fa = O.compute_features(a, op); fb = O.compute_features(b, op)
    if op.multi_stage:
        reference.same('rec_1p1', fa['rec1']); reference.same('rec_1c1', fb['rec1'])
    reference.same('rec_1p2', fa['rec2']); reference.same('rec_1c2', fb['rec2'])
    eff = op.effective()
    dims = fa['dims']
    planes = dict(du1p=fa['du_full'] if op.half_resolution else fa['du'], dv1p=fa['dv_full'] if op.half_resolution else fa['dv'],
                  du1c=fb['du_full'] if op.half_resolution else fb['du'], dv1c=fb['dv_full'] if op.half_resolution else fb['dv'])
    if op.multi_stage:
        got1 = O.matching(0, fa['rec1'], None, fb['rec1'], None, dims, eff)
        assert len(got1) > 20
        reference.same('raw1', got1)
        kept = H.Matcher(V.Params(**kw)).remove_outliers(got1, 0)
        got_r = O.prior_statistics(kept, 0, dims, eff)
        reference.same('ranges', got_r.reshape(-1, 4, 4)[:, :, :2])
        got2 = O.matching(0, fa['rec2'], None, fb['rec2'], None, dims, eff, ranges=got_r)
    else:
        got2 = O.matching(0, fa['rec2'], None, fb['rec2'], None, dims, eff)
    assert len(got2) > 100
    reference.same('raw2', got2)
    reference.same('refined2', O.refine_pixel(got2, 0, dims, planes))


def test_quad_matching(reference):
    lp, rpv, lc, rc = synth.blob_quad(401, 240, seed=19)
    kw = dict(nms_n=2, half_resolution=0)
    op = O.Params(**kw)
    f = [O.compute_features(i, op) for i in (lp, rpv, lc, rc)]
    got1 = O.matching(2, f[0]['rec1'], f[1]['rec1'], f[2]['rec1'], f[3]['rec1'], f[0]['dims'], op.effective())
    assert len(got1) > 20
    reference.same('raw1', got1)
    kept = H.Matcher(V.Params(**kw)).remove_outliers(got1, 2)
    ranges = O.prior_statistics(kept, 2, f[0]['dims'], op.effective())
    reference.same('ranges', ranges)
    got2 = O.matching(2, f[0]['rec2'], f[1]['rec2'], f[2]['rec2'], f[3]['rec2'], f[0]['dims'], op.effective(), ranges=ranges)
    assert len(got2) > 100
    reference.same('raw2', got2)
    planes = dict(du1p=f[0]['du'], dv1p=f[0]['dv'], du2p=f[1]['du'], dv2p=f[1]['dv'], du1c=f[2]['du'], dv1c=f[2]['dv'],
                  du2c=f[3]['du'], dv2c=f[3]['dv'])
    reference.same('refined2', O.refine_pixel(got2, 2, f[0]['dims'], planes))


# ------------------------------------------------------------------------------------------------------------------------
# Stereo matching, motion-predicted quad matching and sub-pixel refinement have no counterpart in the reference shim: the
# oracle's restatement is pinned against the reference results stored for the host-layer GPU tests instead, on the same
# inputs.  The chain is the Matcher's: pass 0, removeOutliers (the host layer's, pinned by tests/test_host_cpu.py), prior
# statistics, pass 1 with them, refinement, removeOutliers.
def _host_layer(case):
    return refgold.Reference('test_gpu_host_layer', case)


def oracle_chain(method, imgs, kw, tr_delta=None):
    """(survivors of pass 0, survivors of pass 1) of Matcher::matchFeatures(method) on imgs = (1p, 2p, 1c, 2c), None for
    an image the method does not use; kw: Matcher parameters (match_radius as given to the constructor)."""
    op = O.Params(**kw)
    eff = op.effective()
    f = [None if i is None else O.compute_features(i, op) for i in imgs]
    dims = next(x for x in f if x is not None)['dims']
    recs = lambda r: [None if x is None else x[r] for x in f]
    hm = H.Matcher(V.Params(**kw))
    kept1 = hm.remove_outliers(O.matching(method, *recs('rec1'), dims, eff, tr_delta=tr_delta), method)
    ranges = O.prior_statistics(kept1, method, dims, eff)
    raw2 = O.matching(method, *recs('rec2'), dims, eff, ranges=ranges, tr_delta=tr_delta)
    planes = {}
    for name, x in zip(('1p', '2p', '1c', '2c'), f):
        if x is not None:
            planes['du' + name] = x['du_full'] if op.half_resolution else x['du']
            planes['dv' + name] = x['dv_full'] if op.half_resolution else x['dv']
    if op.refinement == 2:
        raw2, keep, _ = O.refine_subpixel(raw2, method, dims, planes)
        raw2 = raw2[keep]
    elif op.refinement == 1:
        raw2 = O.refine_pixel(raw2, method, dims, planes)
    return kept1, hm.remove_outliers(raw2, method)


def test_stereo_matching_priors_refinement():
    """Method 1 (matcher.cpp:1045-1084): matching, its prior statistics and pixel refinement of (u2c, v2c), bit-exact
    against both modes of test_matcher_stereo_method1."""
    lp, rpv, lc, rc = synth.blob_quad(1244, 376, seed=47)
    ref = _host_layer('test_matcher_stereo_method1')
    for mode, kw in (('fullres', dict(half_resolution=0)), ('defaults', dict())):
        kept1, kept2 = oracle_chain(1, (None, None, lc, rc), kw)
        assert len(kept2) > 1000 and np.all(kept2['u1c'] >= kept2['u2c'])
        ref.same(mode + '_matches1', kept1)
        ref.same(mode + '_matches2', kept2)


def test_quad_matching_with_motion_prediction():
    """Tr_delta-predicted quad matching (matcher.cpp:1112-1138, cost SAD + 4 * distance in double precision), bit-exact
    against test_quad_matching_with_motion_prediction (reference built with -ffp-contract=off)."""
    lp, rpv, lc, rc = synth.blob_quad(1242, 376, seed=53, shift=(3, 1), disparity=12)
    Tr = np.eye(4); Tr[0, 3] = 0.02; Tr[2, 3] = -0.3; Tr[0, 2] = 0.01; Tr[2, 0] = -0.01
    kw = dict(nms_n=2, half_resolution=0, f=645.2, cu=635.9, cv=194.1, base=0.54)
    kept1, kept2 = oracle_chain(2, (lp, rpv, lc, rc), kw, tr_delta=Tr)
    assert len(kept2) > 500
    _host_layer('test_quad_matching_with_motion_prediction').same('matches2', kept2)
    # the prediction changes the result: without it the list differs
    assert kept2.tobytes() != oracle_chain(2, (lp, rpv, lc, rc), kw)[1].tobytes()


def test_subpixel_refinement():
    """parabolicFitting (matcher.cpp:1379-1454) with a least-squares solve per match: integer fields and the kept set
    bit-exact against test_matcher_subpixel_refinement, the stored coordinate samples within 1e-4 pixel."""
    ref = _host_layer('test_matcher_subpixel_refinement')
    sample = lambda n: np.sort(np.random.default_rng(0).choice(n, min(n, 512), replace=False))
    a, b = synth.blob_pair(1242, 376, seed=49)
    _, got = oracle_chain(0, (a, None, b, None), dict(nms_n=4, refinement=2, half_resolution=0))
    assert len(got) > 1000
    ref.same('flow_integer', np.stack([got[f] for f in ('i1p', 'i1c', 'u1c', 'v1c')], 1))
    rows = sample(len(got))
    for f in ('u1p', 'v1p'):
        assert np.abs(got[f][rows] - ref.value('flow_' + f)).max() < 1e-4
    lp, rpv, lc, rc = synth.blob_quad(1242, 376, seed=51)
    _, got = oracle_chain(2, (lp, rpv, lc, rc), dict(nms_n=2, refinement=2, half_resolution=0))
    assert len(got) > 500
    ref.same('quad_integer', np.stack([got[f] for f in ('i1p', 'i2p', 'i1c', 'i2c', 'u1c', 'v1c')], 1))
    rows = sample(len(got))
    for f in ('u1p', 'v1p', 'u2p', 'v2p', 'u2c', 'v2c'):
        assert np.abs(got[f][rows] - ref.value('quad_' + f)).max() < 1e-4


def _unit(F):
    F = F / np.linalg.norm(F)
    return F * np.sign(F.flat[np.argmax(np.abs(F))])


def test_ransac_pieces(reference):
    """FP64: F from the 8-point fit to 1e-9 (unit norm, fixed sign), inlier sets identical for the same F, RANSAC winner
    and inlier set identical, per-hypothesis counts equal for >= 99% of the hypotheses.  The reference side is the build
    without FMA contraction (-ffp-contract=off)."""
    rng = np.random.default_rng(3)
    n = 300
    # synthetic two-view geometry: points in front of two cameras, 30% gross outliers, already Hartley-scaled
    X = np.stack([rng.uniform(-2, 2, n), rng.uniform(-1, 1, n), rng.uniform(4, 12, n)], 1)
    R = np.array([[0.9998, 0.0, 0.02], [0, 1, 0], [-0.02, 0, 0.9998]]); t = np.array([0.05, 0.01, -0.8])
    x1 = X[:, :2] / X[:, 2:]; X2 = X @ R.T + t; x2 = X2[:, :2] / X2[:, 2:]
    bad = rng.random(n) < 0.3
    x2[bad] += rng.normal(0, 0.2, (bad.sum(), 2))
    m = np.zeros(n, pyref.P_MATCH)
    m['u1p'], m['v1p'], m['u1c'], m['v1c'] = 500 * x1[:, 0] + 600, 500 * x1[:, 1] + 180, 500 * x2[:, 0] + 600, 500 * x2[:, 1] + 180
    ok2, mn2, Tp2, Tc2 = O.normalize(m)
    assert ok2
    reference.same('normalized', mn2)
    assert np.allclose(Tp2, reference.value('Tp'), rtol=0, atol=1e-12) and np.allclose(Tc2, reference.value('Tc'), rtol=0, atol=1e-12)
    for k in range(20):
        act = rng.choice(n, 8, replace=False).astype(np.int32)
        Fo = O.fundamental(mn2, act)
        Fr = reference.value('F%d' % k)
        assert np.abs(_unit(Fr) - _unit(Fo)).max() < 1e-9
        reference.same('inliers%d' % k, O.get_inlier(mn2, Fr))
    samples = np.stack([rng.choice(n, 8, replace=False) for _ in range(500)]).astype(np.int32)
    got = O.ransac(mn2, samples)
    assert (reference.value('counts') != got['counts']).mean() <= 0.01
    assert int(reference.value('best_iter')) == got['best_iter']
    reference.same('inliers', got['inliers'])
    assert np.abs(_unit(reference.value('F')) - _unit(got['F'])).max() < 1e-8
