"""GPU parity tests proper: the CUDA path, called through the C-ABI of include/visocu.h, against the outputs of the
unmodified reference CPU path on identical synthetic inputs (stored under tests/golden/reference, see oracle/refgold.py).
Integer stages are compared bit-exactly, list order included (SURVEY.md 8d checkpoints P1-P6, P8)."""
import numpy as np
import pytest

import synth
import pyoracle as O
import visocu_py as V
import host_py as H

pytestmark = pytest.mark.gpu


def params(**kw):
    """C-ABI params: the Matcher constructor halves match_radius at half resolution (matcher.cpp:59-60); the C-ABI takes
    the effective value."""
    vp = V.Params(**kw)
    if vp.half_resolution:
        vp.match_radius = vp.match_radius // 2
    return vp


def valid(plane, w):
    return plane[2:-2, 2:w - 2]


def comparable(rec, wm, scale):
    """Feature records are compared bit-exactly, except for the last descriptor word of a maximum sitting at
    u = w-7: its two samples at u+5 read Sobel column w-2, which in the reference depends on the uninitialised
    pad bytes behind each image row (matcher.cpp:170-174), so the reference itself is not reproducible there."""
    r = rec.copy()
    r[(r[:, 0] // scale) >= wm - 7, 11] = 0
    return r


CASES = [
    dict(width=1241, height=376, half_resolution=1),
    dict(width=1241, height=376, half_resolution=0),
    dict(width=1241, height=376, half_resolution=0, nms_n=4),      # flow demo setting: sparse n = 10
    dict(width=337, height=211, half_resolution=0, nms_n=2),       # quad demo setting, ragged size
    dict(width=640, height=480, half_resolution=1, nms_n=5, nms_tau=30),
    dict(width=130, height=70, half_resolution=0, multi_stage=0),
]


@pytest.mark.parametrize('case', CASES, ids=lambda c: '-'.join('%s%s' % (k[:4], v) for k, v in c.items()))
def test_features_match_reference(ctx, reference, case):
    case = dict(case)
    w, h = case.pop('width'), case.pop('height')
    vp = params(**case)
    a, b = synth.blob_pair(w, h, seed=7)
    ctx.configure(vp, w, h, 2)
    ns, nd = ctx.push_frames([0, 1], [a, b])
    reference.same('counts', np.array([ns.tolist(), nd.tolist()], np.int64))
    for frame, tag in ((0, '1p'), (1, '1c')):
        scale = 2 if vp.half_resolution else 1
        if vp.multi_stage:
            reference.same('rec_' + tag + '1', comparable(ctx.features(frame, 0), w // scale, scale))
        reference.same('rec_' + tag + '2', comparable(ctx.features(frame, 1), w // scale, scale))
        gdu, (gw, gh, gbpl) = ctx.plane(frame, 0)
        gdv, _ = ctx.plane(frame, 1)
        reference.same('dims_' + tag, np.array([gw, gh, gbpl], np.int64))
        reference.same('du_' + tag, valid(gdu, gw)); reference.same('dv_' + tag, valid(gdv, gw))
        if vp.half_resolution:
            g2, (w2, h2, b2) = ctx.plane(frame, 2)
            g3, _ = ctx.plane(frame, 3)
            reference.same('dims_full_' + tag, np.array([w2, h2, b2], np.int64))
            reference.same('du_full_' + tag, valid(g2, w2)); reference.same('dv_full_' + tag, valid(g3, w2))


def test_half_image(ctx, reference):
    vp = params(half_resolution=1)
    a, _ = synth.blob_pair(1241, 376, seed=3)
    ctx.configure(vp, 1241, 376, 1)
    ctx.push_frames([0], [a])
    g, (gw, gh, gb) = ctx.plane(0, 5)
    reference.same('dims', np.array([gw, gh, gb], np.int64))
    reference.same('half', g[:, :gw])


def test_standalone_filters(ctx, reference):
    img = synth.blob_pair(320, 200, seed=5)[0]
    du, dv = ctx.sobel5x5(img)
    reference.same('sobel5x5_du', du[2:-2, 2:-2]); reference.same('sobel5x5_dv', dv[2:-2, 2:-2])
    du, dv = ctx.sobel3x3(img)
    reference.same('sobel3x3_du', du[1:-1, 1:-1]); reference.same('sobel3x3_dv', dv[1:-1, 1:-1])
    f1 = ctx.blob5x5(img)
    reference.same('blob5x5', f1[3:-2, 3:-2])
    f2 = ctx.checkerboard5x5(img)
    reference.same('checkerboard5x5', f2[2:-2, 2:-66])       # the reference's row pass stops short (filter.cpp:268)
    # NMS on the response maps
    for n in (3, 9):
        reference.same('nms%d' % n, ctx.nms(f1, f2, 320, n, 50))


def _host_priors(first, method, frames, **kw):
    """Prior ranges from a first-pass list through the host stages of the drop-in Matcher, which are the reference's
    (removeOutliers + computePriorStatistics, P5)."""
    hm = H.Matcher(V.Params(**kw))
    if method == 2:
        hm.push(frames[0], frames[1]); hm.push(frames[2], frames[3])
    else:
        hm.push(frames[0]); hm.push(frames[1])
    return hm.prior(hm.remove_outliers(first, method), method)


@pytest.mark.parametrize('half', [1, 0])
@pytest.mark.parametrize('size', [(1241, 376), (400, 300)])
def test_flow_matching_two_pass(ctx, reference, size, half):
    w, h = size
    vp = params(half_resolution=half)
    a, b = synth.blob_pair(w, h, seed=11)
    ctx.configure(vp, w, h, 2)
    ctx.push_frames([0, 1], [a, b])
    quad = (0, -1, 1, -1)
    # pass 1: sparse sets, full search window (P4)
    got1 = ctx.match([quad], 0, 0)[0]
    assert len(got1) > 50
    reference.same('raw1', got1)
    # priors from the host stages (P5), then pass 2 with priors and pixel refinement (P6)
    ranges = _host_priors(got1, 0, [a, b], half_resolution=half)
    got2 = ctx.match([quad], 0, 1, ranges=[ranges])[0]
    assert len(got2) > 200
    reference.same('raw2', got2)
    got3 = ctx.match([quad], 0, 1, ranges=[ranges], refine=True)[0]
    reference.same('refined2', got3)
    assert ctx.refine(quad, 0, got2).tobytes() == got3.tobytes()
    cand, scanned = ctx.match_stats()
    assert cand > 0 and scanned >= cand


@pytest.mark.parametrize('half', [1, 0])
def test_quad_matching_two_pass(ctx, reference, half):
    w, h = 1242, 376        # 1241 with n = 2 would allow maxima at u = w-7 (see comparable)
    vp = params(half_resolution=half, nms_n=2)
    frames = synth.blob_quad(w, h, seed=21)
    ctx.configure(vp, w, h, 4)
    ctx.push_frames([0, 1, 2, 3], list(frames))
    scale = 2 if half else 1
    for frame, tag in ((0, '1p2'), (1, '2p2'), (2, '1c2'), (3, '2c2')):
        reference.same('rec_' + tag, comparable(ctx.features(frame, 1), w // scale, scale))
    quad = (0, 1, 2, 3)
    got1 = ctx.match([quad], 2, 0)[0]
    assert len(got1) > 50
    reference.same('raw1', got1)
    ranges = _host_priors(got1, 2, frames, half_resolution=half, nms_n=2)
    got2 = ctx.match([quad], 2, 1, ranges=[ranges])[0]
    assert len(got2) > 200
    reference.same('raw2', got2)
    got3 = ctx.match([quad], 2, 1, ranges=[ranges], refine=True)[0]
    reference.same('refined2', got3)


def test_batched_jobs_equal_single_jobs(ctx, reference):
    """Batch dimension: 6 frames / 3 independent pairs in one launch give the lists of the reference's single pairs."""
    w, h = 500, 260
    ctx.configure(params(), w, h, 6)
    pairs = [synth.blob_pair(w, h, seed=s) for s in (31, 32, 33)]
    ctx.push_frames(list(range(6)), [im for p in pairs for im in p])
    quads = [(0, -1, 1, -1), (2, -1, 3, -1), (4, -1, 5, -1)]
    batched = ctx.match(quads, 0, 0)
    for k in range(len(pairs)):
        reference.same('raw1_%d' % k, batched[k])
        reference.same('rec_1c2_%d' % k, ctx.features(2 * k + 1, 1))


def _normalized_F(F):
    F = F / np.linalg.norm(F)
    k = np.argmax(np.abs(F))
    return F * np.sign(F.flat[k])


def test_ransac_against_reference(ctx, reference):
    """P8: identical sample table -> per-hypothesis inlier counts, winner, inlier set and F, against the reference built
    without FMA contraction.  The matches come from two odometry frames (the same list as the reference's, see
    test_gpu_host_layer.py), normalised by the plain-C restatement (the reference's bytes, see test_oracle_vs_ref.py).
    Tolerances: F (unit Frobenius norm, fixed sign) to 1e-8 absolute; per-hypothesis counts may differ only for
    hypotheses whose 8-point system is numerically rank deficient (different null-space basis) or whose matches
    sit within rounding of the threshold: at most 1% of hypotheses, each by a bounded amount checked below."""
    seq = synth.corridor_sequence(2, seed=1234)
    hv = H.Mono(H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08,
                             bucket_max_features=2))
    hv.process(seq[0]); hv.process(seq[1])
    pm = hv.matches()
    assert len(pm) > 100
    reference.same('matches', pm)
    ok, pmn, Tp, Tc = O.normalize(pm)
    assert ok
    reference.same('normalized', pmn)
    rng = np.random.default_rng(5)
    iters = 2000
    samples = np.stack([rng.choice(len(pmn), 8, replace=False) for _ in range(iters)]).astype(np.int32)
    uv = np.stack([pmn['u1p'], pmn['v1p'], pmn['u1c'], pmn['v1c']], axis=1)
    got = ctx.ransac([uv], [samples], 1e-5, want_all=True)[0]
    diff = got['counts'] != reference.value('counts')
    assert diff.mean() <= 0.01, 'hypothesis counts differ for %d of %d' % (diff.sum(), iters)
    assert got['best_iter'] == int(reference.value('best_iter'))
    assert got['n_inliers'] == int(reference.value('n_inliers'))
    reference.same('inliers', got['inliers'])
    assert np.abs(_normalized_F(got['F']) - _normalized_F(reference.value('F'))).max() < 1e-8
    # the non-degenerate hypotheses agree to rounding as well (stored for a fixed sample, see oracle/refgold.py)
    rows = np.sort(np.random.default_rng(0).choice(iters, 250, replace=False))
    Fg = np.stack([_normalized_F(f) for f in got['F_all'][rows]])
    Fw = reference.value('F_all_sample')
    same = ~diff[rows]
    assert np.median(np.abs(Fg[same] - Fw[same]).max(axis=(1, 2))) < 1e-10
