"""GPU tests of individual C-ABI entry points: pose helpers against numpy, error and edge behaviour."""
import ctypes as C

import numpy as np
import pytest

import synth
import visocu_py as V

pytestmark = pytest.mark.gpu


def test_triangulate_against_numpy(ctx):
    rng = np.random.default_rng(7)
    n = 500
    K = np.array([[645.2, 0, 635.9], [0, 645.2, 194.1], [0, 0, 1.0]])
    X = np.stack([rng.uniform(-5, 5, n), rng.uniform(-2, 2, n), rng.uniform(4, 40, n), np.ones(n)])
    R = np.array([[0.9998, 0.0, 0.02], [0, 1, 0], [-0.02, 0, 0.9998]]); t = np.array([[0.1], [0.0], [-0.8]])
    P1 = K @ np.hstack([np.eye(3), np.zeros((3, 1))])
    P2 = np.stack([K @ np.hstack([R, s * t]) for s in (1, -1)])
    x1 = P1 @ X; x2 = P2[0] @ X
    uv = np.stack([x1[0] / x1[2], x1[1] / x1[2], x2[0] / x2[2], x2[1] / x2[2]], 1).astype(np.float32)
    Xg, nf = ctx.triangulate(uv, P1, P2)
    assert Xg.shape == (2, 4, n)
    Xn = Xg[0] / Xg[0][3]
    assert np.abs(Xn[:3] - X[:3]).max() / 40 < 2e-3          # float32 pixel coordinates limit the depth accuracy
    assert nf[0] == n and nf[1] < n // 10                     # the true (R|t) puts every point in front of both cameras
    # each column is the null vector of its 4x4 system (tolerance: 1e-9 of the matrix norm)
    for i in range(0, n, 37):
        u1, v1, u2, v2 = uv[i].astype(np.float64)
        J = np.stack([P1[2] * u1 - P1[0], P1[2] * v1 - P1[1], P2[0][2] * u2 - P2[0][0], P2[0][2] * v2 - P2[0][1]])
        x = Xg[0][:, i]
        smin = np.linalg.svd(J, compute_uv=False)[-1]
        assert abs(np.linalg.norm(x) - 1) < 1e-12 and np.linalg.norm(J @ x) <= smin * (1 + 1e-6) + 1e-9 * np.linalg.norm(J)


def test_best_plane_against_numpy(ctx):
    rng = np.random.default_rng(8)
    d = np.concatenate([rng.normal(1.6, 0.02, 150), rng.uniform(0.2, 5, 60)])
    rng.shuffle(d)
    thr, w = 0.5, 1.0 / (2 * 0.05 ** 2)
    sums = np.array([np.exp(-(d - di) ** 2 * w).sum() if di > thr else -1 for di in d])
    got = ctx.best_plane(d, thr, w)
    assert sums[got] >= sums.max() * (1 - 1e-12) and abs(d[got] - 1.6) < 0.05
    assert ctx.best_plane(np.full(10, 0.1), thr, w) == 0        # no candidate above the threshold -> index 0


def test_error_codes_and_edge_inputs(ctx):
    L = V.lib()
    p = V.Params()
    assert L.visocu_configure(ctx.h, C.byref(p), 0, 100, 2) == -1            # VISOCU_EINVAL
    assert b'bad dims' in L.visocu_last_error(ctx.h)
    bad = V.Params(nms_n=40)
    assert L.visocu_configure(ctx.h, C.byref(bad), 640, 480, 2) == -1
    ctx.configure(p, 200, 120, 2)
    img = synth.blob_pair(200, 120, seed=3)[0]
    with pytest.raises(V.VisocuError, match='out of range'):
        ctx.push_frames([5], [img])
    with pytest.raises(V.VisocuError, match='bytes per line'):
        ctx.push_frames([0], [img], bpl_in=100)
    with pytest.raises(V.VisocuError, match='holds no features'):
        ctx.match([(0, -1, 1, -1)], 0, 1)
    # a constant image has no maxima: empty lists everywhere, matching returns nothing instead of failing
    flat = np.full((120, 200), 90, np.uint8)
    ns, nd = ctx.push_frames([0, 1], [flat, flat])
    assert ns.tolist() == [0, 0] and nd.tolist() == [0, 0]
    assert len(ctx.match([(0, -1, 1, -1)], 0, 1)[0]) == 0
    # an image smaller than one NMS cell grid (no cells at all)
    ctx.configure(V.Params(half_resolution=0), 24, 20, 1)
    ns, nd = ctx.push_frames([0], [np.zeros((20, 24), np.uint8)])
    assert ns[0] == 0 and nd[0] == 0


def test_sad_extremes(ctx):
    """maximum SAD (8160) and ties: two identical frames match one-to-one with cost 0, inverted frames still match on
    position only through the bin structure."""
    a, _ = synth.blob_pair(320, 200, seed=9)
    ctx.configure(V.Params(half_resolution=0), 320, 200, 2)
    ctx.push_frames([0, 1], [a, a])
    m = ctx.match([(0, -1, 1, -1)], 0, 1)[0]
    n = len(ctx.features(0, 1))
    assert len(m) > 0.9 * n and np.all(m['i1p'] == m['i1c'])
    cand, scanned = ctx.match_stats()
    assert cand >= 2 * n


def test_fused_submit_collect_and_lanes(ctx, reference):
    """visocu_match_fused_submit / _collect on two lanes of one context: misuse is reported with a status, never a crash,
    and two steps in flight on different lanes deliver the lists of the reference (stored under tests/golden/reference)."""
    import ctypes as C
    lib = V.lib()
    w, h = 500, 260
    p = V.Params(); p.match_radius //= 2
    ctx.configure(p, w, h, 4)
    z = lambda n, t: np.zeros(n, t)
    l1 = (C.c_void_p * 1)(); l2 = (C.c_void_p * 1)()
    n1, n2, d1, d2, cnt = z(1, np.int32), z(1, np.int32), z(1, np.int32), z(1, np.int32), z(4, np.int32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    compact = C.c_int32()
    rc = lib.visocu_match_fused_collect(ctx.h, l1, vp(n1), vp(d1), l2, vp(n2), vp(d2), None, vp(cnt), C.byref(compact))
    assert rc != 0 and b'no fused matching call' in lib.visocu_last_error(ctx.h)
    assert lib.visocu_set_lane(ctx.h, 9) != 0 and b'out of range' in lib.visocu_last_error(ctx.h)
    q = np.zeros(1, V.QUAD); q[0] = (0, -1, 1, -1)
    rc = lib.visocu_match_fused_submit(ctx.h, 1, vp(q), 1, 0, -1)
    assert rc != 0 and b'holds no features' in lib.visocu_last_error(ctx.h)
    # three frames; frames 0, 1 pushed on lane 0, frame 2 on lane 1; pairs (0,1) and (1,2) in flight together
    seq = synth.blob_sequence(3, w, h, seed=77)
    assert lib.visocu_set_lane(ctx.h, 0) == 0
    ctx.push_frames([0, 1], [seq[0], seq[1]], want_counts=False)
    assert lib.visocu_match_fused_submit(ctx.h, 1, vp(q), 1, 0, -1) == 0
    assert lib.visocu_match_fused_submit(ctx.h, 1, vp(q), 1, 0, -1) != 0 and b'not been collected' in lib.visocu_last_error(ctx.h)
    assert lib.visocu_set_lane(ctx.h, 1) == 0
    ctx.push_frames([2], [seq[2]], want_counts=False)
    q2 = np.zeros(1, V.QUAD); q2[0] = (1, -1, 2, -1)
    assert lib.visocu_match_fused_submit(ctx.h, 1, vp(q2), 1, 0, 0) == 0
    def unpack(fmt, addr, n):
        """list 2 of a fused call as p_match records: 1 = six words per match, 2 = three words (16-bit fields)"""
        m = np.zeros(n, V.P_MATCH)
        for f in ('u2p', 'v2p', 'i2p', 'u2c', 'v2c', 'i2c'):
            m[f] = -1
        if fmt == 1:
            half = np.dtype([('u', 'f4'), ('v', 'f4'), ('i', 'i4')])
            raw = np.ctypeslib.as_array((C.c_uint8 * (24 * n)).from_address(addr)).view(half).reshape(-1, 2)
            m['u1p'], m['v1p'], m['i1p'] = raw[:, 0]['u'], raw[:, 0]['v'], raw[:, 0]['i']
            m['u1c'], m['v1c'], m['i1c'] = raw[:, 1]['u'], raw[:, 1]['v'], raw[:, 1]['i']
        else:
            raw = np.ctypeslib.as_array((C.c_uint32 * (3 * n)).from_address(addr)).reshape(-1, 3)
            m['u1p'], m['v1p'] = raw[:, 0] & 0xFFFF, raw[:, 0] >> 16
            m['u1c'], m['v1c'] = raw[:, 1] & 0xFFFF, raw[:, 1] >> 16
            m['i1p'], m['i1c'] = raw[:, 2] & 0xFFFF, raw[:, 2] >> 16
        return m

    got = []
    for lane in (0, 1):
        assert lib.visocu_set_lane(ctx.h, lane) == 0
        assert lib.visocu_match_fused_collect(ctx.h, l1, vp(n1), vp(d1), l2, vp(n2), vp(d2), None, vp(cnt), C.byref(compact)) == 0
        assert d1[0] == 1 and d2[0] == 1 and cnt.min() > 100
        assert compact.value == 2 and not l1[0]                       # pixel refinement: 12 bytes per match; flags 0: list 1 stays on the device
        got.append(unpack(2, l2[0], int(n2[0])))
    assert lib.visocu_set_lane(ctx.h, 0) == 0
    assert len(got[0]) > 300
    reference.same('lane0', got[0]); reference.same('lane1', got[1])
    # sub-pixel refinement is not part of the fused call
    assert lib.visocu_match_fused_submit(ctx.h, 1, vp(q2), 2, 0, -1) != 0 and b'refine must be' in lib.visocu_last_error(ctx.h)
    # more than 65535 records per list: indices no longer fit 16 bits, six words per match
    w2, h2 = 1000, 600
    p2 = V.Params(nms_n=4, half_resolution=0)
    ctx.configure(p2, w2, h2, 2)
    a2, b2 = synth.blob_pair(w2, h2, n_blobs=2500, seed=78)           # few blobs: the lists stay within the outlier kernel
    ctx.push_frames([0, 1], [a2, b2], want_counts=False)
    assert lib.visocu_match_fused_submit(ctx.h, 1, vp(q), 1, 0, -1) == 0
    assert lib.visocu_match_fused_collect(ctx.h, l1, vp(n1), vp(d1), l2, vp(n2), vp(d2), None, vp(cnt), C.byref(compact)) == 0
    assert compact.value == 1 and d2[0] == 1
    wide = unpack(1, l2[0], int(n2[0]))
    assert len(wide) > 300
    reference.same('wide', wide)
