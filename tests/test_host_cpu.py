"""CPU tests of the host-side logic and of the C-ABI surface (no compute calls without a GPU)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import pyref
import visocu_py as V
import host_py as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, 'include', 'visocu.h')).read()
    declared = sorted(set(re.findall(r'\b(visocu_[a-z0-9_]+)\s*\(', hdr)))
    assert len(declared) >= 25
    lib = V.lib()
    for name in declared:
        assert hasattr(lib, name), name + ' is declared in include/visocu.h but not exported by libvisocu.so'
    assert C.sizeof(V.Params) == 72 and V.P_MATCH.itemsize == 48 and V.RANGE.itemsize == 64


def test_no_cpu_fallback_without_gpu():
    """On a box without a GPU the library must refuse loudly instead of computing something on the CPU."""
    h = C.c_void_p()
    rc = V.lib().visocu_create(0, C.byref(h))
    if rc == 0:
        V.lib().visocu_destroy(h)
        pytest.skip('a GPU is present')
    assert rc == -3 and b'no CPU fallback' in V.lib().visocu_last_error(None)


def _random_matches(rng, n, w, h, grid, dup):
    u = (rng.integers(0, w // grid, n) * grid).astype(np.float32); v = (rng.integers(0, h // grid, n) * grid).astype(np.float32)
    if not dup:
        _, idx = np.unique(u * 10000 + v, return_index=True)
        idx.sort(); u = u[idx]; v = v[idx]
    n = len(u)
    m = np.zeros(n, pyref.P_MATCH)
    m['u1c'] = u; m['v1c'] = v
    m['u1p'] = u - rng.integers(-3, 4, n); m['v1p'] = v - rng.integers(-3, 4, n)
    m['u2c'] = u - rng.integers(0, 6, n); m['v2c'] = v
    m['u2p'] = m['u1p'] - rng.integers(0, 6, n); m['v2p'] = m['v1p']
    m['i1c'] = np.arange(n); m['i1p'] = np.arange(n)
    return m


def test_remove_outliers_matches_reference(reference):
    """Matcher::removeOutliers (own exact Delaunay + support vote) against the reference's Triangle-based one on
    grid-heavy point sets: co-circular ties and duplicate pixels must be resolved identically."""
    hm = H.Matcher(V.Params(half_resolution=0))
    rng = np.random.default_rng(1)
    for trial in range(120):
        n = int(rng.integers(4, 1200)); grid = int(rng.choice([1, 1, 2, 4, 8, 16]))
        w = int(rng.integers(40, 1300)); h = int(rng.integers(40, 400)); method = int(rng.choice([0, 2]))
        m = _random_matches(rng, n, w, h, grid, dup=trial % 2 == 0)
        reference.same('trial%d' % trial, hm.remove_outliers(m, method))
    for n, grid, dup in ((7000, 1, False), (9000, 2, True)):      # beyond the ~5700 points the device kernel takes: the host path
        m = _random_matches(rng, n, 1300, 400, grid, dup)
        assert len(m) > 5700
        reference.same('large%d' % n, hm.remove_outliers(m, 0))
    for n in (0, 1, 3, 4):          # tiny inputs: <= 3 matches are returned untouched (matcher.cpp:1210)
        m = _random_matches(rng, 50, 100, 100, 1, False)[:n]
        reference.same('tiny%d' % n, hm.remove_outliers(m, 0))
    line = np.zeros(40, pyref.P_MATCH); line['u1c'] = np.arange(40) * 3; line['v1c'] = 7; line['u1p'] = line['u1c']; line['v1p'] = 7
    reference.same('collinear', hm.remove_outliers(line, 0))       # all collinear


def test_large_list_tree_with_device_nodes(tmp_path):
    """Lists beyond the device kernel (3840x2160): host/delaunay.cpp cuts the divide-and-conquer tree into nodes, takes their
    meshes from the device and merges above them.  Here the device entry point is a stand-in (tests/sim_device_nodes.cpp:
    the host algorithm answering in the device's format), so the cutting, the vertex maps, the import and the top merges run
    on the CPU: same edge list as the all-host triangulation, also when the device fails, declines a node or returns a corrupt mesh."""
    import ctypes as C
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = str(tmp_path / 'libsim_nodes.so')
    subprocess.check_call(['g++', '-O2', '-std=c++14', '-shared', '-fPIC', '-I' + os.path.join(root, 'include'),
                           '-I' + os.path.join(root, 'opencl-structure-from-motion_b200', 'host'),
                           os.path.join(root, 'tests', 'sim_device_nodes.cpp'), '-o', so])
    L = C.CDLL(so)
    calls = C.c_int(); ne = C.c_int()
    cases = [(5000, 1241, 376, 2, 0, 0), (6001, 2000, 300, 1, 0, 1), (7000, 1241, 376, 2, 0, 1), (20000, 3840, 2160, 2, 0, 1),
             (87000, 3840, 2160, 2, 0, 1), (30000, 3840, 2160, 4, 0, 1), (9000, 8000, 200, 1, 0, 1), (9000, 9000, 200, 1, 0, 0),
             (20000, 3840, 2160, 2, 1, 1), (20000, 3840, 2160, 2, 2, 1), (20000, 3840, 2160, 2, 3, 1)]
    for n, w, h, grid, fail, want_calls in cases:
        assert L.sim_check(n, w, h, 11 + n, grid, fail, C.byref(calls), C.byref(ne)) == 0, (n, w, h, grid, fail)
        assert calls.value == want_calls and ne.value > 2.9 * n - 400, (n, w, h, calls.value, ne.value)


def test_delaunay_is_delaunay():
    rng = np.random.default_rng(2)
    key = rng.choice(300 * 200, 500, replace=False)
    x = (key % 300).astype(np.int32); y = (key // 300).astype(np.int32)
    tri = H.delaunay(x, y)
    assert len(tri) >= 2 * 500 - 2 - 60
    P = np.stack([x, y], 1).astype(np.int64)
    for a, b, c in tri[::7]:
        A, B, Cc = P[a], P[b], P[c]
        assert (B[0] - A[0]) * (Cc[1] - A[1]) - (B[1] - A[1]) * (Cc[0] - A[0]) > 0          # counter-clockwise
        d = P - Cc
        al = ((P[a] - P) ** 2).sum(1)
        m = np.stack([A - P, B - P, np.broadcast_to(Cc, P.shape) - P], 1)               # n x 3 x 2
        lift = (m ** 2).sum(2)
        det = (lift[:, 0] * (m[:, 1, 0] * m[:, 2, 1] - m[:, 2, 0] * m[:, 1, 1]) +
               lift[:, 1] * (m[:, 2, 0] * m[:, 0, 1] - m[:, 0, 0] * m[:, 2, 1]) +
               lift[:, 2] * (m[:, 0, 0] * m[:, 1, 1] - m[:, 1, 0] * m[:, 0, 1]))
        assert (det <= 0).all()                                                          # empty circumcircle


def test_matrix_svd_conventions(reference):
    rng = np.random.default_rng(4)
    for m, n in ((8, 9), (3, 3), (4, 4), (20, 9)):
        A = rng.normal(size=(m, n))
        U, W, Vv = H.svd(A)
        k = min(m, n)
        Wr = reference.value('W%dx%d' % (m, n)); Vr = reference.value('V%dx%d' % (m, n))
        assert np.allclose(W, Wr, rtol=1e-12, atol=1e-12)
        assert np.allclose(U[:, :k] * W @ Vv[:, :k].T, A, atol=1e-12)
        assert np.allclose(np.abs(Vv[:, :k]), np.abs(Vr), atol=1e-9)
        assert np.allclose(Vv[:, :k], Vr, atol=1e-9)                                    # same sign convention


def test_bench_rank_aggregation_gloo():
    """N > 1 path of bench.py (max over ranks, whole-job value) with two CPU ranks over gloo."""
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', '29533', os.path.join(ROOT, 'bench.py'), '--gpus', '2', '--steps', '4', '--warmup', '3', '--dry-run']
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1                                   # rank 0 only
    import json
    r = json.loads(lines[0])
    assert r['n_gpus'] == 2 and r['scaling'] == 'weak' and r['config']['frame_pairs_per_step'] == 2 * r['config']['sequences_per_gpu']
    # dry-run ranks report 10 ms and 20 ms per step: the slower rank decides
    assert abs(r['ms_per_step'] - 20.0) < 1e-6
    assert abs(r['value'] - 2 * r['config']['sequences_per_gpu'] / 0.020) < 1e-3
    assert r['gpu_launches'] == 0 and r['data'] == 'dry-run'
    # configs[4] as written: 64 sequences in total over the ranks (strong scaling)
    out = subprocess.run(cmd[:-1] + ['--scaling', 'strong', '--sequences', '64', '--dry-run'], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    r = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][0])
    assert r['scaling'] == 'strong' and r['config']['sequences_per_gpu'] == 32 and r['config']['frame_pairs_per_step'] == 64
    assert abs(r['value'] - 64 / 0.020) < 1e-3


@pytest.mark.parametrize('point_type,min_len,min_angle', [(0, 2, 3.0), (1, 2, 2.0), (2, 3, 1.0)])
def test_reconstruction_matches_reference(reference, point_type, min_len, min_angle):
    """Reconstruction::update (reconstruction.cpp:50-146) on synthetic feature tracks: same tracks end in the same
    frames, so the point lists have the same length and order; coordinates agree to float rounding (the 4x4 null vector
    comes from a different SVD algorithm, then both sides run the same Gauss-Newton to convergence at 1e-5)."""
    import synth
    seq = synth.track_sequence(n_frames=14, n_points=700, seed=21)
    hr = pyref.Recon(H.lib(), 'visob_recon')
    hr.set_calibration(synth.KITTI_F, synth.KITTI_CU, synth.KITTI_CV)
    total = 0
    for k, (m, tr) in enumerate(seq):
        hr.update(m, tr, point_type, min_len, 30.0, min_angle)
        b = hr.points()
        a = reference.value('points%d' % k)
        assert len(a) == len(b)
        if len(a):
            assert np.abs(a - b).max() <= 1e-5 * max(1.0, np.abs(a).max())
        total = len(b)
    assert total > 50


def test_stereo_odometry_from_matches(reference):
    """VisualOdometryStereo::estimateMotion (viso_stereo.cpp:42-145) is host code: fed with the same quad matches, the
    3-point RANSAC over Gauss-Newton fits and the final refinement must pick the same inliers and the same motion as
    the reference.  Synthetic rig: f = 645.2, base 0.54 m, 0.8 m forward with a slight yaw, 0.3 px noise, 15 % outliers.
    Both sides draw the RANSAC samples from a fresh generator (the reference's is process-wide state, viso.cpp:88)."""
    rng = np.random.RandomState(5)
    f, cu, cv, base = 645.2, 635.9, 194.1, 0.54
    kw = dict(f=f, cu=cu, cv=cv, base=base)
    hv = H.Stereo(H.StereoParams(match=V.Params(), **kw))
    for step in range(3):
        n = 400
        P = np.stack([rng.uniform(-10, 10, n), rng.uniform(-3, 1.6, n), rng.uniform(5, 50, n)], 1)
        yaw = 0.01 * (step + 1)
        R = np.array([[np.cos(yaw), 0, np.sin(yaw)], [0, 1, 0], [-np.sin(yaw), 0, np.cos(yaw)]])
        t = np.array([0.02, -0.01, -0.8])
        Q = P @ R.T + t                                        # the same points in the current left camera frame

        def project(X, shift):
            return f * (X[:, 0] - shift) / X[:, 2] + cu, f * X[:, 1] / X[:, 2] + cv

        m = np.zeros(n, pyref.P_MATCH)
        for name in ('i1p', 'i2p', 'i1c', 'i2c'):
            m[name] = np.arange(n)
        m['u1p'], m['v1p'] = project(P, 0.0); m['u2p'], m['v2p'] = project(P, base)
        m['u1c'], m['v1c'] = project(Q, 0.0); m['u2c'], m['v2c'] = project(Q, base)
        for name in ('u1p', 'v1p', 'u2p', 'u1c', 'v1c', 'u2c'):
            m[name] += rng.normal(0, 0.3, n).astype(np.float32)
        m['v2p'] = m['v1p']; m['v2c'] = m['v1c']
        bad = rng.rand(n) < 0.15
        m['u1c'][bad] += rng.uniform(-40, 40, bad.sum()).astype(np.float32)
        assert hv.process_matches(m)
        reference.same('inliers%d' % step, hv.inliers())
        assert len(hv.inliers()) > 250
        Th = hv.motion()
        Tr = reference.value('motion%d' % step)
        assert np.abs(Tr - Th).max() < 1e-9
        assert abs(Th[2, 3] + 0.8) < 0.05


def test_prior_statistics_before_any_push():
    """Matcher::computePriorStatistics on a matcher that has seen no image has no image size to lay its bin grid over:
    it gives no ranges (it used to index a grid of zero bins)."""
    m = np.zeros(3, H.P_MATCH)
    m['u1p'], m['v1p'], m['u1c'], m['v1c'], m['u2c'], m['v2c'] = [10, 20, 30], 5, [12, 21, 33], 6, [4, 9, 20], 6
    for method in (0, 1, 2):
        assert H.Matcher(V.Params()).prior(m, method).shape == (0, 16)
