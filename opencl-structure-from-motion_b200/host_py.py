"""ctypes binding of the C++ host layer (libviso_b200.so: Matcher, filter::, VisualOdometryMono, the sharded
sequence runner) for the tests and bench.py.  Plumbing only."""
import ctypes as C
import os
import numpy as np

from visocu_py import Params, P_MATCH, VisocuError

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libviso_b200.so')


class MonoParams(C.Structure):
    """VisualOdometryMono::parameters flattened (reference viso.h:33-62, viso_mono.h:32-45)."""
    _fields_ = [('match', Params), ('bucket_max_features', C.c_int32), ('bucket_width', C.c_double),
                ('bucket_height', C.c_double), ('f', C.c_double), ('cu', C.c_double), ('cv', C.c_double),
                ('height', C.c_double), ('pitch', C.c_double), ('ransac_iters', C.c_int32),
                ('inlier_threshold', C.c_double), ('motion_threshold', C.c_double)]

    def __init__(self, match=None, **kw):
        super().__init__()
        self.match = match if match is not None else Params()
        d = dict(bucket_max_features=2, bucket_width=50.0, bucket_height=50.0, f=1.0, cu=0.0, cv=0.0,
                 height=1.0, pitch=0.0, ransac_iters=2000, inlier_threshold=0.00001, motion_threshold=100.0)
        d.update(kw)
        for k, v in d.items():
            setattr(self, k, v)


class StereoParams(C.Structure):
    """VisualOdometryStereo::parameters flattened (reference viso.h:33-62, viso_stereo.h:32-46)."""
    _fields_ = [('match', Params), ('bucket_max_features', C.c_int32), ('bucket_width', C.c_double),
                ('bucket_height', C.c_double), ('f', C.c_double), ('cu', C.c_double), ('cv', C.c_double),
                ('base', C.c_double), ('ransac_iters', C.c_int32), ('inlier_threshold', C.c_double), ('reweighting', C.c_int32)]

    def __init__(self, match=None, **kw):
        super().__init__()
        self.match = match if match is not None else Params()
        d = dict(bucket_max_features=2, bucket_width=50.0, bucket_height=50.0, f=1.0, cu=0.0, cv=0.0,
                 base=1.0, ransac_iters=200, inlier_threshold=2.0, reweighting=1)
        d.update(kw)
        for k, v in d.items():
            setattr(self, k, v)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise VisocuError(LIB_PATH + ' is missing: run __graft_entry__.build()')
        L = C.CDLL(LIB_PATH)
        for name in ('visob_matcher_create', 'visob_mono_create', 'visob_mono_matcher', 'visob_runner_create', 'visob_runner_create_stereo', 'visob_stereo_create', 'visob_recon_create', 'visob_sfm_create',
                     'visob_matcher_context'):
            getattr(L, name).restype = C.c_void_p
        L.visob_matcher_gain.restype = C.c_float
        L.visob_runner_step.restype = C.c_double
        L.visob_runner_run.restype = C.c_double
        L.visob_runner_launches.restype = C.c_uint64
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def stage_times(reset=True):
    """Host-layer wall-clock per stage, summed over worker threads: dict name -> (seconds, calls)."""
    sec = np.zeros(8); calls = np.zeros(8, np.int64)
    lib().visob_stage_times(_p(sec), _p(calls), int(reset))
    names = ['pushBack', 'matching_pass1', 'matching_pass2', 'priors', 'removeOutliers_small', 'removeOutliers_large',
             'ransacEstimateF', 'estimateMotion_total']
    return {n: (float(sec[k]), int(calls[k])) for k, n in enumerate(names)}


def set_device(d):
    lib().visob_set_device(int(d))


def _dims(img):
    h, w = img.shape
    return np.array([w, h, w], np.int32)


class Matcher:
    """The C++ Matcher (same semantics as the reference class)."""

    def __init__(self, params, handle=None):
        self.params = params
        self.owned = handle is None
        self.h = C.c_void_p(lib().visob_matcher_create(C.byref(params))) if handle is None else C.c_void_p(handle)

    def __del__(self):
        if getattr(self, 'owned', False) and self.h:
            lib().visob_matcher_destroy(self.h)
            self.h = None

    def push(self, I1, I2=None, replace=False):
        I1 = np.ascontiguousarray(I1, np.uint8)
        if I2 is not None:
            I2 = np.ascontiguousarray(I2, np.uint8)
        lib().visob_matcher_push(self.h, _p(I1), _p(I2), _p(_dims(I1)), int(replace))

    def match_features(self, method, tr_delta=None):
        if tr_delta is None:
            lib().visob_matcher_match_features(self.h, method)
        else:
            lib().visob_matcher_match_features_tr(self.h, method, _p(np.ascontiguousarray(tr_delta, np.float64)))

    def set_intrinsics(self, f, cu, cv, base):
        lib().visob_matcher_set_intrinsics(self.h, C.c_double(f), C.c_double(cu), C.c_double(cv), C.c_double(base))

    def bucket(self, max_features, bw, bh):
        lib().visob_matcher_bucket(self.h, max_features, C.c_float(bw), C.c_float(bh))

    def matches(self, stage=2):
        n = lib().visob_matcher_get_matches(self.h, stage, None, 0)
        out = np.zeros(n, P_MATCH)
        if n:
            lib().visob_matcher_get_matches(self.h, stage, _p(out), n)
        return out

    def counts(self):
        out = np.zeros(8, np.int32)
        lib().visob_matcher_counts(self.h, _p(out))
        return dict(zip(('1p1', '2p1', '1c1', '2c1', '1p2', '2p2', '1c2', '2c2'), out.tolist()))

    def gain(self, inliers):
        a = np.ascontiguousarray(inliers, np.int32)
        return float(lib().visob_matcher_gain(self.h, _p(a), len(a)))

    def remove_outliers(self, matches, method):
        m = np.array(matches, dtype=P_MATCH, copy=True)
        n = lib().visob_matcher_remove_outliers(self.h, _p(m), len(m), method)
        return m[:n].copy()

    def ranges(self):
        """Prior ranges of the last matchFeatures (computed on the device for multi-stage flow matching)."""
        nb = lib().visob_matcher_ranges(self.h, None, 0)
        out = np.zeros((nb, 16), np.float32)
        if nb:
            lib().visob_matcher_ranges(self.h, _p(out), nb)
        return out

    def prior(self, matches, method):
        m = np.ascontiguousarray(matches, dtype=P_MATCH)
        nb = lib().visob_matcher_prior(self.h, _p(m), len(m), method, None, 0)
        out = np.zeros((nb, 16), np.float32)
        lib().visob_matcher_prior(self.h, _p(m), len(m), method, _p(out), nb)
        return out


def filter_call(which, img):
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    a = np.zeros_like(img); b = np.zeros_like(img); o = np.zeros((h, w), np.int16)
    rc = lib().visob_filter(which, _p(img), _p(a), _p(b), _p(o), w, h)
    if rc:
        raise VisocuError('filter:: call failed')
    return (a, b) if which < 2 else o


class Mono:
    def __init__(self, params):
        self.params = params
        self.h = C.c_void_p(lib().visob_mono_create(C.byref(params)))
        self.matcher = Matcher(params.match, handle=lib().visob_mono_matcher(self.h))

    def __del__(self):
        if getattr(self, 'h', None):
            lib().visob_mono_destroy(self.h)
            self.h = None

    def process(self, I, replace=False):
        I = np.ascontiguousarray(I, np.uint8)
        return bool(lib().visob_mono_process(self.h, _p(I), _p(_dims(I)), int(replace)))

    def process_matches(self, matches):
        m = np.ascontiguousarray(matches, dtype=P_MATCH)
        return bool(lib().visob_mono_process_matches(self.h, _p(m), len(m)))

    def motion(self):
        out = np.zeros((4, 4))
        lib().visob_mono_get_motion(self.h, _p(out))
        return out

    def matches(self):
        n = lib().visob_mono_get_matches(self.h, None, 0)
        out = np.zeros(n, P_MATCH)
        if n:
            lib().visob_mono_get_matches(self.h, _p(out), n)
        return out

    def inliers(self):
        n = lib().visob_mono_get_inliers(self.h, None, 0)
        out = np.zeros(n, np.int32)
        if n:
            lib().visob_mono_get_inliers(self.h, _p(out), n)
        return out

    def F(self):
        F = np.zeros((3, 3))
        return F if lib().visob_mono_get_F(self.h, _p(F)) else None

    def samples(self):
        n = lib().visob_mono_get_samples(self.h, None, 0)
        out = np.zeros(n, np.int32)
        if n:
            lib().visob_mono_get_samples(self.h, _p(out), n)
        return out.reshape(-1, 8)


class Stereo:
    def __init__(self, params):
        self.params = params
        self.h = C.c_void_p(lib().visob_stereo_create(C.byref(params)))

    def __del__(self):
        if getattr(self, 'h', None):
            lib().visob_stereo_destroy(self.h)
            self.h = None

    def process(self, I1, I2, replace=False):
        I1 = np.ascontiguousarray(I1, np.uint8); I2 = np.ascontiguousarray(I2, np.uint8)
        return bool(lib().visob_stereo_process(self.h, _p(I1), _p(I2), _p(_dims(I1)), int(replace)))

    def process_matches(self, matches):
        m = np.ascontiguousarray(matches, dtype=P_MATCH)
        return bool(lib().visob_stereo_process_matches(self.h, _p(m), len(m)))

    def motion(self):
        out = np.zeros((4, 4))
        lib().visob_stereo_get_motion(self.h, _p(out))
        return out

    def matches(self):
        n = lib().visob_stereo_get_matches(self.h, None, 0)
        out = np.zeros(n, P_MATCH)
        if n:
            lib().visob_stereo_get_matches(self.h, _p(out), n)
        return out

    def inliers(self):
        n = lib().visob_stereo_get_inliers(self.h, None, 0)
        out = np.zeros(n, np.int32)
        if n:
            lib().visob_stereo_get_inliers(self.h, _p(out), n)
        return out

    def samples(self):
        """The RANSAC sample table of the last estimate (ransac_iters x 3)."""
        n = lib().visob_stereo_get_samples(self.h, None, 0)
        out = np.zeros(n, np.int32)
        if n:
            lib().visob_stereo_get_samples(self.h, _p(out), n)
        return out.reshape(-1, 3)

    def batch_prepare(self, matches):
        """First half of process_matches for a device estimate: keeps the matches and draws the sample table (samples()).
        False if there are fewer than 6 matches."""
        m = np.ascontiguousarray(matches, dtype=P_MATCH)
        return bool(lib().visob_stereo_batch_prepare(self.h, _p(m), len(m)))

    def batch_finish(self, tr6, ok, mask):
        """Second half: the results of visocu_stereo_motion for the prepared matches; returns what process_matches returns."""
        tr6 = np.ascontiguousarray(tr6, np.float64); mask = np.ascontiguousarray(mask, np.uint8)
        return bool(lib().visob_stereo_batch_finish(self.h, _p(tr6), int(ok), _p(mask)))


class Sfm:
    """StructureFromMotion facade (host/sfm.h)."""

    def __init__(self, params, width, height):
        self.dims = np.array([width, height, width], np.int32)
        self.h = C.c_void_p(lib().visob_sfm_create(C.byref(params), _p(self.dims)))

    def __del__(self):
        if getattr(self, 'h', None):
            lib().visob_sfm_destroy(self.h)
            self.h = None

    def update(self, img):
        img = np.ascontiguousarray(img, np.uint8)
        lib().visob_sfm_update(self.h, _p(img))

    def points(self):
        n = lib().visob_sfm_get_points(self.h, None, 0)
        out = np.zeros((n, 3), np.float32)
        if n:
            lib().visob_sfm_get_points(self.h, _p(out), n)
        return out

    def pose(self):
        out = np.zeros((4, 4))
        lib().visob_sfm_get_pose(self.h, _p(out))
        return out


def set_pipeline_depth(depth):
    """Steps that Runner.run keeps in flight per sequence (1 = synchronous, default and maximum 3)."""
    lib().visob_set_pipeline_depth(int(depth))


def delaunay(x, y):
    x = np.ascontiguousarray(x, np.int32); y = np.ascontiguousarray(y, np.int32)
    cap = 2 * len(x) + 8
    tri = np.zeros((cap, 3), np.int32)
    n = lib().visob_delaunay(_p(x), _p(y), len(x), _p(tri), cap)
    return tri[:n].copy()


def delaunay_edges(x, y, ctx=None):
    """(a, b, t) per undirected edge of the triangulation, t = triangles it bounds.  ctx: a visocu_py.Context - inputs of more
    than 6000 points then build the lower levels of their tree on the device.  Returns (edges, nodes built on the device)."""
    import ctypes as C
    x = np.ascontiguousarray(x, np.int32); y = np.ascontiguousarray(y, np.int32)
    cap = 3 * len(x) + 8
    e = np.zeros((cap, 3), np.int32)
    nodes = C.c_int64(0)
    L = lib()
    L.visob_delaunay_edges.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    n = L.visob_delaunay_edges(ctx.h if ctx is not None else None, _p(x), _p(y), len(x), _p(e), cap, C.byref(nodes))
    return e[:n].copy(), int(nodes.value)


def svd(A):
    A = np.ascontiguousarray(A, np.float64)
    m, n = A.shape
    U = np.zeros((m, m)); W = np.zeros(min(m, n)); V = np.zeros((n, n))
    lib().visob_svd(_p(A), m, n, _p(U), _p(W), _p(V))
    return U, W, V


class Runner:
    """S independent sequences on one GPU driven by `threads` host workers (mode 0: Matcher, 1: mono odometry,
    2: stereo odometry - see Runner.stereo)."""

    def __init__(self, device, n_sequences, threads, mode, method, mono_params):
        self.S = n_sequences
        self.mp = mono_params
        self.h = C.c_void_p(lib().visob_runner_create(device, n_sequences, threads, mode, method, C.byref(mono_params)))

    @classmethod
    def stereo(cls, device, n_sequences, threads, stereo_params):
        """Stereo odometry runner: one VisualOdometryStereo per sequence; step() / run() take left and right images."""
        r = cls.__new__(cls)
        r.S = n_sequences
        r.mp = stereo_params
        r.h = C.c_void_p(lib().visob_runner_create_stereo(device, n_sequences, threads, C.byref(stereo_params)))
        return r

    def close(self):
        if getattr(self, 'h', None):
            lib().visob_runner_destroy(self.h)
            self.h = None

    __del__ = close

    def step(self, ptrs, dims, ptrs2=None, on_device=False, bucket=False):
        S = self.S
        a = (C.c_void_p * S)(*ptrs)
        b = (C.c_void_p * S)(*ptrs2) if ptrs2 is not None else None
        nm = np.zeros(S, np.int32); ok = np.zeros(S, np.int32)
        d = np.ascontiguousarray(dims, np.int32)
        secs = lib().visob_runner_step(self.h, a, b, _p(d), int(on_device), int(bucket), _p(nm), _p(ok))
        return secs, nm, ok

    def run(self, ptr_steps, dims, ptr_steps2=None, on_device=False, bucket=False):
        """K steps with no barrier in between; ptr_steps: K lists of S pointers."""
        K, S = len(ptr_steps), self.S
        a = (C.c_void_p * (K * S))(*[p for row in ptr_steps for p in row])
        b = (C.c_void_p * (K * S))(*[p for row in ptr_steps2 for p in row]) if ptr_steps2 is not None else None
        nm = np.zeros((K, S), np.int32); ok = np.zeros((K, S), np.int32)
        d = np.ascontiguousarray(dims, np.int32)
        secs = lib().visob_runner_run(self.h, K, a, b, _p(d), int(on_device), int(bucket), _p(nm), _p(ok))
        return secs, nm, ok

    def matches(self, seq):
        n = lib().visob_runner_get_matches(self.h, seq, None, 0)
        out = np.zeros(max(n, 0), P_MATCH)
        if n > 0:
            lib().visob_runner_get_matches(self.h, seq, _p(out), n)
        return out

    def motion(self, seq):
        out = np.zeros((4, 4))
        lib().visob_runner_get_motion(self.h, seq, _p(out))
        return out

    def inliers(self, seq):
        """Inlier indices of the sequence's last motion estimate (odometry modes)."""
        n = lib().visob_runner_get_inliers(self.h, seq, None, 0)
        out = np.zeros(max(n, 0), np.int32)
        if n > 0:
            lib().visob_runner_get_inliers(self.h, seq, _p(out), n)
        return out

    def launches(self):
        return int(lib().visob_runner_launches(self.h))

    def outlier_stats(self):
        """Device outlier removal: lists handled / declined and mean kernel phase times (microseconds)."""
        out = np.zeros(8, np.uint64)
        lib().visob_runner_outlier_stats(self.h, _p(out))
        n = max(int(out[0]), 1)
        nodes = np.zeros(2, np.uint64)
        lib().visob_runner_node_stats(self.h, _p(nodes))
        return dict(lists=int(out[0]), declined=int(out[1]), declined_lists_built_in_device_nodes=int(nodes[0]), device_nodes=int(nodes[1]), declined_too_long=int(out[2]), declined_duplicates=int(out[3]),
                    declined_guard=int(out[4]), sort_partition_us=round(float(out[5]) / n / 1e3, 1),
                    build_us=round(float(out[6]) / n / 1e3, 1), vote_us=round(float(out[7]) / n / 1e3, 1))

    def transfer_bytes(self):
        a = C.c_uint64(); b = C.c_uint64()
        lib().visob_runner_transfer_bytes(self.h, C.byref(a), C.byref(b))
        return a.value, b.value
