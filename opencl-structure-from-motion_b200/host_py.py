"""ctypes binding of the C++ host layer (libviso_b200.so: Matcher, filter::, VisualOdometryMono, the sharded
sequence runner) for the tests and bench.py.  Plumbing only."""
import ctypes as C
import os
import numpy as np

from visocu_py import Camera, Params, P_MATCH, RECON_FRAME, RECON_TRACK, ReconJob, VisocuError

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


class Rectification(C.Structure):
    """Rectification (host/rectify.h): n_cams cameras (left, right) for raw src_w x src_h images, rectified to out_w x out_h;
    base = rectified baseline (stereo odometry)."""
    _fields_ = [('n_cams', C.c_int32), ('cams', Camera * 2), ('src_w', C.c_int32), ('src_h', C.c_int32),
                ('out_w', C.c_int32), ('out_h', C.c_int32), ('base', C.c_double)]

    def __init__(self, cams, src_w, src_h, out_w, out_h, base=0.0):
        super().__init__()
        self.n_cams = len(cams)
        for k, c in enumerate(cams):
            self.cams[k] = c
        self.src_w, self.src_h, self.out_w, self.out_h, self.base = int(src_w), int(src_h), int(out_w), int(out_h), float(base)


def stereo_rectify(cam0, cam1, R, T, out_w, out_h):
    """Bouguet's rectification of a rig whose camera 1 sees X1 = R X0 + T (host/rectify.h): (rect0, rect1, base), the
    input cameras with their rectifying rotation and common rectified projection."""
    R = np.ascontiguousarray(R, np.float64).reshape(9); T = np.ascontiguousarray(T, np.float64).reshape(3)
    r0, r1, base = Camera(1, 1, 0, 0), Camera(1, 1, 0, 0), C.c_double()
    lib().visob_stereo_rectify(C.byref(cam0), C.byref(cam1), _p(R), _p(T), int(out_w), int(out_h), C.byref(r0), C.byref(r1),
                               C.byref(base))
    return r0, r1, base.value


def rectify_map(cam, src_w, src_h, out_w, out_h):
    """The map visocu_set_rectification builds, computed on the host: (out_h, out_w, 2) int32 in 1/32 pixel; raises
    VisocuError for what the library rejects."""
    out = np.zeros((out_h, out_w, 2), np.int32) if out_w > 0 and out_h > 0 else None
    why = C.create_string_buffer(256)
    rc = lib().visob_rectify_map(C.byref(cam), int(src_w), int(src_h), int(out_w), int(out_h), _p(out), why)
    if rc:
        raise VisocuError('rectify_map: %d %s' % (rc, why.value.decode()))
    return out


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise VisocuError(LIB_PATH + ' is missing: run __graft_entry__.build()')
        L = C.CDLL(LIB_PATH)
        for name in ('visob_matcher_create', 'visob_mono_create', 'visob_mono_matcher', 'visob_runner_create', 'visob_runner_create_stereo', 'visob_runner_create_sfm', 'visob_stereo_create', 'visob_recon_create', 'visob_sfm_create',
                     'visob_matcher_context', 'visob_runner_create_stereo_sfm', 'visob_stereo_sfm_create', 'visob_stereo_sfm_odometry',
                     'visob_stereo_matcher'):
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

    def set_rectification(self, rect):
        """Raw images of rect.src_w x rect.src_h from now on; False (nothing changed) after the first push."""
        return bool(lib().visob_matcher_set_rectification(self.h, C.byref(rect)))

    def set_intrinsics(self, f, cu, cv, base):
        lib().visob_matcher_set_intrinsics(self.h, C.c_double(f), C.c_double(cu), C.c_double(cv), C.c_double(base))

    def bucket(self, max_features, bw, bh):
        lib().visob_matcher_bucket(self.h, max_features, C.c_float(bw), C.c_float(bh))

    def stereo_size(self):
        """(w, h) of the current stereo pair, or None after a mono push or a failed one."""
        f = np.zeros(2, np.int32); wh = np.zeros(2, np.int32)
        return tuple(wh.tolist()) if lib().visob_matcher_stereo_pair(self.h, _p(f), _p(wh)) else None

    def disparity(self, params=None):
        """Matcher::computeDisparity of the current stereo pair: an (h, w) int16 map in 1/16 pixel (-1 = invalid), or
        None after a mono push or when the device call fails."""
        wh = self.stereo_size()
        if wh is None:
            return None
        out = np.zeros((wh[1], wh[0]), np.int16)
        ok = lib().visob_matcher_disparity(self.h, C.byref(_sgm(params)), _p(out), 0)
        return out if ok else None

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

    def set_rectification(self, rect):
        """Raw images, calibration = rectified projection of camera 0; False (nothing changed) after the first frame."""
        return bool(lib().visob_mono_set_rectification(self.h, C.byref(rect)))

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
    def __init__(self, params, handle=None, owner=None):
        """handle: an existing VisualOdometryStereo that `owner` keeps alive (StereoSfm.odometry); not destroyed here."""
        self.params = params
        self.owner = owner
        self.owned = handle is None
        self.h = C.c_void_p(lib().visob_stereo_create(C.byref(params)) if handle is None else handle)

    def __del__(self):
        if getattr(self, 'owned', False) and self.h:
            lib().visob_stereo_destroy(self.h)
            self.h = None

    def process(self, I1, I2, replace=False):
        I1 = np.ascontiguousarray(I1, np.uint8); I2 = np.ascontiguousarray(I2, np.uint8)
        return bool(lib().visob_stereo_process(self.h, _p(I1), _p(I2), _p(_dims(I1)), int(replace)))

    def process_matches(self, matches):
        m = np.ascontiguousarray(matches, dtype=P_MATCH)
        return bool(lib().visob_stereo_process_matches(self.h, _p(m), len(m)))

    def set_rectification(self, rect):
        """Raw stereo pairs (rect.n_cams = 2), calibration and base from rect; False (nothing changed) after the first frame."""
        return bool(lib().visob_stereo_set_rectification(self.h, C.byref(rect)))

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

    def matcher(self):
        """The odometry's Matcher (a view, kept alive by this object)."""
        m = Matcher(self.params, handle=lib().visob_stereo_matcher(self.h))
        m.owner = self
        return m

    def disparity(self, params=None):
        """Dense disparity of the last stereo pair (Matcher.disparity)."""
        return self.matcher().disparity(params)

    def batch_prepare(self, matches):
        """First half of process_matches for a device estimate: keeps the matches and draws the sample table (samples()).
        False if there are fewer than 6 matches."""
        m = np.ascontiguousarray(matches, dtype=P_MATCH)
        return bool(lib().visob_stereo_batch_prepare(self.h, _p(m), len(m)))

    def batch_finish(self, tr6, ok, mask):
        """Second half: the results of visocu_stereo_motion for the prepared matches; returns what process_matches returns."""
        tr6 = np.ascontiguousarray(tr6, np.float64); mask = np.ascontiguousarray(mask, np.uint8)
        return bool(lib().visob_stereo_batch_finish(self.h, _p(tr6), int(ok), _p(mask)))


class Recon:
    """Reconstruction (host/reconstruction.h): update() on the host, or its two halves around an evaluation of the finished
    tracks elsewhere (batch_prepare, batch_job, then host_eval or visocu_py.Context.recon_points, then batch_finish)."""

    def __init__(self, f, cu, cv):
        self.h = C.c_void_p(lib().visob_recon_create())
        lib().visob_recon_set_calibration(self.h, C.c_double(f), C.c_double(cu), C.c_double(cv))

    def __del__(self):
        if getattr(self, 'h', None):
            lib().visob_recon_destroy(self.h)
            self.h = None

    def update(self, matches, tr, point_type=1, min_track_length=2, max_dist=30.0, min_angle=2.0):
        m = np.ascontiguousarray(matches, P_MATCH); tr = np.ascontiguousarray(tr, np.float64)
        lib().visob_recon_update(self.h, _p(m), len(m), _p(tr), int(point_type), int(min_track_length), C.c_double(max_dist),
                                 C.c_double(min_angle))

    def batch_prepare(self, matches, tr, point_type=1, min_track_length=2, max_dist=30.0, min_angle=2.0):
        """update()'s bookkeeping; returns the number of finished tracks to evaluate."""
        m = np.ascontiguousarray(matches, P_MATCH); tr = np.ascontiguousarray(tr, np.float64)
        return lib().visob_recon_batch_prepare(self.h, _p(m), len(m), _p(tr), int(point_type), int(min_track_length),
                                               C.c_double(max_dist), C.c_double(min_angle))

    def batch_prepare_tracks(self, matches, tr, point_type=1, min_track_length=2, max_dist=30.0, min_angle=2.0):
        """batch_prepare without moving the stored points (for points kept in a device store, visocu_py.Context.recon_update);
        returns the number of finished tracks to evaluate."""
        m = np.ascontiguousarray(matches, P_MATCH); tr = np.ascontiguousarray(tr, np.float64)
        return lib().visob_recon_batch_prepare_tracks(self.h, _p(m), len(m), _p(tr), int(point_type), int(min_track_length),
                                                      C.c_double(max_dist), C.c_double(min_angle))

    def batch_job(self):
        """The prepared job as a dict (frames, tracks, cam_road, max_dist, min_angle, point_type), copied out."""
        job = ReconJob()
        lib().visob_recon_batch_job(self.h, C.byref(job), None, None)
        frames = np.zeros(job.n_frames, RECON_FRAME); tracks = np.zeros(job.n_tracks, RECON_TRACK)
        lib().visob_recon_batch_job(self.h, C.byref(job), _p(frames), _p(tracks))
        return dict(frames=frames, tracks=tracks, cam_road=np.array(job.cam_road[:]), max_dist=job.max_dist,
                    min_angle=job.min_angle, point_type=job.point_type)

    def host_eval(self):
        """The host functions on the prepared tracks: (status, xyz) with the meaning of visocu_recon_points."""
        job = ReconJob()
        lib().visob_recon_batch_job(self.h, C.byref(job), None, None)
        status = np.zeros(job.n_tracks, np.int32); xyz = np.zeros((job.n_tracks, 3), np.float32)
        lib().visob_recon_host_eval(self.h, _p(status), _p(xyz))
        return status, xyz

    def batch_finish(self, status, xyz):
        """Appends the points of the prepared tracks whose status is 0."""
        status = np.ascontiguousarray(status, np.int32); xyz = np.ascontiguousarray(xyz, np.float32)
        lib().visob_recon_batch_finish(self.h, _p(status), _p(xyz))

    def points(self):
        n = lib().visob_recon_get_points(self.h, None, 0)
        out = np.zeros((n, 3), np.float32)
        if n:
            lib().visob_recon_get_points(self.h, _p(out), n)
        return out


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
        """One frame; returns whether its odometry succeeded."""
        img = np.ascontiguousarray(img, np.uint8)
        return bool(lib().visob_sfm_update(self.h, _p(img)))

    def set_rectification(self, rect):
        return bool(lib().visob_sfm_set_rectification(self.h, C.byref(rect)))

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


class StereoSfm:
    """StructureFromMotionStereo facade (host/sfm.h): stereo odometry and reconstruction, both estimated on the GPU."""

    def __init__(self, params, width, height):
        self.params = params
        self.dims = np.array([width, height, width], np.int32)
        self.h = C.c_void_p(lib().visob_stereo_sfm_create(C.byref(params), _p(self.dims)))

    def __del__(self):
        if getattr(self, 'h', None):
            lib().visob_stereo_sfm_destroy(self.h)
            self.h = None

    def update(self, left, right):
        """One stereo pair; returns whether its odometry (and, after the first frame, its reconstruction) succeeded."""
        left = np.ascontiguousarray(left, np.uint8); right = np.ascontiguousarray(right, np.uint8)
        return bool(lib().visob_stereo_sfm_update(self.h, _p(left), _p(right)))

    def set_rectification(self, rect):
        """Raw stereo pairs for update(); False (nothing changed) after the first frame."""
        return bool(lib().visob_stereo_sfm_set_rectification(self.h, C.byref(rect)))

    def points(self):
        n = lib().visob_stereo_sfm_get_points(self.h, None, 0)
        out = np.zeros((n, 3), np.float32)
        if n:
            lib().visob_stereo_sfm_get_points(self.h, _p(out), n)
        return out

    def pose(self):
        out = np.zeros((4, 4))
        lib().visob_stereo_sfm_get_pose(self.h, _p(out))
        return out

    def odometry(self):
        """The facade's VisualOdometryStereo (matches, inliers, motion of the last frame) as a Stereo view."""
        return Stereo(self.params, handle=lib().visob_stereo_sfm_odometry(self.h), owner=self)

    def device_points(self):
        """(device address, count) of the points in the facade's device store, valid until the next update."""
        d = C.c_void_p(); n = C.c_int64()
        lib().visob_stereo_sfm_device_points(self.h, C.byref(d), C.byref(n))
        return d.value or 0, n.value

    def points_tensor(self):
        """The points as a float32 CUDA tensor (n x 3) of its own (a copy of the device store)."""
        return _points_tensor(*self.device_points())

    def disparity_tensor(self, params=None):
        """Dense disparity of the last pair as an (h, w) int16 CUDA tensor, written in place by the device; None after a
        failed frame."""
        import torch
        wh = self.odometry().matcher().stereo_size()
        if wh is None:
            return None
        out = torch.empty((wh[1], wh[0]), dtype=torch.int16, device='cuda')
        torch.cuda.current_stream(out.device).synchronize()
        ok = lib().visob_stereo_sfm_disparity(self.h, C.byref(_sgm(params)), C.c_void_p(out.data_ptr()), 1)
        return out if ok else None


class _DevicePoints:
    """A borrowed view of n x 3 device floats for torch (__cuda_array_interface__)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = dict(shape=(n, 3), typestr='<f4', data=(ptr, False), version=3, strides=None)


class _DeviceMap:
    """A borrowed view of an (h, w) int16 device map for torch (__cuda_array_interface__)."""

    def __init__(self, ptr, w, h):
        self.__cuda_array_interface__ = dict(shape=(h, w), typestr='<i2', data=(ptr, False), version=3, strides=None)


def _sgm(params):
    import visocu_py
    return visocu_py.SgmParams() if params is None else params


def disparity_to_points(disp16, f, cu, cv, base):
    """The valid pixels (value > 0) of an (h, w) disparity map in 1/16 pixel (numpy or torch) reprojected into the left
    camera: Z = 16 f base / d, X = (u - cu) Z / f, Y = (v - cv) Z / f.  Returns an (n, 3) float32 torch tensor on the
    map's device, in row-major pixel order."""
    import torch
    d = torch.as_tensor(disp16)
    v, u = torch.nonzero(d > 0, as_tuple=True)
    Z = (16.0 * f * base) / d[v, u].to(torch.float32)
    X = (u.to(torch.float32) - cu) * Z / f
    Y = (v.to(torch.float32) - cv) * Z / f
    return torch.stack([X, Y, Z], 1)


def _points_tensor(ptr, n):
    import torch
    if n == 0:
        return torch.zeros((0, 3), dtype=torch.float32, device='cuda')
    return torch.as_tensor(_DevicePoints(ptr, n), device='cuda').clone()


def affine_points(M, xyz):
    """Reconstruction's affineTransform (host/reconstruction.cpp) on every point: rows 0..2 of the 4x4 M applied to (p, 1)."""
    M = np.ascontiguousarray(M, np.float64); a = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
    out = np.zeros_like(a)
    lib().visob_affine_points(_p(M), _p(a), _p(out), C.c_int64(len(a)))
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
    2: stereo odometry - see Runner.stereo, 3: structure from motion - see Runner.sfm, 4: stereo structure from motion -
    see Runner.stereo_sfm)."""

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

    @classmethod
    def sfm(cls, device, n_sequences, threads, mono_params):
        """Structure-from-motion runner (mode 3): per sequence what the StructureFromMotion facade does (Sfm), with the
        finished tracks of each worker's sequences reconstructed by one device call per step; steps are synchronous."""
        r = cls.__new__(cls)
        r.S = n_sequences
        r.mp = mono_params
        r.h = C.c_void_p(lib().visob_runner_create_sfm(device, n_sequences, threads, C.byref(mono_params)))
        return r

    @classmethod
    def stereo_sfm(cls, device, n_sequences, threads, stereo_params):
        """Stereo structure-from-motion runner (mode 4): per sequence what the StereoSfm facade does, with one
        visocu_stereo_motion and one visocu_recon_points per worker and step; step() / run() take left and right images
        (without right images they return -1 and do nothing) and are synchronous."""
        r = cls.__new__(cls)
        r.S = n_sequences
        r.mp = stereo_params
        r.h = C.c_void_p(lib().visob_runner_create_stereo_sfm(device, n_sequences, threads, C.byref(stereo_params)))
        return r

    def close(self):
        if getattr(self, 'h', None):
            lib().visob_runner_destroy(self.h)
            self.h = None

    __del__ = close

    def set_rectification(self, rect):
        """Raw images for step() / run() (dims = the raw size); False (nothing changed) after the first step."""
        return bool(lib().visob_runner_set_rectification(self.h, C.byref(rect)))

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

    def points(self, seq):
        """The sequence's reconstructed points (structure-from-motion modes)."""
        n = lib().visob_runner_get_points(self.h, seq, None, 0)
        out = np.zeros((max(n, 0), 3), np.float32)
        if n > 0:
            lib().visob_runner_get_points(self.h, seq, _p(out), n)
        return out

    def device_points(self, seq):
        """(device address, count) of the sequence's points in its device store (structure-from-motion modes), valid
        until the next step."""
        d = C.c_void_p(); n = C.c_int64()
        if lib().visob_runner_device_points(self.h, seq, C.byref(d), C.byref(n)):
            raise VisocuError('device_points: not a structure-from-motion runner, or no sequence %d' % seq)
        return d.value or 0, n.value

    def set_disparity(self, params):
        """Stereo modes: compute every sequence's dense disparity at each following step (SgmParams), or stop (None).
        False for another mode or parameters out of range."""
        return bool(lib().visob_runner_set_disparity(self.h, None if params is None else C.byref(params)))

    def disparity_tensor(self, seq):
        """The sequence's disparity map of the last step as an (h, w) int16 CUDA tensor (a copy), or None without one."""
        import torch
        d = C.c_void_p(); w = C.c_int32(); h = C.c_int32()
        if lib().visob_runner_device_disparity(self.h, seq, C.byref(d), C.byref(w), C.byref(h)):
            return None
        return torch.as_tensor(_DeviceMap(d.value, w.value, h.value), device='cuda').clone()

    def points_tensor(self, seq):
        """The sequence's points as a float32 CUDA tensor (n x 3) on the runner's device, a copy of its own."""
        return _points_tensor(*self.device_points(seq))

    def pose(self, seq):
        """The sequence's accumulated pose, first camera -> current camera (structure-from-motion modes)."""
        out = np.zeros((4, 4))
        lib().visob_runner_get_pose(self.h, seq, _p(out))
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
