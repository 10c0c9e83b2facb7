"""ctypes binding of include/visocu.h (libvisocu.so) for the parity tests and bench.py.

This is plumbing, not product logic: the product is the CUDA library and the C++ host layer
(libviso_b200.so, see host_py.py).  Importing this module never builds or falls back to anything --
if the shared library is missing or no sm_100 GPU is present, the calls fail loudly.
"""
import ctypes as C
import os
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libvisocu.so')

P_MATCH = np.dtype([('u1p', 'f4'), ('v1p', 'f4'), ('i1p', 'i4'), ('u2p', 'f4'), ('v2p', 'f4'), ('i2p', 'i4'),
                    ('u1c', 'f4'), ('v1c', 'f4'), ('i1c', 'i4'), ('u2c', 'f4'), ('v2c', 'f4'), ('i2c', 'i4')])
RANGE = np.dtype([('u_min', 'f4', 4), ('u_max', 'f4', 4), ('v_min', 'f4', 4), ('v_max', 'f4', 4)])
QUAD = np.dtype([('f1p', 'i4'), ('f2p', 'i4'), ('f1c', 'i4'), ('f2c', 'i4')])


RECON_FRAME = np.dtype([('proj', 'f8', 12), ('inv', 'f8', 12), ('center', 'f8', 3)])        # visocu_recon_frame
RECON_TRACK = np.dtype([('first', 'i4'), ('n_obs', 'i4'), ('u', 'f4', 6), ('v', 'f4', 6)])   # visocu_recon_track


class ReconJob(C.Structure):
    """visocu_recon_job: the finished tracks of one Reconstruction update and the window they refer to."""
    _fields_ = [('frames', C.c_void_p), ('n_frames', C.c_int32), ('tracks', C.c_void_p), ('n_tracks', C.c_int32),
                ('cam_road', C.c_double * 12), ('max_dist', C.c_double), ('min_angle', C.c_double), ('point_type', C.c_int32)]


class StereoMotionParams(C.Structure):
    """visocu_stereo_params: calibration and RANSAC settings of VisualOdometryStereo::parameters."""
    _fields_ = [(n, C.c_double) for n in ('f', 'cu', 'cv', 'base', 'inlier_threshold')] + \
               [('ransac_iters', C.c_int32), ('reweighting', C.c_int32)]


class Params(C.Structure):
    """Matcher::parameters (reference matcher.h:42-69): same order, same defaults."""
    _fields_ = [(n, C.c_int32) for n in ('nms_n', 'nms_tau', 'match_binsize', 'match_radius', 'match_disp_tolerance',
                                         'outlier_disp_tolerance', 'outlier_flow_tolerance', 'multi_stage',
                                         'half_resolution', 'refinement')] + \
               [(n, C.c_double) for n in ('f', 'cu', 'cv', 'base')]

    def __init__(self, **kw):
        super().__init__()
        d = dict(nms_n=3, nms_tau=50, match_binsize=50, match_radius=200, match_disp_tolerance=2,
                 outlier_disp_tolerance=5, outlier_flow_tolerance=5, multi_stage=1, half_resolution=1,
                 refinement=1, f=1.0, cu=0.0, cv=0.0, base=1.0)
        d.update(kw)
        for k, v in d.items():
            setattr(self, k, v)


class Camera(C.Structure):
    """visocu_camera: raw pinhole K, radial-tangential distortion, rectifying rotation R (row-major) and the rectified
    projection f, cu, cv (host/rectify.h).  Defaults: no distortion, R = I, f = fy, (cu, cv) = (cx, cy)."""
    _fields_ = [(n, C.c_double) for n in ('fx', 'fy', 'cx', 'cy', 'k1', 'k2', 'p1', 'p2', 'k3')] + \
               [('R', C.c_double * 9)] + [(n, C.c_double) for n in ('f', 'cu', 'cv')]

    def __init__(self, fx, fy, cx, cy, k1=0.0, k2=0.0, p1=0.0, p2=0.0, k3=0.0, R=None, f=None, cu=None, cv=None):
        super().__init__()
        for k, v in dict(fx=fx, fy=fy, cx=cx, cy=cy, k1=k1, k2=k2, p1=p1, p2=p2, k3=k3).items():
            setattr(self, k, float(v))
        self.R[:] = [float(x) for x in np.asarray(np.eye(3) if R is None else R, np.float64).reshape(9)]
        self.f = float(fy if f is None else f)
        self.cu = float(cx if cu is None else cu)
        self.cv = float(cy if cv is None else cv)

    def rotation(self):
        return np.array(self.R[:], np.float64).reshape(3, 3)


class SgmParams(C.Structure):
    """visocu_sgm_params: semi-global matching settings of visocu_disparity (include/visocu.h)."""
    _fields_ = [(n, C.c_int32) for n in ('max_disp', 'paths', 'p1', 'p2', 'uniqueness', 'lr_max_diff', 'subpixel')]

    def __init__(self, **kw):
        super().__init__()
        d = dict(max_disp=128, paths=8, p1=10, p2=120, uniqueness=95, lr_max_diff=1, subpixel=1)
        d.update(kw)
        for k, v in d.items():
            setattr(self, k, int(v))


class VisocuError(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise VisocuError(LIB_PATH + ' is missing: run __graft_entry__.build() (make -C opencl-structure-from-motion_b200)')
        _lib = C.CDLL(LIB_PATH)
        _lib.visocu_last_error.restype = C.c_char_p
        _lib.visocu_last_error.argtypes = [C.c_void_p]
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    def __init__(self, device=0):
        self.h = C.c_void_p()
        rc = lib().visocu_create(device, C.byref(self.h))
        if rc:
            raise VisocuError('visocu_create: %d %s' % (rc, lib().visocu_last_error(None).decode()))
        self.params = None
        self.dims = None
        self.device = device

    def close(self):
        if getattr(self, 'h', None) and self.h.value:
            lib().visocu_destroy(self.h)
            self.h = C.c_void_p()

    __del__ = close

    def _ck(self, rc, what):
        if rc:
            raise VisocuError('%s: %d %s' % (what, rc, lib().visocu_last_error(self.h).decode()))

    def device_info(self):
        sm = C.c_int32(); ma = C.c_int32(); mi = C.c_int32(); name = C.create_string_buffer(64)
        self._ck(lib().visocu_device_info(self.h, C.byref(sm), C.byref(ma), C.byref(mi), name), 'device_info')
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), name=name.value.decode())

    def configure(self, params, width, height, n_frames):
        """params.match_radius is taken as given: halve it yourself for half_resolution (matcher.cpp:59-60)."""
        self._ck(lib().visocu_configure(self.h, C.byref(params), width, height, n_frames), 'configure')
        self.params, self.dims, self.n_frames = params, (width, height), n_frames

    def sync(self):
        self._ck(lib().visocu_sync(self.h), 'sync')

    def timer_start(self):
        self._ck(lib().visocu_timer_start(self.h), 'timer_start')

    def timer_stop(self):
        ms = C.c_float()
        self._ck(lib().visocu_timer_stop(self.h, C.byref(ms)), 'timer_stop')
        return ms.value

    def launch_count(self):
        n = C.c_uint64()
        self._ck(lib().visocu_launch_count(self.h, C.byref(n)), 'launch_count')
        return n.value

    def transfer_bytes(self):
        a = C.c_uint64(); b = C.c_uint64()
        self._ck(lib().visocu_transfer_bytes(self.h, C.byref(a), C.byref(b)), 'transfer_bytes')
        return a.value, b.value

    def profile(self, enable=True):
        self._ck(lib().visocu_profile(self.h, int(enable)), 'profile')

    def profile_read(self):
        ms = C.c_double(); n = C.c_uint64(); f = C.c_uint64()
        self._ck(lib().visocu_profile_read(self.h, C.byref(ms), C.byref(n), C.byref(f)), 'profile_read')
        return ms.value, n.value, f.value

    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(lib().visocu_device_alloc(self.h, C.c_size_t(nbytes), C.byref(p)), 'device_alloc')
        return p.value

    def device_free(self, ptr):
        self._ck(lib().visocu_device_free(self.h, C.c_void_p(ptr)), 'device_free')

    def host_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(lib().visocu_host_alloc(self.h, C.c_size_t(nbytes), C.byref(p)), 'host_alloc')
        return p.value

    def host_free(self, ptr):
        self._ck(lib().visocu_host_free(self.h, C.c_void_p(ptr)), 'host_free')

    def memcpy_h2d(self, dptr, arr):
        arr = np.ascontiguousarray(arr)
        self._ck(lib().visocu_memcpy_h2d(self.h, C.c_void_p(dptr), _p(arr), C.c_size_t(arr.nbytes)), 'memcpy_h2d')

    # ---- features
    def push_frames(self, frames, imgs=None, ptrs=None, bpl_in=None, on_device=False, want_counts=True):
        frames = np.ascontiguousarray(frames, np.int32)
        n = len(frames)
        if ptrs is None:
            imgs = [np.ascontiguousarray(i, np.uint8) for i in imgs]
            ptrs = [i.ctypes.data for i in imgs]
            bpl_in = imgs[0].shape[1] if bpl_in is None else bpl_in
        arr = (C.c_void_p * n)(*ptrs)
        ns = np.zeros(n, np.int32); nd = np.zeros(n, np.int32)
        self._ck(lib().visocu_push_frames(self.h, n, _p(frames), arr, int(bpl_in), int(on_device),
                                          _p(ns) if want_counts else None, _p(nd) if want_counts else None), 'push_frames')
        return ns, nd

    def set_rectification(self, cams, src_w, src_h):
        """visocu_set_rectification: maps for raw src_w x src_h images (cams: 0, 1 or 2 Camera)."""
        arr = (Camera * max(1, len(cams)))(*cams)
        self._ck(lib().visocu_set_rectification(self.h, len(cams), arr if cams else None, int(src_w), int(src_h)),
                 'set_rectification')

    def push_frames_rectified(self, frames, cams, imgs=None, ptrs=None, bpl_in=None, on_device=False, want_counts=True):
        """visocu_push_frames_rectified: raw image k resampled with map cams[k] into frame frames[k]."""
        frames = np.ascontiguousarray(frames, np.int32)
        cams = np.ascontiguousarray(cams, np.int32)
        n = len(frames)
        if ptrs is None:
            imgs = [np.ascontiguousarray(i, np.uint8) for i in imgs]
            ptrs = [i.ctypes.data for i in imgs]
            bpl_in = imgs[0].shape[1] if bpl_in is None else bpl_in
        arr = (C.c_void_p * n)(*ptrs)
        ns = np.zeros(n, np.int32); nd = np.zeros(n, np.int32)
        self._ck(lib().visocu_push_frames_rectified(self.h, n, _p(frames), arr, _p(cams), int(bpl_in), int(on_device),
                                                    _p(ns) if want_counts else None, _p(nd) if want_counts else None),
                 'push_frames_rectified')
        return ns, nd

    def rectify_map(self, cam, width, height):
        """The map of camera `cam` for width x height output images: (height, width, 2) int32, x and y in 1/32 pixel."""
        out = np.zeros((height, width, 2), np.int32)
        self._ck(lib().visocu_get_rectify_map(self.h, int(cam), _p(out), C.c_size_t(out.size)), 'get_rectify_map')
        return out

    def features(self, frame, pass_):
        n = C.c_int32()
        self._ck(lib().visocu_get_features(self.h, frame, pass_, None, 0, C.byref(n)), 'get_features')
        out = np.zeros((n.value, 12), np.int32)
        if n.value:
            self._ck(lib().visocu_get_features(self.h, frame, pass_, _p(out), n.value, C.byref(n)), 'get_features')
        return out

    def plane(self, frame, which):
        dims = np.zeros(3, np.int32)
        self._ck(lib().visocu_get_plane(self.h, frame, which, None, C.c_size_t(0), _p(dims)), 'get_plane')
        w, h, bpl = dims.tolist()
        out = np.zeros((h, bpl), np.uint8)
        self._ck(lib().visocu_get_plane(self.h, frame, which, _p(out), C.c_size_t(out.nbytes), _p(dims)), 'get_plane')
        return out, (w, h, bpl)

    def _disparity(self, left, right, params, ptrs, on_device):
        left = np.ascontiguousarray(left, np.int32); right = np.ascontiguousarray(right, np.int32)
        n = len(left)
        params = SgmParams() if params is None else params
        arr = (C.c_void_p * max(n, 1))(*ptrs)
        self._ck(lib().visocu_disparity(self.h, n, _p(left), _p(right), C.byref(params), arr, int(on_device)), 'disparity')

    def disparity(self, left, right, params=None):
        """visocu_disparity of frames left[k] against right[k]: a list of (h, w) int16 maps in 1/16 pixel (-1 = invalid)."""
        w, h = self.dims
        outs = [np.zeros((h, w), np.int16) for _ in range(len(left))]
        self._disparity(left, right, params, [o.ctypes.data for o in outs], 0)
        return outs

    def disparity_tensor(self, left, right, params=None):
        """The same maps as one int16 CUDA tensor (n, h, w), written by the kernels in place."""
        import torch
        w, h = self.dims
        out = torch.empty((len(left), h, w), dtype=torch.int16, device='cuda:%d' % self.device)
        torch.cuda.current_stream(out.device).synchronize()     # the memory may still be in use by torch's stream
        self._disparity(left, right, params, [out[k].data_ptr() for k in range(len(left))], 1)
        return out

    def tile_levels(self, n_launch=1):
        """(levels, pick): the fused filter + NMS kernel's tile configurations, largest first, as dicts (kx, ky, ntx, nty,
        threads), and the level a push launch of n_launch frames runs on."""
        n = C.c_int32(); out = np.zeros(15, np.int32); pick = C.c_int32()
        self._ck(lib().visocu_tile_levels(self.h, int(n_launch), C.byref(n), _p(out), C.byref(pick)), 'tile_levels')
        keys = ('kx', 'ky', 'ntx', 'nty', 'threads')
        return [dict(zip(keys, out[5 * k:5 * k + 5].tolist())) for k in range(n.value)], pick.value

    # ---- filters
    def sobel5x5(self, img):
        img = np.ascontiguousarray(img, np.uint8); h, w = img.shape
        a = np.zeros_like(img); b = np.zeros_like(img)
        self._ck(lib().visocu_sobel5x5(self.h, _p(img), _p(a), _p(b), w, h), 'sobel5x5')
        return a, b

    def sobel3x3(self, img):
        img = np.ascontiguousarray(img, np.uint8); h, w = img.shape
        a = np.zeros_like(img); b = np.zeros_like(img)
        self._ck(lib().visocu_sobel3x3(self.h, _p(img), _p(a), _p(b), w, h), 'sobel3x3')
        return a, b

    def blob5x5(self, img):
        img = np.ascontiguousarray(img, np.uint8); h, w = img.shape
        o = np.zeros((h, w), np.int16)
        self._ck(lib().visocu_blob5x5(self.h, _p(img), _p(o), w, h), 'blob5x5')
        return o

    def checkerboard5x5(self, img):
        img = np.ascontiguousarray(img, np.uint8); h, w = img.shape
        o = np.zeros((h, w), np.int16)
        self._ck(lib().visocu_checkerboard5x5(self.h, _p(img), _p(o), w, h), 'checkerboard5x5')
        return o

    def nms(self, f1, f2, w, n, tau):
        f1 = np.ascontiguousarray(f1, np.int16); f2 = np.ascontiguousarray(f2, np.int16)
        h, bpl = f1.shape
        cap = 4 * (w // (n + 1) + 1) * (h // (n + 1) + 1)
        out = np.zeros((cap, 4), np.int32); cnt = C.c_int32()
        self._ck(lib().visocu_nms(self.h, _p(f1), _p(f2), w, h, bpl, n, tau, _p(out), cap, C.byref(cnt)), 'nms')
        return out[:cnt.value].copy()

    # ---- matching
    def match(self, quads, method, pass_, ranges=None, refine=False, tr_delta=None, outliers=False):
        """quads: list of (f1p, f2p, f1c, f2c).  ranges: list of (ub*vb) RANGE arrays or None.  Returns list of P_MATCH arrays."""
        nj = len(quads)
        q = np.zeros(nj, QUAD)
        for k, t in enumerate(quads):
            q[k] = tuple(t)
        w, h = self.dims
        cap = 4 * (w // 2 + 1) * (h // 2 + 1) // 4 + 64
        outs = [np.zeros(cap, P_MATCH) for _ in range(nj)]
        optr = (C.c_void_p * nj)(*[o.ctypes.data for o in outs])
        caps = np.full(nj, cap, np.int32); nout = np.zeros(nj, np.int32)
        rptr = None
        if ranges is not None:
            ranges = [np.ascontiguousarray(r) for r in ranges]
            rptr = (C.c_void_p * nj)(*[r.ctypes.data for r in ranges])
        tptr = None
        if tr_delta is not None:
            trs = [np.ascontiguousarray(np.asarray(t, np.float64)[:3, :4]) for t in tr_delta]
            tptr = (C.c_void_p * nj)(*[t.ctypes.data for t in trs])
        done = np.zeros(nj, np.int32) if outliers else None
        self._ck(lib().visocu_match(self.h, nj, _p(q), method, pass_, int(ranges is not None), rptr, tptr, int(refine),
                                    optr, _p(caps), _p(nout), _p(done)), 'match')
        res = [outs[k][:nout[k]].copy() for k in range(nj)]
        return (res, done) if outliers else res

    def remove_outliers(self, lists, method):
        """Matcher::removeOutliers on the device for a batch of match lists.  Returns (survivor lists, status array);
        status 1 = not handled by the device path, list returned unchanged."""
        nj = len(lists)
        bufs = [np.array(l, dtype=P_MATCH, copy=True) for l in lists]
        ptr = (C.c_void_p * nj)(*[b.ctypes.data for b in bufs])
        n = np.array([len(b) for b in bufs], np.int32); nout = np.zeros(nj, np.int32); status = np.zeros(nj, np.int32)
        self._ck(lib().visocu_remove_outliers(self.h, nj, method, ptr, _p(n), _p(nout), _p(status)), 'remove_outliers')
        return [bufs[k][:nout[k]].copy() for k in range(nj)], status

    def refine(self, quad, method, matches, mode=1):
        q = np.zeros(1, QUAD); q[0] = tuple(quad)
        m = np.array(matches, dtype=P_MATCH, copy=True)
        n = C.c_int32(len(m))
        self._ck(lib().visocu_refine(self.h, _p(q), method, mode, _p(m), len(m), C.byref(n)), 'refine')
        return m[:n.value].copy()

    def match_stats(self):
        a = C.c_uint64(); b = C.c_uint64()
        self._ck(lib().visocu_match_stats(self.h, C.byref(a), C.byref(b)), 'match_stats')
        return a.value, b.value

    # ---- pose helpers
    def triangulate(self, uv, P1, P2s):
        uv = np.ascontiguousarray(uv, np.float32); N = len(uv)
        P1 = np.ascontiguousarray(P1, np.float64); P2s = np.ascontiguousarray(P2s, np.float64)
        ns = len(P2s)
        X = np.zeros((ns, 4, N)); nf = np.zeros(ns, np.int32)
        self._ck(lib().visocu_triangulate(self.h, _p(uv), N, _p(P1), _p(P2s), ns, _p(X), _p(nf)), 'triangulate')
        return X, nf

    def best_plane(self, d, threshold, weight):
        d = np.ascontiguousarray(d, np.float64); idx = C.c_int32()
        self._ck(lib().visocu_best_plane(self.h, _p(d), len(d), C.c_double(threshold), C.c_double(weight), C.byref(idx)), 'best_plane')
        return idx.value

    # ---- ransac
    def ransac(self, uv_list, samples_list, thresh=1e-5, want_all=False):
        nj = len(uv_list)
        uvs = [np.ascontiguousarray(u, np.float32) for u in uv_list]
        smp = [np.ascontiguousarray(s, np.int32) for s in samples_list]
        iters = len(smp[0])
        N = np.array([len(u) for u in uvs], np.int32)
        F = np.zeros((nj, 9)); ninl = np.zeros(nj, np.int32); best = np.zeros(nj, np.int32)
        masks = [np.zeros(len(u), np.uint8) for u in uvs]
        counts = [np.zeros(iters, np.int32) for _ in range(nj)] if want_all else None
        Fall = [np.zeros((iters, 9)) for _ in range(nj)] if want_all else None
        mk = lambda lst: (C.c_void_p * nj)(*[a.ctypes.data for a in lst]) if lst is not None else None
        self._ck(lib().visocu_ransac_F(self.h, nj, mk(uvs), _p(N), mk(smp), iters, C.c_double(thresh), _p(F), mk(masks),
                                       _p(ninl), _p(best), mk(counts), mk(Fall)), 'ransac_F')
        res = []
        for j in range(nj):
            res.append(dict(F=F[j].reshape(3, 3).copy(), n_inliers=int(ninl[j]), best_iter=int(best[j]),
                            inliers=np.nonzero(masks[j])[0].astype(np.int32),
                            counts=counts[j] if want_all else None, F_all=Fall[j].reshape(-1, 3, 3) if want_all else None))
        return res

    # ---- stereo odometry
    def stereo_motion(self, lists, samples, params, want_all=False):
        """visocu_stereo_motion for a batch of match lists (P_MATCH arrays) and their sample tables (iters x 3).  params: a
        StereoMotionParams or anything with its fields (host_py.StereoParams).  Returns one dict per job."""
        nj = len(lists)
        if not isinstance(params, StereoMotionParams):
            params = StereoMotionParams(f=params.f, cu=params.cu, cv=params.cv, base=params.base,
                                        inlier_threshold=params.inlier_threshold, ransac_iters=params.ransac_iters,
                                        reweighting=int(params.reweighting))
        ms = [np.ascontiguousarray(m, dtype=P_MATCH) for m in lists]
        smp = [np.ascontiguousarray(s, np.int32) for s in samples]
        iters = params.ransac_iters
        N = np.array([len(m) for m in ms], np.int32)
        tr = np.zeros((nj, 6)); ok = np.zeros(nj, np.int32); ninl = np.zeros(nj, np.int32); best = np.zeros(nj, np.int32)
        masks = [np.zeros(len(m), np.uint8) for m in ms]
        counts = [np.zeros(iters, np.int32) for _ in range(nj)] if want_all else None
        trall = [np.zeros((iters, 6)) for _ in range(nj)] if want_all else None
        mk = lambda lst: (C.c_void_p * nj)(*[a.ctypes.data for a in lst]) if lst is not None else None
        self._ck(lib().visocu_stereo_motion(self.h, nj, mk(ms), _p(N), mk(smp), C.byref(params), _p(tr), _p(ok), mk(masks),
                                            _p(ninl), _p(best), mk(counts), mk(trall)), 'stereo_motion')
        return [dict(ok=bool(ok[j]), tr=tr[j].copy(), mask=masks[j], inliers=np.nonzero(masks[j])[0].astype(np.int32),
                     n_inliers=int(ninl[j]), best_iter=int(best[j]), counts=counts[j] if want_all else None,
                     tr_all=trall[j] if want_all else None) for j in range(nj)]

    # ---- reconstruction
    @staticmethod
    def _job_array(jobs):
        """ReconJob array of job dicts (host_py.Recon.batch_job makes them), and the arrays it points into."""
        nj = len(jobs)
        arr = (ReconJob * max(nj, 1))()
        keep = []
        for j, job in enumerate(jobs):
            fr = np.ascontiguousarray(job['frames'], RECON_FRAME); tr = np.ascontiguousarray(job['tracks'], RECON_TRACK)
            keep += [fr, tr]
            a = arr[j]
            a.frames, a.n_frames, a.tracks, a.n_tracks = fr.ctypes.data, len(fr), tr.ctypes.data, len(tr)
            a.cam_road[:] = [float(x) for x in np.ravel(job['cam_road'])]
            a.max_dist, a.min_angle, a.point_type = job['max_dist'], job['min_angle'], int(job['point_type'])
        return arr, keep

    def recon_points(self, jobs):
        """visocu_recon_points for a list of jobs, each a dict with frames (RECON_FRAME array), tracks (RECON_TRACK array),
        cam_road (12), max_dist, min_angle and point_type (host_py.Recon.batch_job makes them).  Returns one
        (status int32 array, xyz float32 n x 3 array) per job."""
        nj = len(jobs)
        arr, keep = self._job_array(jobs)
        status = [np.zeros(arr[j].n_tracks, np.int32) for j in range(nj)]
        xyz = [np.zeros((arr[j].n_tracks, 3), np.float32) for j in range(nj)]
        sp = (C.c_void_p * max(nj, 1))(*[x.ctypes.data for x in status])
        xp = (C.c_void_p * max(nj, 1))(*[x.ctypes.data for x in xyz])
        self._ck(lib().visocu_recon_points(self.h, nj, arr, sp, xp), 'recon_points')
        return list(zip(status, xyz))

    def recon_store(self, initial_capacity=0):
        """A device point store on this context (visocu_recon_store)."""
        return ReconStore(self, initial_capacity)

    def recon_update(self, stores, trs, jobs, want_status=False):
        """visocu_recon_update: per job j, the points of stores[j] move with trs[j] (4x4, or rows 0..2), jobs[j] (a dict
        as for recon_points) is evaluated and its kept points are appended to stores[j].  Returns the kept counts (int32
        array), and with want_status also one (status, xyz) per job as recon_points returns them."""
        nj = len(jobs)
        arr, keep = self._job_array(jobs)
        t = [np.ascontiguousarray(np.asarray(x, np.float64)[:3, :4]) for x in trs]
        tp = (C.c_void_p * max(nj, 1))(*[x.ctypes.data for x in t])
        sp = (C.c_void_p * max(nj, 1))(*[s.h.value for s in stores])
        kept = np.zeros(nj, np.int32)
        status = xyz = None
        if want_status:
            status = [np.zeros(arr[j].n_tracks, np.int32) for j in range(nj)]
            xyz = [np.zeros((arr[j].n_tracks, 3), np.float32) for j in range(nj)]
        mk = lambda lst: None if lst is None else (C.c_void_p * max(nj, 1))(*[x.ctypes.data for x in lst])
        self._ck(lib().visocu_recon_update(self.h, nj, sp, tp, arr, _p(kept), mk(status), mk(xyz)), 'recon_update')
        return (kept, list(zip(status, xyz))) if want_status else kept


class ReconStore:
    """One sequence's reconstructed points (float x, y, z) in device memory of a Context (visocu_recon_store_*)."""

    def __init__(self, ctx, initial_capacity=0):
        self.ctx = ctx
        self.h = C.c_void_p()
        ctx._ck(lib().visocu_recon_store_create(ctx.h, C.c_int64(int(initial_capacity)), C.byref(self.h)), 'recon_store_create')

    def close(self):
        if self.h.value and self.ctx.h.value:
            self.ctx._ck(lib().visocu_recon_store_destroy(self.ctx.h, self.h), 'recon_store_destroy')
        self.h = C.c_void_p()

    def device_pointer(self):
        """(device address, point count); the address stays valid until the next call that changes the store."""
        d = C.c_void_p(); n = C.c_int64()
        if lib().visocu_recon_store_points(self.h, C.byref(d), C.byref(n)):
            raise VisocuError('recon_store_points: no store')
        return d.value or 0, n.value

    @property
    def count(self):
        return self.device_pointer()[1]

    def append(self, xyz):
        a = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
        self.ctx._ck(lib().visocu_recon_store_append(self.ctx.h, self.h, _p(a), C.c_int64(len(a))), 'recon_store_append')

    def read(self, first=0, count=None):
        n = self.count
        count = n - first if count is None else count
        out = np.zeros((max(count, 0), 3), np.float32)
        self.ctx._ck(lib().visocu_recon_store_read(self.ctx.h, self.h, C.c_int64(first), C.c_int64(count), _p(out)),
                     'recon_store_read')
        return out
