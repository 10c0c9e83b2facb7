"""TEST INFRASTRUCTURE ONLY: ctypes binding of oracle/_build/libvisooracle.so (viso_oracle.c, the plain-C
restatement).  Imported by tests/ only."""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
P_MATCH = np.dtype([('u1p', 'f4'), ('v1p', 'f4'), ('i1p', 'i4'), ('u2p', 'f4'), ('v2p', 'f4'), ('i2p', 'i4'),
                    ('u1c', 'f4'), ('v1c', 'f4'), ('i1c', 'i4'), ('u2c', 'f4'), ('v2c', 'f4'), ('i2c', 'i4')])


class Params(C.Structure):
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

    def effective(self):
        """match_radius as the Matcher constructor leaves it (matcher.cpp:59-60)."""
        q = Params(**{n: getattr(self, n) for n, _ in self._fields_})
        if q.half_resolution:
            q.match_radius //= 2
        return q


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


_lib = None


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(HERE, '_build', 'libvisooracle.so')
        if not os.path.exists(path):
            subprocess.run(['make', '-C', HERE, 'oracle'], check=True, stdout=subprocess.DEVNULL)
        _lib = C.CDLL(path)
    return _lib


def bpl(w):
    return w + 15 - (w - 1) % 16


def pad(img):
    h, w = img.shape
    out = np.zeros((h, bpl(w)), np.uint8)
    lib().vo_pad_image(_p(np.ascontiguousarray(img)), w, h, w, _p(out))
    return out


def half_image(Ipad, w):
    h, b = Ipad.shape
    dims = np.array([w, h, b], np.int32); dh = np.zeros(3, np.int32)
    lib().vo_half_dims(_p(dims), _p(dh))
    out = np.zeros((dh[1], dh[2]), np.uint8)
    lib().vo_half_image(_p(np.ascontiguousarray(Ipad)), _p(dims), _p(out))
    return out, tuple(dh.tolist())


def _two8(fn, img):
    img = np.ascontiguousarray(img, np.uint8); h, w = img.shape
    a = np.zeros_like(img); b = np.zeros_like(img)
    fn(_p(img), w, h, _p(a), _p(b))
    return a, b


def sobel5x5(img):
    return _two8(lib().vo_sobel5x5, img)


def sobel3x3(img):
    return _two8(lib().vo_sobel3x3, img)


def blob5x5(img):
    img = np.ascontiguousarray(img, np.uint8); h, w = img.shape
    o = np.zeros((h, w), np.int16)
    lib().vo_blob5x5(_p(img), w, h, _p(o))
    return o


def checkerboard5x5(img):
    img = np.ascontiguousarray(img, np.uint8); h, w = img.shape
    o = np.zeros((h, w), np.int16)
    lib().vo_checkerboard5x5(_p(img), w, h, _p(o))
    return o


def nms(f1, f2, w, n, tau):
    f1 = np.ascontiguousarray(f1, np.int16); f2 = np.ascontiguousarray(f2, np.int16)
    h, b = f1.shape
    dims = np.array([w, h, b], np.int32)
    cap = 4 * (w // (n + 1) + 1) * (h // (n + 1) + 1)
    out = np.zeros((cap, 4), np.int32)
    cnt = lib().vo_nms(_p(f1), _p(f2), _p(dims), n, tau, _p(out), cap)
    return out[:cnt].copy()


def sad(a, b):
    a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
    return lib().vo_sad(_p(a), _p(b), len(a))


def compute_features(img, params):
    """Returns dict(rec1, rec2, du, dv, du_full, dv_full, dims_m)."""
    I = pad(np.ascontiguousarray(img, np.uint8))
    h, b = I.shape
    w = img.shape[1]
    dims = np.array([w, h, b], np.int32)
    if params.half_resolution:
        dh = np.zeros(3, np.int32)
        lib().vo_half_dims(_p(dims), _p(dh))
        wm, hm, bm = dh.tolist()
    else:
        wm, hm, bm = w, h, b
    du = np.zeros((hm, bm), np.uint8); dv = np.zeros((hm, bm), np.uint8)
    duf = np.zeros((h, b), np.uint8); dvf = np.zeros((h, b), np.uint8)
    cap = 4 * (wm // 2 + 1) * (hm // 2 + 1)
    r1 = np.zeros((cap, 12), np.int32); r2 = np.zeros((cap, 12), np.int32)
    n1 = C.c_int32(); n2 = C.c_int32()
    rc = lib().vo_compute_features(_p(I), _p(dims), C.byref(params), _p(du), _p(dv), _p(duf), _p(dvf), _p(r1), cap, C.byref(n1),
                                   _p(r2), cap, C.byref(n2))
    assert rc == 0
    return dict(rec1=r1[:n1.value].copy(), rec2=r2[:n2.value].copy(), du=du, dv=dv, du_full=duf, dv_full=dvf,
                dims=(w, h, b), dims_m=(wm, hm, bm))


def matching(method, m1p, m2p, m1c, m2c, dims_c, params, ranges=None, tr_delta=None, counts=False):
    """params: effective parameters (match_radius already halved for half resolution).  tr_delta: Tr_delta (4x4 or
    3x4, quad matching; the prediction also uses params.f, cu, cv, base).  counts=True also returns (entries of the
    scanned bins, window candidates) over all hops."""
    arrs = [np.ascontiguousarray(m, np.int32) if m is not None else np.zeros((0, 12), np.int32) for m in (m1p, m2p, m1c, m2c)]
    cap = max(len(a) for a in arrs) + 1
    out = np.zeros(cap, P_MATCH)
    d = np.array(dims_c, np.int32)
    r = np.ascontiguousarray(ranges, np.float32) if ranges is not None else None
    t = np.ascontiguousarray(np.asarray(tr_delta, np.float64)[:3, :4]) if tr_delta is not None else None
    c2 = np.zeros(2, np.int64)
    n = lib().vo_matching(method, _p(arrs[0]), len(arrs[0]), _p(arrs[1]), len(arrs[1]), _p(arrs[2]), len(arrs[2]), _p(arrs[3]),
                          len(arrs[3]), _p(d), C.byref(params), int(ranges is not None), _p(r), _p(t), _p(out), cap, _p(c2))
    assert 0 <= n <= cap
    return (out[:n].copy(), (int(c2[0]), int(c2[1]))) if counts else out[:n].copy()


def prior_statistics(matches, method, dims_c, params):
    m = np.ascontiguousarray(matches, dtype=P_MATCH)
    bs = params.match_binsize
    nb = int(np.ceil(np.float32(dims_c[0]) / np.float32(bs))) * int(np.ceil(np.float32(dims_c[1]) / np.float32(bs)))
    out = np.zeros((nb, 16), np.float32)
    d = np.array(dims_c, np.int32)
    n = lib().vo_prior_statistics(_p(m), len(m), method, _p(d), C.byref(params), _p(out))
    assert n == nb
    return out


def _planes(planes):
    g = lambda k: _p(np.ascontiguousarray(planes[k])) if planes.get(k) is not None else None
    return [g(k) for k in ('du1p', 'dv1p', 'du2p', 'dv2p', 'du1c', 'dv1c', 'du2c', 'dv2c')]


def refine_pixel(matches, method, dims, planes):
    """planes: dict with du1p dv1p du2p dv2p du1c dv1c du2c dv2c (full-resolution planes; missing = None)."""
    m = np.array(matches, dtype=P_MATCH, copy=True)
    d = np.array(dims, np.int32)
    lib().vo_refine_pixel(_p(m), len(m), method, _p(d), _p(d), *_planes(planes))
    return m


def refine_subpixel(matches, method, dims, planes):
    """parabolicFitting on every match.  Returns (matches with refined coordinates, keep flags, decision margins): the
    list is not compacted; margin = smallest distance of a float decision to its threshold (+inf: none taken)."""
    m = np.array(matches, dtype=P_MATCH, copy=True)
    d = np.array(dims, np.int32)
    keep = np.zeros(len(m), np.uint8); margin = np.zeros(len(m), np.float64)
    lib().vo_refine_subpixel(_p(m), len(m), method, _p(d), _p(d), *_planes(planes), _p(keep), _p(margin))
    return m, keep.astype(bool), margin


def normalize(matches):
    m = np.array(matches, dtype=P_MATCH, copy=True)
    Tp = np.zeros((3, 3)); Tc = np.zeros((3, 3))
    ok = lib().vo_normalize(_p(m), len(m), _p(Tp), _p(Tc))
    return bool(ok), m, Tp, Tc


def fundamental(matches, active):
    m = np.ascontiguousarray(matches, dtype=P_MATCH); a = np.ascontiguousarray(active, np.int32)
    F = np.zeros((3, 3))
    lib().vo_fundamental(_p(m), _p(a), len(a), _p(F))
    return F


def get_inlier(matches, F, thresh=1e-5):
    m = np.ascontiguousarray(matches, dtype=P_MATCH)
    out = np.zeros(len(m), np.int32)
    n = lib().vo_get_inlier(_p(m), len(m), _p(np.ascontiguousarray(F, np.float64)), C.c_double(thresh), _p(out))
    return out[:n].copy()


def ransac(matches, samples, thresh=1e-5):
    m = np.ascontiguousarray(matches, dtype=P_MATCH); s = np.ascontiguousarray(samples, np.int32)
    iters = len(s)
    F = np.zeros((3, 3)); inl = np.zeros(len(m), np.int32); counts = np.zeros(iters, np.int32)
    Fall = np.zeros((iters, 3, 3)); best = C.c_int32(-1)
    n = lib().vo_ransac(_p(m), len(m), _p(s), iters, C.c_double(thresh), _p(F), _p(inl), _p(counts), _p(Fall), C.byref(best))
    return dict(n_inliers=n, F=F, inliers=inl[:max(n, 0)].copy(), counts=counts, F_all=Fall, best_iter=best.value)
