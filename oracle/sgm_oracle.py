"""TEST INFRASTRUCTURE ONLY: ctypes binding of oracle/_build/libsgmoracle.so (sgm_oracle.c, the plain-C restatement of
visocu_disparity's semi-global matching).  Imported by tests/ only."""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(HERE, '_build', 'libsgmoracle.so')
        if not os.path.exists(path):
            subprocess.run(['make', '-C', HERE, '-f', 'sgm_oracle.mk'], check=True, stdout=subprocess.DEVNULL)
        _lib = C.CDLL(path)
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def sgm(left, right, params, want_S=False):
    """Semi-global matching of sgm_oracle.c on two (h, w) uint8 images.  params: anything with the fields of
    visocu_sgm_params (max_disp, paths, p1, p2, uniqueness, lr_max_diff, subpixel).  Returns the (h, w) int16 map in
    1/16 pixel (-1 = invalid), and with want_S also S as an (h, w, max_disp) uint16 array."""
    L = np.ascontiguousarray(left, np.uint8); R = np.ascontiguousarray(right, np.uint8)
    assert L.shape == R.shape and L.ndim == 2
    h, w = L.shape
    p = np.array([params.max_disp, params.paths, params.p1, params.p2, params.uniqueness, params.lr_max_diff,
                  params.subpixel], np.int32)
    out = np.zeros((h, w), np.int16)
    S = np.zeros((h, w, int(p[0])), np.uint16) if want_S else None
    rc = lib().vo_sgm(_p(L), _p(R), w, h, w, _p(p), _p(out), _p(S))
    if rc:
        raise ValueError('vo_sgm: parameters out of range')
    return (out, S) if want_S else out
