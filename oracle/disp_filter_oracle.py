"""TEST INFRASTRUCTURE ONLY: ctypes binding of oracle/_build/libdispfilteroracle.so (disp_filter_oracle.c, the plain-C
restatement of the disparity post-filters of visocu_disparity and visocu_disparity_filter).  Imported by tests/ only."""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(HERE, '_build', 'libdispfilteroracle.so')
        if not os.path.exists(path):
            subprocess.run(['make', '-C', HERE, '-f', 'disp_filter_oracle.mk'], check=True, stdout=subprocess.DEVNULL)
        _lib = C.CDLL(path)
    return _lib


def filter(disp, median=0, speckle_size=0, speckle_range=0):
    """The post-filters of disp_filter_oracle.c (vo_disp_filter) on a copy of an (h, w) int16 map: returns the filtered
    map."""
    out = np.array(disp, np.int16, order='C', copy=True)
    assert out.ndim == 2
    h, w = out.shape
    rc = lib().vo_disp_filter(out.ctypes.data_as(C.c_void_p), w, h, int(median), int(speckle_size), int(speckle_range))
    if rc:
        raise ValueError('vo_disp_filter: parameters out of range')
    return out
