"""Dense stereo disparity (visocu_disparity, semi-global matching) at 1241x376, D = 128, 8 paths, default parameters:
pairs per second for launches of 1, 16, 64 and 128 pairs (device output, CUDA events on the context's stream around
REPS calls after WARM untimed ones), then the kernels of one 16-pair call per stage from the CUDA activity of
torch.profiler (a separate phase after the timed one: tracing slows the host).  Bytes per pair are computed from the
shapes (see bytes_per_pair); GB/s = those bytes x pairs / time.  The card's name and power limit are read in the same
run.  Prints one JSON line.
usage: python profiles/bench_disparity.py [reps=10]"""
import json
import os
import subprocess
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'opencl-structure-from-motion_b200')]
import ctypes as C
import numpy as np
import synth
import visocu_py as V

W, H, D, PATHS = 1241, 376, 128, 8
REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
WARM = 2
LAUNCHES = (1, 16, 64, 128)
NF = 32                                 # 16 distinct stereo pairs; larger launches reuse them (each pair has its own S)


def bytes_per_pair(w, h, d, paths):
    """Bytes one pair moves, from the shapes: both images read by k_census (1 B / pixel each) and 2 x 8 B of census
    written; every path pass reads both census rows of its line once (16 B / pixel; the D - 1 shifted right-image reads
    of a step hit L1) and S (2 B per pixel and disparity) is written by the first pass and read and written by each of
    the other paths - 1; k_sgm_select reads S once and writes 2 B of output per pixel."""
    px = w * h
    census = 2 * px + 16 * px
    paths_b = paths * 16 * px + (2 + 4 * (paths - 1)) * px * d
    select = 2 * px * d + 2 * px
    return census + paths_b + select


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(',')]
        return name, limit
    except Exception as e:                 # the measurement still stands; the record says the query failed
        return 'unknown (%s)' % e, 'unknown'


ctx = V.Context(0)
info = ctx.device_info()
ctx.configure(V.Params(half_resolution=0), W, H, NF)
imgs = [im for k in range(NF // 2) for im in synth.corridor_stereo_frame(k, W, H, seed=1234 + k)]
ctx.push_frames(np.arange(NF), imgs=imgs)
p = V.SgmParams(max_disp=D, paths=PATHS)
nmax = max(LAUNCHES)
outs = [ctx.device_alloc(W * H * 2) for _ in range(nmax)]
left = np.array([2 * (k % (NF // 2)) for k in range(nmax)], np.int32)
right = left + 1
bpp = bytes_per_pair(W, H, D, PATHS)


def call(n):
    arr = (C.c_void_p * n)(*outs[:n])
    rc = V.lib().visocu_disparity(ctx.h, n, left.ctypes.data_as(C.c_void_p), right.ctypes.data_as(C.c_void_p), C.byref(p), arr, 1)
    if rc:
        raise V.VisocuError('disparity: %d %s' % (rc, V.lib().visocu_last_error(ctx.h).decode()))


rates = {}
for n in LAUNCHES:
    for _ in range(WARM):
        call(n)
    ctx.timer_start()
    for _ in range(REPS):
        call(n)
    ms = ctx.timer_stop() / REPS
    rates[str(n)] = dict(ms_per_call=round(ms, 3), pairs_per_s=round(n * 1e3 / ms, 1), gb_per_s=round(n * bpp / ms / 1e6, 1))

import torch
from torch.profiler import profile, ProfilerActivity
call(16)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    call(16)
    torch.cuda.synchronize()
stages = {}
for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA and ('k_census' in e.name or 'k_sgm_' in e.name):
        key = [k for k in ('k_census', 'k_sgm_rows', 'k_sgm_cols', 'k_sgm_diag', 'k_sgm_antidiag', 'k_sgm_select') if k in e.name][0]
        stages[key] = round(stages.get(key, 0.0) + e.device_time / 1e3, 3)
total = sum(stages.values())
name, limit = card()
print(json.dumps(dict(bench='disparity', size=[W, H], max_disp=D, paths=PATHS, params='defaults (P1 10, P2 120, U 95, lr 1, subpixel 1)',
                      reps=REPS, card=name, power_limit=limit, device=info['name'], sm_count=info['sm_count'],
                      bytes_per_pair=bpp, launches=rates,
                      stage_ms_16_pairs=stages, stage_total_ms_16_pairs=round(total, 3),
                      stage_gb_per_s_16_pairs=round(16 * bpp / total / 1e6, 1) if total else None)))
for o in outs:
    ctx.device_free(o)
ctx.close()
