"""Post-filters of dense disparity (masked 3x3 median, then speckle removal with speckle_size 100, speckle_range 2) on
corridor maps of 1241x376 (SGM at D = 128, 8 paths, default parameters), in four phases of one process:
  1. visocu_disparity_filter on 1, 16 and 128 device maps: CUDA events on the context's stream around each call (the
     maps are restored from an unfiltered copy between calls, outside the timed window), REPS calls after WARM;
  2. the filter kernels of one 128-map call from the CUDA activity of torch.profiler (tracing slows the host);
  3. visocu_disparity at 1 and 128 pairs with the filters off and on, alternated call by call, CUDA events;
  4. the card's name and power limit.
Bytes per map are computed from the shapes (see bytes_per_map).  128 maps are 60 M pixels and 1.5 GB of filter
traffic, more than the 126 MB of L2.  Prints one JSON line.
usage: python profiles/bench_disparity_filter.py [reps=10]"""
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
MEDIAN, SPECKLE_SIZE, SPECKLE_RANGE = 1, 100, 2
REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
WARM = 2
MAPS = (1, 16, 128)
NF = 32                                 # 16 distinct stereo pairs; larger launches reuse them
KERNELS = ('k_disp_median3', 'k_speckle_local', 'k_speckle_merge', 'k_speckle_count', 'k_speckle_apply')


def bytes_per_map(w, h, tw=32, th=32):
    """Bytes one map moves through the filters, from the shapes: k_disp_median3 reads the map (2 B / pixel; the window's
    other 8 reads hit L1) and writes its output (2); k_speckle_local reads that (2) and writes a label and a count (4 + 4);
    k_speckle_merge reads both values and labels of each pixel pair across a tile border (2 x (2 + 4)); k_speckle_count
    reads every count (4); k_speckle_apply reads the value and the label (2 + 4) and writes the map (2).  The root lookups
    (a tile root's label and count, shared by the tile's pixels) are not counted."""
    px = w * h
    pairs = ((w + tw - 1) // tw - 1) * h + ((h + th - 1) // th - 1) * w
    return px * (4 + 10 + 4 + 8) + pairs * 12


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(',')]
        return name, limit
    except Exception as e:                 # the measurement still stands; the record says the query failed
        return 'unknown (%s)' % e, 'unknown'


import torch
ctx = V.Context(0)
info = ctx.device_info()
ctx.configure(V.Params(half_resolution=0), W, H, NF)
imgs = [im for k in range(NF // 2) for im in synth.corridor_stereo_frame(k, W, H, seed=1234 + k)]
ctx.push_frames(np.arange(NF), imgs=imgs)
nmax = max(MAPS)
left = np.array([2 * (k % (NF // 2)) for k in range(nmax)], np.int32)
right = left + 1
p_off = V.SgmParams(max_disp=D, paths=PATHS)
p_on = V.SgmParams(max_disp=D, paths=PATHS, median=MEDIAN, speckle_size=SPECKLE_SIZE, speckle_range=SPECKLE_RANGE)
pristine = ctx.disparity_tensor(left, right, p_off)          # (128, H, W) unfiltered corridor maps
work = pristine.clone()
torch.cuda.synchronize()
bpm = bytes_per_map(W, H)


def filt(n):
    arr = (C.c_void_p * n)(*[work[k].data_ptr() for k in range(n)])
    rc = V.lib().visocu_disparity_filter(ctx.h, n, arr, W, H, 1, MEDIAN, SPECKLE_SIZE, SPECKLE_RANGE)
    if rc:
        raise V.VisocuError('disparity_filter: %d %s' % (rc, V.lib().visocu_last_error(ctx.h).decode()))


def restore():
    work.copy_(pristine)
    torch.cuda.synchronize()


# 1. the stand-alone filter
filter_rates = {}
for n in MAPS:
    for _ in range(WARM):
        restore(); filt(n)
    ms = []
    for _ in range(REPS):
        restore()
        ctx.timer_start(); filt(n); ms.append(ctx.timer_stop())
    m = float(np.mean(ms))
    filter_rates[str(n)] = dict(ms_per_call=round(m, 4), ms_min=round(min(ms), 4), maps_per_s=round(n * 1e3 / m, 1),
                                gb_per_s=round(n * bpm / m / 1e6, 1))
valid_before = float((pristine >= 0).float().mean())
restore(); filt(nmax)
valid_after = float((work >= 0).float().mean())

# 2. the kernels of one 128-map call
from torch.profiler import profile, ProfilerActivity
restore(); filt(nmax)
restore()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    filt(nmax)
    torch.cuda.synchronize()
kernels = {}
for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA:
        for k in KERNELS:
            if k in e.name:
                kernels[k] = round(kernels.get(k, 0.0) + e.device_time / 1e3, 4)
ktotal = sum(kernels.values())

# 3. visocu_disparity with the filters off and on, alternated
outs = [ctx.device_alloc(W * H * 2) for _ in range(nmax)]


def sgm(n, p):
    arr = (C.c_void_p * n)(*outs[:n])
    rc = V.lib().visocu_disparity(ctx.h, n, left.ctypes.data_as(C.c_void_p), right.ctypes.data_as(C.c_void_p), C.byref(p), arr, 1)
    if rc:
        raise V.VisocuError('disparity: %d %s' % (rc, V.lib().visocu_last_error(ctx.h).decode()))


sgm_rates = {}
for n in (1, 128):
    for _ in range(WARM):
        sgm(n, p_off); sgm(n, p_on)
    t = {'off': [], 'on': []}
    for _ in range(REPS):
        for key, p in (('off', p_off), ('on', p_on)):
            ctx.timer_start(); sgm(n, p); t[key].append(ctx.timer_stop())
    off, on = float(np.mean(t['off'])), float(np.mean(t['on']))
    sgm_rates[str(n)] = dict(off_ms=round(off, 3), on_ms=round(on, 3), off_ms_min=round(min(t['off']), 3),
                             on_ms_min=round(min(t['on']), 3), added_pct=round(100.0 * (on - off) / off, 2))

name, limit = card()
print(json.dumps(dict(bench='disparity_filter', size=[W, H], max_disp=D, paths=PATHS,
                      filters=dict(median=MEDIAN, speckle_size=SPECKLE_SIZE, speckle_range=SPECKLE_RANGE), reps=REPS,
                      card=name, power_limit=limit, device=info['name'], sm_count=info['sm_count'],
                      bytes_per_map=bpm, filter_device_maps=filter_rates,
                      valid_fraction_before=round(valid_before, 4), valid_fraction_after=round(valid_after, 4),
                      kernel_ms_128_maps=kernels, kernel_total_ms_128_maps=round(ktotal, 4),
                      kernel_gb_per_s_128_maps=round(128 * bpm / ktotal / 1e6, 1) if ktotal else None,
                      disparity_filters_off_on=sgm_rates)))
for o in outs:
    ctx.device_free(o)
ctx.close()
