"""Rectifying pushes: the sequence runner in modes 0 (flow matching) and 2 (stereo odometry) on 64 sequences of raw
1392x512 images rectified to 1241x376 on the device, against the same modes on pre-rectified 1241x376 images; both
variants alternate in one process, resident in HBM (on_device) and end to end from host memory.  Then k_rectify alone:
device time per push of 128 frames from the CUDA activity of torch.profiler, in a process of its own (tracing slows the
host), and the algorithmic bytes per second (8 B of map + 1 B written per output pixel, each raw byte once).  Prints one
JSON line.
usage: python profiles/bench_rectify.py [sequences=64] [steps=16]   (--kernel: only the k_rectify part, one JSON line)"""
import json
import os
import subprocess
import sys
import time
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'opencl-structure-from-motion_b200')]
import numpy as np
import synth
import host_py as H
import visocu_py as V

KERNEL_ONLY = '--kernel' in sys.argv
ARGS = [a for a in sys.argv[1:] if a != '--kernel']
S = int(ARGS[0]) if len(ARGS) > 0 else 64
K = int(ARGS[1]) if len(ARGS) > 1 else 16
W, Hh, RW, RH = 1241, 376, 1392, 512
SEEDS = 2
WARM = 9                      # the first frame, then 8 steps: every lane of the pipelined mode 0 has captured its graphs
NF = K + WARM


def rig():
    """A KITTI-raw-like rig (radial-tangential distortion, about 1 degree of relative rotation) and its rectification."""
    def rot(axis, deg):
        a = np.asarray(axis, np.float64) / np.linalg.norm(axis); t = np.radians(deg)
        A = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
        return np.eye(3) + np.sin(t) * A + (1 - np.cos(t)) * A @ A
    c0 = V.Camera(959.8, 957.5, 696.0, 224.0, -0.37, 0.20, 1.2e-3, -3.4e-4, -0.07)
    c1 = V.Camera(955.1, 953.0, 690.3, 229.5, -0.365, 0.19, -6e-4, 8e-4, -0.06)
    r0, r1, base = H.stereo_rectify(c0, c1, rot((0.3, 1.0, -0.2), 1.0), np.array([-0.54, 0.01, 0.005]), W, Hh)
    return H.Rectification([r0, r1], RW, RH, W, Hh, base)


RECT = rig()
# raw-sized and rectified-sized corridor drives: the timing does not depend on what the raw pixels show
raw = np.ascontiguousarray(np.stack([np.stack([np.stack(synth.corridor_stereo_frame(k, RW, RH, seed=1234 + q)) for k in range(NF)])
                                     for q in range(SEEDS)]))
pre = np.ascontiguousarray(np.stack([np.stack([np.stack(synth.corridor_stereo_frame(k, W, Hh, seed=1234 + q)) for k in range(NF)])
                                     for q in range(SEEDS)]))
ctx = V.Context(0)
info = ctx.device_info()
dev = {'raw': ctx.device_alloc(raw.nbytes), 'pre': ctx.device_alloc(pre.nbytes)}
ctx.memcpy_h2d(dev['raw'], raw)
ctx.memcpy_h2d(dev['pre'], pre)
host = {'raw': raw, 'pre': pre}
size = {'raw': (RW, RH), 'pre': (W, Hh)}
threads = min(S, os.cpu_count() or 1)


def ptr(variant, resident, s, k, side):
    w, h = size[variant]
    off = (((s % SEEDS) * NF + k) * 2 + side) * w * h
    return dev[variant] + off if resident else host[variant].ctypes.data + off


def run_mode(mode, variant, resident):
    match = V.Params()
    if mode == 0:
        runner = H.Runner(0, S, threads, 0, 0, H.MonoParams(match=match, f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV))
    else:
        runner = H.Runner.stereo(0, S, threads, H.StereoParams(match=match, f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV,
                                                               base=0.54, bucket_max_features=2))
    if variant == 'raw':
        assert runner.set_rectification(RECT)
    w, h = size[variant]
    dims = np.array([w, h, w], np.int32)
    right = (lambda k: [ptr(variant, resident, s, k, 1) for s in range(S)]) if mode == 2 else (lambda k: None)
    runner.step([ptr(variant, resident, s, 0, 0) for s in range(S)], dims, ptrs2=right(0), on_device=resident)
    runner.run([[ptr(variant, resident, s, 1 + k, 0) for s in range(S)] for k in range(WARM - 1)], dims,
               ptr_steps2=[right(1 + k) for k in range(WARM - 1)] if mode == 2 else None, on_device=resident)
    t0 = time.perf_counter()
    secs, nm, ok = runner.run([[ptr(variant, resident, s, WARM + k, 0) for s in range(S)] for k in range(K)], dims,
                              ptr_steps2=[right(WARM + k) for k in range(K)] if mode == 2 else None, on_device=resident)
    rate = S * K / (time.perf_counter() - t0)
    runner.close()
    return rate, int(ok.sum()), float(nm.mean())


def runner_part():
    result = {}
    for mode in (0, 2):
        for resident in (True, False):
            rates = {'raw': [], 'pre': []}
            oks, nms = {}, {}
            for rep in range(2):                                        # alternate the variants
                for variant in ('raw', 'pre') if rep == 0 else ('pre', 'raw'):
                    r, oks[variant], nms[variant] = run_mode(mode, variant, resident)
                    rates[variant].append(r)
            result['mode%d_%s' % (mode, 'resident' if resident else 'end_to_end')] = {
                'rectified_raw_pairs_per_s': [round(x, 1) for x in rates['raw']],
                'pre_rectified_pairs_per_s': [round(x, 1) for x in rates['pre']],
                'ok_pairs': {v: oks[v] for v in oks}, 'matches_per_pair_mean': {v: round(nms[v], 1) for v in nms}}
    return result


def kernel_part():
    """k_rectify alone: 128 frames per push, raw images resident in HBM, two maps."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    N = 128
    ctx.configure(V.Params(), W, Hh, N)
    ctx.set_rectification(list(RECT.cams), RW, RH)
    ptrs = [ptr('raw', True, s % SEEDS, s % NF, s & 1) for s in range(N)]
    cams = np.array([s & 1 for s in range(N)], np.int32)
    frames = np.arange(N)
    for _ in range(3):
        ctx.push_frames_rectified(frames, cams, ptrs=ptrs, bpl_in=RW, on_device=1, want_counts=False)
    ctx.sync()
    REPS = 50
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(REPS):
            ctx.push_frames_rectified(frames, cams, ptrs=ptrs, bpl_in=RW, on_device=1, want_counts=False)
        ctx.sync()
    ks = [e for e in prof.key_averages() if 'k_rectify' in e.key]
    per_push_us = sum(e.device_time_total for e in ks) / REPS
    bytes_push = N * (W * Hh * 9 + RW * RH)
    return {'frames_per_push': N, 'launches_seen': sum(e.count for e in ks), 'us_per_push': round(per_push_us, 2),
            'algorithmic_bytes_per_push': bytes_push,
            'GB_per_s': round(bytes_push / (per_push_us * 1e-6) / 1e9, 1) if per_push_us > 0 else None}


if KERNEL_ONLY:
    print(json.dumps(kernel_part()))
    sys.exit(0)
result = runner_part()
# the profiler in a run of its own, after the timed runs of this process
out = subprocess.run([sys.executable, os.path.abspath(__file__), '--kernel', str(S), str(K)], capture_output=True, text=True)
result['k_rectify'] = json.loads(out.stdout.strip().splitlines()[-1]) if out.returncode == 0 else {'error': out.stderr[-2000:]}

try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True,
                       timeout=30).stdout.strip().splitlines()[0]
except Exception as e:                      # the card name still comes from the context
    q = 'power limit not read: %s' % e
print(json.dumps({'metric': 'runner pairs/s, raw 1392x512 rectified on the device vs pre-rectified 1241x376',
                  'sequences': S, 'steps': K, 'host_threads': threads, 'device': info['name'], 'nvidia_smi': q, **result}))
for d in dev.values():
    ctx.device_free(d)
