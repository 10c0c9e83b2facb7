"""Structure from motion over long drives: does the runner's rate hold up as the reconstructed cloud grows?

Reconstruction keeps every point in current-camera coordinates, so each update moves ALL points stored so far.  On the host
that costs O(points) per frame; with device point stores (visocu_recon_update) the move is a kernel and the host never
touches the cloud.  This script runs runner modes 3 (mono) and 4 (stereo) over 64 corridor drives of 400 frames, resident
in HBM (a pool of 2 seeded drives, as bench_sfm.py uses), 16 host workers, bucket 1000, and reports pairs/s in windows of
25 steps plus the points per sequence at the end.  The runner part uses only API that predates the device stores (Runner.sfm,
Runner.stereo_sfm, run, points), so the same script measures an older tree as well: --parent DIR runs it on both trees in
one session, alternating (mode 3: parent then this tree; mode 4: this tree then parent), each in a fresh process.

On this tree it adds, on the final clouds:
  - one move-only visocu_recon_update over all 64 stores (CUDA events around the C call, median of 20 warm calls; 24 bytes
    per point, far more than the 126 MB of L2), and k_recon_move alone (torch.profiler), as GB/s and as a share of the
    B200's 7.7 TB/s data-sheet HBM bandwidth;
  - the host move of batchPrepare (batch_prepare minus batch_prepare_tracks) on one core for one sequence's final cloud.
Prints one JSON line.
usage: python profiles/bench_sfm_long.py [--parent DIR] [--frames 400] [--sequences 64] [--threads 16]"""
import argparse
import json
import multiprocessing
import os
import statistics
import subprocess
import sys
import tempfile
import time
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
import numpy as np

W, HT = 1241, 376
SEEDS = 2
WINDOW = 25
HBM_BYTES_PER_S = 7.7e12        # HGX B200 data sheet, one GPU


def _paths(tree):
    sys.path[:0] = [tree, os.path.join(tree, 'opencl-structure-from-motion_b200')]


def _frame(args):
    import synth
    k, seed, baseline = args
    return synth.corridor_frame(k, W, HT, seed, baseline_x=baseline)


def make_pool(frames, cache):
    """left[q][k], right[q][k] of the seeded drives as uint8 .npy files (made once, shared by every run)."""
    _paths(ROOT)
    with multiprocessing.Pool(min(32, os.cpu_count() or 1)) as pool:
        for name, baseline in (('left', 0.0), ('right', 0.54)):
            imgs = pool.map(_frame, [(k, 1234 + q, baseline) for q in range(SEEDS) for k in range(frames)])
            np.save(os.path.join(cache, name + '.npy'), np.stack(imgs).reshape(SEEDS, frames, HT, W))


def worker(tree, mode, cache, S, threads):
    _paths(tree)
    import synth
    import host_py as H
    import visocu_py as V
    left = np.load(os.path.join(cache, 'left.npy'))
    right = np.load(os.path.join(cache, 'right.npy'))
    NF = left.shape[1]
    ctx = V.Context(0)
    info = ctx.device_info()
    fb = W * HT
    dl, dr = ctx.device_alloc(left.nbytes), ctx.device_alloc(right.nbytes)
    ctx.memcpy_h2d(dl, left); ctx.memcpy_h2d(dr, right)
    dims = np.array([W, HT, W], np.int32)
    ptr = lambda base, s, k: base + ((s % SEEDS) * NF + k) * fb
    if mode == 3:
        p = H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08,
                         bucket_max_features=1000)
        runner = H.Runner.sfm(0, S, threads, p)
    else:
        p = H.StereoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, base=0.54,
                           bucket_max_features=1000)
        runner = H.Runner.stereo_sfm(0, S, threads, p)
    rates, ok_pairs = [], 0
    for k0 in range(0, NF - NF % WINDOW, WINDOW):
        steps = range(k0, k0 + WINDOW)
        l = [[ptr(dl, s, k) for s in range(S)] for k in steps]
        r = [[ptr(dr, s, k) for s in range(S)] for k in steps] if mode == 4 else None
        t0 = time.perf_counter()
        secs, nm, ok = runner.run(l, dims, ptr_steps2=r, on_device=True)
        rates.append(round(S * WINDOW / (time.perf_counter() - t0), 1))
        ok_pairs += int(ok.sum())
    clouds = [runner.points(s) for s in range(S)]
    out = {'pairs_per_s_windows': rates, 'window_steps': WINDOW, 'ok_pairs': ok_pairs, 'pairs': S * (NF - NF % WINDOW),
           'points_per_sequence_mean': round(float(np.mean([len(c) for c in clouds])), 1),
           'points_per_sequence_max': max(len(c) for c in clouds), 'device': info['name']}
    runner.close()
    ctx.device_free(dl); ctx.device_free(dr)
    if hasattr(V.Context, 'recon_update'):
        out.update(move_timing(ctx, H, V, clouds))
    ctx.close()
    print(json.dumps(out))


def move_timing(ctx, H, V, clouds):
    T = np.eye(4)
    yaw = 0.01
    T[:3, :3] = [[np.cos(yaw), 0, np.sin(yaw)], [0, 1, 0], [-np.sin(yaw), 0, np.cos(yaw)]]
    T[:3, 3] = [0.01, 0.0, -0.8]
    stores = [ctx.recon_store(initial_capacity=len(c)) for c in clouds]
    for s, c in zip(stores, clouds):
        s.append(c)
    r = H.Recon(1.0, 0.0, 0.0)
    r.batch_prepare(np.zeros(0, V.P_MATCH), np.eye(4), 0, 2, 30.0, 3.0)
    empty = r.batch_job()
    # the call's arguments are built once, so that the event interval holds the call and not the Python binding's set-up
    import ctypes as C
    ns = len(stores)
    arr, keep = V.Context._job_array([empty] * ns)
    tr12 = np.ascontiguousarray(T[:3, :4])
    sp, tp = (C.c_void_p * ns)(*[s.h.value for s in stores]), (C.c_void_p * ns)(*[tr12.ctypes.data] * ns)
    call = lambda: V.lib().visocu_recon_update(ctx.h, ns, sp, tp, arr, None, None, None)
    for _ in range(3):
        assert call() == 0
    ms = []
    for _ in range(20):
        ctx.timer_start()
        assert call() == 0
        ms.append(ctx.timer_stop())
    n = sum(len(c) for c in clouds)
    t = statistics.median(ms) * 1e-3
    # the kernel alone: torch.profiler (CUPTI) sees every kernel of the process
    kernel = {}
    try:
        import torch
        from torch.profiler import profile, ProfilerActivity
        torch.zeros(1, device='cuda')
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                call()
            torch.cuda.synchronize()
        us = [getattr(e, 'device_time', None) or e.cuda_time for e in prof.events() if 'k_recon_move' in e.name]
        tk = statistics.median(us) * 1e-6
        kernel = {'k_recon_move_us_median': round(1e6 * tk, 1), 'launches_seen': len(us),
                  'GB_per_s': round(24 * n / tk / 1e9, 1), 'share_of_hbm_7p7TBps': round(24 * n / tk / HBM_BYTES_PER_S, 3)}
    except Exception as e:
        kernel = {'not_measured': repr(e)}
    for s in stores:
        s.close()
    # the host move of one sequence's final cloud: a Reconstruction holding it (all points as tracks of two observations
    # that end at once), then batch_prepare minus batch_prepare_tracks with the same empty match list
    c = max(clouds, key=len)
    m = np.zeros(len(c), V.P_MATCH)
    m['i1p'] = m['i1c'] = np.arange(len(c), dtype=np.int32)
    r = H.Recon(1.0, 0.0, 0.0)
    r.batch_prepare(m, np.eye(4), 0, 2, 30.0, 3.0)
    assert r.batch_prepare(np.zeros(0, V.P_MATCH), np.eye(4), 0, 2, 30.0, 3.0) == len(c)
    r.batch_finish(np.zeros(len(c), np.int32), c)
    assert len(r.points()) == len(c)
    full, tracks = [], []
    for _ in range(15):
        t0 = time.perf_counter(); r.batch_prepare(np.zeros(0, V.P_MATCH), T, 0, 2, 30.0, 3.0); full.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); r.batch_prepare_tracks(np.zeros(0, V.P_MATCH), T, 0, 2, 30.0, 3.0); tracks.append(time.perf_counter() - t0)
    return {'move_only_update': {'points': n, 'bytes': 24 * n, 'call_ms_median': round(1e3 * t, 3),
                                 'call_GB_per_s': round(24 * n / t / 1e9, 1),
                                 'call_share_of_hbm_7p7TBps': round(24 * n / t / HBM_BYTES_PER_S, 3), 'kernel': kernel},
            'host_move_ms_per_frame': {'points': len(c), 'ms_median': round(1e3 * (statistics.median(full) - statistics.median(tracks)), 3)}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--parent', help='an older tree of this project, built, to run beside this one')
    ap.add_argument('--frames', type=int, default=400)
    ap.add_argument('--sequences', type=int, default=64)
    ap.add_argument('--threads', type=int, default=16)
    ap.add_argument('--worker', nargs=3, metavar=('TREE', 'MODE', 'CACHE'), help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        worker(a.worker[0], int(a.worker[1]), a.worker[2], a.sequences, a.threads)
        return
    result = {}
    with tempfile.TemporaryDirectory() as cache:
        t0 = time.perf_counter()
        make_pool(a.frames, cache)
        setup_s = time.perf_counter() - t0
        trees = [('this', ROOT)] + ([('parent', os.path.abspath(a.parent))] if a.parent else [])
        for mode in (3, 4):
            order = trees[::-1] if mode == 3 else trees
            for name, tree in order:
                out = subprocess.run([sys.executable, os.path.abspath(__file__), '--worker', tree, str(mode), cache,
                                      '--sequences', str(a.sequences), '--threads', str(a.threads)],
                                     capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
                result['mode%d_%s' % (mode, name)] = json.loads(out)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:
        q = 'power limit not read: %s' % e
    print(json.dumps({'metric': 'structure from motion pairs/s over long drives (runner modes 3 and 4, bucket 1000, 1241x376 '
                                'corridor drives resident in HBM)', 'sequences': a.sequences, 'frames': a.frames,
                      'host_threads': a.threads, 'nvidia_smi': q, 'frame_synthesis_s': round(setup_s, 1), **result}))


if __name__ == '__main__':
    main()
