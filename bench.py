#!/usr/bin/env python
"""Benchmark of the hot path: matched frame-pairs/s at 1241x376 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload flow|quad|mono|flow4k]
                  [--bucket B] [--scaling weak|strong] [--sequences S] [--no-extra] [--dump-outputs DIR]

A step = one new frame for every one of the S independent sequences of this rank (S frame pairs):
Matcher::pushBack + matchFeatures [+ bucketFeatures + RANSAC/pose for `mono`], results back on the host.
Sequences are sharded over GPUs (one rank per GPU under torchrun, no data-path collective).  --scaling weak: S sequences
per GPU; --scaling strong: S sequences in total, S / N per GPU (BASELINE.json configs[4]: 64 sequences over 1/2/4/8 GPUs).
`value` is measured with the frames already resident in HBM (pushBackDevice); `e2e` repeats the run through the public
host-buffer API (pushBack from pinned host memory, H2D inside the timed region).
Timing: the K timed steps run back to back inside the host library (wall clock of that call, between two barriers with
the device idle on both sides; CUDA events around the same region are reported as `event_ms`), max over ranks.
The rank-0 line also carries the roofline of the fused filter+NMS kernel (timed alone with CUDA events, 128 frames per
launch so that the input exceeds L2; primary leg = the configuration of the workload, i.e. Matcher defaults =
half-resolution mode, second leg = half_resolution 0), the reference CPU path on this box's host cores (`cpu_baseline`),
and, at N = 1, an `extra` object with short runs of the other configurations of BASELINE.json.
--dump-outputs DIR writes what the last timed step delivered to the caller (see dump_outputs).
"""
import argparse
import ctypes as C
import json
import os
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')   # one CUDA stream per lane and host worker: see include/visocu.h
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, 'opencl-structure-from-motion_b200'), os.path.join(ROOT, 'oracle')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = 'matched frame-pairs/sec at 1241x376'
UNIT = 'frame-pairs/s'
KITTI = dict(f=645.2, cu=635.9, cv=194.1, height=1.6, pitch=-0.08)
GRAPH_WARMUP = 16          # untimed steps before the timed region: every lane has run plain, been captured and replayed


def workload_dims(workload):
    return (3840, 2160) if workload == 'flow4k' else (1241, 376)


def measured_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return json.load(f), 'measured'
    except Exception:
        return {'hbm_gbs': 6650.0}, 'fallback'


class ClockSampler:
    """nvidia-smi clocks and throttle reasons during the timed region."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(gpu), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '200'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([time.time()] + [x.strip() for x in line.split(',')])

    def mark(self):
        """start (first call) / end (second call) of the timed region"""
        self.marks = getattr(self, 'marks', []) + [time.time()]

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        marks = getattr(self, 'marks', [])
        rows = self.rows
        if len(marks) == 2:          # samples taken during the timed region (the 200 ms sampling grid is padded by one tick)
            inside = [r for r in rows if marks[0] - 0.25 <= r[0] <= marks[1] + 0.25]
            rows = inside or rows[-1:]
        rows = [r[1:] for r in rows]
        sm = [float(r[0]) for r in rows if len(r) >= 6 and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 6 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith('active')})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(sm)}


def make_pools(workload, n_frames):
    import synth
    W, H = workload_dims(workload)
    if workload == 'mono':
        return [synth.corridor_sequence(n_frames, W, H, seed=1234 + s) for s in range(2)]
    if workload == 'flow4k':
        return [synth.blob_sequence(n_frames, W, H, n_blobs=120000, seed=1234 + s) for s in range(2)]
    return [synth.blob_sequence(n_frames, W, H, seed=1234 + s) for s in range(4)]


def params_for(workload, bucket):
    import visocu_py as V
    import host_py as Hh
    mp = V.Params(nms_n=2) if workload == 'quad' else V.Params()     # quad: matlab/demo_matching_quad.m:12-21 of the reference
    kw = dict(KITTI)
    kw['bucket_max_features'] = bucket
    return Hh.MonoParams(match=mp, **kw)


# ------------------------------------------------------------------------------------------------ reference arm
def reference_run(workload, steps, warmup, bucket, pairs_per_step=6, threads=None):
    """The reference's own CPU implementation (oracle/_ref, unmodified sources) on all host cores: persistent threads, one
    sequence per thread, pairs counted and timed inside the C shim (oracle/ref_shim.cpp: ref_time_parallel).  A step =
    pairs_per_step frame pairs per thread."""
    import pyref
    ref = pyref.RefLib()
    cores = threads or os.cpu_count() or 1
    W, H = workload_dims(workload)
    wl = {'flow': 0, 'flow4k': 0, 'quad': 1, 'mono': 2}[workload]
    if workload == 'flow4k':
        pairs_per_step = 1
    pools = make_pools(workload, 24 if workload != 'flow4k' else 6)
    rp = pyref.MatcherParams(nms_n=2) if workload == 'quad' else pyref.MatcherParams()
    mp = pyref.MonoParams(match=rp, bucket_max_features=bucket, **KITTI)
    imgs = pools[0]
    imgs2 = np.ascontiguousarray(np.roll(imgs, -12, axis=2)) if workload == 'quad' else None
    bk = (bucket, 50.0, 50.0) if workload == 'quad' else None
    wall, done = pyref.time_parallel(ref, mp, wl, imgs, imgs2, cores, max(warmup, 1) * pairs_per_step, steps * pairs_per_step, bucket=bk)
    pairs = int(done.sum())
    return pairs / wall, wall, cores, '%d persistent threads x %d frame pairs per step, %d steps, pairs timed inside the shim ' \
        '(oracle/_ref = unmodified reference sources, g++ -O3 -DUSE_SIMD)' % (cores, pairs_per_step, steps)


# ------------------------------------------------------------------------------------------------ our arm
class Staged:
    """Frames of a workload staged once: pinned host copies (e2e) and device copies (value)."""

    def __init__(self, tctx, workload, n_frames):
        self.tctx = tctx
        self.W, self.H = workload_dims(workload)
        pools = make_pools(workload, n_frames)
        self.npool, self.n_frames, self.fb = len(pools), n_frames, self.W * self.H
        total = self.npool * n_frames * self.fb
        self.pinned = tctx.host_alloc(total)
        self.pin_arr = np.ctypeslib.as_array((C.c_uint8 * total).from_address(self.pinned)).reshape(self.npool, n_frames, self.H, self.W)
        for p in range(self.npool):
            self.pin_arr[p] = pools[p]
        self.dev = tctx.device_alloc(total)
        tctx.memcpy_h2d(self.dev, self.pin_arr)
        self.pinned_r = self.dev_r = None
        if workload == 'quad':
            # right camera = the same field seen 12 px further left (positive disparity), as in the reference arm
            self.pinned_r = tctx.host_alloc(total)
            pin_r = np.ctypeslib.as_array((C.c_uint8 * total).from_address(self.pinned_r)).reshape(self.npool, n_frames, self.H, self.W)
            for p in range(self.npool):
                pin_r[p] = np.roll(pools[p], -12, axis=2)
            self.dev_r = tctx.device_alloc(total)
            tctx.memcpy_h2d(self.dev_r, pin_r)
        self.pageable = None

    def ptrs(self, S, k, where, right=False):
        """pointers of frame k for S sequences; sequence s walks through pool s % npool.  where: 'dev' | 'pinned' | 'pageable'"""
        if where == 'pageable':
            if self.pageable is None:
                self.pageable = np.array(self.pin_arr, copy=True)          # ordinary (pageable) host memory
            base = self.pageable.ctypes.data
        else:
            base = {('dev', False): self.dev, ('dev', True): self.dev_r, ('pinned', False): self.pinned, ('pinned', True): self.pinned_r}[(where, right)]
        return [base + ((s % self.npool) * self.n_frames + k % self.n_frames) * self.fb for s in range(S)]

    def free(self):
        self.tctx.host_free(self.pinned); self.tctx.device_free(self.dev)
        if self.pinned_r:
            self.tctx.host_free(self.pinned_r); self.tctx.device_free(self.dev_r)


def dump_outputs(out_dir, runner, S, mode, prefix):
    """The results of the last step as a caller of the runner receives them: every sequence's final match list (one row per
    match, the twelve fields of p_match in their order, as float64: exact for the float32 coordinates and int32 indices) and,
    for odometry, its 4x4 motion.  Above 64 MB in all, every list keeps the same share of its rows, drawn with a fixed seed."""
    lists = {'%smatches_seq%03d' % (prefix, s): runner.matches(s) for s in range(S)}
    arrays = {k: np.stack([m[f] for f in m.dtype.names], 1).astype(np.float64) if len(m) else np.zeros((0, 12))
              for k, m in lists.items()}
    if mode == 1:
        arrays.update({'%smotion_seq%03d' % (prefix, s): np.asarray(runner.motion(s), np.float64) for s in range(S)})
    share = min(1.0, 64e6 / sum(a.nbytes for a in arrays.values()))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        if share < 1.0 and k.startswith(prefix + 'matches'):
            a = a[np.sort(np.random.default_rng(0).choice(len(a), int(len(a) * share), replace=False))]
        np.save(os.path.join(out_dir, k + '.npy'), a)


def timed_run(tctx, st, workload, S, threads, K, Wm, mp, where, local_rank, barrier, sample_clocks, dump=None):
    import host_py as Hh
    method = 2 if workload == 'quad' else 0
    mode = 1 if workload == 'mono' else 0
    stereo = workload == 'quad'
    dims = np.array([st.W, st.H, st.W], np.int32)
    on_device = where == 'dev'
    runner = Hh.Runner(local_rank, S, threads, mode, method, mp)
    sampler = ClockSampler(local_rank) if sample_clocks else None          # sampling starts before the warm-up
    # warm-up: the first frame, then Wm steps through the same pipelined call as the timed region
    runner.step(st.ptrs(S, 0, where), dims, st.ptrs(S, 0, where, True) if stereo else None, on_device=on_device)
    k = 1
    if Wm > 0:
        w1 = [st.ptrs(S, k + j, where) for j in range(Wm)]
        w2 = [st.ptrs(S, k + j, where, True) for j in range(Wm)] if stereo else None
        runner.run(w1, dims, w2, on_device=on_device, bucket=stereo)
        k += Wm
    l0 = runner.launches(); b0 = runner.transfer_bytes()
    Hh.stage_times(reset=True)
    tctx.sync(); barrier()
    if sampler:
        sampler.mark()
    tctx.timer_start()
    # the K timed steps run back to back inside the host library: every worker walks its own sequences through
    # the K frames, no barrier between steps (the sequences are independent)
    steps1 = [st.ptrs(S, k + j, where) for j in range(K)]
    steps2 = [st.ptrs(S, k + j, where, True) for j in range(K)] if stereo else None
    secs, nm, ok = runner.run(steps1, dims, steps2, on_device=on_device, bucket=stereo)
    tctx.sync()
    ev_ms = tctx.timer_stop()
    if sampler:
        sampler.mark()
    clocks = sampler.stop() if sampler else None
    barrier()
    l1 = runner.launches(); b1 = runner.transfer_bytes()
    ro = runner.outlier_stats()
    stages = {kk: round(1e3 * v[0] / max(v[1], 1), 4) for kk, v in Hh.stage_times().items() if v[1]}
    if dump:
        dump_outputs(dump[0], runner, S, mode, dump[1])
    runner.close()
    return dict(ms=1e3 * secs, event_ms=ev_ms, launches=l1 - l0, h2d=(b1[0] - b0[0]) / K, d2h=(b1[1] - b0[1]) / K,
                matches_per_pair=int(nm.sum()) / float(S * K), ok_frac=int(ok.sum()) / float(S * K), clocks=clocks, stages=stages, outliers=ro)


def roofline_leg(local_rank, st, mp, half, reps):
    """The fused filter+NMS kernel alone: 128 frames per launch (8 at 3840x2160), timed with CUDA events on the launching stream."""
    import visocu_py as V
    nb = 128 if st.W * st.H < 2000000 else 8
    rctx = V.Context(local_rank)
    vp = V.Params(**{f: getattr(mp.match, f) for f, _ in V.Params._fields_})
    vp.half_resolution = half
    if half:
        vp.match_radius //= 2
    rctx.configure(vp, st.W, st.H, nb)
    ptrs = [st.dev + ((i % st.npool) * st.n_frames + (i // st.npool) % st.n_frames) * st.fb for i in range(nb)]
    frames = list(range(nb))
    for _ in range(3):
        rctx.push_frames(frames, ptrs=ptrs, bpl_in=st.W, on_device=True)
    rctx.profile(True)
    for _ in range(reps):
        rctx.push_frames(frames, ptrs=ptrs, bpl_in=st.W, on_device=True)
    fms, nl, nfr = rctx.profile_read()
    rctx.profile(False)
    rctx.close()
    bpl = st.W + 15 - (st.W - 1) % 16
    # algorithmic bytes per frame (SURVEY.md 8d), per pixel of the padded full-resolution image: half_resolution = 0:
    # 1 B read + du + dv written = 3 B; half_resolution = 1: 1 B read + du_full + dv_full (2 B) + half-resolution du, dv
    # (0.5 B) = 3.5 B (the half image itself is never written: the kernel forms it in shared memory).  The 4-byte codes
    # of the maxima are not counted.
    alg = (3.5 if half else 3.0) * bpl * st.H
    peaks, which = measured_peaks()
    achieved = alg * nfr / (fms * 1e-3) / 1e9 if fms > 0 else 0.0
    return {'bound': 'hbm', 'kernel': 'k_filter_nms', 'achieved': round(achieved, 2), 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
            'frac': round(achieved / peaks['hbm_gbs'], 5), 'peak_source': which + ' (MEASURED_PEAKS.json hbm_gbs)',
            'launch_ms': round(fms / max(nl, 1), 5), 'frames_per_launch': nb, 'algorithmic_bytes_per_launch': int(alg * nb),
            'workload': '%d frames of %dx%d per launch, half_resolution=%d (%.0f MB of algorithmic traffic per launch, larger than L2 together '
                        'with the %d MB of frame planes it touches)' % (nb, st.W, st.H, half, alg * nb / 1e6, int(alg * nb / 1e6)),
            'bytes_per_pixel': 3.5 if half else 3.0}


def run_ours(args, rank, world, local_rank):
    import visocu_py as V
    import host_py as Hh
    workload = args.workload
    S = args.sequences if args.scaling == 'weak' else max(1, args.sequences // world)
    K, Wm = args.steps, max(args.warmup, GRAPH_WARMUP)
    # host workers per GPU: one per core of the rank's share, between 6 and 12.  Fewer workers = larger batches per launch
    # and less contention in the driver (frames resident: 63 k pairs/s with 4 - 6 workers, 58 k with 16); the end-to-end leg
    # issues one copy per image and likes more of them (44 k with 4 workers, 54 k with 12 - 16): profiles/r2_pipeline_summary.md
    cores = os.cpu_count() or 1
    if workload == 'flow':
        threads = args.threads or min(12, max(6, cores // max(1, min(world, 8))))
    else:
        # quad, odometry, 4K: the host stages (bucketing, estimateMotion, large-list votes) want every core
        threads = args.threads or min(16, max(8, cores // max(1, min(world, 8))))
    threads = max(1, min(threads, S))
    if threads * world > (os.cpu_count() or 1):
        # more workers than cores: waiting workers sleep between polls instead of yielding
        os.environ.setdefault('VISOCU_WAIT_SLEEP_US', '50')
    mp = params_for(workload, args.bucket)
    Hh.set_device(local_rank)
    tctx = V.Context(local_rank)                       # timing / staging context
    info = tctx.device_info()
    st = Staged(tctx, workload, K + Wm + 2)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()

    dump = (args.dump_outputs, 'rank%d_' % rank if world > 1 else '') if args.dump_outputs else None
    res_dev = timed_run(tctx, st, workload, S, threads, K, Wm, mp, 'dev', local_rank, barrier, rank == 0, dump)
    res_e2e = timed_run(tctx, st, workload, S, threads, K, Wm, mp, 'pinned', local_rank, barrier, False)
    extra = {}
    roof = roof2 = None
    if rank == 0 and not args.no_roofline:
        half = int(mp.match.half_resolution)
        roof = roofline_leg(local_rank, st, mp, half, max(5, min(K, 20)))
        roof2 = roofline_leg(local_rank, st, mp, 1 - half, max(5, min(K, 20)))
        # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed `ncu --set full` captures
        traffic = {(1241, 1): (159603200, 'profiles/r2_filter_nms_summary.md (r2_filter_nms_half_raw.csv)'), (1241, 0): (144969984, 'profiles/r2_filter_nms_summary.md (r2_filter_nms_full_raw.csv)')}
        for r in (roof, roof2):
            tr = traffic.get((st.W, int(r['bytes_per_pixel'] == 3.5)))
            r['traffic'] = tr[0] if tr else None
            r['traffic_source'] = tr[1] if tr else None
    if rank == 0 and world == 1 and not args.no_extra:
        # the drop-in API as a caller uses it: ONE Matcher, one sequence, pageable host images, every call synchronous
        hm = Hh.Matcher(mp.match)
        seq = np.array(st.pin_arr[0][:min(40, st.n_frames)], copy=True)
        hm.push(seq[0]); hm.push(seq[1]); hm.match_features(0)
        t0 = time.perf_counter()
        for k in range(2, len(seq)):
            hm.push(seq[k]); hm.match_features(0); m = hm.matches(2)
        dt = time.perf_counter() - t0
        extra['drop_in_single_matcher'] = {'value': round((len(seq) - 2) / dt, 1), 'unit': UNIT, 'ms_per_pair': round(1e3 * dt / (len(seq) - 2), 3),
                                           'api': 'one Matcher object, pushBack(pageable host image) + matchFeatures(0) + getMatches, synchronous', 'matches': int(len(m))}
        del hm
        # the sharded runner fed from pageable host memory
        rp = timed_run(tctx, st, workload, S, threads, min(K, 30), Wm, mp, 'pageable', local_rank, barrier, False)
        extra['e2e_pageable_host_memory'] = {'value': round(S * min(K, 30) / (rp['ms'] * 1e-3), 1), 'unit': UNIT}
    st.free()
    tctx.close()
    return res_dev, res_e2e, roof, roof2, extra, threads, info, S, Wm


def extra_workloads(args):
    """Short single-GPU runs of the other configurations of BASELINE.json, each in its own process (fresh CUDA state)."""
    out = {}
    todo = [('quad', ['--workload', 'quad']), ('mono', ['--workload', 'mono']), ('mono_bucket1000', ['--workload', 'mono', '--bucket', '1000']),
            ('flow_3840x2160', ['--workload', 'flow4k', '--sequences', '24', '--threads', '24', '--steps', '16'])]
    for name, extra in todo:
        if extra[1] == args.workload and '--bucket' not in extra and int(args.bucket) == 2:
            continue
        cmd = [sys.executable, os.path.abspath(__file__), '--steps', '20', '--warmup', '3', '--no-extra', '--no-cpu-baseline', '--no-roofline'] + extra
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
            line = [l for l in r.stdout.splitlines() if l.startswith('{')][-1]
            d = json.loads(line)
            out[name] = {'value': d['value'], 'e2e': d['e2e']['value'], 'unit': UNIT, 'ms_per_step': d['ms_per_step'], 'steps': d['steps'],
                         'workload': d['config']['workload'], 'sequences': d['config']['sequences_per_gpu'],
                         'matches_per_pair': d['config']['matches_per_pair'], 'process_ok_fraction': d['config']['process_ok_fraction'],
                         'outlier_lists_declined': d['config']['outlier_removal'].get('declined'),
                         'declined_lists_built_in_device_nodes': d['config']['outlier_removal'].get('declined_lists_built_in_device_nodes')}
        except Exception as e:
            out[name] = {'error': str(e)[:200]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='flow', choices=['flow', 'quad', 'mono', 'flow4k'])
    ap.add_argument('--bucket', type=int, default=2, help='bucket.max_features (mono / quad); the reference CLI uses 1000 (main.cpp:71)')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'], help='strong: --sequences is the total over all GPUs (configs[4])')
    ap.add_argument('--sequences', type=int, default=64, help='independent sequences per GPU (weak) or in total (strong)')
    ap.add_argument('--threads', type=int, default=0, help='host worker threads per rank (default: cores / ranks, between 6 and 12)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the single-Matcher / pageable / other-workload figures')
    ap.add_argument('--no-roofline', action='store_true')
    ap.add_argument('--dry-run', action='store_true', help='no GPU work: fake per-rank timings over gloo (tests of the N>1 plumbing)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the results of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    workload_name = {'flow': 'flow_1241x376_matcher_defaults (configs[0]: pushBack + matchFeatures(0), half-res, multi-stage, pixel refinement)',
                     'quad': 'quad_1241x376_nms2 (configs[1]: stereo pushBack + matchFeatures(2) + bucketFeatures)',
                     'mono': 'mono_vo_1241x376 (configs[2]: VisualOdometryMono::process, 2000 RANSAC iterations, bucket.max_features = %d)' % args.bucket,
                     'flow4k': 'flow_3840x2160_120k_blobs (configs[3]: pushBack + matchFeatures(0), Matcher defaults)'}[args.workload]

    if args.impl == 'reference':
        if rank != 0:
            return
        val, secs, cores, sample = reference_run(args.workload, args.steps, args.warmup, args.bucket)
        print(json.dumps({'impl': 'reference', 'metric': METRIC, 'value': round(val, 2), 'unit': UNIT, 'n_gpus': args.gpus,
                          'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(1e3 * secs / args.steps, 3),
                          'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
                          'config': {'workload': workload_name},
                          'cpu_baseline': {'value': round(val, 2), 'unit': UNIT, 'cores': cores, 'kind': 'reference', 'sample': sample},
                          'e2e': {'value': round(val, 2), 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))
        return

    tdev = 'cpu' if args.dry_run else 'cuda'
    if world > 1:
        import torch
        import torch.distributed as dist
        if args.dry_run:
            dist.init_process_group('gloo')
        else:
            torch.cuda.set_device(local_rank)
            dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    if args.dry_run:
        ms = 10.0 * (rank + 1) * args.steps
        S = args.sequences if args.scaling == 'weak' else max(1, args.sequences // world)
        fake = dict(ms=ms, event_ms=ms, launches=0, h2d=0, d2h=0, matches_per_pair=0.0, ok_frac=0.0, clocks=None)
        res_dev, res_e2e, roof, roof2, extra, threads, info, Wm = fake, dict(fake), None, None, {}, 1, {'name': 'none (dry run)'}, args.warmup
    else:
        res_dev, res_e2e, roof, roof2, extra, threads, info, S, Wm = run_ours(args, rank, world, local_rank)
    ms_dev, ms_e2e = res_dev['ms'], res_e2e['ms']
    launches = res_dev['launches']
    if world > 1:
        import torch
        import torch.distributed as dist
        t = torch.tensor([ms_dev, ms_e2e], dtype=torch.float64, device=tdev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e = float(t[0]), float(t[1])
        l = torch.tensor([launches], dtype=torch.int64, device=tdev)
        dist.all_reduce(l, op=dist.ReduceOp.SUM)
        launches = int(l[0])
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    K = args.steps
    pairs = S * world * K
    cores = os.cpu_count() or 1
    line = {'metric': METRIC, 'value': round(pairs / (ms_dev * 1e-3), 2), 'unit': UNIT, 'n_gpus': world, 'steps': K,
            'warmup': Wm, 'ms_per_step': round(ms_dev / K, 4), 'higher_is_better': True, 'scaling': args.scaling,
            'vs_baseline': None, 'dtype': 'u8', 'data': 'dry-run' if args.dry_run else 'synthetic',
            'config': {'workload': workload_name, 'sequences_per_gpu': S, 'frame_pairs_per_step': S * world,
                       'host_threads_per_gpu': threads, 'host_cores': cores,
                       'steps_in_flight_per_sequence': int(os.environ.get('VISOB_DEPTH', '3')) if args.workload in ('flow', 'mono', 'flow4k') else 1,
                       'timing': 'wall clock of the K steps inside the host library between barriers, device idle on both sides (event_ms = CUDA '
                                 'events around the same region: %.3f)' % res_dev.get('event_ms', 0.0),
                       'inputs': 'frames resident in HBM (pushBackDevice); every step uses new frames, %d sequences x %.2f MB per step, L2 not flushed '
                                 'between steps (the working set of a step, frame planes and record lists of all sequences, exceeds L2 only at 4K)' % (S, workload_dims(args.workload)[0] * workload_dims(args.workload)[1] / 1e6),
                       'device': info['name'], 'matches_per_pair': round(res_dev['matches_per_pair'], 1),
                       'process_ok_fraction': res_dev['ok_frac'],
                       'host_ms_per_call': res_dev.get('stages'),
                       'outlier_removal': dict(where='device (csrc/outliers.cu); a list too long for one CTA (3840x2160) is declined as a whole: its triangulation tree is cut into nodes the same kernel builds, the few merges above them and the vote run on the host',
                                               **res_dev.get('outliers', {}))},
            'clocks': res_dev['clocks'],
            'e2e': {'value': round(pairs / (ms_e2e * 1e-3), 2), 'unit': UNIT, 'h2d_bytes_per_step': int(res_e2e['h2d'] * world),
                    'd2h_bytes_per_step': int(res_e2e['d2h'] * world),
                    'api': 'Matcher::pushBack(host image, pinned) + matchFeatures + getMatches through the sharded runner'},
            'gpu_launches': launches, 'roofline': roof}
    if roof2:
        line['roofline_other_mode'] = roof2
    if not args.no_cpu_baseline and not args.dry_run:
        try:
            val, secs, ncores, sample = reference_run(args.workload, 5, 1, args.bucket)
            line['cpu_baseline'] = {'value': round(val, 2), 'unit': UNIT, 'cores': ncores, 'kind': 'reference', 'sample': sample}
        except Exception as e:     # the checker library is prebuilt; say so instead of inventing a number
            line['cpu_baseline'] = {'value': None, 'unit': UNIT, 'cores': 0, 'kind': 'reference', 'sample': 'unavailable: %s' % e}
    if extra or (world == 1 and not args.no_extra and not args.dry_run):
        if world == 1 and not args.no_extra and not args.dry_run:
            extra.update(extra_workloads(args))
        line['extra'] = extra
    print(json.dumps(line))


if __name__ == '__main__':
    main()
