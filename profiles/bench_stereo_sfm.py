"""Stereo structure-from-motion throughput: the sequence runner's stereo SfM mode (mode 4: quad matching with motion
prediction, then per worker and step ONE visocu_stereo_motion and ONE visocu_recon_points) next to mode 2 (stereo odometry
only), on 64 sequences of 1241x376 stereo corridor drives resident in HBM, at bucket 2 and bucket 1000.  Beside it, per
frame on one core and the same drives: the StructureFromMotionStereo facade's update (its estimate and reconstruction on
the device) against the host composition VisualOdometryStereo::process + Reconstruction::update; and the host half of the
batched reconstruction (Reconstruction::batchPrepare and batchFinish, timed separately) on the match lists of modes 3 (mono)
and 4 (stereo).  Prints one JSON line.
usage: python profiles/bench_stereo_sfm.py [sequences=64] [steps=8]"""
import json
import os
import statistics
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

S = int(sys.argv[1]) if len(sys.argv) > 1 else 64
K = int(sys.argv[2]) if len(sys.argv) > 2 else 8
W, Hh = 1241, 376
SEEDS = 2                     # a small seeded pool: sequence s drives through corridor (1234 + s % SEEDS)
NF = K + 6                    # six warm-up steps (the track window fills up over six frames), then K timed steps
stereo_pool = np.ascontiguousarray(np.stack([np.stack([np.stack(synth.corridor_stereo_frame(k, W, Hh, seed=1234 + q))
                                                       for k in range(NF)]) for q in range(SEEDS)]))   # SEEDS x NF x 2 x H x W
mono_pool = np.ascontiguousarray(np.stack([np.stack(synth.corridor_sequence(NF, W, Hh, seed=1234 + q)) for q in range(SEEDS)]))
ctx = V.Context(0)
info = ctx.device_info()
dev_stereo = ctx.device_alloc(stereo_pool.nbytes)
ctx.memcpy_h2d(dev_stereo, stereo_pool)
dev_mono = ctx.device_alloc(mono_pool.nbytes)
ctx.memcpy_h2d(dev_mono, mono_pool)
fb = W * Hh
sptr = lambda s, k, side: dev_stereo + (((s % SEEDS) * NF + k) * 2 + side) * fb
mptr = lambda s, k: dev_mono + ((s % SEEDS) * NF + k) * fb
threads = min(S, os.cpu_count() or 1)
dims = np.array([W, Hh, W], np.int32)
RECON = (0, 2, 30.0, 3.0)     # the facades' constants: point type, min track length, max distance, min angle
TIMED = range(NF - K, NF)


def stereo_params(bucket):
    return H.StereoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, base=0.54,
                          bucket_max_features=bucket)


def mono_params(bucket):
    return H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08,
                        bucket_max_features=bucket)


def timed(fn, *args):
    t0 = time.perf_counter()
    out = fn(*args)
    return out, 1e3 * (time.perf_counter() - t0)


def stats(ms):
    return {'median': round(statistics.median(ms), 3), 'max': round(max(ms), 3)}


def runner_rate(runner):
    steps = lambda ks, side: [[sptr(s, k, side) for s in range(S)] for k in ks]
    runner.run(steps(range(NF - K), 0), dims, ptr_steps2=steps(range(NF - K), 1), on_device=True)
    t0 = time.perf_counter()
    secs, nm, ok = runner.run(steps(TIMED, 0), dims, ptr_steps2=steps(TIMED, 1), on_device=True)
    return S * K / (time.perf_counter() - t0), ok


def recon_halves(frames):
    """Reconstruction of one sequence's (matches, motion) per frame (None: failed frame) through batchPrepare, one
    visocu_recon_points and batchFinish; the host halves timed per timed frame (ms)."""
    r = H.Recon(synth.KITTI_F, synth.KITTI_CU, synth.KITTI_CV)
    prep, fin = [], []
    for k, f in enumerate(frames):
        if f is None:
            continue
        _, tp = timed(r.batch_prepare, f[0], f[1], *RECON)
        status, xyz = ctx.recon_points([r.batch_job()])[0]
        _, tf = timed(r.batch_finish, status, xyz)
        if k in TIMED:
            prep.append(tp); fin.append(tf)
    return prep, fin


result = {}
for bucket in (2, 1000):
    p = stereo_params(bucket)
    r2 = H.Runner.stereo(0, S, threads, p)
    rate2, ok2 = runner_rate(r2)
    r2.close()
    r4 = H.Runner.stereo_sfm(0, S, threads, p)
    rate4, ok4 = runner_rate(r4)
    npts = [len(r4.points(s)) for s in range(S)]
    r4.close()
    # one core, per frame: the facade against the host composition on the same host images; the host composition's
    # matches and motions feed the timing of the batch halves (mode 4's lists: the facade's are byte-identical)
    facade_ms, host_ms, process_ms, update_ms, matches = [], [], [], [], []
    prep4, fin4 = [], []
    for q in range(SEEDS):
        sfm, vo, recon = H.StereoSfm(p, W, Hh), H.Stereo(p), H.Recon(synth.KITTI_F, synth.KITTI_CU, synth.KITTI_CV)
        replace, frames = False, []
        for k in range(NF):
            left, right = stereo_pool[q, k, 0], stereo_pool[q, k, 1]
            _, tf = timed(sfm.update, left, right)
            ok, tp = timed(vo.process, left, right, replace)
            tu = 0.0
            if k > 0 and ok:
                _, tu = timed(recon.update, vo.matches(), vo.motion(), *RECON)
            replace = k > 0 and not ok
            frames.append((vo.matches(), vo.motion()) if k > 0 and ok else None)
            if k in TIMED:
                facade_ms.append(tf); host_ms.append(tp + tu); process_ms.append(tp); update_ms.append(tu)
                matches.append(len(vo.matches()))
        a, b = recon_halves(frames)
        prep4 += a; fin4 += b
    # mode 3's lists: a mono odometry runner stepped frame by frame over the mono drives
    mp = mono_params(bucket)
    rs = H.Runner(0, SEEDS, 1, 1, 0, mp)
    mono_frames = [[] for _ in range(SEEDS)]
    for k in range(NF):
        secs, nm, ok = rs.step([mptr(s, k) for s in range(SEEDS)], dims, on_device=True)
        for s in range(SEEDS):
            mono_frames[s].append((rs.matches(s), rs.motion(s)) if ok[s] and k > 0 else None)
    rs.close()
    prep3, fin3 = [], []
    for s in range(SEEDS):
        a, b = recon_halves(mono_frames[s])
        prep3 += a; fin3 += b
    result['bucket%d' % bucket] = {
        'runner_stereo_sfm_pairs_per_s': round(rate4, 1), 'runner_stereo_odometry_pairs_per_s': round(rate2, 1),
        'ok_pairs_stereo_sfm': int(ok4.sum()), 'ok_pairs_stereo_odometry': int(ok2.sum()), 'pairs': int(ok4.size),
        'points_per_sequence_mean': round(float(np.mean(npts)), 1),
        'matches_per_pair_mean': round(float(np.mean(matches)), 1),
        'facade_update_ms_per_frame': stats(facade_ms),
        'host_composition_ms_per_frame': stats(host_ms),
        'host_stereo_process_ms_per_frame': stats(process_ms), 'host_recon_update_ms_per_frame': stats(update_ms),
        'mode4_batch_prepare_ms': stats(prep4), 'mode4_batch_finish_ms': stats(fin4),
        'mode3_batch_prepare_ms': stats(prep3), 'mode3_batch_finish_ms': stats(fin3),
    }

try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True,
                       timeout=30).stdout.strip().splitlines()[0]
except Exception as e:                      # the card name still comes from the context
    q = 'power limit not read: %s' % e
print(json.dumps({'metric': 'stereo structure from motion pairs/s (runner mode 4, 1241x376 stereo corridor drives resident in HBM)',
                  'sequences': S, 'steps': K, 'host_threads': threads, 'device': info['name'], 'nvidia_smi': q, **result}))
ctx.device_free(dev_mono)
ctx.device_free(dev_stereo)
