"""Structure-from-motion throughput: the sequence runner's SfM mode (mode 3: flow matching, mono odometry, then per worker
and step ONE visocu_recon_points for the finished tracks of its sequences) next to mode 1 (odometry only), on 64 sequences
of 1241x376 corridor drives resident in HBM, at bucket 2 and bucket 1000.  Beside it: the host Reconstruction::update per
frame on the same match lists (one core, the facade's constants), and one warm visocu_recon_points call for 1 job, for one
worker's share and for all sequences.  Prints one JSON line.
usage: python profiles/bench_sfm.py [sequences=64] [steps=8]"""
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
pool = np.ascontiguousarray(np.stack([np.stack(synth.corridor_sequence(NF, W, Hh, seed=1234 + q)) for q in range(SEEDS)]))
ctx = V.Context(0)
info = ctx.device_info()
dev = ctx.device_alloc(pool.nbytes)
ctx.memcpy_h2d(dev, pool)
fb = W * Hh
ptr = lambda s, k: dev + ((s % SEEDS) * NF + k) * fb
threads = min(S, os.cpu_count() or 1)
dims = np.array([W, Hh, W], np.int32)
RECON = (0, 2, 30.0, 3.0)     # StructureFromMotion's constants: point type, min track length, max distance, min angle


def params(bucket):
    return H.MonoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, height=1.6, pitch=-0.08,
                        bucket_max_features=bucket)


def median_seconds(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def runner_rate(runner):
    for k in range(NF - K):
        runner.step([ptr(s, k) for s in range(S)], dims, on_device=True)
    t0 = time.perf_counter()
    secs, nm, ok = runner.run([[ptr(s, NF - K + k) for s in range(S)] for k in range(K)], dims, on_device=True)
    return S * K / (time.perf_counter() - t0), ok


result = {}
for bucket in (2, 1000):
    p = params(bucket)
    r1 = H.Runner(0, S, threads, 1, 0, p)
    rate1, ok1 = runner_rate(r1)
    r1.close()
    H.set_pipeline_depth(1)                 # mode 1 with one step in flight: synchronous steps, as mode 3 runs them
    r1 = H.Runner(0, S, threads, 1, 0, p)
    rate1_sync, _ = runner_rate(r1)
    r1.close()
    H.set_pipeline_depth(3)
    r3 = H.Runner.sfm(0, S, threads, p)
    rate3, ok3 = runner_rate(r3)
    npts = [len(r3.points(s)) for s in range(S)]
    r3.close()
    # the match lists and motions of the seeded drives (mode-1 runner stepped frame by frame), then Reconstruction on them:
    # update() timed per frame on the host; the batch halves give the jobs of the last step for the device call
    rs = H.Runner(0, SEEDS, 1, 1, 0, p)
    steps = []
    for k in range(NF):
        secs, nm, ok = rs.step([ptr(s, k) for s in range(SEEDS)], dims, on_device=True)
        steps.append([(rs.matches(s), rs.motion(s)) if ok[s] and k > 0 else None for s in range(SEEDS)])
    rs.close()
    host_ms, tracks, last_jobs = [], [], []
    for s in range(SEEDS):
        hr, br = H.Recon(synth.KITTI_F, synth.KITTI_CU, synth.KITTI_CV), H.Recon(synth.KITTI_F, synth.KITTI_CU, synth.KITTI_CV)
        job = None
        for k in range(NF):
            if steps[k][s] is None:
                continue
            m, T = steps[k][s]
            t0 = time.perf_counter(); hr.update(m, T, *RECON); dt = time.perf_counter() - t0
            if k >= NF - K:
                host_ms.append(1e3 * dt)
            br.batch_prepare(m, T, *RECON)
            job = br.batch_job()
            if k >= NF - K:
                tracks.append(len(job['tracks']))
            br.batch_finish(*br.host_eval())
        last_jobs.append(job)
    jobs = [last_jobs[s % SEEDS] for s in range(S)]
    per_worker = (S + threads - 1) // threads
    dev_one = median_seconds(lambda: ctx.recon_points(jobs[:1]), 20)
    dev_worker = median_seconds(lambda: ctx.recon_points(jobs[:per_worker]), 20)
    dev_all = median_seconds(lambda: ctx.recon_points(jobs), 20)
    result['bucket%d' % bucket] = {
        'runner_sfm_pairs_per_s': round(rate3, 1), 'runner_odometry_pairs_per_s': round(rate1, 1),
        'runner_odometry_synchronous_pairs_per_s': round(rate1_sync, 1),
        'ok_pairs_sfm': int(ok3.sum()), 'ok_pairs_odometry': int(ok1.sum()), 'pairs': int(ok3.size),
        'points_per_sequence_mean': round(float(np.mean(npts)), 1),
        'matches_per_pair_mean': round(float(np.mean([len(x[0]) for row in steps[NF - K:] for x in row if x is not None])), 1),
        'finished_tracks_per_update_mean': round(float(np.mean(tracks)), 1),
        'host_update_ms_per_frame': {'median': round(statistics.median(host_ms), 3), 'max': round(max(host_ms), 3)},
        'device_call_ms': {'jobs_1': round(1e3 * dev_one, 3), 'jobs_%d' % per_worker: round(1e3 * dev_worker, 3),
                           'jobs_%d' % S: round(1e3 * dev_all, 3)},
        'device_call_tracks': {'job_1': len(jobs[0]['tracks']), 'all': int(sum(len(j['tracks']) for j in jobs))},
    }

try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True,
                       timeout=30).stdout.strip().splitlines()[0]
except Exception as e:                      # the card name still comes from the context
    q = 'power limit not read: %s' % e
print(json.dumps({'metric': 'structure from motion pairs/s (runner mode 3, 1241x376 corridor drives resident in HBM)',
                  'sequences': S, 'steps': K, 'host_threads': threads, 'device': info['name'], 'nvidia_smi': q, **result}))
ctx.device_free(dev)
