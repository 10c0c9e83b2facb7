"""Stereo odometry throughput: the sequence runner's stereo mode (quad matching with motion prediction + ONE
visocu_stereo_motion per worker and step) on 64 sequences of 1241x376 corridor drives resident in HBM, at bucket 2 and
bucket 1000, next to the host estimate (VisualOdometryStereo::estimateMotion through process_matches) and one warm
visocu_stereo_motion call on the same matches.  Prints one JSON line.
usage: python profiles/bench_stereo.py [sequences=64] [steps=8]"""
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
NF = K + 2                    # two warm-up steps (the first pair has no motion yet), then K timed steps
pool = np.ascontiguousarray(np.stack([np.stack([np.stack(synth.corridor_stereo_frame(k, W, Hh, seed=1234 + q)) for k in range(NF)])
                                      for q in range(SEEDS)]))         # SEEDS x NF x 2 x H x W
ctx = V.Context(0)
info = ctx.device_info()
dev = ctx.device_alloc(pool.nbytes)
ctx.memcpy_h2d(dev, pool)
fb = W * Hh
ptr = lambda s, k, side: dev + (((s % SEEDS) * NF + k) * 2 + side) * fb
threads = min(S, os.cpu_count() or 1)
dims = np.array([W, Hh, W], np.int32)


def params(bucket):
    return H.StereoParams(match=V.Params(), f=synth.KITTI_F, cu=synth.KITTI_CU, cv=synth.KITTI_CV, base=0.54,
                          bucket_max_features=bucket)


def median_seconds(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


result = {}
for bucket in (2, 1000):
    p = params(bucket)
    runner = H.Runner.stereo(0, S, threads, p)
    for k in range(2):
        runner.step([ptr(s, k, 0) for s in range(S)], dims, ptrs2=[ptr(s, k, 1) for s in range(S)], on_device=True)
    t0 = time.perf_counter()
    secs, nm, ok = runner.run([[ptr(s, 2 + k, 0) for s in range(S)] for k in range(K)], dims,
                              ptr_steps2=[[ptr(s, 2 + k, 1) for s in range(S)] for k in range(K)], on_device=True)
    rate = S * K / (time.perf_counter() - t0)
    lists = [runner.matches(s) for s in range(S)]
    runner.close()
    # the host estimate on the matches of the last step (one core, the default 200 iterations)
    host_s = []
    for s in range(min(S, 8)):
        h = H.Stereo(p)
        host_s.append(median_seconds(lambda: h.process_matches(lists[s]), 5))
    # one device call, warm, host clock around the synchronous call: one worker's share of the sequences, and one job
    tables = []
    for ml in lists:
        h = H.Stereo(p)
        h.batch_prepare(ml)
        tables.append(h.samples())
    per_worker = (S + threads - 1) // threads
    dev_worker = median_seconds(lambda: ctx.stereo_motion(lists[:per_worker], tables[:per_worker], p), 20)
    dev_one = median_seconds(lambda: ctx.stereo_motion(lists[:1], tables[:1], p), 20)
    dev_all = median_seconds(lambda: ctx.stereo_motion(lists, tables, p), 20)
    n = [len(x) for x in lists]
    result['bucket%d' % bucket] = {
        'runner_pairs_per_s': round(rate, 1), 'ok_pairs': int(ok.sum()), 'pairs': int(ok.size),
        'matches_per_pair_mean': round(float(np.mean(n)), 1),
        'host_estimate_ms_per_frame': round(1e3 * statistics.median(host_s), 3),
        'device_call_ms': {'jobs_%d' % per_worker: round(1e3 * dev_worker, 3), 'jobs_1': round(1e3 * dev_one, 3),
                           'jobs_%d' % S: round(1e3 * dev_all, 3)},
        'device_call_N': {'min': int(min(n)), 'max': int(max(n)), 'job_1': int(n[0])},
    }

try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True,
                       timeout=30).stdout.strip().splitlines()[0]
except Exception as e:                      # the card name still comes from the context
    q = 'power limit not read: %s' % e
print(json.dumps({'metric': 'stereo odometry pairs/s (runner mode 2, 1241x376 corridor drives resident in HBM)',
                  'sequences': S, 'steps': K, 'host_threads': threads, 'ransac_iters': 200, 'device': info['name'],
                  'nvidia_smi': q, **result}))
ctx.device_free(dev)
