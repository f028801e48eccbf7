"""Transformation-matrix fitting benchmark: FlowBatch.matrix on N device-resident frames (default 32 x 1080p) against
OpenCV on the host, for every dof x method.

    python tools/matrixbench.py [N] [H] [W] [--cv2-frames F] [--out PATH]   (default PATH: profiles/r05_matrixbench_b32.txt)

Input: homography fields (a different matrix per frame) with 30 % outliers (uniform +-20 px) and 2 % mask holes,
N x 16.6 MB of flow, more than the 126 MB L2.
  device : FlowBatch.matrix with the default 1024 hypotheses, default stream; CUDA events around one call, after a
           warm-up call, median of 10 windows; reported per frame.
  cv2    : the reference's route (cv2.estimateAffinePartial2D / estimateAffine2D / findHomography on every valid point
           pair, float32, default OpenCV threads), host clock, F frames (default 2), median per frame.
  scoring: the scoring kernels' hypothesis x point evaluations per second, from their summed time in a separate
           torch.profiler pass (RANSAC: one pass over the points; LMedS: three radix-selection passes, each counted).
The output names the card and its power limit, read in the same run.
"""
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oflibnumpy_b200 as of  # noqa: E402
from oflibnumpy_b200 import device  # noqa: E402
from oflibnumpy_b200.device import Event  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith('--')]
OUT = os.path.join(ROOT, 'profiles', 'r05_matrixbench_b32.txt')
CV2_FRAMES = 2
for flag in ('--out', '--cv2-frames'):
    if flag in sys.argv:
        val = sys.argv[sys.argv.index(flag) + 1]
        args.remove(val)
        if flag == '--out':
            OUT = val
        else:
            CV2_FRAMES = int(val)
N = int(args[0]) if len(args) > 0 else 32
H = int(args[1]) if len(args) > 1 else 1080
W = int(args[2]) if len(args) > 2 else 1920
K = 1024
WINDOWS = 10
CASES = [(4, 'ransac'), (4, 'lmeds'), (6, 'ransac'), (6, 'lmeds'), (8, 'lms'), (8, 'ransac'), (8, 'lmeds')]
lines = []


def emit(line):
    print(line, flush=True)
    lines.append(line)


def gpu_name_and_power():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                            str(device.get_device())], capture_output=True, text=True, timeout=60)
        return r.stdout.strip() or 'unknown (nvidia-smi printed nothing)'
    except (OSError, subprocess.SubprocessError) as e:
        return 'unknown ({})'.format(e)


def make_fields(rng):
    y, x = np.mgrid[:H, :W].astype(np.float64)
    P = np.stack([x, y, np.ones_like(x)], -1)
    vecs = np.empty((N, H, W, 2), np.float32)
    for i in range(N):
        M = np.array([[1.0 + 0.01 * np.sin(i), 0.02, 3.5 + 0.1 * i], [-0.015, 0.99, -2.0], [1e-6 * i, -2e-6, 1.0]])
        Q = P @ M.T
        v = Q[..., :2] / Q[..., 2:] - P[..., :2]
        o = rng.random((H, W)) < 0.3
        v[o] += rng.uniform(-20, 20, (int(o.sum()), 2))
        vecs[i] = v
    return vecs, rng.random((N, H, W)) > 0.02


def cv2_frame(vecs, mask, dof, method):
    import cv2
    y, x = np.mgrid[:H, :W].astype(np.float32)
    src = np.stack([x[mask], y[mask]], -1)
    dst = np.stack([x[mask] + vecs[..., 0][mask], y[mask] + vecs[..., 1][mask]], -1)
    if dof == 8:
        return cv2.findHomography(src, dst, {'lms': 0, 'ransac': cv2.RANSAC, 'lmeds': cv2.LMEDS}[method])
    est = cv2.estimateAffinePartial2D if dof == 4 else cv2.estimateAffine2D
    return est(src, dst, method={'ransac': cv2.RANSAC, 'lmeds': cv2.LMEDS}[method])


def time_device(fn):
    fn()
    device.synchronize()
    e0, e1 = Event(), Event()
    ts = []
    for _ in range(WINDOWS):
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_ms(e1))
    return statistics.median(ts)


def scoring_seconds(fn):
    """Summed CUDA time of the scoring kernels in one call, from torch.profiler (None if it is unavailable)."""
    try:
        import torch
        from torch.profiler import profile, ProfilerActivity
    except ImportError:
        return None
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        device.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if 'score_kernel' in e.key)
    return us * 1e-6 if us > 0 else None


device.require_gpu()
device.set_stream(None)
rng = np.random.default_rng(0)
vecs, masks = make_fields(rng)
fb = of.FlowBatch(vecs, 's', masks)
m_valid = masks.reshape(N, -1).sum(1)
emit("GPU: {} | N={} H={} W={} | hypotheses {} | 30 % outliers, 2 % mask holes".format(gpu_name_and_power(), N, H, W,
                                                                                     K))
emit("{:<14} {:>16} {:>18} {:>10} {:>22}".format('dof / method', 'device ms/frame', 'cv2 ms/frame (host)', 'speed-up',
                                                  'scoring eval/s'))
for dof, method in CASES:
    call = lambda: fb.matrix(dof, method)  # noqa: E731
    dev_ms = time_device(call) / N
    host = []
    for i in range(CV2_FRAMES):
        t0 = time.perf_counter()
        cv2_frame(vecs[i], masks[i], dof, method)
        host.append((time.perf_counter() - t0) * 1e3)
    host_ms = statistics.median(host)
    rate = 'n/a (no sampling)'
    if method != 'lms':
        sec = scoring_seconds(call)
        evals = K * float(m_valid.sum()) * (1 if method == 'ransac' else 3)
        rate = 'not measured' if sec is None else '{:.3e}'.format(evals / sec)
    emit("{:<14} {:>16.3f} {:>18.1f} {:>9.0f}x {:>22}".format('{} {}'.format(dof, method), dev_ms, host_ms,
                                                            host_ms / dev_ms, rate))
os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
with open(OUT, 'w') as fh:
    fh.write('\n'.join(lines) + '\n')
