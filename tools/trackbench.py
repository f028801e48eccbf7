"""Batched point tracking benchmark: N frames (default 32 x 1080p) of device-resident flows, P points per frame
(default 4096), six routes, two ways.

    python tools/trackbench.py [N] [H] [W] [P] [--out PATH]      (default PATH: profiles/r04_trackbench_b32.txt)

  loop  : Flow.track frame by frame -- the only way before FlowBatch.track. Each call ends in downloads (and blocks on
          the zero test first), so a host clock times it: median of 5 runs.
  batch : FlowBatch.track with the (N,P,2) host points, default stream; CUDA events around 10 back-to-back calls, median
          of 10 such windows. The points are inside the frames, so no call synchronises (they all pass the host range
          tests); the time includes the upload of the points.

Routes: 's' float points, 's' int64 points, 's' float + get_valid_status, 's' s_exact_mode, 't', 't' + get_valid_status.
The flows are smooth affine fields (rotation, scaling and translation per frame, as bench.py's workload); N x 16.6 MB
exceeds the 126 MB L2. Both legs are first checked to give equal bytes. The output names the card and its power limit,
read in the same run.
"""
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import golden_inputs as gi  # noqa: E402
import oflibnumpy_b200 as of  # noqa: E402
from oflibnumpy_b200 import _lib, device  # noqa: E402
from oflibnumpy_b200.device import Event  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith('--')]
OUT = os.path.join(ROOT, 'profiles', 'r04_trackbench_b32.txt')
if '--out' in sys.argv:
    OUT = sys.argv[sys.argv.index('--out') + 1]
    args.remove(OUT)
N = int(args[0]) if len(args) > 0 else 32
H = int(args[1]) if len(args) > 1 else 1080
W = int(args[2]) if len(args) > 2 else 1920
P = int(args[3]) if len(args) > 3 else 4096
WINDOWS, CALLS = 10, 10
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


of.device.require_gpu()
of.device.set_stream(None)       # on another stream the upload of pageable points would synchronise it
rng = np.random.default_rng(0)
masks = rng.random((N, H, W)) > 0.02
batches = {}
for ref in ('s', 't'):
    fb = of.FlowBatch.from_transforms([gi.cfg4_transforms(i) for i in range(N)], (H, W), ref)
    batches[ref] = of.FlowBatch(fb.vecs, ref, masks, validate=False)
fpts = rng.uniform(0, 1, (N, P, 2)) * [H - 1, W - 1]
ipts = np.round(fpts).astype(np.int64)
ROUTES = [("'s' float", 's', fpts, {}), ("'s' int", 's', ipts, {}),
          ("'s' float + status", 's', fpts, {'get_valid_status': True}),
          ("'s' exact", 's', fpts, {'s_exact_mode': True}), ("'t'", 't', fpts, {}),
          ("'t' + status", 't', fpts, {'get_valid_status': True})]


def loop(ref, pts, kw):
    fb = batches[ref]
    return [fb[i].track(pts[i], **kw) for i in range(N)]


def batch(ref, pts, kw):
    return batches[ref].track(pts, **kw)


for name, ref, pts, kw in ROUTES:
    want = loop(ref, pts, kw)
    got = batch(ref, pts, kw)
    if kw.get('get_valid_status'):
        assert np.array_equal(got[1].numpy().view(bool), np.stack([w[1] for w in want])), name
        got, want = got[0], [w[0] for w in want]
    g = got.numpy()
    assert g.dtype == want[0].dtype and g.tobytes() == np.stack(want).tobytes(), name
emit("outputs equal on every route (loop of Flow.track, FlowBatch.track)")


def time_events(fn):
    """Per call: median and best over WINDOWS event windows, each around CALLS back-to-back calls."""
    fn()
    fn()
    device.synchronize()
    e0, e1 = Event(), Event()
    ts = []
    for _ in range(WINDOWS):
        e0.record()
        for _ in range(CALLS):
            fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_ms(e1) / CALLS)
    return statistics.median(ts), min(ts)


def time_host(fn, reps=5):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), min(ts)


def launches(fn):
    before = _lib.load().ofk_rt_launch_count()
    fn()
    return _lib.load().ofk_rt_launch_count() - before


emit("GPU: {} | N={} H={} W={} P={} | library {}".format(gpu_name_and_power(), N, H, W, P,
                                                        os.path.relpath(_lib.library_path(), ROOT)))
emit("{:<22} {:>14} {:>14} {:>16} {:>9} {:>9}".format('route', 'loop ms/frame', 'batch ms/frame', 'batch ms/call',
                                                      'speed-up', 'launches'))
for name, ref, pts, kw in ROUTES:
    lmed, _ = time_host(lambda: loop(ref, pts, kw))
    bmed, bbest = time_events(lambda: batch(ref, pts, kw))
    emit("{:<22} {:>14.4f} {:>14.5f} {:>16.4f} {:>8.1f}x {:>9}".format(
        name, lmed / N, bmed / N, bmed, lmed / bmed, launches(lambda: batch(ref, pts, kw))))
os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
with open(OUT, 'w') as fh:
    fh.write('\n'.join(lines) + '\n')
