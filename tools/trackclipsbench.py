"""Trajectory benchmark: FlowBatch.track_clips against the loop users write today, a Flow.track call per step with the
lost points dropped on the host, at 1080p.

    python tools/trackclipsbench.py [--out PATH]   (default PATH: profiles/r10_trackclipsbench.txt)

Inputs: device-resident 1080p flows, smooth swirls of up to ~5 px (8 distinct fields repeated over the batch), all
pixels valid, no keep plane; 16.6 MB per frame, so every batch (64 or 128 frames) is larger than the 126 MB L2. Routes
's' (float64 bilinear), 's' exact (mesh on the undisplaced grid) and 't' (mesh p - flow); clip shapes (S, L) = (1, 64)
and (16, 8); points: P = 4096 random points, or a dense grid every 4 px (270 x 480 = 129,600 points), the same points
in every clip.
  track_clips : one call on device points (float64), CUDA events around 3 back-to-back calls after a warm-up call,
                median of 5 windows, on the default stream; launches per call from the library's launch counter.
  loop        : for every clip and step, the rules of track_clips on the host: the rounded points tested in numpy,
                Flow.track(q, get_valid_status=True) ('s') or Flow.track(q) and the valid_target plane ('t'), the lost
                points dropped before the next step. Host clock around the whole loop, which ends with host arrays
                (a synchronisation), second of two runs.
After the timing the loop's positions and alive flags are compared with the call's byte for byte. The output names the
card and its power limit, read in the same run.
"""
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oflibnumpy_b200 import _lib, device  # noqa: E402
from oflibnumpy_b200.batch import FlowBatch  # noqa: E402
from oflibnumpy_b200.device import DeviceArray, Event  # noqa: E402

OUT = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else os.path.join(ROOT, 'profiles',
                                                                                     'r10_trackclipsbench.txt')
H, W = 1080, 1920
CALLS, WINDOWS = 3, 5
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


def swirl(seed):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[:H, :W].astype(np.float32)
    a, b = rng.uniform(0.3, 0.9, 2) * min(H, W) / 4
    return np.stack([4 * np.sin(xx / a + seed) * np.cos(yy / b) + 0.002 * (xx - W / 2),
                     3 * np.cos(xx / b + 1) * np.sin(yy / a) - 0.003 * (yy - H / 2)], -1).astype(np.float32)


def in_frame(q):
    with np.errstate(invalid='ignore'):
        r = np.round(q)
    return (r[:, 0] >= 0) & (r[:, 0] <= H - 1) & (r[:, 1] >= 0) & (r[:, 1] <= W - 1)


def user_loop(fb, pts, L, exact):
    """track_clips' rules as a loop of single-frame Flow.track calls (zero frames do not occur in these inputs)."""
    n, p = len(fb), len(pts)
    pos, alive = np.full((n, p, 2), np.nan), np.zeros((n, p), np.uint8)
    for s in range(n // L):
        q, live = pts.astype(np.float64), np.ones(p, bool)
        for k in range(L):
            f = fb[s * L + k]
            live &= in_frame(q)
            idx = np.flatnonzero(live)
            if idx.size == 0:
                continue                                # pos and alive stay NaN and 0
            if fb.ref == 's':
                qi = q[idx]
                if exact:
                    new, st = f.track(qi, get_valid_status=True, s_exact_mode=True)
                    ok = st & ~(new == 0).all(1)
                else:                                   # Flow.track raises IndexError outside [0,H-1]x[0,W-1]
                    ok = (0 <= qi[:, 0]) & (qi[:, 0] <= H - 1) & (0 <= qi[:, 1]) & (qi[:, 1] <= W - 1)
                    new = np.zeros_like(qi)
                    new[ok], st = f.track(qi[ok], get_valid_status=True)
                    ok[ok] &= st
            else:
                new = f.track(q[idx])
                ok = ~(new == 0).all(1)
            live[idx[~ok]] = False
            q[idx[ok]] = new[ok]
            live &= in_frame(q)
            if fb.ref == 't' and live.any():
                idx = np.flatnonzero(live)
                target = f.valid_target()
                live[idx[~target[np.round(q[idx, 0]).astype(int), np.round(q[idx, 1]).astype(int)]]] = False
            pos[s * L + k][live] = q[live]
            alive[s * L + k] = live
    return pos, alive


def time_call(fn):
    fn()
    device.synchronize()
    ms = []
    for _ in range(WINDOWS):
        e0, e1 = Event(), Event()
        e0.record()
        for _ in range(CALLS):
            fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_ms(e1) / CALLS)
    return statistics.median(ms)


def main():
    device.require_gpu()
    emit("GPU: {} | {} x {} | track_clips: CUDA events, {} back-to-back calls per window, median of {} windows; loop: "
         "host clock, second of two runs".format(gpu_name_and_power(), H, W, CALLS, WINDOWS))
    fields = [swirl(i) for i in range(8)]
    rng = np.random.default_rng(0)
    random_pts = rng.uniform(0, 1, (4096, 2)) * [H - 1, W - 1]
    gy, gx = np.mgrid[0:H:4, 0:W:4]
    grid_pts = np.stack([gy.ravel(), gx.ravel()], 1).astype(np.float64)
    emit("{:<44} {:>12} {:>10} {:>9} {:>9} {:>8} {:>7}".format('configuration', 'track_clips', 'loop', 'speed-up',
                                                                 'launches', 'alive', 'equal'))
    for S, L in ((1, 64), (16, 8)):
        vecs = DeviceArray.from_numpy(np.stack([fields[i % 8] for i in range(S * L)]))
        for ref, exact in (('s', False), ('s', True), ('t', False)):
            fb = FlowBatch(vecs, ref)
            for pname, pts in (('P=4096 random', random_pts), ('grid every 4 px', grid_pts)):
                dpts = DeviceArray.from_numpy(pts)
                ms = time_call(lambda: fb.track_clips(dpts, L, s_exact_mode=exact))
                before = _lib.call('ofk_rt_launch_count')
                got = fb.track_clips(dpts, L, s_exact_mode=exact)
                launches = _lib.call('ofk_rt_launch_count') - before
                got = (got[0].numpy(), got[1].numpy())
                user_loop(fb, pts, L, exact)
                t0 = time.perf_counter()
                want = user_loop(fb, pts, L, exact)
                loop_ms = (time.perf_counter() - t0) * 1e3
                equal = got[0].tobytes() == want[0].tobytes() and np.array_equal(got[1], want[1])
                name = "S={} L={} {}{} | {}".format(S, L, ref, ' exact' if exact else '', pname)
                emit("{:<44} {:>9.3f} ms {:>7.1f} ms {:>8.0f}x {:>9d} {:>7.1f}% {:>7}".format(
                    name, ms, loop_ms, loop_ms / ms, launches, 100 * got[1][L - 1::L].mean(), 'yes' if equal else 'NO'))
        del vecs
    emit("alive: share of the trajectories alive at the end of their clip; equal: positions byte for byte and alive "
         "flags of the call and the loop")
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, 'w') as fh:
        fh.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
