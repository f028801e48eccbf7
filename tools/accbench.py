"""Accumulation benchmark: FlowBatch.accumulate against the loop of FlowBatch.combine_with(., 3) it replaces, at 1080p.

    python tools/accbench.py [--out PATH]   (default PATH: profiles/r07_accbench_folds.txt)

Configurations: (S = 1, L = 64) and (S = 32, L = 8) clips of device-resident 1080p flows (rotations, scalings and
translations, a different one per frame; 1.2 GB and 4.8 GB of flow and mask, more than the 126 MB L2), all four
(ref, fold) combinations, cumulative and final-only; plus (S = 32, L = 8) with one cancelling clip (a translation
followed by its inverse, where the fold meets it first), which prices the repair path of the walked folds.
  loop       : the steps laid out as L contiguous S-frame FlowBatches, prepared outside the timed region; the left fold
               runs acc = acc.combine_with(step[k], 3), the right fold acc = step[j].combine_with(acc, 3). Each step
               writes a full output, so the loop's time is the same whether the intermediates are kept or not.
  accumulate : FlowBatch.accumulate(L, cumulative, fold=fold).
After the timing, the final-only result is compared with the loop's, byte for byte.
Timing: CUDA events around 3 back-to-back calls after a warm-up call, median of 7 windows, on the default stream.
Reported per frame-step (one composition step of one clip, S * (L - 1) per call), with the algorithmic bytes: the
loop 27 B/px per step (running flow and next flow read, result written); the walked folds ('s' left, 't' right)
9 B/px in per input frame plus 9 B/px out per output frame; the sampled folds ('t' left, 's' right) 27 B/px per
step like the loop, plus the copy of the anchor frame (18 B/px per clip) when cumulative. Also the share of the
7.7 TB/s HBM3e bandwidth of the data sheet that the bytes over the time correspond to. The output names the card and
its power limit, read in the same run.
"""
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oflibnumpy_b200 import _lib, _ops, device  # noqa: E402
from oflibnumpy_b200.batch import FlowBatch  # noqa: E402
from oflibnumpy_b200.device import DeviceArray, Event  # noqa: E402

OUT = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else os.path.join(ROOT, 'profiles',
                                                                                     'r07_accbench_folds.txt')
H, W = 1080, 1920
CALLS, WINDOWS = 3, 7
PEAK = 7.7e12
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


def transform(rng):
    c = np.cos(np.radians(rng.uniform(-3, 3)))
    s = np.sin(np.radians(rng.uniform(-3, 3)))
    k = rng.uniform(0.97, 1.03)
    cx, cy = W / 2, H / 2
    m = np.array([[k * c, -k * s, 0], [k * s, k * c, 0], [0, 0, 1.0]])
    m[:2, 2] = [cx - m[0, 0] * cx - m[0, 1] * cy + rng.uniform(-6, 6), cy - m[1, 0] * cx - m[1, 1] * cy +
                rng.uniform(-6, 6)]
    return m


def make_batch(n, rng, cancel_clip=None, clip=None, fold='left'):
    mats = np.stack([transform(rng) for _ in range(n)])
    if cancel_clip is not None:                  # +(3, 2) then -(3, 2) at the start (left) or end (right) of that clip
        first = cancel_clip * clip + (0 if fold == 'left' else clip - 2)
        for i, (u, v) in enumerate(((3, 2), (-3, -2))):
            mats[first + i] = np.array([[1, 0, u], [0, 1, v], [0, 0, 1.0]])
    vecs = _ops.from_matrix(DeviceArray.from_numpy(mats), (H, W), 1.0)
    masks = DeviceArray.empty((n, H, W), np.uint8)
    _lib.call('ofk_rt_memset', masks.ptr, 1, masks.nbytes, device.current_stream())
    return vecs, masks


def steps_of(vecs, masks, s, clip, ref):
    """The L contiguous S-frame batches of the loop: step k holds frame k of every clip."""
    out = []
    for k in range(clip):
        v = DeviceArray.empty((s, H, W, 2), np.float32)
        m = DeviceArray.empty((s, H, W), np.uint8)
        for c in range(s):
            v.frames(c, c + 1).copy_from(vecs.frames(c * clip + k, c * clip + k + 1))
            m.frames(c, c + 1).copy_from(masks.frames(c * clip + k, c * clip + k + 1))
        out.append(FlowBatch._wrap(v, ref, m))
    return out


def loop(steps, fold):
    if fold == 'left':
        acc = steps[0]
        for k in range(1, len(steps)):
            acc = acc.combine_with(steps[k], 3)
    else:
        acc = steps[-1]
        for j in range(len(steps) - 2, -1, -1):
            acc = steps[j].combine_with(acc, 3)
    return acc


def time_ms(fn):
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
    return statistics.median(ts)


def row(name, ms, frame_steps, nbytes):
    per = ms / frame_steps
    rate = nbytes / (ms * 1e-3)
    emit("{:<52} {:>12.4f} {:>10.2f} {:>9.0f} {:>8.1f} %".format(name, per, nbytes / 1e9, rate / 1e9,
                                                                   100 * rate / PEAK))
    return per


device.require_gpu()
device.set_stream(None)
rng = np.random.default_rng(0)
px = H * W
emit("GPU: {} | {} x {} | CUDA events, {} back-to-back calls per window, median of {} windows".format(
    gpu_name_and_power(), H, W, CALLS, WINDOWS))
emit("{:<52} {:>12} {:>10} {:>9} {:>10}".format('configuration / leg', 'ms/frame-step', 'GB (alg.)', 'GB/s',
                                                 'of 7.7TB/s'))
for s, clip, cancel in ((1, 64, None), (32, 8, None), (32, 8, 5)):
    fs = s * (clip - 1)
    for fold in ('left', 'right'):
        vecs, masks = make_batch(s * clip, rng, cancel, clip, fold)
        for ref in ('s', 't'):
            walked = (ref == 's') == (fold == 'left')
            tag = "S={} L={} ref '{}' {}{}".format(s, clip, ref, fold, ', clip {} cancels'.format(cancel) if cancel
                                                   else '')
            steps = steps_of(vecs, masks, s, clip, ref)
            loop_ms = time_ms(lambda: loop(steps, fold))
            t_loop = row(tag + ' | loop', loop_ms, fs, 27.0 * px * fs)
            want = loop(steps, fold)
            del steps
            fb = FlowBatch._wrap(vecs, ref, masks)
            for cumulative in (True, False):
                acc_ms = time_ms(lambda: fb.accumulate(clip, cumulative, fold=fold))
                if walked:
                    nbytes = 9.0 * px * s * clip + 9.0 * px * (s * clip if cumulative else s)
                else:
                    nbytes = 27.0 * px * fs + (18.0 * px * s if cumulative else 0.0)
                t_acc = row(tag + (' | accumulate cumulative' if cumulative else ' | accumulate final-only'), acc_ms,
                            fs, nbytes)
                emit("{:<52} {:>11.2f}x".format('   speed-up over the loop', t_loop / t_acc))
            got = fb.accumulate(clip, False, fold=fold)
            same = got.vecs.numpy().tobytes() == want.vecs.numpy().tobytes() and \
                np.array_equal(got.masks.numpy(), want.masks.numpy())
            emit("   final-only equals the loop's result byte for byte: {}".format('yes' if same else 'NO'))
            del want, got
        del vecs, masks
os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
with open(OUT, 'w') as fh:
    fh.write('\n'.join(lines) + '\n')
