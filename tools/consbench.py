"""Consistency benchmark: FlowBatch.consistent_with against combine_with(., 3) on the same pair and against the unfused
recipe of existing calls, at 1080p.

    python tools/consbench.py [--out PATH]   (default PATH: profiles/r08_consbench.txt)

Inputs: device-resident 1080p batches of N = 16, 64 and 256 forward flows F (a smooth transform per frame: rotation,
scaling, translation) and backward flows G (the inverse transforms), both refs, all pixels valid. The 'boundaries'
version adds 50 x 50 px blocks that move by another (+-9, +-5) px in F and not in G: motion boundaries and occlusions
(tiles whose box does not cover every tap). 16 MB per frame of flows: every batch is larger than the 126 MB L2.
  consistent_with        : F.consistent_with(G), and with return_valid_area.
  combine_with(., 3)     : the composition of the same pair (F.combine_with(G, 3) for 's', G.combine_with(F, 3) for
                           't'), the yardstick: 27 B/px, plus its zero-test and exit launches.
  unfused recipe         : that composition, the sampled backward flow (F.invert('t').apply(G.vecs) for 's',
                           F.apply(G.vecs) for 't') and the criterion in torch element-wise operations.
Timing: CUDA events around 3 back-to-back calls after a warm-up call, median of 7 windows, on the default stream.
Reported: ms per call, Gpx/s, the algorithmic bytes per pixel (consistent_with: 18 B/px in, 1 out, 2 with the valid
area; combine_with: 27 B/px), and the share of the 7.7 TB/s HBM3e bandwidth of the data sheet that those bytes over the
time correspond to. After the timing the fused outputs are compared with the unfused recipe byte for byte. The output
names the card and its power limit, read in the same run.
"""
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oflibnumpy_b200 import _lib, _ops, device  # noqa: E402
from oflibnumpy_b200.batch import FlowBatch  # noqa: E402
from oflibnumpy_b200.device import DeviceArray, Event  # noqa: E402

OUT = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else os.path.join(ROOT, 'profiles',
                                                                                     'r08_consbench.txt')
H, W = 1080, 1920
CALLS, WINDOWS = 3, 7
PEAK = 7.7e12
A1, A2 = 0.01, 0.5
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


def make_pair(n, ref, boundaries, rng):
    mats = np.stack([transform(rng) for _ in range(n)])
    inv = np.stack([np.linalg.inv(m) for m in mats])
    sign = 1.0 if ref == 's' else -1.0
    f = _ops.from_matrix(DeviceArray.from_numpy(mats if ref == 's' else inv), (H, W), sign)
    g = _ops.from_matrix(DeviceArray.from_numpy(inv if ref == 's' else mats), (H, W), sign)
    if boundaries:   # the same block pattern added to every frame of F: blocks move on their own, G does not follow
        yy, xx = np.mgrid[0:H, 0:W]
        on = ((xx // 50) + (yy // 50)) % 2 == 1
        extra = np.zeros((1, H, W, 2), np.float32)
        extra[0, on] = (9.0, 5.0)
        extra[0, on & ((yy // 100) % 2 == 1)] = (-9.0, -5.0)
        tf = torch.as_tensor(f, device='cuda')
        tf += torch.as_tensor(DeviceArray.from_numpy(extra), device='cuda')
    masks = []
    for _ in range(2):
        m = DeviceArray.empty((n, H, W), np.uint8)
        _lib.call('ofk_rt_memset', m.ptr, 1, m.nbytes, device.current_stream())
        masks.append(m)
    return FlowBatch._wrap(f, ref, masks[0]), FlowBatch._wrap(g, ref, masks[1])


def composition(F, G):
    return F.combine_with(G, 3) if F.ref == 's' else G.combine_with(F, 3)


def unfused(F, G):
    comp = composition(F, G)
    s = (F.invert('t') if F.ref == 's' else F).apply(G.vecs)
    r, w, s = (torch.as_tensor(x, device='cuda') for x in (comp.vecs, F.vecs, s))
    valid = torch.as_tensor(comp.masks, device='cuda').bool()
    lhs = r[..., 0] * r[..., 0] + r[..., 1] * r[..., 1]
    rhs = A1 * ((w[..., 0] * w[..., 0] + w[..., 1] * w[..., 1]) + (s[..., 0] * s[..., 0] + s[..., 1] * s[..., 1])) + A2
    return valid & (lhs < rhs), valid


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


def row(name, ms, px, bpp):
    rate = bpp * px / (ms * 1e-3) if bpp else None
    emit("{:<58} {:>9.3f} {:>8.2f} {:>6} {:>9} {:>8}".format(
        name, ms, px / (ms * 1e-3) / 1e9, '{:.0f}'.format(bpp) if bpp else '-',
        '{:.0f}'.format(rate / 1e9) if rate else '-', '{:.1f} %'.format(100 * rate / PEAK) if rate else '-'))


device.require_gpu()
device.set_stream(None)
assert torch.cuda.current_stream().cuda_stream == 0     # torch and the library share the legacy default stream
rng = np.random.default_rng(0)
emit("GPU: {} | {} x {} | CUDA events, {} back-to-back calls per window, median of {} windows".format(
    gpu_name_and_power(), H, W, CALLS, WINDOWS))
emit("{:<58} {:>9} {:>8} {:>6} {:>9} {:>8}".format('configuration / leg', 'ms/call', 'Gpx/s', 'B/px', 'GB/s',
                                                  'of 7.7TB/s'))
summary = []
for n in (16, 64, 256):
    for boundaries in (False, True):
        for ref in ('s', 't'):
            F, G = make_pair(n, ref, boundaries, rng)
            px = n * H * W
            tag = "N={} ref '{}' {}".format(n, ref, 'boundaries' if boundaries else 'smooth')
            t_comb = time_ms(lambda: composition(F, G))
            t_cons = time_ms(lambda: F.consistent_with(G))
            t_both = time_ms(lambda: F.consistent_with(G, return_valid_area=True))
            t_unf = time_ms(lambda: unfused(F, G))
            row(tag + ' | consistent_with', t_cons, px, 19)
            row(tag + ' | consistent_with, return_valid_area', t_both, px, 20)
            row(tag + ' | combine_with(., 3)', t_comb, px, 27)
            row(tag + ' | unfused recipe', t_unf, px, None)
            c, v = F.consistent_with(G, return_valid_area=True)
            wc, wv = unfused(F, G)
            same = np.array_equal(c.numpy(), wc.cpu().numpy().view(np.uint8)) and \
                np.array_equal(v.numpy(), wv.cpu().numpy().view(np.uint8))
            frac = 1.0 - float(c.numpy().mean())
            emit("   fused / combine_with: {:.2f}   fused / unfused: {:.2f}   inconsistent: {:.1f} %   equal to the "
                 "unfused recipe byte for byte: {}".format(t_cons / t_comb, t_cons / t_unf, 100 * frac,
                                                           'yes' if same else 'NO'))
            summary.append((tag, t_cons / t_comb, same))
            del F, G, c, v, wc, wv
            torch.cuda.empty_cache()
emit("consistent_with no slower than combine_with(., 3) in {} of {} configurations; outputs equal in {} of {}".format(
    sum(r <= 1.0 for _, r, _ in summary), len(summary), sum(s for _, _, s in summary), len(summary)))
os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
with open(OUT, 'w') as fh:
    fh.write('\n'.join(lines) + '\n')
