"""Evaluation benchmark: FlowBatch.evaluate against Flow - Flow on the same pair and against a torch recipe of the same
metrics, at 1080p; and the host entry evaluate_flows_host.

    python tools/evalbench.py [--out PATH]   (default PATH: profiles/r09_evalbench.txt)

Inputs: device-resident 1080p batches of N = 16, 64 and 256 ground-truth flows T (a smooth transform per frame:
rotation, scaling, translation) and estimates E = T + Gaussian noise (sigma 1.5 px), the truth masked at a density of
5 % invalid pixels, the estimate all valid. 16.6 MB per frame of flows: every batch is larger than the 126 MB L2, and
256 frames of both flows are 8.5 GB.
  evaluate               : E.evaluate(T): 16 B/px of flows and 2 B/px of masks in, 104 B per frame out.
  evaluate, return_epe   : the same and the EPE map (+4 B/px).
  Flow - Flow            : _ops.addsub of the same pair with both masks, the yardstick: 27 B/px.
  torch recipe           : the definitions of include/oflib_b200.h in torch element-wise float32 operations and
                           float64 reductions per frame.
  evaluate_flows_host    : the same batch from pinned host buffers through the ring (N = 16 and 64 only: the pinned
                           copies of N = 256 would be 9.5 GB of host memory). 18 B/px go up, the rows come back.
Timing: CUDA events around 3 back-to-back calls after a warm-up call, median of 7 windows, on the default stream; the
host entry, which is synchronous, by the host clock, median of 3 calls after a warm-up. Reported: ms per call, Gpx/s,
the algorithmic bytes per pixel, and the share of the 7.7 TB/s HBM3e bandwidth of the data sheet that those bytes over
the time correspond to (for the host entry: the upload rate in GB/s). After the timing the rows of evaluate are compared
with the torch recipe: counts equal, sums within 1e-12 relative. The output names the card and its power limit, read
in the same run.
"""
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oflibnumpy_b200 import _lib, _ops, device  # noqa: E402
from oflibnumpy_b200.batch import FlowBatch, evaluate_flows_host  # noqa: E402
from oflibnumpy_b200.device import DeviceArray, Event  # noqa: E402

OUT = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else os.path.join(ROOT, 'profiles',
                                                                                     'r09_evalbench.txt')
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
    k = rng.uniform(0.9, 1.1)
    cx, cy = W / 2, H / 2
    m = np.array([[k * c, -k * s, 0], [k * s, k * c, 0], [0, 0, 1.0]])
    m[:2, 2] = [cx - m[0, 0] * cx - m[0, 1] * cy + rng.uniform(-30, 30), cy - m[1, 0] * cx - m[1, 1] * cy +
                rng.uniform(-30, 30)]
    return m


def make_pair(n, rng):
    t = _ops.from_matrix(DeviceArray.from_numpy(np.stack([transform(rng) for _ in range(n)])), (H, W), 1.0)
    tt = torch.as_tensor(t, device='cuda')
    gen = torch.Generator(device='cuda').manual_seed(n)
    et = tt + 1.5 * torch.randn(tt.shape, device='cuda', generator=gen)
    tm = (torch.rand((n, H, W), device='cuda', generator=gen) >= 0.05).to(torch.uint8)
    em = torch.ones((n, H, W), dtype=torch.uint8, device='cuda')
    E = FlowBatch._wrap(device.as_device(et), 's', device.as_device(em))
    T = FlowBatch._wrap(t, 's', device.as_device(tm))
    return E, T, (et, em, tt, tm)


def torch_recipe(et, em, tt, tm):
    ue, ve, ug, vg = et[..., 0], et[..., 1], tt[..., 0], tt[..., 1]
    du, dv = ue - ug, ve - vg
    d2 = du * du + dv * dv
    epe = torch.sqrt(d2)
    mg = torch.sqrt(ug * ug + vg * vg)
    ev = (em & tm).bool()
    fl = (epe > 3) & (epe / mg > 0.05)
    cz = ue * vg - ve * ug
    cr = torch.sqrt(d2 + cz * cz)
    dot = (1 + ue * ug) + ve * vg
    ae = torch.atan2(cr, dot) * 57.29578
    b0 = mg < 10
    b2 = ~(mg < 40)
    b1 = ~b0 & ~b2
    dims = (1, 2)
    counts = torch.stack([ev.sum(dims), (ev & fl).sum(dims), (ev & (epe > 1)).sum(dims), (ev & (epe > 3)).sum(dims),
                          (ev & (epe > 5)).sum(dims), (ev & b0).sum(dims), (ev & b1).sum(dims), (ev & b2).sum(dims)], 1)
    e64 = torch.where(ev, epe, 0).double()
    sums = torch.stack([e64.sum(dims), torch.where(ev, ae, 0).double().sum(dims), torch.where(b0, e64, 0).sum(dims),
                        torch.where(b1, e64, 0).sum(dims), torch.where(b2, e64, 0).sum(dims)], 1)
    return counts, sums


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


def row(name, ms, px, bpp, host=False):
    rate = bpp * px / (ms * 1e-3) if bpp else None
    share = ('{:.0f} GB/s up'.format(18 * px / (ms * 1e-3) / 1e9) if host else
             '{:.1f} %'.format(100 * rate / PEAK) if rate else '-')
    emit("{:<46} {:>9.3f} {:>8.2f} {:>6} {:>9} {:>12}".format(
        name, ms, px / (ms * 1e-3) / 1e9, '{:.0f}'.format(bpp) if bpp else '-',
        '{:.0f}'.format(rate / 1e9) if rate and not host else '-', share))


device.require_gpu()
device.set_stream(None)
assert torch.cuda.current_stream().cuda_stream == 0     # torch and the library share the legacy default stream
rng = np.random.default_rng(0)
emit("GPU: {} | {} x {} | CUDA events, {} back-to-back calls per window, median of {} windows".format(
    gpu_name_and_power(), H, W, CALLS, WINDOWS))
emit("{:<46} {:>9} {:>8} {:>6} {:>9} {:>12}".format('configuration / leg', 'ms/call', 'Gpx/s', 'B/px', 'GB/s',
                                                   'of 7.7TB/s'))
summary = []
for n in (16, 64, 256):
    E, T, tensors = make_pair(n, rng)
    px = n * H * W
    tag = "N={}".format(n)
    t_eval = time_ms(lambda: E.evaluate(T))
    t_map = time_ms(lambda: E.evaluate(T, return_epe=True))
    t_sub = time_ms(lambda: _ops.addsub(_lib.OP_SUB, E.vecs, E.masks, T.vecs, T.masks))
    t_torch = time_ms(lambda: torch_recipe(*tensors))
    row(tag + ' | evaluate', t_eval, px, 18)
    row(tag + ' | evaluate, return_epe', t_map, px, 22)
    row(tag + ' | Flow - Flow', t_sub, px, 27)
    row(tag + ' | torch recipe', t_torch, px, None)
    t_host = None
    if n <= 64:
        host = []
        keep = []
        for x in tensors:
            a, k = device.pinned_empty(tuple(x.shape), np.float32 if x.dtype == torch.float32 else np.bool_)
            a.view(np.uint8 if x.dtype != torch.float32 else np.float32)[...] = x.cpu().numpy()
            host.append(a)
            keep.append(k)
        et_h, em_h, tt_h, tm_h = host
        evaluate_flows_host(et_h, tt_h, em_h, tm_h)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            hc, hs = evaluate_flows_host(et_h, tt_h, em_h, tm_h)
            ts.append((time.perf_counter() - t0) * 1e3)
        t_host = statistics.median(ts)
        row(tag + ' | evaluate_flows_host, pinned', t_host, px, 18, host=True)
    counts, sums = E.evaluate(T).numpy()
    wc, ws = (x.cpu().numpy() for x in torch_recipe(*tensors))
    same_counts = np.array_equal(counts, wc)
    rel = np.abs(sums - ws) / np.maximum(np.abs(ws), 1e-300)
    ok = same_counts and bool((rel <= 1e-12).all())
    if t_host is not None:
        ok = ok and hc.tobytes() == counts.tobytes() and hs.tobytes() == sums.tobytes()
    s = E.evaluate(T).summary()
    emit("   evaluate / Flow - Flow: {:.2f}   torch / evaluate: {:.1f}   EPE {:.4f}  AE {:.4f}  Fl {:.4f} over {} px"
         .format(t_eval / t_sub, t_torch / t_eval, s['epe'], s['ae'], s['fl'], s['pixels']))
    emit("   rows against the torch recipe: counts equal: {}; largest relative difference of the sums (epe, ae, "
         "bands): "
         "{}; within 1e-12{}: {}".format('yes' if same_counts else 'NO', ' '.join('{:.1e}'.format(r) for r in
                                                                                   rel.max(0)),
                                         ', host rows equal' if t_host is not None else '', 'yes' if ok else 'NO'))
    summary.append((tag, t_eval / t_sub, ok))
    del E, T, tensors
    torch.cuda.empty_cache()
emit("evaluate no slower than Flow - Flow in {} of {} batch sizes; rows agree in {} of {}".format(
    sum(r <= 1.0 for _, r, _ in summary), len(summary), sum(s for _, _, s in summary), len(summary)))
os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
with open(OUT, 'w') as fh:
    fh.write('\n'.join(lines) + '\n')
