"""Batched flow visualisation benchmark: N frames (default 32 x 1080p, 'rgb' with the mask shown) four ways.

    python tools/visbench.py [N] [H] [W]

  loop         : Flow.visualise frame by frame (per frame: magnitude, selection, host blend and read-back, colourise,
                 synchronous download) -- the only way before FlowBatch.visualise
  batch        : FlowBatch.visualise, default range (found on the device) and a given range; device-resident inputs
                 and output, CUDA events on the library's stream around 10 back-to-back calls, median of 10 such windows
  host pinned  : batch.visualise_flows_host on pinned numpy buffers (ring: uploads, kernels, downloads overlapped)
  host pageable: the same on ordinary numpy arrays

All paths are first checked to give equal bytes. Device legs report bytes per pixel and the share of the HBM roofline
(7.7 TB/s, NVIDIA's data sheet for one HGX B200 GPU) at the 12 B/px the operation must move (flow 8, mask 1, image 3);
the host legs report the share of the upload ceiling (DESIGN.md section 5: ~49 GB/s per direction with copies both
ways at once; 9 B/px in -> ~5.4 Gpx/s). The N flows (530 MB at 32 x 1080p) exceed the 126 MB L2.
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
from oflibnumpy_b200.batch import visualise_flows_host  # noqa: E402
from oflibnumpy_b200.device import Event, Stream  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 32
H = int(sys.argv[2]) if len(sys.argv) > 2 else 1080
W = int(sys.argv[3]) if len(sys.argv) > 3 else 1920
HBM_GBS = 7700.0
UPLOAD_GBS = 49.0
MODE, KW, RANGE = 'rgb', {'show_mask': True}, 12.0
WINDOWS, CALLS = 10, 10      # device legs: 10 event windows of 10 back-to-back calls each (5 to 10 ms per window)


def gpu_name_and_power():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                            str(device.get_device())], capture_output=True, text=True, timeout=60)
        return r.stdout.strip() or 'unknown (nvidia-smi printed nothing)'
    except (OSError, subprocess.SubprocessError) as e:
        return 'unknown ({})'.format(e)


of.device.require_gpu()
st = Stream()
of.device.set_stream(st)
rng = np.random.default_rng(0)
px = N * H * W

fb = of.FlowBatch.from_transforms([gi.cfg4_transforms(i) for i in range(N)], (H, W), 't')
masks = rng.random((N, H, W)) > 0.02
fb = of.FlowBatch(fb.vecs, 't', masks, validate=False)
host_vecs, _ = fb.numpy()
pin_vecs, keep_v = device.pinned_empty(host_vecs.shape, np.float32)
pin_vecs[...] = host_vecs
pin_masks, keep_m = device.pinned_empty(masks.shape, np.bool_)
pin_masks[...] = masks
pin_out, keep_o = device.pinned_empty((N, H, W, 3), np.uint8)


def loop(range_max=None):
    return np.stack([fb[i].visualise(MODE, range_max=range_max, **KW) for i in range(N)])


def batch(range_max=None):
    return fb.visualise(MODE, range_max=range_max, **KW)


# equal bytes on every path
for r in (None, RANGE):
    want = loop(r)
    got = batch(r).numpy()
    assert np.array_equal(got, want), ('batch', r)
    assert np.array_equal(visualise_flows_host(host_vecs, MODE, masks, range_max=r, **KW), want), ('host pageable', r)
    assert np.array_equal(visualise_flows_host(pin_vecs, MODE, pin_masks, range_max=r, out=pin_out, **KW), want), \
        ('host pinned', r)
print("outputs equal on all paths (loop, batch, host pinned, host pageable; default and given range)")


def time_events(fn):
    """Per call: median and best over WINDOWS event windows, each around CALLS back-to-back calls."""
    fn()
    fn()
    st.synchronize()
    e0, e1 = Event(), Event()
    ts = []
    for _ in range(WINDOWS):
        e0.record(st)
        for _ in range(CALLS):
            fn()
        e1.record(st)
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


print("GPU: {} | N={} H={} W={} | mode '{}' {} | library {}".format(gpu_name_and_power(), N, H, W, MODE, KW,
                                                                 os.path.relpath(_lib.library_path(), ROOT)))


def report(name, med, best, ceiling_gbs, bpp, ceiling_name):
    mpx = px / (med * 1e-3) / 1e6
    gbs = px * bpp / (med * 1e-3) / 1e9
    line = "{:<42} {:9.3f} ms/call {:8.4f} ms/frame {:10.1f} Mpx/s {:8.1f} GB/s at {:>2} B/px = {:5.1f} % of {} " \
           "(best {:.3f} ms)".format(name, med, med / N, mpx, gbs, bpp, 100 * gbs / ceiling_gbs, ceiling_name, best)
    print(line)


report("loop of Flow.visualise, default range", *time_host(loop), HBM_GBS, 12, "HBM 7.7 TB/s")
report("loop of Flow.visualise, range given", *time_host(lambda: loop(RANGE)), HBM_GBS, 12, "HBM 7.7 TB/s")
report("FlowBatch.visualise, default range", *time_events(batch), HBM_GBS, 12, "HBM 7.7 TB/s")
report("FlowBatch.visualise, range given", *time_events(lambda: batch(RANGE)), HBM_GBS, 12, "HBM 7.7 TB/s")
# With a range given the call is the colourise kernel alone. 'hsv' skips the float64 HSV->RGB conversion and the mask
# options add little arithmetic; the same bytes at different arithmetic separate the two costs.
report("  colourise only: 'hsv', mask shown", *time_events(lambda: fb.visualise('hsv', range_max=RANGE, **KW)),
       HBM_GBS, 12, "HBM 7.7 TB/s")
report("  colourise only: 'rgb', no mask options", *time_events(lambda: fb.visualise('rgb', range_max=RANGE)),
       HBM_GBS, 12, "HBM 7.7 TB/s")
report("  colourise only: 'hsv', no mask options", *time_events(lambda: fb.visualise('hsv', range_max=RANGE)),
       HBM_GBS, 12, "HBM 7.7 TB/s")
for r, rname in ((None, 'default range'), (RANGE, 'range given')):
    report("visualise_flows_host pinned, " + rname,
           *time_host(lambda: visualise_flows_host(pin_vecs, MODE, pin_masks, range_max=r, out=pin_out, **KW)),
           UPLOAD_GBS, 9, "upload 49 GB/s")
    report("visualise_flows_host pageable, " + rname,
           *time_host(lambda: visualise_flows_host(host_vecs, MODE, masks, range_max=r, **KW)), UPLOAD_GBS, 9,
           "upload 49 GB/s")


def launches(fn):
    before = _lib.load().ofk_rt_launch_count()
    fn()
    return _lib.load().ofk_rt_launch_count() - before


print("kernel launches per FlowBatch.visualise call: default range {}, range given {}".format(
    launches(batch), launches(lambda: batch(RANGE))))
