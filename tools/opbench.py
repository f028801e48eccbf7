"""Op-level device benchmark of the SURVEY section 8d rows (algorithmic GB/s against the measured HBM peak).

    python tools/opbench.py [N] [H] [W]

Device-resident inputs, CUDA events on the library's stream, best of `reps` after warm-up. Prints one line per op and
a JSON summary (copied to profiles/ by hand).
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import golden_inputs as gi  # noqa: E402
import oflibnumpy_b200 as of  # noqa: E402
from oflibnumpy_b200 import _lib, _ops  # noqa: E402
from oflibnumpy_b200.device import DeviceArray, Event, Stream  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 32
H = int(sys.argv[2]) if len(sys.argv) > 2 else 1080
W = int(sys.argv[3]) if len(sys.argv) > 3 else 1920
PEAK = 6544.0
pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
if os.path.exists(pk):
    PEAK = float(json.load(open(pk))['hbm_gbs'])

of.device.require_gpu()
st = Stream()
of.device.set_stream(st)
rng = np.random.default_rng(0)
px = N * H * W

ta, tb = zip(*[(gi.cfg4_transforms(i), gi.cfg4_transforms(i + 100000)) for i in range(N)])
fa = of.FlowBatch.from_transforms(list(ta), (H, W), 't')
fb = of.FlowBatch.from_transforms(list(tb), (H, W), 't')
m1 = (rng.random((1, H, W)) > 0.02).astype(np.uint8)
for fl in (fa, fb):
    for i in range(N):
        d = fl.masks.frames(i, i + 1)
        _lib.call('ofk_rt_memcpy_h2d', d.ptr, m1.ctypes.data, d.nbytes, st.handle)
img1 = rng.integers(0, 256, (1, H, W, 3), dtype=np.uint8)
imgs = DeviceArray.empty((N, H, W, 3), np.uint8)
imgf = DeviceArray.empty((N, H, W, 3), np.float32)
img1f = img1.astype(np.float32)
for i in range(N):
    _lib.call('ofk_rt_memcpy_h2d', imgs.frames(i, i + 1).ptr, img1.ctypes.data, img1.nbytes, st.handle)
    _lib.call('ofk_rt_memcpy_h2d', imgf.frames(i, i + 1).ptr, img1f.ctypes.data, img1f.nbytes, st.handle)
st.synchronize()
o_img = DeviceArray.empty((N, H, W, 3), np.uint8)
o_imgf = DeviceArray.empty((N, H, W, 3), np.float32)
o_v = DeviceArray.empty((N, H, W, 2), np.float32)
o_m = DeviceArray.empty((N, H, W), np.uint8)
flags = DeviceArray.empty((N, 2), np.int32)
ws_bytes = _lib.call('ofk_forward_s_workspace', N, H, W)
ws = DeviceArray.empty((max(ws_bytes, 16),), np.uint8)
s = st.handle
results = []


def timeit(name, bytes_px, fn, reps=5):
    for _ in range(2):
        fn()
    st.synchronize()
    best = 1e30
    for _ in range(reps):
        e0, e1 = Event(), Event()
        e0.record(st)
        fn()
        e1.record(st)
        st.synchronize()
        best = min(best, e0.elapsed_ms(e1))
    gbs = px * bytes_px / best / 1e6
    print("%-52s %8.3f ms %9.1f Mpx/s %8.1f GB/s  %5.1f %% of %.0f" % (name, best, px / best / 1e3, gbs,
                                                                      100 * gbs / PEAK, PEAK))
    results.append({"op": name, "ms": best, "mpx_s": px / best / 1e3, "bytes_per_px": bytes_px, "gbs": gbs,
                    "frac": gbs / PEAK})


c = _lib.call
timeit("apply 't' u8x3, no valid area (14 B/px)", 14,
       lambda: c('ofk_warp_t', imgs.ptr, _lib.U8, 3, _lib.ARITH_NATIVE, fa.vecs.ptr, -1.0, None, None, o_img.ptr, None,
                 _lib.RULE_STRICT, N, H, W, H, W, 0, 0, 1, s))
timeit("apply 't' u8x3 + valid area (16 B/px)", 16,
       lambda: c('ofk_warp_t', imgs.ptr, _lib.U8, 3, _lib.ARITH_RINT, fa.vecs.ptr, -1.0, None, fa.masks.ptr, o_img.ptr,
                 o_m.ptr, _lib.RULE_GT_HALF, N, H, W, H, W, 0, 0, 1, s))
timeit("apply 't' u8x3 + target mask + valid (17 B/px)", 17,
       lambda: c('ofk_warp_t', imgs.ptr, _lib.U8, 3, _lib.ARITH_NATIVE, fa.vecs.ptr, -1.0, fb.masks.ptr, fa.masks.ptr,
                 o_img.ptr, o_m.ptr, _lib.RULE_GE_HALF, N, H, W, H, W, 0, 0, 1, s))
timeit("apply 't' f32x3 (32 B/px)", 32,
       lambda: c('ofk_warp_t', imgf.ptr, _lib.F32, 3, _lib.ARITH_NATIVE, fa.vecs.ptr, -1.0, None, None, o_imgf.ptr, None,
                 _lib.RULE_STRICT, N, H, W, H, W, 0, 0, 1, s))
img1c = DeviceArray.empty((N, H, W, 1), np.uint8)
o_img1c = DeviceArray.empty((N, H, W, 1), np.uint8)
img4c = DeviceArray.empty((N, H, W, 4), np.uint8)
o_img4c = DeviceArray.empty((N, H, W, 4), np.uint8)
imgf1 = DeviceArray.empty((N, H, W, 1), np.float32)
o_imgf1 = DeviceArray.empty((N, H, W, 1), np.float32)
timeit("apply 't' u8x1 + valid area (8+1+1+1+1 = 12 B/px)", 12,
       lambda: c('ofk_warp_t', img1c.ptr, _lib.U8, 1, _lib.ARITH_RINT, fa.vecs.ptr, -1.0, None, fa.masks.ptr, o_img1c.ptr,
                 o_m.ptr, _lib.RULE_GT_HALF, N, H, W, H, W, 0, 0, 1, s))
timeit("apply 't' u8x4 (8+4+4 = 16 B/px)", 16,
       lambda: c('ofk_warp_t', img4c.ptr, _lib.U8, 4, _lib.ARITH_NATIVE, fa.vecs.ptr, -1.0, None, None, o_img4c.ptr, None,
                 _lib.RULE_STRICT, N, H, W, H, W, 0, 0, 1, s))
timeit("apply 't' f32x1 + valid area (8+4+4+1+1 = 18 B/px)", 18,
       lambda: c('ofk_warp_t', imgf1.ptr, _lib.F32, 1, _lib.ARITH_NATIVE, fa.vecs.ptr, -1.0, None, fa.masks.ptr, o_imgf1.ptr,
                 o_m.ptr, _lib.RULE_STRICT, N, H, W, H, W, 0, 0, 1, s))
timeit("Flow.apply(Flow) 't' (27 B/px)", 27,
       lambda: c('ofk_warp_t', fb.vecs.ptr, _lib.F32, 2, _lib.ARITH_NATIVE, fa.vecs.ptr, -1.0, fb.masks.ptr, fa.masks.ptr,
                 o_v.ptr, o_m.ptr, _lib.RULE_STRICT, N, H, W, H, W, 0, 0, 1, s))
timeit("combine_with mode 3 't' (27 B/px)", 27,
       lambda: c('ofk_combine3', fa.vecs.ptr, fa.masks.ptr, fb.vecs.ptr, fb.masks.ptr, ord('t'), 0.0, o_v.ptr, o_m.ptr,
                 flags.ptr, N, H, W, s))
timeit("combine_with mode 3 's' (27 B/px)", 27,
       lambda: c('ofk_combine3', fa.vecs.ptr, fa.masks.ptr, fb.vecs.ptr, fb.masks.ptr, ord('s'), 0.0, o_v.ptr, o_m.ptr,
                 flags.ptr, N, H, W, s))
timeit("combine_flows mode 3 't', no masks (25 B/px)", 25,
       lambda: c('ofk_combine3', fa.vecs.ptr, None, fb.vecs.ptr, None, ord('t'), 0.0, o_v.ptr, o_m.ptr, flags.ptr, N, H,
                 W, s))
timeit("valid_target 't' (10 B/px)", 10,
       lambda: c('ofk_valid_geom_t', fa.vecs.ptr, -1.0, fa.masks.ptr, o_m.ptr, N, H, W, s))
mats = np.tile(np.eye(3)[None], (N, 1, 1))
mats[:, 0, 2] = 3.5
timeit("from_matrix (8 B/px)", 8, lambda: _ops.from_matrix(mats, (H, W), -1.0), reps=3)
timeit("Flow + Flow (27 B/px)", 27,
       lambda: c('ofk_addsub', _lib.OP_ADD, fa.vecs.ptr, fa.masks.ptr, fb.vecs.ptr, fb.masks.ptr, o_v.ptr, o_m.ptr, N, H,
                 W, s))
timeit("is_zero masked (9 B/px)", 9,
       lambda: c('ofk_nonzero_flags', fa.vecs.ptr, fa.masks.ptr, 0.0, flags.ptr, N, H, W, s))
timeit("switch_ref / invert same-ref: forward_s of vecs||mask (18 B/px)", 18,
       lambda: c('ofk_forward_s', fa.vecs.ptr, 2, fa.vecs.ptr, 1.0, fa.masks.ptr, None, o_v.ptr, o_m.ptr, _lib.RULE_STRICT,
                 N, H, W, ws.ptr, ws_bytes, s))
timeit("apply 's' f32x3 + valid (8+12+12+1 = 33 B/px)", 33,
       lambda: c('ofk_forward_s', imgf.ptr, 3, fa.vecs.ptr, 1.0, None, None, o_imgf.ptr, o_m.ptr, _lib.RULE_STRICT, N, H,
                 W, ws.ptr, ws_bytes, s))
# Flow.visualise is a per-frame call: ofk_visualise_batch of one frame, default range (magnitudes + exact 99th
# percentile by radix selection, on the device) + colourise
px_all, px = px, H * W
vis = DeviceArray.empty((H, W, 3), np.uint8)
vws_b = c('ofk_visualise_batch_workspace', 1, H, W)
vws = DeviceArray.empty((vws_b,), np.uint8)
timeit("visualise 'rgb', ONE frame, default range (8+1+3 = 12 B/px)", 12,
       lambda: c('ofk_visualise_batch', fa.vecs.ptr, fa.masks.ptr, 1e-3, 1, 1, 1, 0.0, vis.ptr, 1, H, W, vws.ptr, vws_b,
                 s))
timeit("visualise 'rgb', ONE frame, range_max given (12 B/px)", 12,
       lambda: c('ofk_visualise_batch', fa.vecs.ptr, fa.masks.ptr, 1e-3, 1, 1, 1, 25.0, vis.ptr, 1, H, W, None, 0, s))
px = px_all
print(json.dumps({"N": N, "H": H, "W": W, "peak_gbs": PEAK, "ops": results}))
