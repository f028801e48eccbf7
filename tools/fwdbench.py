"""Device benchmark of the source-referenced resampler (ofk_forward_s) over the regimes that matter:

    python tools/fwdbench.py [N] [H] [W]

rotation-type flows (cfg 4 transforms) without / with 2 % of the points removed (`consider_mask`), a smooth
non-affine field (curved frame border -> hull pockets), and a folding field (an occlusion band: the frame is
triangulated as a whole) as one frame and as a batch of 16. Device-resident inputs, CUDA events on the library's
stream.
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
from oflibnumpy_b200 import _lib  # noqa: E402
from oflibnumpy_b200.device import DeviceArray, Event, Stream  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 16
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
fa = of.FlowBatch.from_transforms([gi.cfg4_transforms(i) for i in range(N)], (H, W), 's')
sm = np.ascontiguousarray(np.broadcast_to(gi.smooth_field(H, W)[None], (N, H, W, 2)))
fsm = of.FlowBatch(sm, 's')
mask = DeviceArray.from_numpy(np.ascontiguousarray(np.broadcast_to((rng.random((1, H, W)) > 0.02), (N, H, W))).view(np.uint8))
imgf = DeviceArray.from_numpy((rng.random((N, H, W, 3)) * 255).astype(np.float32))
o_v = DeviceArray.empty((N, H, W, 2), np.float32)
o_f = DeviceArray.empty((N, H, W, 3), np.float32)
o_m = DeviceArray.empty((N, H, W), np.uint8)
ws_bytes = _lib.call('ofk_forward_s_workspace', N, H, W)
ws = DeviceArray.empty((max(ws_bytes, 16),), np.uint8)
s = st.handle
c = _lib.call
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
    print("%-64s %9.3f ms %9.1f Mpx/s %8.1f GB/s  %5.1f %% of %.0f" % (name, best, px / best / 1e3, gbs,
                                                                      100 * gbs / PEAK, PEAK), flush=True)
    results.append({"op": name, "ms": best, "mpx_s": px / best / 1e3, "bytes_per_px": bytes_px, "gbs": gbs,
                    "frac": gbs / PEAK})


def fwd(payload, C, flow, pm, pt, out):
    return lambda: c('ofk_forward_s', payload.ptr if payload is not None else None, C, flow.ptr, 1.0,
                     pm.ptr if pm is not None else None, pt.ptr if pt is not None else None,
                     out.ptr if out is not None else None, o_m.ptr, _lib.RULE_STRICT, N, H, W, ws.ptr, ws_bytes, s)


stats0 = [c('ofk_rt_path_count', k) for k in range(6, 10)]
timeit("rotation: invert / switch_ref, full masks (18 B/px)", 18, fwd(fa.vecs, 2, fa.vecs, fa.masks, None, o_v))
timeit("rotation: apply 's' f32x3 + valid (33 B/px)", 33, fwd(imgf, 3, fa.vecs, None, None, o_f))
timeit("rotation: valid_target 's' (8+1+1 = 10 B/px)", 10, fwd(None, 0, fa.vecs, fa.masks, None, None))
timeit("smooth field: invert as Flow.invert() calls it (all-true point mask)", 18, fwd(fsm.vecs, 2, fsm.vecs, fsm.masks, fsm.masks, o_v), reps=3)
timeit("rotation: invert, 2 % points removed, consider_mask (18 B/px)", 18, fwd(fa.vecs, 2, fa.vecs, mask, mask, o_v))
timeit("rotation: invert, 2 % masked, consider_mask=False (18 B/px)", 18, fwd(fa.vecs, 2, fa.vecs, mask, None, o_v))
timeit("smooth field: invert, full masks (18 B/px)", 18, fwd(fsm.vecs, 2, fsm.vecs, fsm.masks, None, o_v), reps=3)
timeit("smooth field: invert, 2 % points removed (18 B/px)", 18, fwd(fsm.vecs, 2, fsm.vecs, mask, mask, o_v), reps=3)
stats1 = [c('ofk_rt_path_count', k) for k in range(6, 10)]


def folds(vecs):
    """Cells of the displaced grid that are not positively oriented convex quadrilaterals (a folding field)."""
    y, x = np.mgrid[:vecs.shape[0], :vecs.shape[1]].astype(np.float64)
    px, py = x + vecs[..., 0].astype(np.float64), y + vecs[..., 1].astype(np.float64)
    a, b, cc, d = [(px[i:i + vecs.shape[0] - 1, j:j + vecs.shape[1] - 1], py[i:i + vecs.shape[0] - 1, j:j + vecs.shape[1] - 1])
                   for i, j in ((0, 0), (0, 1), (1, 0), (1, 1))]

    def orient(p, q, r):
        return (q[0] - p[0]) * (r[1] - p[1]) - (q[1] - p[1]) * (r[0] - p[0])
    ok = (orient(a, b, d) > 0) & (orient(a, d, cc) > 0) & (orient(a, b, cc) > 0) & (orient(b, d, cc) > 0)
    return int((~ok).sum())


# the fields of bench.py's forward_s block must not fold (a folding frame is triangulated as a whole, far slower)
print("cells that fold: rotation %d, smooth %d" % (sum(folds(v) for v in fa.vecs.numpy()), folds(gi.smooth_field(H, W))),
      flush=True)


def fold_field(h, w):
    """An occlusion band moving 6 px over a slightly sheared background, as estimated flows have them."""
    y, x = np.mgrid[:h, :w].astype(np.float64)
    band = (x > 0.4 * w) & (x < 0.65 * w)
    return np.dstack([np.where(band, 6.0, 0.3) + 0.02 * y + 0.013 * x, 0.1 + 0.01 * x + 0.017 * y]).astype(np.float32)


for nf in (1, 16):
    fv = DeviceArray.from_numpy(np.ascontiguousarray(np.broadcast_to(fold_field(H, W)[None], (nf, H, W, 2))))
    fo = DeviceArray.empty((nf, H, W, 2), np.float32)
    fm = DeviceArray.empty((nf, H, W), np.uint8)
    fws_bytes = _lib.call('ofk_forward_s_workspace', nf, H, W)
    fws = DeviceArray.empty((max(fws_bytes, 16),), np.uint8)
    run = (lambda nf=nf, fv=fv, fo=fo, fm=fm, fws=fws, fws_bytes=fws_bytes:
           c('ofk_forward_s', fv.ptr, 2, fv.ptr, 1.0, None, None, fo.ptr, fm.ptr, _lib.RULE_STRICT, nf, H, W, fws.ptr,
             fws_bytes, s))
    px_all = px
    px = nf * H * W
    timeit("folding field (occlusion band): invert, %d frame%s (18 B/px)" % (nf, "s" if nf > 1 else ""), 18, run, reps=3)
    px = px_all
print(json.dumps({"N": N, "H": H, "W": W, "peak_gbs": PEAK, "ops": results,
                  "irregular_pixels": dict(zip(("located", "outside_by_search", "failed", "hull_rejected"),
                                               [b - a for a, b in zip(stats0, stats1)]))}))
