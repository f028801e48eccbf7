"""Device-level operations on batched DeviceArrays: one function per C-ABI hot-path entry point.

Shapes: flow vectors [N,H,W,2] float32, masks [N,H,W] uint8 (0/1), payloads [N,H,W,C]. Everything is asynchronous on
the current stream (device.set_stream) unless a result has to be read on the host.
"""
import numpy as np

from . import _lib
from . import device as dev
from .device import DeviceArray
from .validation import DEFAULT_THRESHOLD

DTYPE_CODES = {np.dtype('uint8'): _lib.U8, np.dtype('int16'): _lib.I16, np.dtype('uint16'): _lib.U16,
               np.dtype('float32'): _lib.F32, np.dtype('float64'): _lib.F64}


def _p(a):
    return None if a is None else a.ptr


def dtype_code(dtype):
    try:
        return DTYPE_CODES[np.dtype(dtype)]
    except KeyError:
        raise TypeError("Error applying flow: target dtype {} is not supported by the bilinear warp (supported: "
                        "uint8, int16, uint16, float32, float64 -- the dtypes cv2.remap accepts)".format(dtype))


def promoted_rule(payload_dtype, mask_is_bool):
    """(arith, mask_rule) of Flow.apply's `payload || mask` concatenation (flow_class.py:615,626,644): the numpy
    promotion of the payload dtype with int8 (no target_mask: np.ones(..., 'b')) or bool (target_mask given) decides
    which cv2.remap arithmetic samples both image and mask."""
    dt = np.dtype(payload_dtype)
    if dt == np.uint8:
        return (_lib.ARITH_NATIVE, _lib.RULE_GE_HALF) if mask_is_bool else (_lib.ARITH_RINT, _lib.RULE_GT_HALF)
    if dt == np.int16:
        return _lib.ARITH_NATIVE, _lib.RULE_GT_HALF
    if dt == np.uint16:
        if not mask_is_bool:
            raise TypeError("Error applying flow: a uint16 target with return_valid_area needs a boolean target_mask "
                            "(uint16 || int8 promotes to int32, which the bilinear warp -- like cv2.remap -- rejects)")
        return _lib.ARITH_NATIVE, _lib.RULE_GT_HALF
    if dt in (np.float32, np.float64):
        return _lib.ARITH_NATIVE, _lib.RULE_STRICT
    dtype_code(dt)  # raises
    raise AssertionError


def warp_t(flow, sign, payload=None, payload_mask=None, flow_mask=None, want_mask=False, arith=_lib.ARITH_NATIVE,
           rule=_lib.RULE_STRICT, placement=None, cut=True):
    """Backward warp (ofk_warp_t_ex). placement = (top, left) of the flow frame inside the payload frame. Frames of a
    float payload whose flow is zero below the threshold pass the payload through, as apply_flow does
    (utils.py:215-216), decided on the device; integer payloads come out of the identity taps unchanged anyway."""
    n, h, w = flow.shape[:3]
    if payload is not None:
        hs, ws, c = payload.shape[1:4]
        code = dtype_code(payload.dtype)
    else:
        hs, ws = (payload_mask.shape[1:3] if payload_mask is not None else (h, w))
        c, code = 0, _lib.U8
    top, left = placement if placement is not None else (0, 0)
    ho, wo = (h, w) if cut else (hs, ws)
    out = DeviceArray.empty((n, ho, wo, c), payload.dtype) if payload is not None else None
    omask = DeviceArray.empty((n, ho, wo), np.uint8) if want_mask else None
    nz = None
    if payload is not None and n and code in (_lib.F32, _lib.F64):
        nz = nonzero_flags_device(flow, None, DEFAULT_THRESHOLD)
    _lib.call('ofk_warp_t_ex', _p(payload), code, c, arith, flow.ptr, float(sign), _p(payload_mask), _p(flow_mask),
              _p(nz), _p(out), _p(omask), rule, n, h, w, hs, ws, top, left, 1 if cut else 0, dev.current_stream())
    return out, omask


def combine3(a, am, b, bm, ref, thr=0.0, want_flags=True):
    n, h, w = a.shape[:3]
    out = DeviceArray.empty((n, h, w, 2), np.float32)
    omask = DeviceArray.empty((n, h, w), np.uint8)
    flags = DeviceArray.empty((n, 2), np.int32) if want_flags else None
    _lib.call('ofk_combine3', a.ptr, _p(am), b.ptr, _p(bm), ord(ref), float(thr), out.ptr, omask.ptr, _p(flags), n, h,
              w, dev.current_stream())
    return out, omask, flags


def valid_geom_t(flow, sign, flow_mask):
    n, h, w = flow.shape[:3]
    out = DeviceArray.empty((n, h, w), np.uint8)
    _lib.call('ofk_valid_geom_t', flow.ptr, float(sign), _p(flow_mask), out.ptr, n, h, w, dev.current_stream())
    return out


def from_matrix(mats, shape, sign):
    """mats: numpy (N,3,3) float64 on the host (N <= 64) or a DeviceArray (N,3,3) float64."""
    h, w = shape
    if isinstance(mats, DeviceArray):
        n = mats.shape[0]
        out = DeviceArray.empty((n, h, w, 2), np.float32)
        _lib.call('ofk_from_matrix', mats.ptr, 0, float(sign), out.ptr, n, h, w, dev.current_stream())
        return out
    m = np.ascontiguousarray(mats, dtype=np.float64).reshape(-1, 3, 3)
    n = m.shape[0]
    if n > 64:
        return from_matrix(DeviceArray.from_numpy(m), shape, sign)
    out = DeviceArray.empty((n, h, w, 2), np.float32)
    _lib.call('ofk_from_matrix', m.ctypes.data, 1, float(sign), out.ptr, n, h, w, dev.current_stream())
    return out


def addsub(op, a, am, b, bm, want_mask=True):
    n, h, w = a.shape[:3]
    out = DeviceArray.empty((n, h, w, 2), np.float32)
    omask = DeviceArray.empty((n, h, w), np.uint8) if want_mask else None
    _lib.call('ofk_addsub', op, a.ptr, _p(am), b.ptr, _p(bm), out.ptr, _p(omask), n, h, w, dev.current_stream())
    return out, omask


def scale(op, a, su, sv, in_f64):
    out = DeviceArray.empty(a.shape, np.float32)
    _lib.call('ofk_scale', op, a.ptr, float(su), float(sv), 1 if in_f64 else 0, out.ptr, a.size // 2,
              dev.current_stream())
    return out


def scale_array(op, a, m, channels):
    out = DeviceArray.empty(a.shape, np.float32)
    _lib.call('ofk_scale_array', op, a.ptr, m.ptr, channels, out.ptr, a.size // 2, dev.current_stream())
    return out


def nonzero_flags(flow, mask, thr):
    """Host numpy int32 [N]: 1 where the frame has a non-zero (resp. >= thr) vector on a valid pixel. Synchronises."""
    n, h, w = flow.shape[:3]
    flags = DeviceArray.empty((n,), np.int32)
    _lib.call('ofk_nonzero_flags', flow.ptr, _p(mask), float(thr), flags.ptr, n, h, w, dev.current_stream())
    return flags.numpy()


def all_finite(arr):
    flag = DeviceArray.empty((1,), np.int32)
    _lib.call('ofk_check_finite', arr.ptr, arr.size, flag.ptr, dev.current_stream())
    return int(flag.numpy()[0]) == 0


def pad(vecs, mask, padding, mode):
    top, bottom, left, right = padding
    n, h, w = (vecs if vecs is not None else mask).shape[:3]
    ho, wo = h + top + bottom, w + left + right
    ov = DeviceArray.empty((n, ho, wo, 2), np.float32) if vecs is not None else None
    om = DeviceArray.empty((n, ho, wo), np.uint8)
    _lib.call('ofk_pad', _p(vecs), _p(mask), _p(ov), om.ptr, _lib.PAD_MODES[mode], n, h, w, top, bottom, left, right,
              dev.current_stream())
    return ov, om


def mask_and(a, b):
    out = DeviceArray.empty(a.shape, np.uint8)
    _lib.call('ofk_mask_and', a.ptr, b.ptr, out.ptr, a.size, dev.current_stream())
    return out


def crop(arr, y0, x0, h, w):
    """Cut [N,H,W,...] to [N,h,w,...]."""
    n, hh, ww = arr.shape[:3]
    inner = int(np.prod(arr.shape[3:], dtype=np.int64)) * arr.dtype.itemsize
    out = DeviceArray.empty((n, h, w) + arr.shape[3:], arr.dtype)
    _lib.call('ofk_crop', arr.ptr, out.ptr, inner, n, hh, ww, y0, x0, h, w, dev.current_stream())
    return out


def extent(flow, mask, sign, thr):
    n, h, w = flow.shape[:3]
    out = DeviceArray.empty((n, 4), np.float32)
    _lib.call('ofk_extent', flow.ptr, _p(mask), float(sign), float(thr), out.ptr, n, h, w, dev.current_stream())
    return out.numpy()


def vis_range_arg(range_max):
    """The range_max argument of ofk_visualise_batch / ofh_visualise: 0 for None (each frame's default range, found
    on the device), else the float32 value. A positive range that float32 cannot hold (rounds to 0) becomes -1, which
    the library rejects, instead of silently taking the default range."""
    if range_max is None:
        return 0.0
    r = float(np.float32(range_max))
    return r if r != 0 else -1.0


def visualise_batch(flow, mask, mode_code, show_mask, show_mask_borders, range_max, thr):
    """Flow.visualise of every frame in one ofk_visualise_batch call: flow [N,H,W,2], mask [N,H,W] or None. With
    range_max None the default range of each frame is found on the device (no read-back). Returns a device uint8
    [N,H,W,3] array; asynchronous."""
    n, h, w = flow.shape[:3]
    out = DeviceArray.empty((n, h, w, 3), np.uint8)
    ws, ws_bytes = None, 0
    if range_max is None:
        ws_bytes = _lib.call('ofk_visualise_batch_workspace', n, h, w)
        ws = DeviceArray.empty((max(ws_bytes, 16),), np.uint8)
    _lib.call('ofk_visualise_batch', flow.ptr, _p(mask), float(thr), mode_code, int(show_mask), int(show_mask_borders),
              vis_range_arg(range_max), out.ptr, n, h, w, _p(ws), ws_bytes, dev.current_stream())
    return out


def points_inside_area(pts, shape):
    p = np.ascontiguousarray(pts, dtype=np.float64)
    d = DeviceArray.from_numpy(p)
    out = DeviceArray.empty((p.shape[0],), np.uint8)
    _lib.call('ofk_points_inside_area', d.ptr, p.shape[0], int(shape[0]), int(shape[1]), out.ptr, dev.current_stream())
    return out.numpy().astype(bool)


def cast(arr, dtype, round_ints=True):
    """Device dtype conversion to / from float32 (ofk_cast)."""
    dtype = np.dtype(dtype)
    out = DeviceArray.empty(arr.shape, dtype)
    _lib.call('ofk_cast', arr.ptr, dtype_code(arr.dtype), out.ptr, dtype_code(dtype), arr.size, dev.current_stream())
    return out


def and_flags(a, b):
    """Element-wise AND of two device int32 0/1 flag arrays."""
    out = DeviceArray.empty(a.shape, np.int32)
    _lib.call('ofk_mask_and', a.ptr, b.ptr, out.ptr, a.nbytes, dev.current_stream())
    return out


def nonzero_flags_device(flow, mask, thr):
    """Device int32 [N] version of nonzero_flags (no synchronisation)."""
    n, h, w = flow.shape[:3]
    flags = DeviceArray.empty((n,), np.int32)
    _lib.call('ofk_nonzero_flags', flow.ptr, _p(mask), float(thr), flags.ptr, n, h, w, dev.current_stream())
    return flags


def forward_s(flow, sign, payload, payload_mask=None, point_mask=None, want_mask=True, rule=_lib.RULE_STRICT,
              flow_nonzero=None):
    """Forward (source-referenced) resampling of a float32 payload [N,H,W,C] (ofk_forward_s_ex). flow_nonzero: device
    int32 [N]; frames with 0 are passed through (apply_flow's early return for a thresholded-zero flow)."""
    n, h, w = flow.shape[:3]
    c = payload.shape[3] if payload is not None else 0
    out = DeviceArray.empty((n, h, w, c), np.float32) if c else None
    omask = DeviceArray.empty((n, h, w), np.uint8) if want_mask else None
    ws_bytes = _lib.call('ofk_forward_s_workspace', n, h, w)
    ws = DeviceArray.empty((max(ws_bytes, 16),), np.uint8)
    _lib.call('ofk_forward_s_ex', _p(payload), c, flow.ptr, float(sign), _p(payload_mask), _p(point_mask),
              _p(flow_nonzero), _p(out), _p(omask), rule, n, h, w, ws.ptr, ws_bytes, dev.current_stream())
    return out, omask


def combine12(mode, ref, a, am, b, bm):
    """combine_with modes 1 / 2 as one device-resident chain (ofk_combine12): flows [N,H,W,2], masks [N,H,W]."""
    n, h, w = a.shape[:3]
    out = DeviceArray.empty((n, h, w, 2), np.float32)
    omask = DeviceArray.empty((n, h, w), np.uint8)
    ws_bytes = _lib.call('ofk_combine12_workspace', mode, ord(ref), n, h, w)
    ws = DeviceArray.empty((max(ws_bytes, 16),), np.uint8)
    _lib.call('ofk_combine12', mode, ord(ref), a.ptr, _p(am), b.ptr, _p(bm), out.ptr, omask.ptr, n, h, w, ws.ptr,
              ws_bytes, dev.current_stream())
    return out, omask


def mesh_sample(mesh_flow, mesh_sign, payload, payload_mask, query_flow=None, query_sign=1.0, query_pts=None,
                pos_f32=False, want_mask=True, want_found=False):
    """Scattered-to-scattered interpolation on the displaced-grid mesh (ofk_mesh_sample)."""
    n, h, w = mesh_flow.shape[:3]
    c = payload.shape[3] if payload is not None else 0
    if query_pts is not None:
        q = query_pts.shape[1]
        oshape = (n, q)
    else:
        q = h * w
        oshape = (n, h, w)
    out = DeviceArray.empty(oshape + (c,), np.float32) if c else None
    mval = DeviceArray.empty(oshape, np.float32) if want_mask else None
    found = DeviceArray.empty(oshape, np.uint8) if want_found else None
    _lib.call('ofk_mesh_sample', mesh_flow.ptr, float(mesh_sign), 1 if pos_f32 else 0, _p(payload), c,
              _p(payload_mask), _p(query_flow), float(query_sign), _p(query_pts), q, _p(out), _p(mval), _p(found), n, h,
              w, dev.current_stream())
    return out, mval, found


def greater(values, thr):
    out = DeviceArray.empty(values.shape, np.uint8)
    _lib.call('ofk_greater', values.ptr, float(thr), out.ptr, values.size, dev.current_stream())
    return out


TRACK_PTS_CODES = {np.dtype('float32'): _lib.F32, np.dtype('float64'): _lib.F64, np.dtype('int32'): _lib.I32,
                   np.dtype('int64'): _lib.I64}


def track(flow, mask, ref, exact, flow_nonzero, pts, arith_dtype, int_out, status_plane=None, want_status=False):
    """Flow.track of every frame in one ofk_track call: flow [N,H,W,2], pts device [N,P,2] or [P,2] of a
    TRACK_PTS_CODES dtype. Returns device arrays (tracked [N,P,2] of arith_dtype or int32, status uint8 [N,P] or None,
    error words int32 [N]); asynchronous."""
    n, h, w = flow.shape[:3]
    p = pts.shape[-2]
    out = DeviceArray.empty((n, p, 2), np.int32 if int_out else arith_dtype)
    status = DeviceArray.empty((n, p), np.uint8) if want_status else None
    errors = DeviceArray.empty((n,), np.int32)
    _lib.call('ofk_track', flow.ptr, _p(mask), ord(ref), int(exact), flow_nonzero.ptr, pts.ptr,
              TRACK_PTS_CODES[pts.dtype], int(pts.ndim == 2), p, DTYPE_CODES[np.dtype(arith_dtype)], int(int_out),
              out.ptr, _p(status_plane), _p(status), errors.ptr, n, h, w, dev.current_stream())
    return out, status, errors


def track_clips(flow, mask, ref, exact, flow_nonzero, pts, s, l, keep):
    """Trajectories through S clips of L frames in one ofk_track_clips call: flow [S*L,H,W,2], pts device float32 /
    float64 [S,P,2] or [P,2], keep uint8 [S*L,H,W] or None. Returns device arrays (positions float64 [S*L,P,2], alive
    uint8 [S*L,P]); asynchronous."""
    n, h, w = flow.shape[:3]
    p = pts.shape[-2]
    out = DeviceArray.empty((n, p, 2), np.float64)
    alive = DeviceArray.empty((n, p), np.uint8)
    _lib.call('ofk_track_clips', flow.ptr, _p(mask), ord(ref), int(exact), flow_nonzero.ptr, pts.ptr,
              TRACK_PTS_CODES[pts.dtype], int(pts.ndim == 2), s, l, p, _p(keep), out.ptr, alive.ptr, h, w,
              dev.current_stream())
    return out, alive


def resize_flow(vecs, mask, fy, fx):
    """cv2.resize semantics: output size = round-half-even(size * scale) (ofk_resize_flow)."""
    n, h, w = (vecs if vecs is not None else mask).shape[:3]
    ho, wo = int(np.rint(h * float(fy))), int(np.rint(w * float(fx)))
    if ho < 1 or wo < 1:
        raise ValueError("Error resizing flow: Scale values result in an empty flow field")
    ov = DeviceArray.empty((n, ho, wo, 2), np.float32) if vecs is not None else None
    om = DeviceArray.empty((n, ho, wo), np.uint8) if mask is not None else None
    _lib.call('ofk_resize_flow', _p(vecs), _p(mask), _p(ov), _p(om), n, h, w, ho, wo, float(fy), float(fx),
              dev.current_stream())
    return ov, om


def fit_matrix(flow, mask, ref, dof, method, hypotheses, thr, masked, want_inliers):
    """Flow.matrix of every frame in one ofk_fit_matrix call: flow [N,H,W,2], mask [N,H,W]. Returns device arrays
    (matrices float64 [N,3,3], inliers uint8 [N,H,W] or None, counts int32 [N]); asynchronous."""
    n, h, w = flow.shape[:3]
    code = _lib.FIT_METHODS[method]
    mats = DeviceArray.empty((n, 3, 3), np.float64)
    inliers = DeviceArray.empty((n, h, w), np.uint8) if want_inliers else None
    counts = DeviceArray.empty((n,), np.int32)
    ws_bytes = _lib.call('ofk_fit_matrix_workspace', dof, code, hypotheses, n, h, w)
    ws = DeviceArray.empty((max(ws_bytes, 16),), np.uint8)
    _lib.call('ofk_fit_matrix', flow.ptr, _p(mask), ord(ref), dof, code, hypotheses, float(thr), int(masked), mats.ptr,
              _p(inliers), counts.ptr, n, h, w, ws.ptr, ws_bytes, dev.current_stream())
    return mats, inliers, counts


def accumulate(flow, mask, ref, thr, s, l, cumulative, fold):
    """Mode-3 composition folded ('left' or 'right') over S clips of L frames in one ofk_accumulate_fold call: flow
    [S*L,H,W,2], mask [S*L,H,W]. Returns device arrays (vecs [S*L or S,H,W,2] float32, masks uint8 of the same
    frames); asynchronous."""
    h, w = flow.shape[1:3]
    n_out = s * l if cumulative else s
    out = DeviceArray.empty((n_out, h, w, 2), np.float32)
    omask = DeviceArray.empty((n_out, h, w), np.uint8)
    ws_bytes = _lib.call('ofk_accumulate_fold_workspace', ord(ref), ord(fold[0]), s, l, h, w, int(cumulative))
    ws = DeviceArray.empty((max(ws_bytes, 16),), np.uint8)
    _lib.call('ofk_accumulate_fold', flow.ptr, mask.ptr, ord(ref), ord(fold[0]), float(thr), s, l, h, w,
              int(cumulative), out.ptr, omask.ptr, ws.ptr, ws_bytes, dev.current_stream())
    return out, omask


def consistency(f, fm, g, gm, ref, alpha_1, alpha_2, want_valid):
    """Forward-backward consistency of every frame in one ofk_consistency call: forward flow f and backward flow g
    [N,H,W,2] with masks [N,H,W]. Returns device uint8 arrays (consistent [N,H,W], valid [N,H,W] or None);
    asynchronous, no launch for N = 0."""
    n, h, w = f.shape[:3]
    out = DeviceArray.empty((n, h, w), np.uint8)
    valid = DeviceArray.empty((n, h, w), np.uint8) if want_valid else None
    if n:
        _lib.call('ofk_consistency', f.ptr, _p(fm), g.ptr, _p(gm), ord(ref), float(np.float32(alpha_1)),
                  float(np.float32(alpha_2)), out.ptr, _p(valid), n, h, w, dev.current_stream())
    return out, valid


def evaluate(est, est_mask, truth, truth_mask, region, want_epe):
    """Error metrics of every frame in one ofk_evaluate call: estimates and truth [N,H,W,2], masks and region [N,H,W]
    or None. Returns device arrays (counts int64 [N,8], sums float64 [N,5], EPE map float32 [N,H,W] or None);
    asynchronous, no launch for N = 0."""
    n, h, w = est.shape[:3]
    counts = DeviceArray.empty((n, 8), np.int64)
    sums = DeviceArray.empty((n, 5), np.float64)
    epe = DeviceArray.empty((n, h, w), np.float32) if want_epe else None
    if n:
        ws_bytes = _lib.call('ofk_evaluate_workspace', n, h, w)
        ws = DeviceArray.empty((ws_bytes,), np.uint8)
        _lib.call('ofk_evaluate', est.ptr, _p(est_mask), truth.ptr, _p(truth_mask), _p(region), _p(epe), counts.ptr,
                  sums.ptr, n, h, w, ws.ptr, ws_bytes, dev.current_stream())
    return counts, sums, epe
