"""Batched extension of the API: N independent flow fields of one shape processed by single kernel launches.

The reference has no batch axis (SURVEY section 2.2); ``FlowBatch`` is how batches of frame / flow pairs are sharded
over GPUs (one process per GPU, contiguous split of the batch axis, no data-path collective). Frame ``i`` of every
result equals what the single-frame :class:`Flow` method returns for frame ``i`` of the inputs.
"""
import numpy as np

from . import _lib
from . import _ops
from . import device as dev
from .device import DeviceArray
from .flow import Flow
from .validation import get_valid_ref, validate_shape, validate_transform_list, validate_visualise_args, \
    validate_track_args, validate_track_dtype, validate_matrix_args, validate_accumulate_args, \
    validate_consistency_args, validate_evaluate_args, validate_track_clips_args, DEFAULT_THRESHOLD

__all__ = ['FlowBatch', 'FlowErrors', 'shard_range', 'apply_flow_host', 'combine_flows_host', 'apply_combine_host',
           'visualise_flows_host', 'evaluate_flows_host']


def shard_range(n, rank, world):
    """Contiguous split of ``n`` frames over ``world`` ranks -> [start, stop) of ``rank`` (sizes differ by <= 1)."""
    base, rem = divmod(n, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def _to_device(x, dtype=None):
    if isinstance(x, np.ndarray):
        return DeviceArray.from_numpy(x, dtype)
    return dev.as_device(x, dtype)


class FlowBatch(object):
    def __init__(self, vecs, ref=None, masks=None, validate=True):
        """:param vecs: (N,H,W,2) float32 numpy or device array; :param masks: (N,H,W) bool/uint8 or None"""
        self.ref = get_valid_ref(ref)
        if isinstance(vecs, np.ndarray):
            if vecs.ndim != 4 or vecs.shape[3] != 2:
                raise ValueError("Error setting flow vectors: batch input needs shape (N,H,W,2)")
        v = _to_device(vecs, np.float32) if not isinstance(vecs, np.ndarray) else \
            DeviceArray.from_numpy(vecs, np.float32)
        if v.ndim != 4 or v.shape[3] != 2:
            raise ValueError("Error setting flow vectors: batch input needs shape (N,H,W,2)")
        if validate and not _ops.all_finite(v):
            raise ValueError("Error setting flow vectors: Input contains NaN, Inf or -Inf values")
        self.vecs = v
        if masks is None:
            m = DeviceArray.empty(v.shape[:3], np.uint8)
            _lib.call('ofk_rt_memset', m.ptr, 1, m.nbytes, dev.current_stream())
        elif isinstance(masks, np.ndarray):
            if masks.shape != v.shape[:3]:
                raise ValueError("Error setting flow mask: Input has a different shape than the flow vectors")
            if masks.dtype != np.bool_ and ((masks != 0) & (masks != 1)).any():
                raise ValueError("Error setting flow mask: Values must be 0 or 1")
            m = DeviceArray.from_numpy(masks.astype(np.bool_).view(np.uint8))
        else:
            d = dev.as_device(masks)
            if d.shape != v.shape[:3] or d.dtype not in (np.uint8, np.bool_):
                raise ValueError("Error setting flow mask: device mask needs shape (N,H,W) and dtype bool/uint8")
            m = DeviceArray(d.ptr, d.shape, np.uint8, owner=d)
        self.masks = m

    @classmethod
    def _wrap(cls, vecs, ref, masks):
        b = cls.__new__(cls)
        b.vecs, b.ref, b.masks = vecs, ref, masks
        return b

    # ------------------------------------------------------------------------------------------------ basics
    def __len__(self):
        return self.vecs.shape[0]

    @property
    def shape(self):
        return tuple(self.vecs.shape[1:3])

    def __getitem__(self, i):
        """Frame ``i`` as a single :class:`Flow` (device view, no copy); a slice gives a FlowBatch view."""
        n = len(self)
        if isinstance(i, slice):
            start, stop, step = i.indices(n)
            if step != 1:
                raise IndexError("FlowBatch slices need unit step")
            return FlowBatch._wrap(self.vecs.frames(start, stop), self.ref, self.masks.frames(start, stop))
        if i < 0:
            i += n
        if not 0 <= i < n:
            raise IndexError("frame index out of range")
        return Flow._wrap(self.vecs.frames(i, i + 1), self.ref, self.masks.frames(i, i + 1))

    def shard(self, rank, world):
        start, stop = shard_range(len(self), rank, world)
        return self[start:stop]

    def numpy(self):
        return self.vecs.numpy(), self.masks.numpy().view(np.bool_)

    @classmethod
    def from_transforms(cls, transform_lists, shape, ref=None, masks=None):
        """One transform list per frame (Flow.from_transforms semantics, evaluated by one launch)."""
        from .ops import matrix_from_transforms
        validate_shape(shape)
        ref = get_valid_ref(ref)
        mats = []
        for tl in transform_lists:
            validate_transform_list(tl)
            m = matrix_from_transforms(tl)
            mats.append(m if ref == 's' else np.linalg.pinv(m))
        v = _ops.from_matrix(np.stack(mats), shape, 1.0 if ref == 's' else -1.0)
        b = cls._wrap(v, ref, None)
        if masks is None:
            m = DeviceArray.empty(v.shape[:3], np.uint8)
            _lib.call('ofk_rt_memset', m.ptr, 1, m.nbytes, dev.current_stream())
            b.masks = m
        else:
            b.masks = cls(v, ref, masks, validate=False).masks
        return b

    # ------------------------------------------------------------------------------------------------ hot path
    def apply(self, targets, target_masks=None, return_valid_area=False, consider_mask=True):
        """Warp images (N,H,W,C) [numpy or device] frame by frame with this batch, like ``Flow.apply`` (ref 't':
        ofk_warp_t, ref 's': ofk_forward_s). Returns device arrays (``.numpy()`` to download): images in the dtype of
        the targets (ref 's' resamples in float32 and rounds integer targets like the reference), and the valid areas
        if requested."""
        payload = _to_device(targets)
        if payload.ndim == 3:
            payload = payload.reshape(payload.shape + (1,))
        if payload.shape[:3] != self.vecs.shape[:3]:
            raise ValueError("Error applying flow: Flow shape does not match target shape")
        if self.ref == 's':
            return self._apply_s(payload, target_masks, return_valid_area, consider_mask)
        pmask = None
        if return_valid_area:
            arith, rule = _ops.promoted_rule(payload.dtype, target_masks is not None)
            if target_masks is not None:
                pmask = _to_device(target_masks.view(np.uint8) if isinstance(target_masks, np.ndarray) else
                                   target_masks)
        else:
            arith, rule = _lib.ARITH_NATIVE, _lib.RULE_STRICT
        out, omask = _ops.warp_t(self.vecs, -1.0, payload, pmask, self.masks if return_valid_area else None,
                                 return_valid_area, arith, rule)
        return (out, omask) if return_valid_area else out

    def _zero_flags(self):
        """Device int32 [N]: 0 where the flow is zero below the threshold (apply_flow passes its target through)."""
        return _ops.nonzero_flags_device(self.vecs, None, DEFAULT_THRESHOLD)

    def _apply_s(self, payload, target_masks, return_valid_area, consider_mask):
        out_dtype = payload.dtype
        is_int = np.issubdtype(out_dtype, np.integer)
        pay32 = payload if out_dtype == np.float32 else _ops.cast(payload, np.float32)
        pmask = None
        if return_valid_area:
            pmask = self.masks
            if target_masks is not None:
                tm = _to_device(target_masks.view(np.uint8) if isinstance(target_masks, np.ndarray) else target_masks)
                pmask = _ops.mask_and(DeviceArray(tm.ptr, tm.shape, np.uint8, owner=tm), self.masks)
        rule = _lib.RULE_GT_HALF if is_int else _lib.RULE_STRICT
        out, omask = _ops.forward_s(self.vecs, 1.0, pay32, pmask, self.masks if consider_mask else None,
                                    return_valid_area, rule, flow_nonzero=self._zero_flags())
        if out_dtype != np.float32:
            out = _ops.cast(out, out_dtype, round_ints=True)
        return (out, omask) if return_valid_area else out

    def apply_to_flows(self, other, consider_mask=True):
        """``self[i].apply(other[i])`` for every frame: warp a batch of flows (vectors and masks) with this batch."""
        if self.ref != 't':
            pm = _ops.mask_and(other.masks, self.masks)
            out, omask = _ops.forward_s(self.vecs, 1.0, other.vecs, pm, self.masks if consider_mask else None, True,
                                        _lib.RULE_STRICT, flow_nonzero=self._zero_flags())
            return FlowBatch._wrap(out, other.ref, omask)
        out, omask = _ops.warp_t(self.vecs, -1.0, other.vecs, other.masks, self.masks, True, _lib.ARITH_NATIVE,
                                 _lib.RULE_STRICT)
        return FlowBatch._wrap(out, other.ref, omask)

    def combine_with(self, other, mode, thresholded=False, return_flags=False):
        """Frame-wise ``self[i].combine_with(other[i], mode)``; mode 3 is one fused launch for the whole batch, the
        zero-flow early exits of the reference are resolved on the device (no host round trip)."""
        if not isinstance(other, FlowBatch):
            raise TypeError("Error combining flows: Flow need to be of type 'FlowBatch'")
        if self.vecs.shape != other.vecs.shape:
            raise ValueError("Error combining flows: Flow fields need to have the same shape")
        if self.ref != other.ref:
            raise ValueError("Error combining flows: Flow fields need to have the same reference")
        if mode not in (1, 2, 3):
            raise ValueError("Error combining flows: Mode needs to be 1, 2 or 3")
        thr = DEFAULT_THRESHOLD if thresholded else 0.0
        if mode == 3:
            v, m, flags = _ops.combine3(self.vecs, self.masks, other.vecs, other.masks, self.ref, thr)
            res = FlowBatch._wrap(v, self.ref, m)
            return (res, flags) if return_flags else res
        # modes 1 and 2: one device-resident chain for the whole batch (ofk_combine12). The reference's early exits
        # (self zero -> flow, flow zero -> self.invert(); flow_class.py:1338-1354) are rare: the two zero tests are
        # read back once and those frames redone through the single-frame path
        v, m = _ops.combine12(mode, self.ref, self.vecs, self.masks, other.vecs, other.masks)
        a_nz = _ops.nonzero_flags(self.vecs, self.masks, thr)
        b_nz = _ops.nonzero_flags(other.vecs, other.masks, thr)
        res = FlowBatch._wrap(v, self.ref, m)
        for i in np.flatnonzero((a_nz == 0) | (b_nz == 0)):
            one = self[int(i)].combine_with(other[int(i)], mode, thresholded)
            res.vecs.frames(int(i), int(i) + 1).copy_from(one._vd())
            res.masks.frames(int(i), int(i) + 1).copy_from(one._md())
        flags = np.stack([a_nz, b_nz], 1)
        return (res, flags) if return_flags else res

    def valid_target(self, consider_mask=True):
        """Device uint8 (N,H,W): Flow.valid_target frame by frame (flow_class.py:1113-1151)."""
        if self.ref == 't':
            return _ops.valid_geom_t(self.vecs, -1.0, self.masks)
        _, area = _ops.forward_s(self.vecs, 1.0, None, self.masks, self.masks if consider_mask else None,
                                 flow_nonzero=self._zero_flags())
        return area

    def valid_source(self, consider_mask=True):
        if self.ref == 's':
            return _ops.valid_geom_t(self.vecs, 1.0, self.masks)
        _, area = _ops.forward_s(self.vecs, -1.0, None, self.masks, self.masks if consider_mask else None,
                                 flow_nonzero=self._zero_flags())
        return area

    def _negated(self):
        return _ops.scale(_lib.OP_MUL, self.vecs, -1.0, -1.0, False)

    def switch_ref(self, mode='valid'):
        """Frame-wise Flow.switch_ref (flow_class.py:697-733): one forward resampling of vectors and mask; frames whose
        flow is exactly zero on its valid pixels, or zero below the threshold everywhere, are only relabelled (the two
        tests run on the device)."""
        other = 't' if self.ref == 's' else 's'
        if mode == 'invalid':
            return FlowBatch._wrap(self.vecs, other, self.masks)
        if mode != 'valid':
            raise ValueError("Error switching flow reference: Mode not recognised, should be 'valid' or 'invalid'")
        active = _ops.and_flags(self._zero_flags(), _ops.nonzero_flags_device(self.vecs, self.masks, 0.0))
        out, omask = _ops.forward_s(self.vecs, 1.0 if self.ref == 's' else -1.0, self.vecs, self.masks, self.masks,
                                    True, _lib.RULE_STRICT, flow_nonzero=active)
        return FlowBatch._wrap(out, other, omask)

    def invert(self, ref=None):
        """Frame-wise Flow.invert (flow_class.py:735-753): cross-reference = negate + relabel, same reference = one
        forward resampling (s -> s: self.apply(-self); t -> t: self.invert('s').switch_ref())."""
        ref = self.ref if ref is None else get_valid_ref(ref)
        if ref != self.ref:
            return FlowBatch._wrap(self._negated(), ref, self.masks)
        if self.ref == 's':
            neg = self._negated()
            out, omask = _ops.forward_s(self.vecs, 1.0, neg, self.masks, self.masks, True, _lib.RULE_STRICT,
                                        flow_nonzero=self._zero_flags())
            return FlowBatch._wrap(out, 's', omask)
        return FlowBatch._wrap(self._negated(), 's', self.masks).switch_ref()

    def visualise(self, mode, show_mask=None, show_mask_borders=None, range_max=None):
        """Frame-wise ``Flow.visualise`` (flow_class.py:869-951) in one ofk_visualise_batch call: frame ``i`` is
        ``self[i].visualise(mode, show_mask, show_mask_borders, range_max)``, bit for bit. The default range of each
        frame (99th percentile of its magnitudes, else the maximum, else 1) is found on the device: no synchronisation,
        no read-back. Returns a device uint8 array (N,H,W,3) (``.numpy()`` to download)."""
        code, show_mask, show_mask_borders = validate_visualise_args(mode, show_mask, show_mask_borders, range_max)
        return _ops.visualise_batch(self.vecs, self.masks, code, show_mask, show_mask_borders, range_max,
                                    DEFAULT_THRESHOLD)

    def track(self, pts, int_out=None, get_valid_status=None, s_exact_mode=None):
        """Frame-wise ``Flow.track`` (flow_class.py:755-795) in one ofk_track call. ``pts`` (row, col) is (N,P,2), frame
        ``i`` using ``pts[i]``, or (P,2), the same points in every frame; a numpy array or a device array
        (``DeviceArray``, any ``__cuda_array_interface__`` exporter such as a torch.cuda tensor; float32, float64, int32
        or int64). Frame ``i`` of the result is ``self[i].track(pts_i, int_out, False, s_exact_mode)`` bit for bit, in
        the dtype ``Flow.track`` gives a frame with non-zero flow (integer points on an 's' flow:
        ``np.result_type(pts.dtype, np.float32)``; otherwise float64; int32 with ``int_out``). Frames whose flow is zero
        below the threshold hold their points converted to that dtype.

        Returns a device array (N,P,2), and with ``get_valid_status`` also a device uint8 (N,P) of 0/1, the status
        ``self[i].track(pts_i, get_valid_status=True)`` returns (``.numpy()`` to download, ``.view(bool)`` for numpy's
        type). Ref 't' status reads the batch's valid_source plane (one forward resampling per frame).

        Raises IndexError where a loop of ``Flow.track`` would, for the lowest such frame. Host points are range-tested
        in numpy first: when they all pass, the call returns without synchronising. Otherwise, and always for device
        points, the per-frame error words of the kernel are read back, which synchronises with the device."""
        host = isinstance(pts, np.ndarray)
        if not host and dev.is_device_array(pts):
            pts = dev.as_device(pts)
        n, (h, w) = len(self), self.shape
        int_out, get_valid_status, s_exact_mode = validate_track_args(pts, int_out, get_valid_status, s_exact_mode, n)
        validate_track_dtype(pts.dtype)
        is_int = np.issubdtype(pts.dtype, np.integer)
        lookup = self.ref == 's' and (is_int or not s_exact_mode)        # Flow.track looks integer points up
        arith = np.result_type(pts.dtype, np.float32) if lookup and is_int else np.dtype(np.float64)
        if host:
            if pts.dtype not in _ops.TRACK_PTS_CODES:           # int8 ... uint16 -> int32 (arith float32 if lookup)
                pts = pts.astype(np.int32 if is_int and pts.dtype.itemsize < 4 else
                                 (np.int64 if is_int else np.float64))
            bad = _track_range_fails(pts, lookup, is_int, get_valid_status, h, w)
            dpts = DeviceArray.from_numpy(pts)
        else:
            if pts.dtype not in _ops.TRACK_PTS_CODES:
                raise TypeError("Error tracking points: device points need dtype float32, float64, int32 or int64, not "
                                "{}".format(pts.dtype))
            bad, dpts = True, pts
        p = pts.shape[-2]
        if n == 0 or p == 0:
            out = DeviceArray.empty((n, p, 2), np.int32 if int_out else arith)
            return (out, DeviceArray.empty((n, p), np.uint8)) if get_valid_status else out
        plane = self.valid_source() if get_valid_status and self.ref == 't' else None
        out, status, errors = _ops.track(self.vecs, self.masks, self.ref, s_exact_mode, self._zero_flags(), dpts,
                                         arith, int_out, plane, get_valid_status)
        if bad:
            _raise_track_error(errors.numpy(), h, w)
        return (out, status) if get_valid_status else out

    def track_clips(self, pts, clip_length=None, keep=None, s_exact_mode=None):
        """Point trajectories through clips (Sundaram, Brox & Keutzer, ECCV 2010) in one ofk_track_clips launch: each
        point is chained through the frames of its clip by ``Flow.track`` steps and dropped where a step fails. The
        batch is clip-major as for ``accumulate``: N / L clips of L = ``clip_length`` frames (default: one clip of
        all N), frame ``s*L + k`` the flow from frame k to frame k+1 of clip s.

        ``pts`` (row, col) in frame 0 is (S,P,2), points per clip, or (P,2), the same points in every clip; a numpy
        array of a float or int dtype (integers are tracked as their float64 values, not looked up as ``Flow.track``
        does), or a float32 / float64 device array (``DeviceArray``, any ``__cuda_array_interface__`` exporter such as
        a torch.cuda tensor). ``keep`` (N,H,W) bool / uint8, numpy or device, on the grid of each frame of the batch:
        ``fw.consistent_with(bw)`` stops trajectories at occlusions. ``s_exact_mode`` as in ``Flow.track``.

        One step of a live point q (float64) through frame F = ``self[s*L + k]``, with round half to even and "in
        frame" meaning 0 <= y <= H-1 and 0 <= x <= W-1 (no wrap of negative indices):

        ref 's' (F on frame k's grid):
            1. (y, x) = round(q); lost unless in frame, ``F.track(q, get_valid_status=True)``'s status is 1 (the
               vector lands strictly inside the frame, AND the mask) and ``keep[s*L + k][y, x]`` (when given) is not 0.
            2. q' = q if F is zero below the threshold, else ``F.track(q, s_exact_mode=s_exact_mode)`` bit for bit;
               lost where the bilinear would raise IndexError or the mesh finds no triangle.
            3. lost unless round(q') is in frame.
        ref 't' (F on frame k+1's grid):
            1. lost unless round(q) is in frame.
            2. q' = q if F is zero below the threshold, else ``F.track(q)`` (the mesh) bit for bit; lost where no
               triangle contains q.
            3. (y', x') = round(q'); lost unless in frame, ``F.valid_target()[y', x']`` is 1 and ``keep[s*L + k][y',
               x']`` (when given) is not 0.

        Every test is on the flow's own grid, as in ``consistent_with``. The 's' bilinear keeps Flow.track's clipped
        weights: on the last row or column they are all 0, so a point there does not move.

        Returns device arrays (``.numpy()`` to download): ``positions`` float64 (N,P,2), row ``s*L + k`` the position
        of each point in frame k+1 of clip s, and ``alive`` uint8 (N,P) of 0/1. A lost point is NaN and 0 from the
        step where it is lost to the end of its clip. The call never raises for a point's position, never
        synchronises and reads nothing back; N = 0 or P = 0 launches nothing."""
        n, (h, w) = len(self), self.shape
        clip, s_exact_mode = validate_track_clips_args(pts, clip_length, keep, s_exact_mode, n, (h, w))
        p = pts.shape[-2]
        if n == 0 or p == 0:
            return DeviceArray.empty((n, p, 2), np.float64), DeviceArray.empty((n, p), np.uint8)
        if isinstance(pts, np.ndarray):
            dpts = DeviceArray.from_numpy(pts if pts.dtype in (np.float32, np.float64) else pts.astype(np.float64))
        else:
            dpts = dev.as_device(pts)
        return _ops.track_clips(self.vecs, self.masks, self.ref, s_exact_mode, self._zero_flags(), dpts, n // clip,
                                clip, _region_device(keep))


    def matrix(self, dof=None, method=None, masked=None, *, hypotheses=None, return_inliers=False):
        """Frame-wise ``Flow.matrix`` (flow_class.py:797-867) fitted on the device in one ofk_fit_matrix call: frame
        ``i`` is the 3x3 transform from the src to the dst points of ``self[i]`` (ref 's': src = grid, dst = grid +
        flow; ref 't': src = grid - flow, dst = grid; the valid pixels only when ``masked``) with ``dof`` 4
        (similarity), 6 (affine) or 8 (homography) and ``method`` 'lms', 'ransac' or 'lmeds'; the defaults are the
        reference's (8, 'ransac', True). 'ransac' and 'lmeds' score ``hypotheses`` (default 1024) minimal samples per
        frame and refine the best on its inliers (reprojection error at most 3 px for 'ransac', the LMedS threshold
        from the median otherwise); 'lms' fits every valid point. No synchronisation and no read-back.

        Returns a device float64 array (N,3,3) (``.numpy()`` to download): the bottom row is [0, 0, 1] for dof 4 and 6,
        H[2,2] = 1 for dof 8. A frame whose flow is zero below the threshold gives the identity; a degenerate frame (too
        few valid points, no non-degenerate sample, a singular refinement) gives NaN. With ``return_inliers`` also a
        device uint8 (N,H,W) of 0/1, the inliers the refinement used, and a device int32 (N,) of their counts (0 for
        zero and degenerate frames). The hypotheses come from a fixed counter-based generator: frame ``i`` does not
        depend on the rest of the batch, and two calls give the same result."""
        dof, method, masked, hypotheses = validate_matrix_args(dof, method, masked, hypotheses)
        mats, inliers, counts = _ops.fit_matrix(self.vecs, self.masks, self.ref, dof, method, hypotheses,
                                                DEFAULT_THRESHOLD, masked, return_inliers)
        return (mats, inliers, counts) if return_inliers else mats

    def accumulate(self, clip_length=None, cumulative=True, thresholded=False, fold=None):
        """Mode-3 composition (``combine_with(., 3)``) folded over clips, in one ofk_accumulate_fold call. The N frames
        are N / ``clip_length`` clips of L = ``clip_length`` consecutive frames (default: one clip of all N),
        clip-major: frame ``s*L + k`` is step k of clip s. Clips are independent.

        ``fold='left'``: A_0 = B_0, A_k = A_{k-1}.combine_with(B_k, 3), the loop ``acc = F[0]; acc =
        acc.combine_with(F[k], 3, thresholded)``. For ref 's' A_k is the flow from frame 0 to frame k+1 on frame 0's
        grid; for ref 't' the flow from frame 0 to frame k+1 on frame k+1's grid, so that ``A_k.apply(frame 0)`` warps
        the keyframe into frame k+1 (keyframe or label propagation).
        ``fold='right'``: A_{L-1} = B_{L-1}, A_j = B_j.combine_with(A_{j+1}, 3), the loop ``acc = F[L-1]; acc =
        F[j].combine_with(acc, 3, thresholded)``. For ref 't' A_j is the flow from frame j to frame L on frame L's
        grid; for ref 's' the flow from frame j to frame L on frame j's grid: where each pixel of frame j ends up in
        the last frame.
        ``fold=None`` is 'left' for ref 's' and 'right' for ref 't'.

        Every step takes combine_with's early exits ("zero" is ``is_zero(thresholded, masked=True)`` of the whole
        frame, self tested first), so each result frame equals the loop, vectors and mask byte for byte. ('s', 'left')
        and ('t', 'right') walk each tile through the clip in a fixed number of launches; ('t', 'left') and ('s',
        'right') sample the previous composite at every step and make one launch per step for all clips.

        Returns a device-resident FlowBatch of the same ref, without synchronisation or read-back: with ``cumulative``
        N frames in the input's layout (frame ``s*L + k`` is A_k), otherwise N / L frames, the whole-clip composite
        (A_{L-1} for the left fold, A_0 for the right). Frames are always new arrays, also where an exit returns an
        input."""
        n, (h, w) = len(self), self.shape
        clip = validate_accumulate_args(clip_length, cumulative, thresholded, n, fold=fold)
        if n == 0:
            return FlowBatch._wrap(DeviceArray.empty((0, h, w, 2), np.float32), self.ref,
                                   DeviceArray.empty((0, h, w), np.uint8))
        if fold is None:
            fold = 'left' if self.ref == 's' else 'right'
        v, m = _ops.accumulate(self.vecs, self.masks, self.ref, DEFAULT_THRESHOLD if thresholded else 0.0, n // clip,
                               clip, cumulative, fold)
        return FlowBatch._wrap(v, self.ref, m)

    def consistent_with(self, other, alpha_1=None, alpha_2=None, return_valid_area=False):
        """Forward-backward consistency check (Sundaram, Brox & Keutzer, ECCV 2010) of this batch, the forward flows
        (frame 1 -> frame 2), with ``other``, the backward flows (frame 2 -> frame 1) of the same shape and ref, in one
        ofk_consistency launch. For every pixel p, with w = self[p] and s = other sampled at p + w (ref 's') or p - w
        (ref 't') the way ``combine_with(., 3)`` samples it:

            consistent = valid & (|w + s|^2 < alpha_1 (|w|^2 + |s|^2) + alpha_2)

        in float32, every operation rounded on its own; the defaults are alpha_1 = 0.01 and alpha_2 = 0.5. The result
        is on self's grid: for ref 's' frame 1's, where 1 means the pixel of frame 1 is visible in frame 2; for ref 't'
        frame 2's, where 1 means the pixel of frame 2 has a consistent source in frame 1. ``valid`` is the mask of
        ``self.combine_with(other, 3)`` for ref 's' and of ``other.combine_with(self, 3)`` for ref 't' (self's mask
        and other's mask at the taps, which must lie inside the frame); ``w + s`` are the vectors of that composition.
        There are no early exits: zero flows go through the same formula, so with alpha_2 = 0 a zero pair is not
        consistent (0 < 0 is false).

        Returns a device uint8 array (N,H,W) of 0/1 (``.numpy()`` to download), and with ``return_valid_area`` also
        ``valid``; the pixels occluded in the frame are ``valid & ~consistent``. No synchronisation, no read-back."""
        a1, a2 = validate_consistency_args(self, other, alpha_1, alpha_2, return_valid_area, FlowBatch)
        out, valid = _ops.consistency(self.vecs, self.masks, other.vecs, other.masks, self.ref, a1, a2,
                                      return_valid_area)
        return (out, valid) if return_valid_area else out

    def evaluate(self, truth, region=None, return_epe=False):
        """Error metrics of this batch, the estimated flows, against ``truth``, the ground truth of the same shape and
        ref, in one ofk_evaluate call (two launches whatever N, none for N = 0; no synchronisation, no read-back).
        Evaluated pixels are ``self.mask & truth.mask & region``: KITTI's valid channel or Sintel's invalid-pixel mask
        come in as ``truth``'s mask, ``region`` (N,H,W) bool / uint8, numpy or device, restricts the metrics further
        (KITTI's noc / occ split, or the occluded / visible split of ``consistent_with``). The ref is not used in the
        arithmetic: the flows are compared pixel by pixel on their common grid. For every pixel, in float32 with every
        operation rounded on its own, with (ue, ve) the estimate and (ug, vg) the truth:

            epe = sqrt((ue - ug)^2 + (ve - vg)^2);  mg = sqrt(ug^2 + vg^2)
            fl = epe > 3 and epe / mg > 0.05 (KITTI 2015);  out_k = epe > k for k = 1, 3, 5
            band = 0 if mg < 10, 1 if mg < 40, else 2 (Sintel s0-10, s10-40, s40+)
            ae = atan2(sqrt(d2 + cz^2), (1 + ue ug) + ve vg) in degrees, d2 = epe^2 before the root, cz = ue vg - ve ug:
                 the angle between (ue, ve, 1) and (ug, vg, 1) (Barron et al.), 0 for a perfect estimate

        Returns a :class:`FlowErrors` of device arrays: per-frame ``counts`` and ``sums`` (the float32 values added in
        float64 in a fixed order, so a frame's rows do not depend on the batch it is in), and with ``return_epe`` the
        EPE of every pixel, evaluated or not. ``.summary()`` gives the pixel-weighted figures of the whole batch."""
        validate_evaluate_args(self, truth, region, return_epe, FlowBatch)
        counts, sums, epe = _ops.evaluate(self.vecs, self.masks, truth.vecs, truth.masks, _region_device(region),
                                          return_epe)
        return FlowErrors(counts, sums, epe)


def _region_device(region):
    """A validated region (numpy or device, bool / uint8 0/1) as a device uint8 array, or None."""
    if region is None:
        return None
    if isinstance(region, np.ndarray):
        return DeviceArray.from_numpy(np.ascontiguousarray(region, dtype=np.bool_).view(np.uint8))
    d = dev.as_device(region)
    return DeviceArray(d.ptr, d.shape, np.uint8, owner=d)


class FlowErrors(object):
    """Error metrics of :meth:`FlowBatch.evaluate`, one row per frame:

    ``counts`` int64 (N, 8): evaluated pixels, KITTI Fl outliers, pixels with EPE > 1, > 3, > 5, and evaluated pixels
    in the Sintel bands s0-10, s10-40, s40+ (by the magnitude of the truth).
    ``sums`` float64 (N, 5): EPE, angular error (degrees), EPE over the bands s0-10, s10-40, s40+.
    ``epe`` float32 (N, H, W) or None: the EPE of every pixel.

    The rows are kept so that callers can form frame-averaged figures, or add the rows of several GPUs' shards, which
    ``summary`` does not do."""
    COUNTS = ('evaluated', 'fl', 'out1', 'out3', 'out5', 's0-10', 's10-40', 's40+')
    SUMS = ('epe', 'ae', 's0-10', 's10-40', 's40+')

    def __init__(self, counts, sums, epe=None):
        self.counts, self.sums, self.epe = counts, sums, epe

    def numpy(self):
        """Host copies: (counts, sums), and the EPE map as a third item when there is one."""
        host = tuple(x if isinstance(x, np.ndarray) else x.numpy() for x in (self.counts, self.sums))
        if self.epe is None:
            return host
        return host + (self.epe if isinstance(self.epe, np.ndarray) else self.epe.numpy(),)

    def summary(self):
        """Pixel-weighted figures of all frames as a host dict: 'epe', 'ae' (mean EPE and angular error), 'fl',
        'out1', 'out3', 'out5' (fractions of the evaluated pixels), 's0-10', 's10-40', 's40+' (mean EPE in each band)
        and 'pixels'. The per-frame rows are added in frame order in float64; a figure over no pixels is NaN."""
        counts, sums = self.numpy()[:2]
        c = [sum(int(v) for v in counts[:, k]) for k in range(8)]
        s = []
        for k in range(5):
            t = 0.0
            for v in sums[:, k]:
                t += float(v)
            s.append(t)

        def ratio(a, b):
            return a / b if b else float('nan')

        n = c[0]
        return {'epe': ratio(s[0], n), 'ae': ratio(s[1], n), 'fl': ratio(c[1], n), 'out1': ratio(c[2], n),
                'out3': ratio(c[3], n), 'out5': ratio(c[4], n), 's0-10': ratio(s[2], c[5]),
                's10-40': ratio(s[3], c[6]), 's40+': ratio(s[4], c[7]), 'pixels': n}


def _track_range_fails(pts, lookup, is_int, status, h, w):
    """True if a host point fails a range test of Flow.track (the tests ofk_track repeats per frame), which only
    depend on the points and the frame size: float points on an 's' flow outside [0,H-1]x[0,W-1], integer points on an
    's' flow outside [-H,H-1]x[-W,W-1], and with status the rounded points outside that range."""
    r, c = pts[..., 0], pts[..., 1]
    if lookup and is_int:
        fails = (r < -h) | (r >= h) | (c < -w) | (c >= w)
    elif lookup:
        r, c = r.astype(np.float64), c.astype(np.float64)
        fails = ~((0 <= r) & (r <= h - 1) & (0 <= c) & (c <= w - 1))
    else:
        fails = np.zeros(r.shape, bool)
    if status:
        with np.errstate(invalid='ignore'):                   # NaN and huge values become INT_MIN, as in Flow.track
            ri, ci = np.round(r).astype('i'), np.round(c).astype('i')
        fails |= (ri < -h) | (ri >= h) | (ci < -w) | (ci >= w)
    return bool(fails.any())


def _raise_track_error(errors, h, w):
    """Raises the IndexError of the lowest frame whose error word (ofk_track) is set, as a loop of Flow.track would."""
    flagged = np.flatnonzero(errors)
    if flagged.size == 0:
        return
    i = int(flagged[0])
    e = int(errors[i])
    if e & 1:
        raise IndexError("Some points are outside of the data area.")
    if e & 2:
        raise IndexError("Error tracking points: Pts of frame {} index outside of the flow field of shape {}".format(
            i, (h, w)))
    raise IndexError("Error tracking points: Rounded pts of frame {} for the valid status lie outside of the flow "
                     "field of shape {}".format(i, (h, w)))


# ---------------------------------------------------------------------------------------------------- host-buffer calls
def _c(a, dtype=None):
    return np.ascontiguousarray(a, dtype=dtype)


def _check_out(arr, shape, dtype, name):
    """Caller-supplied output buffers become raw pointers for the copy engines: shape, dtype and layout must be exact."""
    if not isinstance(arr, np.ndarray) or arr.shape != tuple(shape) or arr.dtype != np.dtype(dtype) or \
            not arr.flags.c_contiguous or not arr.flags.writeable:
        raise ValueError("{} needs to be a writeable C-contiguous numpy array of shape {} and dtype {}".format(
            name, tuple(shape), np.dtype(dtype)))


def apply_flow_host(flows, images, flow_masks=None, target_masks=None, return_valid_area=False, out=None,
                    out_valid=None, device=None):
    """Batched ``Flow(flows[i], 't', flow_masks[i]).apply(images[i], target_masks[i], return_valid_area)`` on HOST
    arrays through ofh_warp_t: frames stream through a device ring, host<->device copies overlap the kernels.
    Pass pinned arrays (device.pinned_empty) for full-rate copies. Returns numpy arrays."""
    flows = _c(flows, np.float32)
    images = _c(images)
    if flows.ndim != 4 or flows.shape[3] != 2:
        raise ValueError("Error applying flow: flows need shape (N,H,W,2)")
    if images.ndim == 3:
        images = images[..., None]
    n, h, w = flows.shape[:3]
    if images.shape[:3] != (n, h, w):
        raise ValueError("Error applying flow: Flow shape does not match target shape")
    code = _ops.dtype_code(images.dtype)
    if return_valid_area:
        arith, rule = _ops.promoted_rule(images.dtype, target_masks is not None)
    else:
        arith, rule = _lib.ARITH_NATIVE, _lib.RULE_STRICT
    if out is None:
        out = np.empty_like(images)
    else:
        _check_out(out, images.shape if out.ndim == 4 else images.shape[:3], images.dtype, 'out')
    pm = fm = om = None
    if return_valid_area:
        if out_valid is None:
            out_valid = np.empty((n, h, w), np.bool_)
        else:
            _check_out(out_valid, (n, h, w), np.bool_, 'out_valid')
        om = out_valid.ctypes.data
        if target_masks is not None:
            target_masks = _c(target_masks, np.bool_)
            pm = target_masks.ctypes.data
        if flow_masks is not None:
            flow_masks = _c(flow_masks, np.bool_)
            fm = flow_masks.ctypes.data
    device = dev.get_device() if device is None else device
    _lib.call('ofh_warp_t', images.ctypes.data, code, images.shape[3], arith, flows.ctypes.data, -1.0, pm, fm,
              out.ctypes.data, om, rule, n, h, w, device)
    return (out, out_valid) if return_valid_area else out


def combine_flows_host(flows_1, flows_2, mode, ref, masks_1=None, masks_2=None, thresholded=False, out=None,
                       out_masks=None, device=None):
    """Batched ``combine_flows(flows_1[i], flows_2[i], mode, ref)`` / ``Flow.combine_with`` on HOST arrays. Mode 3
    streams through ofh_combine3 (pinned ring, copies overlapped with the kernel); modes 1 / 2 upload the batch, run the
    device chain of FlowBatch.combine_with and download. Returns (vecs (N,H,W,2) float32, masks (N,H,W) bool)."""
    if mode not in (1, 2, 3):
        raise ValueError("Error combining flows: Mode needs to be 1, 2 or 3")
    ref = get_valid_ref(ref)
    if mode != 3:
        res = FlowBatch(flows_1, ref, masks_1).combine_with(FlowBatch(flows_2, ref, masks_2), mode, thresholded)
        v, m = res.numpy()
        if out is not None:
            _check_out(out, v.shape, np.float32, 'out')
            out[...] = v
            v = out
        if out_masks is not None:
            _check_out(out_masks, m.shape, np.bool_, 'out_masks')
            out_masks[...] = m
            m = out_masks
        return v, m
    a, b = _c(flows_1, np.float32), _c(flows_2, np.float32)
    if a.shape != b.shape or a.ndim != 4 or a.shape[3] != 2:
        raise ValueError("Error combining flows: Flow fields need to have the same shape (N,H,W,2)")
    n, h, w = a.shape[:3]
    am = None if masks_1 is None else _c(masks_1, np.bool_)
    bm = None if masks_2 is None else _c(masks_2, np.bool_)
    if out is None:
        out = np.empty_like(a)
    else:
        _check_out(out, a.shape, np.float32, 'out')
    if out_masks is None:
        out_masks = np.empty((n, h, w), np.bool_)
    else:
        _check_out(out_masks, (n, h, w), np.bool_, 'out_masks')
    flags = np.empty((n, 2), np.int32)
    device = dev.get_device() if device is None else device
    _lib.call('ofh_combine3', a.ctypes.data, None if am is None else am.ctypes.data, b.ctypes.data,
              None if bm is None else bm.ctypes.data, ord(ref), DEFAULT_THRESHOLD if thresholded else 0.0,
              out.ctypes.data, out_masks.ctypes.data, flags.ctypes.data, n, h, w, device)
    return out, out_masks


def apply_combine_host(flows_1, flows_2, images, ref='t', masks_1=None, masks_2=None, thresholded=False, out_images=None,
                       out_valid=None, out=None, out_masks=None, device=None):
    """The pair of calls of a frame pipeline on HOST arrays in one pass (ofh_apply_combine3), with
    ``A = Flow(flows_1[i], ref, masks_1[i])``: ``A.apply(images[i], return_valid_area=True)`` for ref 't',
    ``A.invert('t').apply(images[i], return_valid_area=True)`` for ref 's' (the images are sampled at
    p + flows_1[i][p]), and ``A.combine_with(Flow(flows_2[i], ref, masks_2[i]), 3)``. ``flows_1`` and ``masks_1`` are
    uploaded once for both kernels (apply_flow_host + combine_flows_host upload them twice). Returns (images, valid
    areas, vecs, masks)."""
    ref = get_valid_ref(ref)
    a, b = _c(flows_1, np.float32), _c(flows_2, np.float32)
    images = _c(images)
    if a.shape != b.shape or a.ndim != 4 or a.shape[3] != 2:
        raise ValueError("Error combining flows: Flow fields need to have the same shape (N,H,W,2)")
    if images.ndim == 3:
        images = images[..., None]
    n, h, w = a.shape[:3]
    if images.shape[:3] != (n, h, w):
        raise ValueError("Error applying flow: Flow shape does not match target shape")
    code = _ops.dtype_code(images.dtype)
    arith, rule = _ops.promoted_rule(images.dtype, False)
    am = None if masks_1 is None else _c(masks_1, np.bool_)
    bm = None if masks_2 is None else _c(masks_2, np.bool_)
    for name, arr, shape, dt in (('out_images', out_images, images.shape, images.dtype),
                                 ('out_valid', out_valid, (n, h, w), np.bool_), ('out', out, a.shape, np.float32),
                                 ('out_masks', out_masks, (n, h, w), np.bool_)):
        if arr is not None:
            _check_out(arr, shape, dt, name)
    out_images = np.empty_like(images) if out_images is None else out_images
    out_valid = np.empty((n, h, w), np.bool_) if out_valid is None else out_valid
    out = np.empty_like(a) if out is None else out
    out_masks = np.empty((n, h, w), np.bool_) if out_masks is None else out_masks
    flags = np.empty((n, 2), np.int32)
    device = dev.get_device() if device is None else device
    _lib.call('ofh_apply_combine3', images.ctypes.data, code, images.shape[3], arith, rule, a.ctypes.data,
              None if am is None else am.ctypes.data, b.ctypes.data, None if bm is None else bm.ctypes.data, ord(ref),
              DEFAULT_THRESHOLD if thresholded else 0.0, out_images.ctypes.data, out_valid.ctypes.data, out.ctypes.data,
              out_masks.ctypes.data, flags.ctypes.data, n, h, w, device)
    return out_images, out_valid, out, out_masks


def visualise_flows_host(flows, mode, masks=None, show_mask=False, show_mask_borders=False, range_max=None, out=None,
                         device=None):
    """Batched ``Flow(flows[i], 't', masks[i]).visualise(mode, show_mask, show_mask_borders, range_max)`` on HOST
    arrays through ofh_visualise: frames stream through the device ring, copies overlap the kernels, the default range
    of each frame is found on the device. Pass pinned arrays (device.pinned_empty) for full-rate copies. Returns a
    numpy uint8 array (N,H,W,3)."""
    code, show_mask, show_mask_borders = validate_visualise_args(mode, show_mask, show_mask_borders, range_max)
    flows = _c(flows, np.float32)
    if flows.ndim != 4 or flows.shape[3] != 2:
        raise ValueError("Error visualising flow: flows need shape (N,H,W,2)")
    n, h, w = flows.shape[:3]
    if masks is not None:
        masks = _c(masks, np.bool_)
        if masks.shape != (n, h, w):
            raise ValueError("Error setting flow mask: Input has a different shape than the flow vectors")
    if out is None:
        out = np.empty((n, h, w, 3), np.uint8)
    else:
        _check_out(out, (n, h, w, 3), np.uint8, 'out')
    device = dev.get_device() if device is None else device
    _lib.call('ofh_visualise', flows.ctypes.data, None if masks is None else masks.ctypes.data, DEFAULT_THRESHOLD,
              code, int(show_mask), int(show_mask_borders), _ops.vis_range_arg(range_max), out.ctypes.data, n, h, w,
              device)
    return out


def evaluate_flows_host(estimates, truths, est_masks=None, truth_masks=None, regions=None, out_epe=None, device=None):
    """``FlowBatch(estimates, masks=est_masks).evaluate(FlowBatch(truths, masks=truth_masks), regions)`` on HOST
    arrays through ofh_evaluate: frames stream through the device ring, and only the per-frame rows (104 bytes per
    frame) come back, plus the EPE map when ``out_epe`` (float32 (N,H,W)) is given. Pass pinned arrays
    (device.pinned_empty) for full-rate copies. Returns numpy (counts (N,8) int64, sums (N,5) float64), and ``out_epe``
    as a third item when given."""
    est, tru = _c(estimates, np.float32), _c(truths, np.float32)
    if est.ndim != 4 or est.shape[3] != 2 or tru.shape != est.shape:
        raise ValueError("Error evaluating flow: estimates and truths need the same shape (N,H,W,2)")
    n, h, w = est.shape[:3]
    planes = []
    for name, m in (('Est_masks', est_masks), ('Truth_masks', truth_masks), ('Regions', regions)):
        if m is not None:
            m = _c(m, np.bool_)
            if m.shape != (n, h, w):
                raise ValueError("Error evaluating flow: {} need shape {}".format(name, (n, h, w)))
        planes.append(m)
    if out_epe is not None:
        _check_out(out_epe, (n, h, w), np.float32, 'out_epe')
    counts, sums = np.empty((n, 8), np.int64), np.empty((n, 5), np.float64)
    device = dev.get_device() if device is None else device
    em, tm, rg = (None if m is None else m.ctypes.data for m in planes)
    _lib.call('ofh_evaluate', est.ctypes.data, em, tru.ctypes.data, tm, rg,
              None if out_epe is None else out_epe.ctypes.data, counts.ctypes.data, sums.ctypes.data, n, h, w, device)
    return (counts, sums) if out_epe is None else (counts, sums, out_epe)
