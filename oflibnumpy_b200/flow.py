"""Device-resident ``Flow`` with the public surface of oflibnumpy's ``Flow`` (reference: flow_class.py:29-1424).

Vectors and mask live in HBM as float32 ``[1,H,W,2]`` / uint8 ``[1,H,W]``; every method that the reference implements
through ``cv2.remap`` / ``griddata`` / numpy full-frame expressions calls one CUDA entry point of liboflib_b200.so
instead (see ``_ops``). numpy views are produced lazily by the ``vecs`` / ``mask`` properties.

Argument checks, defaults (``None`` means default), exception types and messages follow the reference so its tests
read the same against this class. Deliberate differences are listed in DESIGN.md ("Behavioural notes").
"""
import math
import warnings

import numpy as np

from . import _lib
from . import _ops
from . import device as dev
from .device import DeviceArray
from .validation import get_valid_ref, get_valid_padding, validate_shape, validate_visualise_args, \
    validate_track_args, validate_consistency_args, validate_evaluate_args, DEFAULT_THRESHOLD

__all__ = ['Flow']


def _is_dev(x):
    return dev.is_device_array(x)


class _HostView(np.ndarray):
    """The numpy array handed out by ``Flow.vecs`` / ``Flow.mask``.

    In the reference these arrays ARE the flow's storage and its tests and docs edit them in place
    (``flow.vecs[~mask] = 0``, ``flow.mask[:, 200:] = False``; tests/test_flow_class.py:399,580,1003, docs/usage.rst:316).
    Here the storage lives on the device, so the host copy must be uploaded again after such an edit -- but only then:
    the buffer is kept read-only and the two ways numpy writes in place from Python (item assignment and ufuncs with
    ``out=`` / augmented assignment) are intercepted to mark the owning Flow dirty. Every other writer (``np.copyto``,
    ``arr.fill``, ``arr.sort``, a C extension writing into the buffer ...) hits the read-only flag and raises instead of
    silently leaving the device copy stale; assign through the property (``flow.vecs = new_array``) in that case.
    Slices and views share the buffer and the tracking; results of arithmetic are plain, writeable ndarrays."""

    _dirty_cell = None      # one-element list shared with the owning Flow, or None for arrays that own nothing

    def __array_finalize__(self, obj):
        self._dirty_cell = None
        if isinstance(obj, _HostView) and obj._dirty_cell is not None and self.base is not None and \
                np.shares_memory(self, obj):
            self._dirty_cell = obj._dirty_cell

    def _writable(self):
        """Context manager: temporarily lift the read-only flag of the underlying buffer for an intercepted write."""
        return _Unlock(self)

    def __setitem__(self, key, value):
        if self._dirty_cell is None:
            return super().__setitem__(key, value)
        with _Unlock(self):
            super().__setitem__(key, value)
        self._dirty_cell[0] = True

    def __array_ufunc__(self, ufunc, method, *inputs, out=None, **kwargs):
        plain = tuple(np.asarray(x) if isinstance(x, _HostView) else x for x in inputs)
        if out is None:
            return getattr(ufunc, method)(*plain, **kwargs)
        tracked = [o for o in out if isinstance(o, _HostView) and o._dirty_cell is not None]
        outs = tuple(o.view(np.ndarray) if isinstance(o, _HostView) else o for o in out)
        locks = [_Unlock(o) for o in tracked]
        for lk in locks:
            lk.__enter__()
        try:
            # views taken before unlocking keep the read-only flag: take them again now
            outs = tuple(o.view(np.ndarray) if isinstance(o, _HostView) else o for o in out)
            res = getattr(ufunc, method)(*plain, out=outs, **kwargs)
        finally:
            for lk in reversed(locks):
                lk.__exit__(None, None, None)
        for o in tracked:
            o._dirty_cell[0] = True
        if isinstance(res, tuple):
            return tuple(o_in if r is o_plain else r for r, o_plain, o_in in zip(res, outs, out))
        return out[0] if res is outs[0] else res


class _Unlock(object):
    """Lifts ``writeable=False`` along the base chain of a _HostView for the duration of one intercepted write."""

    def __init__(self, arr):
        chain, a = [], arr
        while isinstance(a, np.ndarray):
            chain.append(a)
            a = a.base
        self.chain = chain[::-1]          # owner first: a view can only be made writeable if its base is

    def __enter__(self):
        self.was = [a.flags.writeable for a in self.chain]
        for a in self.chain:
            a.flags.writeable = True
        return self

    def __exit__(self, *exc):
        for a, w in zip(reversed(self.chain), reversed(self.was)):
            a.flags.writeable = w
        return False


def _tracked_view(arr, dirty_cell):
    """Read-only _HostView of a freshly downloaded array, reporting in-place edits to `dirty_cell`."""
    arr.flags.writeable = False
    v = arr.view(_HostView)
    v._dirty_cell = dirty_cell
    return v


class Flow(object):
    def __init__(self, flow_vectors, ref=None, mask=None):
        """:param flow_vectors: numpy array (H,W,2), channel 0 horizontal (+right), channel 1 vertical (+down);
            also accepts a device array (``__cuda_array_interface__``, float32, (H,W,2)) which is adopted without copy
        :param ref: ``'t'`` (default) or ``'s'``
        :param mask: numpy / device array (H,W) of 0/1 or bool; defaults to all valid
        """
        self._dv = self._dm = None
        self._hv = self._hm = None
        self._vdirty, self._mdirty = [False], [False]
        self.vecs = flow_vectors
        self.ref = ref
        self.mask = mask

    # ------------------------------------------------------------------------------------------ internal plumbing
    @classmethod
    def _wrap(cls, dvecs, ref, dmask=None):
        """Adopt device results ([1,H,W,2] float32, [1,H,W] uint8) without validation or copies."""
        f = cls.__new__(cls)
        f._dv, f._dm, f._hv, f._hm = dvecs, dmask, None, None
        f._vdirty, f._mdirty = [False], [False]
        f._ref = ref
        if dmask is None:
            f._dm = _ones_mask(dvecs.shape[1:3])
        return f

    def _vd(self):
        """Device vectors. A host view handed out by ``.vecs`` may have been edited in place (the reference's array
        IS its storage): it reports such edits (see _HostView) and is uploaded again only then."""
        if self._hv is not None and self._vdirty[0]:
            self._dv = DeviceArray.from_numpy(np.asarray(self._hv)[None], np.float32)
            self._vdirty[0] = False
        return self._dv

    def _md(self):
        if self._hm is not None and self._mdirty[0]:
            self._dm = DeviceArray.from_numpy(np.asarray(self._hm)[None].view(np.uint8))
            self._mdirty[0] = False
        return self._dm

    # ------------------------------------------------------------------------------------------ attributes
    @property
    def vecs(self):
        """Flow vectors as a float32 numpy array (H,W,2) (device -> host copy on first access)."""
        if self._hv is None:
            self._vdirty = [False]
            self._hv = _tracked_view(self._dv.numpy()[0], self._vdirty)
        return self._hv

    @vecs.setter
    def vecs(self, input_vecs):
        if _is_dev(input_vecs) and not isinstance(input_vecs, np.ndarray):
            d = dev.as_device(input_vecs)
            if d.ndim != 3:
                raise ValueError("Error setting flow vectors: Input not 3-dimensional")
            if d.shape[2] != 2:
                raise ValueError("Error setting flow vectors: Input does not have 2 channels")
            if d.dtype != np.float32:
                raise TypeError("Error setting flow vectors: Device input needs to be float32")
            d = d.reshape((1,) + d.shape)
            if not _ops.all_finite(d):
                raise ValueError("Error setting flow vectors: Input contains NaN, Inf or -Inf values")
            self._dv, self._hv = d, None
            return
        if not isinstance(input_vecs, np.ndarray):
            raise TypeError("Error setting flow vectors: Input is not a numpy array")
        if not input_vecs.ndim == 3:
            raise ValueError("Error setting flow vectors: Input not 3-dimensional")
        if not input_vecs.shape[2] == 2:
            raise ValueError("Error setting flow vectors: Input does not have 2 channels")
        if input_vecs.dtype == np.float32:
            d = DeviceArray.from_numpy(input_vecs[None])
            if not _ops.all_finite(d):          # finite test on the device (reference: flow_class.py:78-79)
                raise ValueError("Error setting flow vectors: Input contains NaN, Inf or -Inf values")
        else:
            # other dtypes are tested before the float32 cast, as the reference does
            if not np.isfinite(input_vecs).all():
                raise ValueError("Error setting flow vectors: Input contains NaN, Inf or -Inf values")
            d = DeviceArray.from_numpy(input_vecs[None], np.float32)
        self._dv, self._hv = d, None

    @property
    def ref(self):
        return self._ref

    @ref.setter
    def ref(self, input_ref=None):
        self._ref = get_valid_ref(input_ref)

    @property
    def mask(self):
        """Validity mask as a bool numpy array (H,W) (device -> host copy on first access)."""
        if self._hm is None:
            self._mdirty = [False]
            self._hm = _tracked_view(self._dm.numpy()[0].view(np.bool_), self._mdirty)
        return self._hm

    @mask.setter
    def mask(self, input_mask=None):
        if input_mask is None:
            self._dm, self._hm = _ones_mask(self.shape), None
            return
        if _is_dev(input_mask) and not isinstance(input_mask, np.ndarray):
            d = dev.as_device(input_mask)
            if d.ndim != 2:
                raise ValueError("Error setting flow mask: Input not 2-dimensional")
            if d.shape != self.shape:
                raise ValueError("Error setting flow mask: Input has a different shape than the flow vectors")
            if d.dtype not in (np.uint8, np.bool_):
                raise TypeError("Error setting flow mask: Device input needs to be bool or uint8 (0/1)")
            self._dm, self._hm = DeviceArray(d.ptr, (1,) + d.shape, np.uint8, owner=d), None
            return
        if not isinstance(input_mask, np.ndarray):
            raise TypeError("Error setting flow mask: Input is not a numpy array")
        if not input_mask.ndim == 2:
            raise ValueError("Error setting flow mask: Input not 2-dimensional")
        if not input_mask.shape == self.shape:
            raise ValueError("Error setting flow mask: Input has a different shape than the flow vectors")
        if input_mask.dtype != np.bool_ and ((input_mask != 0) & (input_mask != 1)).any():
            raise ValueError("Error setting flow mask: Values must be 0 or 1")
        m = np.ascontiguousarray(input_mask, dtype=np.bool_)      # no host copy for a contiguous bool array: the upload copies
        self._dm, self._hm = DeviceArray.from_numpy(m[None].view(np.uint8)), None

    @property
    def shape(self):
        return tuple(self._dv.shape[1:3])

    # device accessors (extension): zero-copy handles for torch / further kernels
    @property
    def vecs_device(self):
        """DeviceArray [H,W,2] float32 (``torch.as_tensor(flow.vecs_device, device='cuda')`` is zero-copy)."""
        d = self._vd()
        return d.reshape(d.shape[1:])

    @property
    def mask_device(self):
        d = self._md()
        return d.reshape(d.shape[1:])

    # ------------------------------------------------------------------------------------------ constructors
    @classmethod
    def zero(cls, shape, ref=None, mask=None):
        validate_shape(shape)
        f = cls._wrap(DeviceArray.zeros((1, shape[0], shape[1], 2), np.float32), get_valid_ref(ref))
        f.mask = mask
        return f

    @classmethod
    def from_matrix(cls, matrix, shape, ref=None, mask=None):
        from .ops import _from_matrix_device
        r = get_valid_ref(ref)
        f = cls._wrap(_from_matrix_device(matrix, shape, r), r)
        f.mask = mask
        return f

    @classmethod
    def from_transforms(cls, transform_list, shape, ref=None, mask=None):
        from .ops import _from_transforms_device
        r = get_valid_ref(ref)
        f = cls._wrap(_from_transforms_device(transform_list, shape, r), r)
        f.mask = mask
        return f

    @classmethod
    def from_kitti(cls, path, load_valid=None):
        """Flow from a KITTI uint16 PNG (flow_class.py:237-256, utils.py:426-445). The file is decoded on the host by
        OpenCV; the raw uint16 pixels (6 B/px instead of 8 + 1) go to the device and are converted there."""
        from .io import read_kitti_raw
        load_valid = True if load_valid is None else load_valid
        if not isinstance(load_valid, bool):
            raise TypeError("Error loading flow from KITTI data: Load_valid needs to be boolean")
        raw = read_kitti_raw(path)                                   # (H, W, 3) uint16, BGR as OpenCV decodes it
        h, w = raw.shape[:2]
        d_raw = DeviceArray.from_numpy(raw)
        vecs = DeviceArray.empty((1, h, w, 2), np.float32)
        mask = DeviceArray.empty((1, h, w), np.uint8) if load_valid else None
        _lib.call('ofk_decode_kitti', d_raw.ptr, vecs.ptr, mask.ptr if mask is not None else None, h * w,
                  dev.current_stream())
        return cls._wrap(vecs, 's', mask)

    @classmethod
    def from_sintel(cls, path, inv_path=None):
        """Flow from a Sintel .flo file and, optionally, its invalid-pixel PNG (flow_class.py:258-275,
        utils.py:448-490); the mask is inverted on the device."""
        from .io import load_sintel, read_sintel_invalid_raw
        flow = load_sintel(path)
        f = cls(flow, 's')
        if inv_path is not None:
            raw = read_sintel_invalid_raw(inv_path)                  # (H, W) uint8
            if raw.shape != f.shape:
                raise ValueError("Error setting flow mask: Input has a different shape than the flow vectors")
            d_raw = DeviceArray.from_numpy(raw)
            mask = DeviceArray.empty((1,) + raw.shape, np.uint8)
            _lib.call('ofk_decode_sintel_mask', d_raw.ptr, mask.ptr, raw.size, dev.current_stream())
            f._dm, f._hm = mask, None
        return f

    def copy(self):
        """Deep copy (device-to-device)."""
        return Flow._wrap(self._vd().copy(), self._ref, self._md().copy())

    def __str__(self):
        return "Flow object, reference {}, shape {}*{}; ".format(self._ref, *self.shape) + self.__repr__()

    def __getitem__(self, item):
        # contiguous 2-D windows are cut on the device; anything else goes through numpy indexing like the reference
        win = _as_window(item, self.shape)
        if win is not None:
            y0, x0, h, w = win
            return Flow._wrap(_ops.crop(self._vd(), y0, x0, h, w), self._ref, _ops.crop(self._md(), y0, x0, h, w))
        return Flow(self.vecs.__getitem__(item), self._ref, self.mask.__getitem__(item))

    # ------------------------------------------------------------------------------------------ arithmetic
    def _addsub(self, other, op, name, who, whom):
        if not isinstance(other, (np.ndarray, Flow)):
            raise TypeError("Error {} flow: {} is not a flow object or a numpy array".format(name, who))
        if isinstance(other, Flow):
            if self.shape != other.shape:
                raise ValueError("Error {} flow: {} flow objects are not the same shape".format(name, whom))
            v, m = _ops.addsub(op, self._vd(), self._md(), other._vd(), other._md())
            if not _ops.all_finite(v):      # the sum of two finite float32 fields can overflow
                raise ValueError("Error setting flow vectors: Input contains NaN, Inf or -Inf values")
            return Flow._wrap(v, self._ref, m)
        if self.shape != other.shape[:2] or other.ndim != 3 or other.shape[2] != 2:
            raise ValueError("Error {} flow: {} numpy array needs to have the same shape as the flow "
                             "object, 3 dimensions overall, and a channel length of 2".format(name, who))
        if other.dtype == np.float32:
            v, _ = _ops.addsub(op, self._vd(), None, DeviceArray.from_numpy(other[None]), None, want_mask=False)
        else:  # numpy promotes to float64, then the Flow constructor rounds to float32
            v = _ops.scale_array(op, self._vd(), DeviceArray.from_numpy(other[None], np.float64), 2)
        return self._checked(v)

    def _checked(self, v):
        if not _ops.all_finite(v):
            raise ValueError("Error setting flow vectors: Input contains NaN, Inf or -Inf values")
        return Flow._wrap(v, self._ref, self._md().copy())

    def __add__(self, other):
        return self._addsub(other, _lib.OP_ADD, 'adding to', 'Addend', 'Augend and addend')

    def __sub__(self, other):
        return self._addsub(other, _lib.OP_SUB, 'subtracting from', 'Subtrahend', 'Minuend and subtrahend')

    def _scale(self, other, op, verb, noun):
        try:
            s = float(other)
        except TypeError:
            s = None
        if s is not None:
            return self._checked(_ops.scale(op, self._vd(), s, s, False))
        if isinstance(other, list):
            if len(other) != 2:
                raise ValueError("Error {} flow: {} list not length 2".format(verb, noun))
            pair = np.array(other)
            return self._checked(_ops.scale(op, self._vd(), float(pair[0]), float(pair[1]), True))
        if isinstance(other, np.ndarray):
            if other.ndim == 1 and other.size == 2:
                return self._checked(_ops.scale(op, self._vd(), float(other[0]), float(other[1]),
                                                other.dtype != np.float32))
            if other.ndim == 2 and other.shape == self.shape[:2]:
                ch = 1
            elif other.shape == self.shape + (2,):
                ch = 2
            else:
                raise ValueError("Error {} flow: {} array is not one of the following: size 2, "
                                 "shape of the flow object, shape of the flow vectors".format(verb, noun))
            m = DeviceArray.from_numpy(other[None], np.float64)
            return self._checked(_ops.scale_array(op, self._vd(), m, ch))
        raise TypeError("Error {} flow: {} cannot be converted to float, "
                        "or isn't a list or numpy array".format(verb, noun))

    def __mul__(self, other):
        return self._scale(other, _lib.OP_MUL, 'multiplying', 'Multiplier')

    def __truediv__(self, other):
        return self._scale(other, _lib.OP_DIV, 'dividing', 'Divisor')

    def __pow__(self, other):
        return self._scale(other, _lib.OP_POW, 'exponentiating', 'Exponent')

    def __neg__(self):
        return self * -1

    # ------------------------------------------------------------------------------------------ resize / pad
    def resize(self, scale):
        from .ops import _resize_device
        v, m = _resize_device(self._vd(), self._md(), scale)
        return Flow._wrap(v, self._ref, m)

    def pad(self, padding=None, mode=None):
        mode = 'constant' if mode is None else mode
        if mode not in ['constant', 'edge', 'symmetric']:
            raise ValueError("Error padding flow: Mode should be one of "
                             "'constant', 'edge', 'symmetric', but instead got '{}'".format(mode))
        padding = get_valid_padding(padding, "Error padding flow: ")
        v, m = _ops.pad(self._vd(), self._md(), padding, mode)
        return Flow._wrap(v, self._ref, m)

    # ------------------------------------------------------------------------------------------ apply
    def apply(self, target, target_mask=None, return_valid_area=None, consider_mask=None, padding=None, cut=None):
        """Warp ``target`` (numpy array (H,W[,C]) or Flow) with this flow; semantics of the reference's
        ``Flow.apply`` (flow_class.py:528-695). ref 't' -> ofk_warp_t, ref 's' -> ofk_forward_s."""
        return_valid_area = False if return_valid_area is None else return_valid_area
        if not isinstance(return_valid_area, bool):
            raise TypeError("Error applying flow: Return_valid_area needs to be a boolean")
        consider_mask = True if consider_mask is None else consider_mask
        if not isinstance(consider_mask, bool):
            raise TypeError("Error applying flow: Consider_mask needs to be a boolean")
        cut = True if cut is None else cut
        if not isinstance(cut, bool):
            raise TypeError("Error applying flow: Cut needs to be a boolean")
        if not isinstance(target, (Flow, np.ndarray)):
            raise ValueError("Error applying flow: Target needs to be either a flow object, or a numpy ndarray")
        fh, fw = self.shape
        if padding is None:
            if fh != target.shape[0] or fw != target.shape[1]:
                raise ValueError("Error applying flow: Flow shape does not match target shape")
        else:
            padding = get_valid_padding(padding, "Error applying flow: ")
            if fh + sum(padding[:2]) != target.shape[0] or fw + sum(padding[2:]) != target.shape[1]:
                raise ValueError("Error applying flow: Padding values do not match flow and target shape difference")

        return_2d = False
        host_tmask = None
        if isinstance(target, Flow):
            return_flow = True
            payload, pmask = target._vd(), target._md()
            out_dtype = None
        else:
            return_flow = False
            if target.ndim == 3:
                t = target
            elif target.ndim == 2:
                return_2d = True
                t = target[..., np.newaxis]
            else:
                raise ValueError("Error applying flow: Target needs to have the shape H-W (2 dimensions) "
                                 "or H-W-C (3 dimensions)")
            if target_mask is not None:
                if not isinstance(target_mask, np.ndarray):
                    raise TypeError("Error applying flow: Target_mask needs to be a numpy ndarray")
                if target_mask.shape != target.shape[:2]:
                    raise ValueError("Error applying flow: Target_mask needs to match the target shape")
                if target_mask.dtype != bool:
                    raise TypeError("Error applying flow: Target_mask needs to have dtype 'bool'")
                if not return_valid_area:
                    warnings.warn("Warning applying flow: a mask is passed, but return_valid_area is False - so the "
                                  "mask passed will not affect the output, but possibly make the function slower.")
                host_tmask = target_mask
            out_dtype = target.dtype
            _ops.dtype_code(out_dtype)           # TypeError for dtypes the warp (like cv2.remap) does not take
            payload, pmask = t, None
        want_mask = return_flow or return_valid_area
        placement = None if padding is None else (padding[0], padding[2])

        if self._ref == 't':
            warped, wmask = self._apply_t(payload, pmask, host_tmask, return_flow, return_valid_area, placement, cut)
        else:
            warped, wmask = self._apply_s(payload, pmask, host_tmask, return_flow, want_mask, consider_mask, padding,
                                          cut)
        if return_flow:
            return Flow._wrap(warped, target._ref, wmask)
        img = warped.numpy()[0] if isinstance(warped, DeviceArray) else np.array(warped[0])
        if img.dtype != out_dtype:               # ref 's' resamples in float32
            if np.issubdtype(out_dtype, np.integer):
                img = np.round(img)
            img = img.astype(out_dtype)
        if return_2d:
            img = img[:, :, 0]
        if return_valid_area:
            return img, wmask.numpy()[0].view(np.bool_)
        return img

    def _apply_t(self, payload, pmask, host_tmask, return_flow, return_valid_area, placement, cut):
        if return_flow:
            arith, rule = _lib.ARITH_NATIVE, _lib.RULE_STRICT
        else:
            if return_valid_area:
                arith, rule = _ops.promoted_rule(payload.dtype, host_tmask is not None)
                pmask = None if host_tmask is None else DeviceArray.from_numpy(host_tmask[None].view(np.uint8))
            else:
                arith, rule = _lib.ARITH_NATIVE, _lib.RULE_STRICT
            payload = DeviceArray.from_numpy(payload[None])
        want_mask = return_flow or return_valid_area
        return _ops.warp_t(self._vd(), -1.0, payload, pmask, self._md() if want_mask else None, want_mask, arith,
                           rule, placement, cut)

    def _apply_s(self, payload, pmask, host_tmask, return_flow, want_mask, consider_mask, padding, cut):
        out_is_float = return_flow or np.issubdtype(payload.dtype, np.floating)
        host_payload = None
        if not return_flow:
            host_payload = payload[None]                   # kept for the zero-flow pass-through (any dtype, exact)
            payload = DeviceArray.from_numpy(payload[None], np.float32)
            pmask = None if host_tmask is None else DeviceArray.from_numpy(host_tmask[None].view(np.uint8))
        flow_v, flow_m = self._vd(), self._md()
        if padding is not None:
            flow_v, flow_m = _ops.pad(flow_v, flow_m, padding, 'edge')      # flow_class.py:652-660
        res_mask = None
        if want_mask:                                                        # :634-643, AND before warping
            res_mask = flow_m if pmask is None else _ops.mask_and(pmask, flow_m)
            if padding is not None and host_tmask is not None:
                # the reference overwrites the caller's target_mask in place here (flow_class.py:639-641)
                host_tmask[...] = res_mask.numpy()[0].view(np.bool_)
        # integer payloads: the reference rounds the interpolated payload||mask array before `== 1` (utils.py:256-258)
        rule = _lib.RULE_STRICT if (return_flow or out_is_float) else _lib.RULE_GT_HALF
        if int(_ops.nonzero_flags(flow_v, None, DEFAULT_THRESHOLD)[0]) == 0:
            # apply_flow returns its target untouched for a flow that is zero below the threshold (utils.py:215-216):
            # nothing is resampled, the warped mask is the mask that went in
            warped = payload.copy() if return_flow else host_payload
            wmask = res_mask.copy() if (want_mask and res_mask is not None) else None
        else:
            warped, wmask = _ops.forward_s(flow_v, 1.0, payload, res_mask, flow_m if consider_mask else None,
                                           want_mask, rule)
        if padding is not None and cut:
            fh, fw = self.shape
            if isinstance(warped, np.ndarray):
                warped = warped[:, padding[0]:padding[0] + fh, padding[2]:padding[2] + fw]
            else:
                warped = _ops.crop(warped, padding[0], padding[2], fh, fw)
            if wmask is not None:
                wmask = _ops.crop(wmask, padding[0], padding[2], fh, fw)
        return warped, wmask

    # ------------------------------------------------------------------------------------------ ref switching
    def switch_ref(self, mode=None):
        mode = 'valid' if mode is None else mode
        if mode == 'valid':
            if self.is_zero(thresholded=False):
                return self.switch_ref(mode='invalid')
            if self._ref == 's':
                switched = self.apply(self)
                switched._ref = 't'
                return switched
            as_s = self.switch_ref(mode='invalid')
            return (-as_s).apply(as_s)
        elif mode == 'invalid':
            return Flow._wrap(self._vd().copy(), 't' if self._ref == 's' else 's', self._md().copy())
        raise ValueError("Error switching flow reference: Mode not recognised, should be 'valid' or 'invalid'")

    def invert(self, ref=None):
        ref = self._ref if ref is None else get_valid_ref(ref)
        if self._ref == ref == 's':
            return self.apply(-self)
        if self._ref == ref == 't':
            return self.invert('s').switch_ref()
        # cross-reference inversion is a negation plus relabelling (flow_class.py:748,751)
        return Flow._wrap(_ops.scale(_lib.OP_MUL, self._vd(), -1.0, -1.0, False), ref, self._md().copy())

    def track(self, pts, int_out=None, get_valid_status=None, s_exact_mode=None):
        from .ops import _track_device
        int_out, get_valid_status, s_exact_mode = validate_track_args(pts, int_out, get_valid_status, s_exact_mode)
        warped = _track_device(self, pts, int_out, s_exact_mode)
        if get_valid_status:
            status = self.valid_source()[np.round(pts[..., 0]).astype('i'), np.round(pts[..., 1]).astype('i')]
            return warped, status
        return warped

    # ------------------------------------------------------------------------------------------ valid areas
    def valid_target(self, consider_mask=None):
        consider_mask = True if consider_mask is None else consider_mask
        if not isinstance(consider_mask, bool):
            raise TypeError("Error applying flow: Consider_mask needs to be a boolean")
        if self._ref == 's':
            if int(_ops.nonzero_flags(self._vd(), None, DEFAULT_THRESHOLD)[0]) == 0:
                return np.array(self.mask)      # apply_flow hands the mask back for a thresholded-zero flow
            _, area = _ops.forward_s(self._vd(), 1.0, None, self._md(), self._md() if consider_mask else None)
        else:
            area = _ops.valid_geom_t(self._vd(), -1.0, self._md())
        return area.numpy()[0].view(np.bool_)

    def valid_source(self, consider_mask=None):
        consider_mask = True if consider_mask is None else consider_mask
        if not isinstance(consider_mask, bool):
            raise TypeError("Error applying flow: Consider_mask needs to be a boolean")
        if self._ref == 's':
            area = _ops.valid_geom_t(self._vd(), 1.0, self._md())
        else:
            if int(_ops.nonzero_flags(self._vd(), None, DEFAULT_THRESHOLD)[0]) == 0:
                return np.array(self.mask)
            _, area = _ops.forward_s(self._vd(), -1.0, None, self._md(), self._md() if consider_mask else None)
        return area.numpy()[0].view(np.bool_)

    def visualise(self, mode, show_mask=None, show_mask_borders=None, range_max=None):
        """Flow as an rgb / bgr / hsv image (flow_class.py:869-951): hue = direction, saturation = magnitude scaled to
        `range_max` (default: 99th percentile of the magnitudes, found by radix selection on the device), optionally
        invalid areas greyed out and the mask outline in black. Returns a numpy uint8 array (H, W, 3)."""
        _, show_mask, show_mask_borders = validate_visualise_args(mode, show_mask, show_mask_borders, range_max)
        return _ops.visualise(self._vd(), self._md(), mode, show_mask, show_mask_borders, range_max, DEFAULT_THRESHOLD)

    # ---- host-side presentation / estimation (SURVEY section 2 rows 19-20: not on the hot path, delegated)
    def _host_reference(self):
        """The same flow as an object of the reference package on a host copy: `matrix` (OpenCV's robust estimators),
        `visualise_arrows` and the `show*` GUI helpers are OpenCV drawing / windows on the host and are not rebuilt
        here. Needs `oflibnumpy` importable next to this package."""
        try:
            import oflibnumpy
        except ImportError as e:
            raise ImportError("oflibnumpy_b200 delegates matrix / visualise_arrows / show* to the reference package on "
                              "a host copy of the flow: install oflibnumpy to use them") from e
        return oflibnumpy.Flow(np.array(self.vecs), self._ref, np.array(self.mask))

    def matrix(self, dof=None, method=None, masked=None):
        """flow_class.py:797-867 on a host copy (cv2.estimateAffinePartial2D / estimateAffine2D / findHomography)."""
        return self._host_reference().matrix(dof, method, masked)

    def visualise_arrows(self, grid_dist=None, img=None, scaling=None, show_mask=None, show_mask_borders=None,
                         colour=None, thickness=None):
        """flow_class.py:953-1059 on a host copy (OpenCV drawing)."""
        return self._host_reference().visualise_arrows(grid_dist, img, scaling, show_mask, show_mask_borders, colour,
                                                       thickness)

    def show(self, wait=None, show_mask=None, show_mask_borders=None):
        """flow_class.py:1061-1077 on a host copy (cv2.imshow)."""
        return self._host_reference().show(wait, show_mask, show_mask_borders)

    def show_arrows(self, wait=None, grid_dist=None, img=None, scaling=None, show_mask=None, show_mask_borders=None,
                    colour=None):
        """flow_class.py:1079-1111 on a host copy (cv2.imshow)."""
        return self._host_reference().show_arrows(wait, grid_dist, img, scaling, show_mask, show_mask_borders, colour)

    def get_padding(self):
        """[top, bottom, left, right] as in the reference (flow_class.py:1197-1228); masked min/max on the device."""
        mny, mxy, mnx, mxx = (float(x) for x in _ops.extent(self._vd(), self._md(), 1.0 if self._ref == 't' else -1.0,
                                                            DEFAULT_THRESHOLD)[0])
        h, w = self.shape
        if not math.isfinite(mny):   # empty mask: the reference fails on min() of an empty selection
            raise ValueError("zero-size array to reduction operation minimum which has no identity")
        p = [max(-mny, 0), max(mxy - (h - 1), 0), max(-mnx, 0), max(mxx - (w - 1), 0)]
        return [int(math.ceil(x)) for x in p]

    def is_zero(self, thresholded=None, masked=None):
        masked = True if masked is None else masked
        if not isinstance(masked, bool):
            raise TypeError("Error checking whether flow is zero: Masked needs to be a boolean")
        thresholded = True if thresholded is None else thresholded
        if not isinstance(thresholded, bool):
            raise TypeError("Error checking whether flow is zero: Thresholded needs to be a boolean")
        flags = _ops.nonzero_flags(self._vd(), self._md() if masked else None,
                                   DEFAULT_THRESHOLD if thresholded else 0.0)
        return bool(flags[0] == 0)

    # ------------------------------------------------------------------------------------------ combination
    def combine_with(self, flow, mode, thresholded=None):
        """``flow_1 (+) flow_2 = flow_3`` algebra of the reference (flow_class.py:1247-1424). Mode 3 is one fused
        kernel (ofk_combine3); modes 1 and 2 chain the forward / backward warps on the device."""
        if not isinstance(flow, Flow):
            raise TypeError("Error combining flows: Flow need to be of type 'Flow'")
        if not self.shape == flow.shape:
            raise ValueError("Error combining flows: Flow fields need to have the same shape")
        if not self.ref == flow.ref:
            raise ValueError("Error combining flows: Flow fields need to have the same reference")
        if mode not in [1, 2, 3]:
            raise ValueError("Error combining flows: Mode needs to be 1, 2 or 3")
        thresholded = False if thresholded is None else thresholded
        if not isinstance(thresholded, bool):
            raise TypeError("Error combining flows: Thresholded needs to be a boolean")
        thr = DEFAULT_THRESHOLD if thresholded else 0.0

        if mode == 3:
            # speculative fused composition; the zero tests ride along and decide which object is returned
            v, m, flags = _ops.combine3(self._vd(), self._md(), flow._vd(), flow._md(), self._ref, thr)
            a_nz, b_nz = (int(x) for x in flags.numpy()[0])
            if not a_nz:
                return flow
            if not b_nz:
                return self
            return Flow._wrap(v, self._ref, m)

        if self.is_zero(thresholded=thresholded):
            return flow
        if flow.is_zero(thresholded=thresholded):
            return self.invert()
        # the chains of flow_class.py:1357-1410 (switch_ref / invert / apply / + / -) run as one device-resident
        # sequence behind ofk_combine12, including the zero-flow tests inside switch_ref and apply_flow
        v, m = _ops.combine12(mode, self._ref, self._vd(), self._md(), flow._vd(), flow._md())
        return Flow._wrap(v, self._ref, m)

    def consistent_with(self, flow, alpha_1=None, alpha_2=None, return_valid_area=None):
        """Forward-backward consistency check of this flow (forward, frame 1 -> frame 2) with ``flow`` (backward, frame
        2 -> frame 1): ``FlowBatch.consistent_with`` of the one frame, through the same call. Returns a numpy bool
        array (H,W), and with ``return_valid_area`` also the valid area."""
        return_valid_area = False if return_valid_area is None else return_valid_area
        a1, a2 = validate_consistency_args(self, flow, alpha_1, alpha_2, return_valid_area, Flow)
        out, valid = _ops.consistency(self._vd(), self._md(), flow._vd(), flow._md(), self._ref, a1, a2,
                                      return_valid_area)
        out = out.numpy()[0].view(np.bool_)
        return (out, valid.numpy()[0].view(np.bool_)) if return_valid_area else out

    def evaluate(self, truth, region=None):
        """Error metrics of this flow, the estimate, against ``truth``, the ground truth of the same shape and ref:
        ``FlowBatch.evaluate(...).summary()`` of the one frame, through the same call. ``region`` (H,W) bool / uint8,
        numpy or device, restricts the evaluated pixels (``self.mask & truth.mask & region``). Returns a dict of 'epe',
        'ae', 'fl', 'out1', 'out3', 'out5', 's0-10', 's10-40', 's40+' and 'pixels'."""
        from .batch import FlowBatch
        validate_evaluate_args(self, truth, region, False, Flow)
        if region is not None:
            region = region[None] if isinstance(region, np.ndarray) else \
                dev.as_device(region).reshape((1,) + self.shape)
        batch = FlowBatch._wrap(self._vd(), self._ref, self._md())
        return batch.evaluate(FlowBatch._wrap(truth._vd(), truth._ref, truth._md()), region).summary()


def _ones_mask(shape):
    m = DeviceArray.empty((1, shape[0], shape[1]), np.uint8)
    _lib.call('ofk_rt_memset', m.ptr, 1, m.nbytes, dev.current_stream())
    return m


def _as_window(item, shape):
    """(y0, x0, h, w) if ``item`` selects a contiguous, non-empty 2-D window with unit steps, else None."""
    if not isinstance(item, tuple):
        item = (item,)
    if len(item) > 2 or not all(isinstance(s, slice) for s in item):
        return None
    item = item + (slice(None),) * (2 - len(item))
    out = []
    for s, n in zip(item, shape):
        start, stop, step = s.indices(n)
        if step != 1 or stop <= start:
            return None
        out.append((start, stop - start))
    return out[0][0], out[1][0], out[0][1], out[1][1]
