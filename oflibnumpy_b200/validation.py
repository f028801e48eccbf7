"""Argument validators of the public API. Types of exception and message texts are the reference's
(utils.py:25-88 of oflibnumpy) because they are part of the drop-in contract; the checks run on the host before any
device call."""
import numbers
import warnings

import numpy as np

DEFAULT_THRESHOLD = 1e-3  # utils.py:22


def get_valid_ref(ref):
    if ref is None:
        return 't'
    if not isinstance(ref, str):
        raise TypeError("Error setting flow reference: Input is not a string")
    if ref not in ('s', 't'):
        raise ValueError("Error setting flow reference: Input is not 's' or 't', but {}".format(ref))
    return ref


def get_valid_padding(padding, error_string=None):
    prefix = error_string or ''
    if not isinstance(padding, (list, tuple)):
        raise TypeError(prefix + "Padding needs to be a tuple or a list list of values [top, bot, left, right]")
    if len(padding) != 4:
        raise ValueError(prefix + "Padding list needs to be a list or tuple of length 4 [top, bot, left, right]")
    if any(not isinstance(p, int) for p in padding):
        raise ValueError(prefix + "Padding list [top, bot, left, right] items need to be integers")
    if any(p < 0 for p in padding):
        raise ValueError(prefix + "Padding list [top, bot, left, right] items need to be 0 or larger")
    return padding


def validate_shape(shape):
    if not isinstance(shape, (list, tuple)):
        raise TypeError("Error creating flow from matrix: Dims need to be a list or a tuple")
    if len(shape) != 2:
        raise ValueError("Error creating flow from matrix: Dims need to be a list or a tuple of length 2")
    if any((item <= 0 or not isinstance(item, int)) for item in shape):
        raise ValueError("Error creating flow from matrix: Dims need to be a list or a tuple of integers above zero")


def validate_flow_array(flow, error_string=None, finite_on_device=False):
    """Host-side shape/type checks of a flow ndarray; returns it as C-contiguous float32. The NaN / Inf test
    (utils.py:55-56) runs here unless `finite_on_device` is set and the array is float32 already: the caller then
    uploads first and tests on the device (upload_flow_array) -- np.isfinite costs more than the upload at megapixel
    sizes. Other dtypes are always tested before the float32 cast, as the reference does."""
    prefix = error_string or ''
    if not isinstance(flow, np.ndarray):
        raise TypeError(prefix + "Flow is not a numpy array")
    if flow.ndim != 3:
        raise ValueError(prefix + "Flow array is not 3-dimensional")
    if flow.shape[2] != 2:
        raise ValueError(prefix + "Flow array does not have 2 channels")
    if not (finite_on_device and flow.dtype == np.float32) and not np.isfinite(flow).all():
        raise ValueError(prefix + "Flow array contains NaN or Inf values")
    return np.ascontiguousarray(flow, dtype=np.float32)


VIS_MODES = {'hsv': 0, 'rgb': 1, 'bgr': 2}


def validate_visualise_args(mode, show_mask, show_mask_borders, range_max):
    """Checks of Flow.visualise (flow_class.py:893-905), shared by Flow.visualise, FlowBatch.visualise and
    batch.visualise_flows_host. Returns (mode code, show_mask, show_mask_borders); None stands for False."""
    show_mask = False if show_mask is None else show_mask
    show_mask_borders = False if show_mask_borders is None else show_mask_borders
    if not isinstance(show_mask, bool):
        raise TypeError("Error visualising flow: Show_mask needs to be boolean")
    if not isinstance(show_mask_borders, bool):
        raise TypeError("Error visualising flow: Show_mask_borders needs to be boolean")
    if range_max is not None:
        if not isinstance(range_max, (float, int)):
            raise TypeError("Error visualising flow: Range_max needs to be an integer or a float")
        if range_max <= 0:
            raise ValueError("Error visualising flow: Range_max needs to be larger than zero")
    if mode not in ('hsv', 'rgb', 'bgr'):                    # a tuple: an unhashable mode raises ValueError too
        raise ValueError("Error visualising flow: Mode needs to be either 'bgr', 'rgb', or 'hsv'")
    return VIS_MODES[mode], show_mask, show_mask_borders


def validate_track_args(pts, int_out, get_valid_status, s_exact_mode, batch_size=None):
    """Checks of Flow.track (flow_class.py:755-795, utils.py:547-622), shared by Flow.track, track_pts and
    FlowBatch.track. Returns (int_out, get_valid_status, s_exact_mode); None stands for False. With batch_size (a
    FlowBatch's N), pts may also be a device array (``__cuda_array_interface__``) and of shape (N,P,2) as well as
    (P,2)."""
    get_valid_status = False if get_valid_status is None else get_valid_status
    if not isinstance(get_valid_status, bool):
        raise TypeError("Error tracking points: Get_tracked needs to be a boolean")
    if not isinstance(pts, np.ndarray) and (batch_size is None or not hasattr(pts, '__cuda_array_interface__')):
        raise TypeError("Error tracking points: Pts needs to be a numpy array")
    if batch_size is None:
        if len(pts.shape) != 2:
            raise ValueError("Error tracking points: Pts needs to have shape N-2")
        if pts.shape[1] != 2:
            raise ValueError("Error tracking points: Pts needs to have shape N-2")
    elif not (len(pts.shape) == 2 or (len(pts.shape) == 3 and pts.shape[0] == batch_size)) or pts.shape[-1] != 2:
        raise ValueError("Error tracking points: Pts needs to have shape ({},P,2) or (P,2)".format(batch_size))
    int_out = False if int_out is None else int_out
    s_exact_mode = False if s_exact_mode is None else s_exact_mode
    if not isinstance(int_out, bool):
        raise TypeError("Error tracking points: Int_out needs to be a boolean")
    if not isinstance(s_exact_mode, bool):
        raise TypeError("Error tracking points: S_exact_mode needs to be a boolean")
    return int_out, get_valid_status, s_exact_mode


def validate_track_dtype(dtype):
    """Point dtypes Flow.track accepts for an 's' flow (utils.py:600-602); FlowBatch.track applies it to both refs."""
    if not (np.issubdtype(dtype, np.integer) or np.issubdtype(dtype, np.floating)):
        raise TypeError("Error tracking points: Pts numpy array needs to have a float or int dtype")


def validate_transform_list(transform_list):
    """Checks of from_transforms (utils.py:363-388)."""
    pre = "Error creating flow from transforms: "
    if not isinstance(transform_list, list):
        raise TypeError(pre + "Transform_list needs to be a list")
    if not all(isinstance(item, list) for item in transform_list):
        raise TypeError(pre + "Transform_list needs to be a list of lists")
    if not all(len(item) > 1 for item in transform_list):
        raise ValueError(pre + "Invalid transforms passed")
    expected = {'translation': 2, 'rotation': 3, 'scaling': 3}
    for t in transform_list:
        if t[0] not in expected:
            raise ValueError(pre + "Transform '{}' not recognised".format(t[0]))
        if len(t) - 1 != expected[t[0]]:
            raise ValueError(pre + "Not enough transform values passed for '{}' - expected {}, got {}"
                             .format(t[0], expected[t[0]], len(t) - 1))
        if not all(isinstance(item, (float, int)) for item in t[1:]):
            raise ValueError(pre + "Transform values for '{}' need to be integers or floats".format(t[0]))


def validate_matrix_args(dof, method, masked, hypotheses):
    """Checks of Flow.matrix (flow_class.py:797-867) plus the hypothesis count of FlowBatch.matrix. Returns (dof, method,
    masked, hypotheses) with the reference's defaults for None (8, 'ransac', True) and 1024 hypotheses. 'lms' with dof
    4 or 6 warns and becomes 'ransac', as in the reference (only findHomography has a plain least-squares method)."""
    pre = "Error fitting transformation matrix to flow: "
    dof = 8 if dof is None else dof
    method = 'ransac' if method is None else method
    masked = True if masked is None else masked
    hypotheses = 1024 if hypotheses is None else hypotheses
    if dof not in (4, 6, 8):
        raise ValueError(pre + "Dof needs to be 4, 6 or 8")
    if method not in ('lms', 'ransac', 'lmeds'):
        raise ValueError(pre + "Method needs to be 'lms', 'ransac', or 'lmeds'")
    if not isinstance(masked, bool):
        raise TypeError(pre + "Masked needs to be boolean")
    if isinstance(hypotheses, bool) or not isinstance(hypotheses, int):
        raise TypeError(pre + "Hypotheses needs to be an integer")
    if not 1 <= hypotheses <= 65536:
        raise ValueError(pre + "Hypotheses needs to be between 1 and 65536")
    if method == 'lms' and dof != 8:
        warnings.warn("Method 'lms' (least mean squares) not supported for fitting a transformation matrix with 4 or 6 "
                      "degrees of freedom to the flow. Method 'ransac' used instead.")
        method = 'ransac'
    return dof, method, masked, hypotheses


def validate_accumulate_args(clip_length, cumulative, thresholded, batch_size, fold=None):
    """Checks of FlowBatch.accumulate. Returns the clip length L: ``clip_length``, or the whole batch for None (1 for
    an empty batch)."""
    pre = "Error accumulating flows: "
    if not isinstance(cumulative, bool):
        raise TypeError(pre + "Cumulative needs to be a boolean")
    if not isinstance(thresholded, bool):
        raise TypeError(pre + "Thresholded needs to be a boolean")
    if fold is not None and not (isinstance(fold, str) and fold in ('left', 'right')):
        raise ValueError(pre + "Fold needs to be 'left' or 'right', not {!r}".format(fold))
    if clip_length is None:
        return max(batch_size, 1)
    if isinstance(clip_length, bool) or not isinstance(clip_length, (int, np.integer)) or clip_length < 1 or \
            batch_size % clip_length != 0:
        raise ValueError(pre + "Clip_length needs to be a positive integer that divides the batch size {}, not {!r}"
                         .format(batch_size, clip_length))
    return int(clip_length)


def validate_consistency_args(flow, other, alpha_1, alpha_2, return_valid_area, flow_type):
    """Checks of Flow.consistent_with / FlowBatch.consistent_with: ``other`` an instance of ``flow_type`` of the same
    shape and reference as ``flow``, alphas real, finite and non-negative (also once rounded to float32, the precision
    of the check), ``return_valid_area`` a boolean. Returns (alpha_1, alpha_2) as floats, with the defaults of Sundaram
    et al. (0.01, 0.5) for None."""
    pre = "Error checking flow consistency: "
    if not isinstance(other, flow_type):
        raise TypeError(pre + "Flow need to be of type '{}'".format(flow_type.__name__))
    def full_shape(f):   # (N, H, W) of a FlowBatch, (H, W) of a Flow
        return ((len(f),) if hasattr(f, '__len__') else ()) + tuple(f.shape)

    if full_shape(flow) != full_shape(other):
        raise ValueError(pre + "Flow fields need to have the same shape")
    if flow.ref != other.ref:
        raise ValueError(pre + "Flow fields need to have the same reference")
    alphas = []
    for name, a, default in (('Alpha_1', alpha_1, 0.01), ('Alpha_2', alpha_2, 0.5)):
        a = default if a is None else a
        ok = not isinstance(a, (bool, np.bool_)) and isinstance(a, numbers.Real)
        if ok:
            with np.errstate(over='ignore'):
                ok = bool(np.isfinite(float(a)) and float(a) >= 0 and np.isfinite(np.float32(a)))
        if not ok:
            raise ValueError(pre + "{} needs to be a non-negative finite number, not {!r}".format(name, a))
        alphas.append(float(a))
    if not isinstance(return_valid_area, bool):
        raise TypeError(pre + "Return_valid_area needs to be a boolean")
    return alphas[0], alphas[1]


def validate_evaluate_args(flow, truth, region, return_epe, flow_type):
    """Checks of Flow.evaluate / FlowBatch.evaluate: ``truth`` an instance of ``flow_type`` of the same shape and
    reference as ``flow``; ``region`` None, or a numpy or device (``__cuda_array_interface__``) array of the flow's full
    shape ((N,H,W) for a FlowBatch, (H,W) for a Flow) and dtype bool / uint8, a numpy one holding only 0 and 1;
    ``return_epe`` a boolean."""
    pre = "Error evaluating flow: "
    if not isinstance(truth, flow_type):
        raise TypeError(pre + "Truth needs to be of type '{}'".format(flow_type.__name__))
    shape = ((len(flow),) if hasattr(flow, '__len__') else ()) + tuple(flow.shape)
    if ((len(truth),) if hasattr(truth, '__len__') else ()) + tuple(truth.shape) != shape:
        raise ValueError(pre + "Flow fields need to have the same shape")
    if flow.ref != truth.ref:
        raise ValueError(pre + "Flow fields need to have the same reference")
    if region is not None:
        if isinstance(region, np.ndarray):
            r_shape, r_dtype = region.shape, region.dtype
        elif hasattr(region, '__cuda_array_interface__'):
            cai = region.__cuda_array_interface__
            r_shape, r_dtype = tuple(cai['shape']), np.dtype(cai['typestr'])
        else:
            raise TypeError(pre + "Region needs to be a numpy or device array")
        if tuple(r_shape) != shape or r_dtype not in (np.bool_, np.uint8):
            raise ValueError(pre + "Region needs shape {} and dtype bool or uint8".format(shape))
        if isinstance(region, np.ndarray) and r_dtype != np.bool_ and ((region != 0) & (region != 1)).any():
            raise ValueError(pre + "Region values must be 0 or 1")
    if not isinstance(return_epe, bool):
        raise TypeError(pre + "Return_epe needs to be a boolean")
