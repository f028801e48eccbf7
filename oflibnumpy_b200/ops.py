"""Array-in / array-out functions of the public API (reference: utils.py and flow_operations.py of oflibnumpy).

Each takes and returns numpy arrays like the reference, uploads once, runs the CUDA entry point(s) and downloads the
result. For pipelines, keep data on the device with :class:`Flow` / :class:`FlowBatch` instead.
"""
import math

import numpy as np

from . import _lib
from . import _ops
from .device import DeviceArray
from .flow import Flow
from .validation import (get_valid_ref, validate_shape, validate_flow_array, validate_transform_list,
                         validate_track_args, validate_track_dtype, DEFAULT_THRESHOLD)

__all__ = ['apply_flow', 'combine_flows', 'invert_flow', 'switch_flow_ref', 'valid_target', 'valid_source',
           'get_flow_padding', 'from_matrix', 'from_transforms', 'matrix_from_transforms', 'matrix_from_transform',
           'is_zero_flow', 'threshold_vectors', 'points_inside_area', 'resize_flow', 'track_pts', 'load_kitti',
           'load_sintel', 'load_sintel_mask', 'visualise_flow', 'get_flow_matrix', 'visualise_flow_arrows', 'show_flow',
           'show_flow_arrows', 'visualise_definition']

from .io import load_kitti, load_sintel, load_sintel_mask  # noqa: E402,F401


# ------------------------------------------------------------------------------------------------- field generators
def matrix_from_transform(transform, values):
    """3x3 matrix of one transform (utils.py:131-158). The image y axis points down, hence the rotation signs."""
    m = np.identity(3)
    if transform == 'translation':
        m[0, 2], m[1, 2] = values[0], values[1]
    elif transform in ('scaling', 'rotation'):
        pre = matrix_from_transform('translation', [-values[0], -values[1]])
        post = matrix_from_transform('translation', values[:2])
        if transform == 'scaling':
            m[0, 0] = m[1, 1] = values[2]
        else:
            r = math.radians(values[2])
            m[0:2, 0:2] = [[math.cos(r), math.sin(r)], [-math.sin(r), math.cos(r)]]
        m = post @ m @ pre
    return m


def matrix_from_transforms(transform_list):
    m = np.identity(3)
    for t in reversed(transform_list):
        m = m @ matrix_from_transform(t[0], t[1:])
    return m


def _from_matrix_device(matrix, shape, ref):
    validate_shape(shape)
    if not isinstance(matrix, np.ndarray):
        raise TypeError("Error creating flow from matrix: Matrix needs to be a numpy array")
    if matrix.shape != (3, 3):
        raise ValueError("Error creating flow from matrix: Matrix needs to be a numpy array of shape (3, 3)")
    ref = get_valid_ref(ref)
    if ref == 's':
        return _ops.from_matrix(matrix[None], shape, 1.0)
    return _ops.from_matrix(np.linalg.pinv(matrix)[None], shape, -1.0)      # utils.py:343


def _from_transforms_device(transform_list, shape, ref):
    validate_shape(shape)
    validate_transform_list(transform_list)
    ref = get_valid_ref(ref)
    return _from_matrix_device(matrix_from_transforms(transform_list), shape, ref)


def from_matrix(matrix, shape, ref):
    """Flow field (H,W,2) float32 of a 3x3 transformation matrix (utils.py:319-344)."""
    return _from_matrix_device(matrix, shape, ref).numpy()[0]


def from_transforms(transform_list, shape, ref):
    """Flow field (H,W,2) float32 of a list of transforms (utils.py:347-423)."""
    return _from_transforms_device(transform_list, shape, ref).numpy()[0]


# ------------------------------------------------------------------------------------------------- warp
def upload_flow_array(flow, error_string):
    """validate_flow_array + upload; float32 input is tested for NaN / Inf on the device after the upload."""
    on_device = isinstance(flow, np.ndarray) and flow.dtype == np.float32
    flow = validate_flow_array(flow, error_string, finite_on_device=True)
    d = DeviceArray.from_numpy(flow[None])
    if on_device and not _ops.all_finite(d):
        raise ValueError(error_string + "Flow array contains NaN or Inf values")
    return flow, d


def apply_flow(flow, target, ref, mask=None):
    """Warp ``target`` (H,W[,C]) with ``flow`` (H,W,2): reference ``apply_flow`` (utils.py:199-261)."""
    ref = get_valid_ref(ref)
    flow, dflow = upload_flow_array(flow, "Error applying flow to a target: ")
    if int(_ops.nonzero_flags(dflow, None, DEFAULT_THRESHOLD)[0]) == 0:
        return target          # the reference returns the very same object (utils.py:215-216), before any other check
    if not isinstance(target, np.ndarray):
        raise TypeError("Error applying flow to a target: Target needs to be a numpy array")
    if target.ndim < 2 or target.ndim > 3:
        raise ValueError("Error applying flow to a target: Target array needs to have shape H-W or H-W-C")
    if target.shape[:2] != flow.shape[:2]:
        raise ValueError("Error applying flow to a target: Target height and width needs to match flow field array")
    if mask is not None:
        if not isinstance(mask, np.ndarray):
            raise TypeError("Error applying flow to a target: Mask needs to be a numpy array")
        if mask.shape != flow.shape[:2]:
            raise ValueError("Error applying flow to a target: Mask height and width needs to match flow field array")
        if mask.dtype != bool:
            raise TypeError("Error applying flow to a target: Mask needs to be boolean")
    t = target[..., None] if target.ndim == 2 else target
    if ref == 't':
        _ops.dtype_code(t.dtype)
        out, _ = _ops.warp_t(dflow, -1.0, DeviceArray.from_numpy(t[None]))
        res = out.numpy()[0]
    else:
        pm = None if mask is None else DeviceArray.from_numpy(mask[None].view(np.uint8))
        out, _ = _ops.forward_s(dflow, 1.0, DeviceArray.from_numpy(t[None], np.float32), None, pm, want_mask=False)
        res = out.numpy()[0]
        if np.issubdtype(target.dtype, np.integer):
            res = np.round(res)
        res = res.astype(target.dtype)
    return res[..., 0] if target.ndim == 2 else res


# ------------------------------------------------------------------------------------------------- flow algebra
def combine_flows(input_1, input_2, mode, ref=None, thresholded=None):
    """Combination of two flows, ``flow_1 (+) flow_2 = flow_3`` (flow_operations.py:70-161)."""
    if isinstance(input_1, Flow) and isinstance(input_2, Flow):
        print("AVOID - future deprecation warning: using combine_flows(flow_obj1, flow_obj2) is deprecated and may "
              "not work anymore in future versions - use flow_obj1.combine_with(flow_obj2) instead. combine_flows() "
              "will be reserved for use with NumPy arrays only.")
        return input_1.combine_with(input_2, mode=mode, thresholded=thresholded)
    return Flow(input_1, ref).combine_with(Flow(input_2, ref), mode=mode, thresholded=thresholded).vecs


def switch_flow_ref(flow, input_ref):
    return Flow(flow, input_ref).switch_ref().vecs


def invert_flow(flow, input_ref, output_ref=None):
    output_ref = input_ref if output_ref is None else output_ref
    return Flow(flow, input_ref).invert(output_ref).vecs


def valid_target(flow, ref):
    return Flow(flow, ref).valid_target()


def valid_source(flow, ref):
    return Flow(flow, ref).valid_source()


def get_flow_padding(flow, ref):
    return Flow(flow, ref).get_padding()


def is_zero_flow(flow, thresholded=None):
    """True if every vector is zero, optionally below the 1e-3 threshold (utils.py:527-544)."""
    flow, dflow = upload_flow_array(flow, "Error checking whether flow is zero: ")
    thresholded = True if thresholded is None else thresholded
    if not isinstance(thresholded, bool):
        raise TypeError("Error checking whether flow is zero: Thresholded needs to be a boolean")
    flags = _ops.nonzero_flags(dflow, None, DEFAULT_THRESHOLD if thresholded else 0.0)
    return bool(flags[0] == 0)


def threshold_vectors(vecs, threshold=None, use_mag=None):
    """Host helper kept for API parity (utils.py:298-316); the device paths threshold inside their kernels."""
    threshold = DEFAULT_THRESHOLD if threshold is None else threshold
    use_mag = False if use_mag is None else use_mag
    f = vecs.copy()
    if use_mag:
        f[np.linalg.norm(vecs, axis=-1) < threshold] = 0
    else:
        f[(vecs < threshold) & (vecs > -threshold)] = 0
    return f


def points_inside_area(pts, shape):
    """True for points (row, col) that round into the (H,W) area (utils.py:283-295)."""
    return _ops.points_inside_area(pts, shape)


# ------------------------------------------------------------------------------------------------- "next" rows
def _valid_scale(scale):
    if isinstance(scale, (float, int)):
        scale = [scale, scale]
    elif isinstance(scale, (tuple, list)):
        if len(scale) != 2:
            raise ValueError("Error resizing flow: Scale {} must have a length of 2".format(type(scale)))
        if not all(isinstance(item, (float, int)) for item in scale):
            raise ValueError("Error resizing flow: Scale {} items must be integers or floats".format(type(scale)))
    else:
        raise TypeError("Error resizing flow: "
                        "Scale must be an integer, float, or list or tuple of integers or floats")
    if any(s <= 0 for s in scale):
        raise ValueError("Error resizing flow: Scale values must be larger than 0")
    return scale


def _resize_device(vecs, mask, scale):
    scale = _valid_scale(scale)
    return _ops.resize_flow(vecs, mask, scale[0], scale[1])


def resize_flow(flow, scale):
    """Resize a flow field array, scaling the vector values accordingly (utils.py:493-524)."""
    flow, dflow = upload_flow_array(flow, "Error resizing flow: ")
    scale = _valid_scale(scale)
    out, _ = _ops.resize_flow(dflow, None, scale[0], scale[1])
    return out.numpy()[0]


def _track_device(flow, pts, int_out, s_exact_mode):
    """Point tracking (utils.py:547-622) on the device. `flow` is a Flow object; the arguments have passed
    validate_track_args."""
    vecs = flow._vd()
    if int(_ops.nonzero_flags(vecs, None, DEFAULT_THRESHOLD)[0]) == 0:      # thresholded-zero flow: points unchanged
        warped = pts
    else:
        if flow.ref == 's' and np.issubdtype(pts.dtype, np.integer):
            # direct lookup of the vectors at integer positions: a gather through the same mesh sampler would be
            # overkill; the points are few, so index a (lazy) host view like the reference does
            d = vecs.numpy()[0][pts[:, 0], pts[:, 1], ::-1]
            warped = pts + d
        elif flow.ref == 's' and not np.issubdtype(pts.dtype, np.floating):
            validate_track_dtype(pts.dtype)
        elif flow.ref == 's' and not s_exact_mode:
            warped, outside = _ops.track_bilinear(vecs, pts)
            if outside:
                raise IndexError("Some points are outside of the data area.")
        else:
            # 's' exact mode: interpolate the flow on the undisplaced grid; 't': on the grid displaced by -flow
            zero = DeviceArray.zeros(vecs.shape, np.float32) if flow.ref == 's' else None
            mesh = zero if flow.ref == 's' else vecs
            q = DeviceArray.from_numpy(np.ascontiguousarray(pts, dtype=np.float64)[None])
            vals, _, found = _ops.mesh_sample(mesh, -1.0, vecs, None, query_pts=q, want_mask=False, want_found=True)
            d = vals.numpy()[0].astype(np.float64)[:, ::-1]
            warped = pts + d
            warped[found.numpy()[0] == 0] = 0                               # NaN rows of griddata -> 0 (utils.py:616-618)
    if int_out:
        warped = np.round(warped).astype('i')
    return warped


def track_pts(flow, ref, pts, int_out=None, s_exact_mode=None):
    """Warp points (N,2) given as (row, col) with a flow field (utils.py:547-622)."""
    flow = validate_flow_array(flow, "Error tracking points: ")
    flow = Flow(flow, ref)
    int_out, _, s_exact_mode = validate_track_args(pts, int_out, None, s_exact_mode)
    return _track_device(flow, pts, int_out, s_exact_mode)


def _combine2_t_device(a, b):
    """combine_with(mode=2) for ref 't' (flow_class.py:1398-1410): A, resampled from its source positions
    grid - A to the source positions grid - B of B, is subtracted from B."""
    vals, mval, _ = _ops.mesh_sample(a._vd(), -1.0, a._vd(), a._md(), query_flow=b._vd(), query_sign=-1.0,
                                     pos_f32=True)
    resampled = Flow._wrap(vals, 't', _ops.greater(mval, 0.99))
    return b - resampled


# ---- host-side presentation / estimation wrappers of flow_operations.py:25-68,251-350 (SURVEY section 2 row 21: not on
# ---- the hot path). visualise_flow runs on the device like Flow.visualise; the others delegate like the Flow methods.
def visualise_flow(flow, mode, range_max=None):
    """flow_operations.py:274-284."""
    return Flow(flow).visualise(mode, range_max=range_max)


def get_flow_matrix(flow, ref, dof=None, method=None):
    """flow_operations.py:251-271."""
    return Flow(flow, ref).matrix(
        dof, method, masked=False)


def visualise_flow_arrows(flow, ref, grid_dist=None, img=None, scaling=None, colour=None):
    """flow_operations.py:287-312."""
    return Flow(flow, ref).visualise_arrows(
        grid_dist, img, scaling, False, False, colour)


def show_flow(flow, wait=None):
    """flow_operations.py:315-323."""
    return Flow(flow).show(wait)


def show_flow_arrows(flow, ref, wait=None, grid_dist=None, img=None, scaling=None, colour=None):
    """flow_operations.py:326-350."""
    return Flow(flow, ref).show_arrows(wait, grid_dist, img, scaling,
                                                                                         False, False, colour)


def visualise_definition(mode, shape=None, insert_text=None):
    """flow_operations.py:25-67: the colour-wheel legend, drawn by the reference package on the host."""
    try:
        from oflibnumpy import visualise_definition as ref_visualise_definition
    except ImportError as e:
        raise ImportError("oflibnumpy_b200 delegates visualise_definition to the reference package: install oflibnumpy "
                          "to use it") from e
    return ref_visualise_definition(mode, shape, insert_text)
