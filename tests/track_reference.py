"""The single-frame point tracking of Flow.track (utils.py:547-622), restated for the tests without the package's
Flow.track or ofk_track: the reference that FlowBatch.track, FlowBatch.track_clips and Flow.track are compared with.

Each route is computed as the package computed it before its single-frame path ran through the batched kernel:

  zero flow        : numpy's threshold test (oracle.flowref.is_zero_array); the points come back as the same object
  's' int points   : ``pts + vecs[r, c, ::-1]`` on the host (float32 vectors, numpy's dtype promotion and index wrap)
  's' float points : oracle.flowref.bilinear_at in float64 (IndexError outside [0,H-1]x[0,W-1])
  's' exact, 't'   : ofk_mesh_sample at the float64 points, on the undisplaced grid (a zero mesh) for 's' and on the
                     grid displaced by -flow for 't'; rows where no triangle contains the point are 0 (griddata's NaN)
  int_out          : ``np.round(x).astype('i')``
  status           : ``Flow(...).valid_source()`` indexed at the rounded points
"""
import numpy as np

from oracle import flowref as R


def track(flow, pts, int_out=False, get_valid_status=False, s_exact_mode=False):
    """``flow.track(pts, int_out, get_valid_status, s_exact_mode)`` for an oflibnumpy_b200 Flow and numpy points
    (P,2) whose arguments are valid."""
    from oflibnumpy_b200 import _ops
    from oflibnumpy_b200.device import DeviceArray
    vecs = np.asarray(flow.vecs)
    if R.is_zero_array(vecs):
        warped = pts
    elif flow.ref == 's' and np.issubdtype(pts.dtype, np.integer):
        warped = pts + vecs[pts[:, 0], pts[:, 1], ::-1]
    elif flow.ref == 's' and not np.issubdtype(pts.dtype, np.floating):
        raise TypeError("Error tracking points: Pts numpy array needs to have a float or int dtype")
    elif flow.ref == 's' and not s_exact_mode:
        p = pts.astype(np.float64)
        warped = p + R.bilinear_at(vecs[..., ::-1], p)
    else:
        dvecs = flow._vd()
        mesh = DeviceArray.zeros(dvecs.shape, np.float32) if flow.ref == 's' else dvecs
        q = DeviceArray.from_numpy(np.ascontiguousarray(pts, dtype=np.float64)[None])
        vals, _, found = _ops.mesh_sample(mesh, -1.0, dvecs, None, query_pts=q, want_mask=False, want_found=True)
        warped = pts + vals.numpy()[0].astype(np.float64)[:, ::-1]
        warped[found.numpy()[0] == 0] = 0
    if int_out:
        warped = np.round(warped).astype('i')
    if get_valid_status:
        return warped, flow.valid_source()[np.round(pts[..., 0]).astype('i'), np.round(pts[..., 1]).astype('i')]
    return warped
