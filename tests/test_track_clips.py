"""Point trajectories through clips: FlowBatch.track_clips (ofk_track_clips). Its oracle is the loop a user writes
today, in this file: ``q = F[k].track(q)`` for every step, with the step rules of the docstring applied on the host
through the single-frame tracking and status of ``track_reference``, ``FlowBatch.valid_target()`` and numpy indexing,
and the lost points dropped between the steps. On the CPU the same loop runs on ``oracle.flowref`` and is pinned on hand-made
cases; on the GPU the kernel must give its positions byte for byte and its alive flags exactly."""
import numpy as np
import pytest

import track_reference
from oracle import flowref as R


@pytest.fixture(scope='module')
def of():
    import oflibnumpy_b200 as of
    of.device.require_gpu()
    return of


@pytest.fixture(scope='module')
def lib():
    from oflibnumpy_b200 import _lib, build
    build.build()
    return _lib


def fake_batch(n=4, h=5, w=6, ref='s'):
    """A FlowBatch whose arrays are never touched: for checks that must fail before any device work."""
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    return FlowBatch._wrap(DeviceArray(0, (n, h, w, 2), np.float32), ref, DeviceArray(0, (n, h, w), np.uint8))


# ------------------------------------------------------------------------------------------------------ the oracle
def rounded_in_frame(q, h, w):
    with np.errstate(invalid='ignore'):
        r = np.round(q)
        return (r[:, 0] >= 0) & (r[:, 0] <= h - 1) & (r[:, 1] >= 0) & (r[:, 1] <= w - 1)


def rounded(q):
    return np.round(q[:, 0]).astype(np.int64), np.round(q[:, 1]).astype(np.int64)


class HostFrame(object):
    """One frame of the loop through oracle.flowref."""

    def __init__(self, vecs, ref, mask):
        self.f = R.make(vecs, ref, mask)
        self.zero = R.is_zero_array(self.f.vecs)
        self.target = R.valid_target(self.f) if ref == 't' else None
        self.source = R.valid_source(self.f) if ref == 's' else None

    def track(self, q, exact):
        return R.track(self.f, q, s_exact_mode=exact)

    def status(self, q):
        y, x = rounded(q)
        return self.source[y, x]


class DeviceFrame(object):
    """One frame of the loop through the single-frame tracking of track_reference (device mesh, host bilinear)."""

    def __init__(self, flow, zero, target):
        self.f, self.zero, self.target = flow, zero, target

    def track(self, q, exact):
        return track_reference.track(self.f, q, s_exact_mode=exact)

    def status(self, q):
        # exact mode never raises, and the status does not depend on the mode
        return track_reference.track(self.f, q, get_valid_status=True, s_exact_mode=True)[1]


def loop_oracle(frames, pts, ref, exact, keep, h, w):
    """One clip: frames[k] is step k, pts (P,2), keep a list of (H,W) planes or None. Returns (positions (L,P,2),
    alive (L,P) uint8). Flow.track returns (0, 0) where no triangle contains a point (griddata's NaN rows), so a mesh
    result of exactly (0, 0) counts as lost; the inputs here never track a point to (0, 0) exactly."""
    q = np.array(pts, np.float64)
    live = np.ones(len(q), bool)
    pos, alive = np.full((len(frames), len(q), 2), np.nan), np.zeros((len(frames), len(q)), np.uint8)
    for k, fr in enumerate(frames):
        live &= rounded_in_frame(q, h, w)
        if ref == 's':
            idx = np.flatnonzero(live)
            if idx.size:
                ok = fr.status(q[idx]).astype(bool)
                if keep is not None:
                    ok &= keep[k][rounded(q[idx])] != 0
                live[idx[~ok]] = False
        idx = np.flatnonzero(live)
        if idx.size and not fr.zero:
            qi = q[idx]
            if ref == 's' and not exact:                  # where the bilinear would raise IndexError
                inside = (0 <= qi[:, 0]) & (qi[:, 0] <= h - 1) & (0 <= qi[:, 1]) & (qi[:, 1] <= w - 1)
                live[idx[~inside]] = False
                idx, qi = idx[inside], qi[inside]
                if idx.size:
                    q[idx] = fr.track(qi, False)
            else:
                new = fr.track(qi, exact)
                lost = (new == 0).all(1)
                live[idx[lost]] = False
                q[idx[~lost]] = new[~lost]
        live &= rounded_in_frame(q, h, w)
        if ref == 't':
            idx = np.flatnonzero(live)
            if idx.size:
                ok = fr.target[rounded(q[idx])].astype(bool)
                if keep is not None:
                    ok &= keep[k][rounded(q[idx])] != 0
                live[idx[~ok]] = False
        pos[k][live] = q[live]
        alive[k] = live
    return pos, alive


def host_loop(vecs, ref, masks, pts, L, exact=False, keep=None):
    """The loop on oracle.flowref over a clip-major batch: pts (S,P,2) or (P,2)."""
    n, h, w = vecs.shape[:3]
    frames = [HostFrame(vecs[i], ref, None if masks is None else masks[i]) for i in range(n)]
    return run_loop(frames, pts, ref, exact, keep, L, h, w)


def run_loop(frames, pts, ref, exact, keep, L, h, w):
    outs = [loop_oracle(frames[s * L:(s + 1) * L], pts if pts.ndim == 2 else pts[s], ref, exact,
                        None if keep is None else keep[s * L:(s + 1) * L], h, w) for s in range(len(frames) // L)]
    return np.concatenate([o[0] for o in outs]), np.concatenate([o[1] for o in outs])


# ------------------------------------------------------------------------------------------------- hand-made cases
H, W = 5, 8
NAN = np.nan


def const(u, v, n=1):
    return np.tile(np.array([u, v], np.float32), (n, H, W, 1))


def hand_cases():
    """(name, vecs, ref, masks, keep, pts, L, exact, expected positions, expected alive)"""
    cases = []
    # 't' translation by half a pixel: the mesh p - flow covers x <= W - 1.5 = 6.5, so 6.75 finds no triangle at step 3
    pos = np.array([[[2, 5.75]], [[2, 6.25]], [[2, 6.75]], [[NAN, NAN]], [[NAN, NAN]]])
    cases.append(('t half-pixel leaves', const(0.5, 0, 5), 't', None, None, np.array([[2, 5.25]]), 5, False, pos,
                  [[1], [1], [1], [0], [0]]))
    # 's' translation by -0.5: pixel 0 sends its vector outside (status 0), so the point is lost at step 2
    for exact in (False, True):
        pos = np.array([[[2, 0.75]], [[2, 0.25]], [[NAN, NAN]], [[NAN, NAN]]])
        cases.append(('s half-pixel leaves', const(-0.5, 0, 4), 's', None, None, np.array([[2, 1.25]]), 4, exact, pos,
                      [[1], [1], [0], [0]]))
    # ties to even: keep has a hole at (2, 2); 2.5 and 1.5 round to 2 (lost), 3.5 to 4 (alive)
    keep = np.ones((1, H, W), bool)
    keep[0, 2, 2] = False
    for ref in ('s', 't'):
        pos = np.array([[[NAN, NAN], [2, 3.5], [NAN, NAN]]])
        cases.append(('ties ' + ref, const(0.0, 0.0), ref, None, keep, np.array([[2, 2.5], [2, 3.5], [2, 1.5]]), 1,
                      False, pos, [[0, 1, 0]]))
    # a masked pixel: 's' tests it at the start of the step, 't' at the end
    masks = np.ones((1, H, W), bool)
    masks[0, 1, 1] = False
    cases.append(('mask s', const(1.0, 0), 's', masks, None, np.array([[1, 1.2], [1, 0.2]]), 1, False,
                  np.array([[[NAN, NAN], [1, 1.2]]]), [[0, 1]]))
    cases.append(('mask t', const(1.0, 0), 't', masks, None, np.array([[1, 1.2], [1, 0.2]]), 1, False,
                  np.array([[[1, 2.2], [NAN, NAN]]]), [[1, 0]]))
    # a keep hole on the second frame
    keep = np.ones((2, H, W), bool)
    keep[1, 3, 4] = False
    cases.append(('keep hole s', const(1.0, 0.5, 2), 's', None, keep, np.array([[2.5, 3], [1.5, 1]]), 2, False,
                  np.array([[[3, 4], [2, 2]], [[NAN, NAN], [2.5, 3]]]), [[1, 1], [0, 1]]))
    # a zero frame (below the 1e-3 threshold) between two moves: the point stays put for a step
    vecs = np.concatenate([const(1.0, 0.0), const(4e-4, -4e-4), const(1.0, 0.0)])
    for ref in ('s', 't'):
        cases.append(('zero frame ' + ref, vecs, ref, None, None, np.array([[2, 2.25]]), 3, False,
                      np.array([[[2, 3.25]], [[2, 3.25]], [[2, 4.25]]]), [[1], [1], [1]]))
    # Flow.track's bilinear on the last row: the clipped weights are all 0, so the point does not move
    pos = np.array([[[4, 3], [2.5, 3]], [[4, 3], [2, 3]]])
    cases.append(('last row', const(0.0, -0.5, 2), 's', None, None, np.array([[4, 3], [3, 3]]), 2, False, pos,
                  [[1, 1], [1, 1]]))
    return cases


@pytest.mark.parametrize('case', hand_cases(), ids=lambda c: c[0] + (' exact' if c[7] else ''))
def test_loop_oracle_on_hand_made_cases(case):
    name, vecs, ref, masks, keep, pts, L, exact, want_pos, want_alive = case
    pos, alive = host_loop(vecs, ref, masks, pts, L, exact, keep)
    np.testing.assert_allclose(pos, want_pos, rtol=0, atol=1e-12, err_msg=name)    # griddata's weights round
    np.testing.assert_array_equal(alive, np.array(want_alive, np.uint8), err_msg=name)


def test_points_outside_are_lost_at_step_zero_in_the_oracle():
    pts = np.array([[-0.6, 3], [3, W - 0.4], [1e300, 0], [NAN, 2], [-np.inf, 0], [2, 3]])
    for ref, exact in (('s', False), ('s', True), ('t', False)):
        pos, alive = host_loop(const(0.25, 0.25, 2), ref, None, pts, 2, exact)
        assert alive[:, :5].sum() == 0 and np.isnan(pos[:, :5]).all()
        np.testing.assert_array_equal(alive[:, 5], [1, 1])


# ------------------------------------------------------------------------------------------------------------- CPU
def test_c_entry_refuses_bad_arguments_without_a_gpu(lib):
    """ofk_track_clips checks every argument before a stream or the device is touched."""
    good = dict(flow=16, mask=None, ref=ord('s'), exact=0, nz=16, pts=16, pts_dtype=lib.F64, shared=0, S=2, L=3, P=8,
                keep=None, out=16, alive=16, H=4, W=4, stream=None)
    for change, msg in (({'flow': None}, "NULL pointer"), ({'nz': None}, "NULL pointer"), ({'pts': None}, "NULL pointer"),
                        ({'out': None}, "NULL pointer"), ({'alive': None}, "NULL pointer"),
                        ({'ref': ord('x')}, "ref must be 's' or 't'"), ({'pts_dtype': lib.I32}, "pts_dtype must be"),
                        ({'pts_dtype': lib.I64}, "pts_dtype must be"), ({'S': -1}, "bad shape"), ({'L': 0}, "bad shape"),
                        ({'P': -1}, "bad shape"), ({'H': 0}, "bad shape"), ({'W': -2}, "bad shape"),
                        ({'S': 1 << 16, 'L': 1 << 15}, "S\\*L must not exceed INT_MAX"),
                        ({'ref': ord('t'), 'H': 1}, "the mesh route needs"), ({'exact': 1, 'W': 1}, "the mesh route needs"),
                        ({'ref': ord('t'), 'H': 1 << 15, 'W': 1 << 15}, "the mesh route needs")):
        args = dict(good, **change)
        with pytest.raises(lib.OflibCudaError, match="ofk_track_clips: " + msg):
            lib.call('ofk_track_clips', *args.values())
    # the 's' bilinear route takes any frame size
    args = dict(good, H=1, W=1, S=0)
    assert lib.call('ofk_track_clips', *args.values()) == 0


BAD_ARGS = [
    # (pts, clip_length, keep, s_exact_mode) on a batch of 4 frames of 5 x 6 -> exception, message
    ((np.zeros((3, 2)), 3, None, None), ValueError, "Clip_length needs to be a positive integer that divides the batch "
                                                    "size 4, not 3"),
    ((np.zeros((3, 2)), 0, None, None), ValueError, "not 0"),
    ((np.zeros((3, 2)), True, None, None), ValueError, "not True"),
    ((np.zeros((3, 2)), 2.0, None, None), ValueError, "not 2.0"),
    (([[1.0, 2.0]], None, None, None), TypeError, "Pts needs to be a numpy or device array"),
    ((np.zeros(4), None, None, None), ValueError, "Pts needs to have shape (1,P,2) or (P,2)"),
    ((np.zeros((3, 3)), None, None, None), ValueError, "Pts needs to have shape (1,P,2) or (P,2)"),
    ((np.zeros((4, 3, 2)), 2, None, None), ValueError, "Pts needs to have shape (2,P,2) or (P,2)"),
    ((np.zeros((3, 2), bool), None, None, None), TypeError, "Pts numpy array needs to have a float or int dtype"),
    ((np.zeros((3, 2), complex), None, None, None), TypeError, "Pts numpy array needs to have a float or int dtype"),
    ((np.zeros((3, 2)), None, [[0]], None), TypeError, "Keep needs to be a numpy or device array"),
    ((np.zeros((3, 2)), None, np.ones((1, 5, 6), bool), None), ValueError, "Keep needs shape (4, 5, 6) and dtype bool "
                                                                           "or uint8"),
    ((np.zeros((3, 2)), None, np.ones((4, 5, 6), np.float32), None), ValueError, "Keep needs shape (4, 5, 6)"),
    ((np.zeros((3, 2)), None, np.full((4, 5, 6), 2, np.uint8), None), ValueError, "Keep values must be 0 or 1"),
    ((np.zeros((3, 2)), None, None, 1), TypeError, "S_exact_mode needs to be a boolean"),
]


@pytest.mark.parametrize('args,exc,msg', BAD_ARGS)
def test_arguments_are_rejected_before_any_device_work(lib, args, exc, msg):
    with pytest.raises(exc) as e:
        fake_batch().track_clips(*args)
    assert str(e.value).startswith("Error tracking points through clips: ")
    assert msg in str(e.value)


def test_device_points_need_a_float_dtype(lib):
    class Dev(object):
        def __init__(self, typestr):
            self.__cuda_array_interface__ = {'shape': (3, 2), 'typestr': typestr, 'data': (0, False), 'version': 3}

    for typestr in ('<i4', '<i8', '<f2'):
        with pytest.raises(TypeError, match="Device pts need dtype float32 or float64"):
            fake_batch().track_clips(Dev(typestr))


def test_accumulate_keeps_its_clip_length_message(lib):
    from oflibnumpy_b200.validation import validate_accumulate_args
    with pytest.raises(ValueError) as e:
        validate_accumulate_args(3, True, False, 4)
    assert str(e.value) == "Error accumulating flows: Clip_length needs to be a positive integer that divides the " \
                           "batch size 4, not 3"


# ------------------------------------------------------------------------------------------------------------- GPU
def swirl(h, w, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[:h, :w].astype(np.float32)
    a, b = rng.uniform(0.3, 0.9, 2) * min(h, w) / 4
    v = np.stack([4 * np.sin(xx / a + seed) * np.cos(yy / b) + 0.002 * (xx - w / 2),
                  3 * np.cos(xx / b + 1) * np.sin(yy / a) - 0.003 * (yy - h / 2)], -1)
    return (v * scale).astype(np.float32)


def make_clips(h, w, S, L, seed):
    """S clips of L frames: smooth swirls at several scales, a rough (white noise, +-3 px at 1080p) frame, and a frame
    below the 1e-3 threshold in every clip; masks with ~2 % holes. Motions shrink with frames smaller than 200 px, so
    that some trajectories last a clip. Returns the forward flows, a backward batch for keep (the forward flows
    negated, plus noise) and the masks."""
    rng = np.random.default_rng(seed)
    amp = min(1.0, min(h, w) / 200)
    frames = []
    for s in range(S):
        for k in range(L):
            if k == 2:
                frames.append(rng.uniform(-5e-4, 5e-4, (h, w, 2)).astype(np.float32))
            elif k == 4:
                frames.append(rng.uniform(-3 * amp, 3 * amp, (h, w, 2)).astype(np.float32))
            else:
                frames.append(swirl(h, w, 10 * s + k, scale=amp * (0.3, 1.0, 2.5)[k % 3]))
    fw = np.stack(frames)
    bw = (-fw + rng.normal(0, 0.3, fw.shape)).astype(np.float32)
    masks = rng.random(fw.shape[:3]) > 0.02
    return fw, bw, masks


def make_points(h, w, S, P, seed):
    """(S, P + 10, 2) float64: random points inside the frame, the borders and the corners."""
    rng = np.random.default_rng(seed)
    edge = [[0, 0], [0, w - 1], [h - 1, 0], [h - 1, w - 1], [0, w / 3], [h - 1, w / 2], [h / 2, 0], [h / 3, w - 1],
            [h - 1.5, w - 1.5], [0.5, 0.5]]
    return np.concatenate([np.tile(np.array(edge, np.float64), (S, 1, 1)),
                           rng.uniform(0, 1, (S, P, 2)) * [h - 1, w - 1]], 1)


def device_loop(of, fb, vecs, pts, L, exact, keep):
    """The loop of single-frame tracking steps (track_reference) over the batch fb (host vecs for the zero test)."""
    target = fb.valid_target().numpy() if fb.ref == 't' else [None] * len(fb)
    frames = [DeviceFrame(fb[i], R.is_zero_array(vecs[i]), target[i]) for i in range(len(fb))]
    h, w = fb.shape
    return run_loop(frames, pts, fb.ref, exact, keep, L, h, w)


def check_parity(got, want, what):
    pos, alive = got[0].numpy(), got[1].numpy()
    assert pos.dtype == np.float64 and alive.dtype == np.uint8
    np.testing.assert_array_equal(alive, want[1], err_msg=str(what))
    assert pos.tobytes() == want[0].tobytes(), what


ROUTES = [('s', False), ('s', True), ('t', False)]


@pytest.mark.gpu
@pytest.mark.parametrize('ref,exact', ROUTES, ids=['s', 's-exact', 't'])
@pytest.mark.parametrize('size', [(1080, 1920, 4096), (37, 53, 300)], ids=['1080p', '37x53'])
def test_clips_match_the_loop_of_flow_track(of, ref, exact, size):
    from oflibnumpy_b200.batch import FlowBatch
    h, w, P = size
    S, L = 2, 8
    fw, bw, masks = make_clips(h, w, S, L, seed=h)
    fb = FlowBatch(fw, ref, masks)
    keep = fb.consistent_with(FlowBatch(bw, ref, masks))
    keep_host = keep.numpy()
    assert 0 < keep_host.mean() < 1
    pts = make_points(h, w, S, P, seed=w)
    for dt, shared, use_keep in ((np.float64, False, True), (np.float32, True, True), (np.float64, True, False),
                                 (np.float32, False, False)):
        p = (pts[0] if shared else pts).astype(dt)
        got = fb.track_clips(p, L, keep=keep if use_keep else None, s_exact_mode=exact)
        want = device_loop(of, fb, fw, p, L, exact, keep_host if use_keep else None)
        check_parity(got, want, (ref, exact, dt, shared, use_keep))
        assert 0 < want[1][L - 1::L].mean() < 1               # some trajectories survive, some are lost


@pytest.mark.gpu
def test_hand_made_cases_on_the_device(of):
    from oflibnumpy_b200.batch import FlowBatch
    for name, vecs, ref, masks, keep, pts, L, exact, want_pos, want_alive in hand_cases():
        got = FlowBatch(vecs, ref, masks).track_clips(pts, L, keep=keep, s_exact_mode=exact)
        np.testing.assert_array_equal(got[0].numpy(), want_pos, err_msg=name)   # the float32 vector rounds to 1/2
        np.testing.assert_array_equal(got[1].numpy(), np.array(want_alive, np.uint8), err_msg=name)


@pytest.mark.gpu
@pytest.mark.parametrize('ref,exact', ROUTES, ids=['s', 's-exact', 't'])
def test_one_step_clips_equal_flowbatch_track(of, ref, exact):
    from oflibnumpy_b200.batch import FlowBatch
    h, w = 120, 160
    fw, _, masks = make_clips(h, w, 1, 6, seed=3)
    fb = FlowBatch(fw, ref, masks)
    pts = make_points(h, w, 6, 500, seed=4)
    pos, alive = (a.numpy() for a in fb.track_clips(pts, 1, s_exact_mode=exact))
    want = fb.track(pts, s_exact_mode=exact).numpy()
    live = alive.astype(bool)
    assert live.mean() > 0.5
    assert pos[live].tobytes() == want[live].tobytes()
    assert np.isnan(pos[~live]).all()


@pytest.mark.gpu
@pytest.mark.parametrize('ref,exact', ROUTES, ids=['s', 's-exact', 't'])
def test_a_clip_alone_equals_the_clip_in_a_batch(of, ref, exact):
    from oflibnumpy_b200.batch import FlowBatch
    h, w, S, L = 64, 96, 3, 5
    fw, bw, masks = make_clips(h, w, S, L, seed=5)
    fb = FlowBatch(fw, ref, masks)
    keep = fb.consistent_with(FlowBatch(bw, ref, masks)).numpy()
    pts = make_points(h, w, S, 400, seed=6)
    pos, alive = (a.numpy() for a in fb.track_clips(pts, L, keep=keep, s_exact_mode=exact))
    for s in range(S):
        sl = slice(s * L, (s + 1) * L)
        one = fb[sl].track_clips(pts[s], L, keep=keep[sl], s_exact_mode=exact)
        assert one[0].numpy().tobytes() == pos[sl].tobytes()
        np.testing.assert_array_equal(one[1].numpy(), alive[sl])
    # one clip of the whole batch is the default
    whole = fb.track_clips(pts[0], s_exact_mode=exact)
    assert whole[0].shape == (S * L, pts.shape[1], 2)


@pytest.mark.gpu
def test_device_points_give_the_bytes_of_host_points(of):
    import torch
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    h, w, S, L = 60, 84, 2, 4
    fw, bw, masks = make_clips(h, w, S, L, seed=7)
    pts = make_points(h, w, S, 300, seed=8)
    for ref, exact in ROUTES:
        fb = FlowBatch(fw, ref, masks)
        keep = fb.consistent_with(FlowBatch(bw, ref, masks))
        for p in (pts, pts.astype(np.float32), pts[1], pts[1].astype(np.float32)):
            want = fb.track_clips(p, L, keep=keep.numpy(), s_exact_mode=exact)
            for dp in (DeviceArray.from_numpy(p), torch.as_tensor(p, device='cuda')):
                for k in (keep, torch.as_tensor(keep.numpy().view(bool), device='cuda')):
                    got = fb.track_clips(dp, L, keep=k, s_exact_mode=exact)
                    assert got[0].numpy().tobytes() == want[0].numpy().tobytes()
                    assert got[1].numpy().tobytes() == want[1].numpy().tobytes()
        # integer points are their float64 values
        ints = np.round(pts).astype(np.int32)
        got = fb.track_clips(ints, L, s_exact_mode=exact)
        want = fb.track_clips(ints.astype(np.float64), L, s_exact_mode=exact)
        assert got[0].numpy().tobytes() == want[0].numpy().tobytes()


@pytest.mark.gpu
def test_empty_inputs_and_points_outside(of):
    from oflibnumpy_b200.batch import FlowBatch
    h, w = 37, 53
    fw, _, masks = make_clips(h, w, 1, 4, seed=9)
    for ref, exact in ROUTES:
        fb = FlowBatch(fw, ref, masks)
        for p, shape in ((np.zeros((0, 2)), (4, 0)), (np.zeros((2, 0, 2), np.float32), (4, 0))):
            before = of._lib.call('ofk_rt_launch_count')
            pos, alive = fb.track_clips(p, 2)
            assert of._lib.call('ofk_rt_launch_count') == before
            assert pos.shape == shape + (2,) and pos.dtype == np.float64
            assert alive.shape == shape and alive.dtype == np.uint8
        empty = fb[0:0]
        pos, alive = empty.track_clips(np.zeros((5, 2)))
        assert pos.shape == (0, 5, 2) and alive.shape == (0, 5)
        out = np.array([[-0.6, 3], [3, w - 0.4], [1e300, 0], [np.nan, 2], [-np.inf, 0], [h, 0], [0, -1]])
        pts = np.concatenate([out, make_points(h, w, 1, 50, seed=10)[0]])
        got = fb.track_clips(pts, 2, s_exact_mode=exact)
        alive = got[1].numpy()
        assert alive[:, :len(out)].sum() == 0 and np.isnan(got[0].numpy()[:, :len(out)]).all()
        check_parity(got, device_loop(of, fb, fw, pts, 2, exact, None), (ref, exact))


@pytest.mark.gpu
def test_batches_over_4_gib_use_64_bit_offsets(of):
    """34 copies of one 8-frame 1080p clip (4.5 GB of flows): the clips past 4 GiB give the bytes of the first."""
    import torch
    from oflibnumpy_b200.batch import FlowBatch
    h, w, L, S = 1080, 1920, 8, 34
    assert (S - 1) * L * h * w * 8 > 1 << 32
    fw, _, masks = make_clips(h, w, 1, L, seed=11)
    pts = make_points(h, w, 1, 4096, seed=12)[0]
    for ref, exact in ROUTES:
        big = torch.as_tensor(fw, device='cuda').repeat(S, 1, 1, 1)
        big_m = torch.as_tensor(masks, device='cuda').repeat(S, 1, 1)
        fb = FlowBatch(big, ref, big_m)
        pos, alive = fb.track_clips(pts, L, s_exact_mode=exact)
        want = FlowBatch(fw, ref, masks).track_clips(pts, L, s_exact_mode=exact)
        want_p, want_a = want[0].numpy(), want[1].numpy()
        for s in (S - 2, S - 1):
            assert pos.frames(s * L, (s + 1) * L).numpy().tobytes() == want_p.tobytes()
            np.testing.assert_array_equal(alive.frames(s * L, (s + 1) * L).numpy(), want_a)
        del fb, big, big_m, pos, alive
        torch.cuda.empty_cache()


@pytest.mark.gpu
def test_launch_count_does_not_grow_with_the_clips(of):
    from oflibnumpy_b200 import _ops
    from oflibnumpy_b200.batch import FlowBatch
    h, w = 37, 53
    fw, bw, masks = make_clips(h, w, 16, 40, seed=13)
    pts = make_points(h, w, 1, 100, seed=14)[0]
    flags = FlowBatch(fw[:2], 's', masks[:2])
    before = of._lib.call('ofk_rt_launch_count')
    _ops.nonzero_flags_device(flags.vecs, None, 1e-3)
    zero_test = of._lib.call('ofk_rt_launch_count') - before

    def launches(fb, L, **kw):
        fb.track_clips(pts, L, **kw)
        before = of._lib.call('ofk_rt_launch_count')
        fb.track_clips(pts, L, **kw)
        return of._lib.call('ofk_rt_launch_count') - before

    for ref, exact in ROUTES:
        small = FlowBatch(fw[:2], ref, masks[:2])
        big = FlowBatch(fw, ref, masks)
        keep = big.consistent_with(FlowBatch(bw, ref, masks))
        assert launches(small, 2, s_exact_mode=exact) == zero_test + 1
        assert launches(big, 40, s_exact_mode=exact, keep=keep) == zero_test + 1


@pytest.mark.gpu
def test_the_call_does_not_synchronise(of, monkeypatch):
    """No download, no synchronisation, no read-back, for host and device points and keep planes."""
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    h, w, S, L = 60, 84, 2, 3
    fw, bw, masks = make_clips(h, w, S, L, seed=15)
    pts = make_points(h, w, S, 100, seed=16)
    pts[0, 0] = [-5, 1e9]                                   # a point outside: still no read-back
    batches = {r: FlowBatch(fw, r, masks) for r in ('s', 't')}
    keeps = {r: batches[r].consistent_with(FlowBatch(bw, r, masks)) for r in ('s', 't')}
    dpts = DeviceArray.from_numpy(pts)
    of.device.set_stream(None)                  # on a non-default stream the upload of pageable points synchronises
    real_call = _lib.call

    def no_sync(name, *args):
        assert name not in ('ofk_rt_memcpy_d2h', 'ofk_rt_stream_sync', 'ofk_rt_device_sync', 'ofk_rt_event_sync'), name
        return real_call(name, *args)

    def no_numpy(self, out=None):
        raise AssertionError("DeviceArray.numpy called")

    results = []
    monkeypatch.setattr(_lib, 'call', no_sync)
    monkeypatch.setattr(DeviceArray, 'numpy', no_numpy)
    for ref, exact in ROUTES:
        for p in (pts, pts[0].astype(np.int64), dpts):
            results.append(batches[ref].track_clips(p, L, keep=keeps[ref], s_exact_mode=exact))
    monkeypatch.undo()
    assert len(results) == 9
