"""Batched point tracking: FlowBatch.track (ofk_track). Frame i of the result must equal the single-frame tracking of
Flow(vecs[i], ref, masks[i]) as track_reference restates it, byte for byte, dtype included, on every route: 's' integer
lookup, 's' float bilinear, 's' exact, 't', zero-flow frames and int_out; the status equals the reference's. IndexError
is raised where a loop of Flow.track would raise, for the lowest such frame. Flow.track itself, the one-frame case of
FlowBatch.track, is held to the same reference."""
import itertools

import numpy as np
import pytest

import track_reference
from conftest import load_golden
from oracle import flowref as R

PT_DTYPES = (np.float64, np.float32, np.int64, np.int32, np.int16)


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


def fake_batch(n=3, h=4, w=5, ref='s'):
    """A FlowBatch whose arrays are never touched: for checks that must fail before any device work."""
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    return FlowBatch._wrap(DeviceArray(0, (n, h, w, 2), np.float32), ref, DeviceArray(0, (n, h, w), np.uint8))


# ------------------------------------------------------------------------------------------------------------- CPU
def test_bad_arguments_are_rejected_without_a_gpu(lib):
    """ofk_track checks every argument before a stream or the device is touched."""
    s, t = ord('s'), ord('t')
    good = dict(flow=16, mask=None, ref=s, exact=0, nz=16, pts=16, pts_dtype=lib.F64, shared=0, P=8, arith=lib.F64,
                int_out=0, out=16, plane=None, status=None, errors=16, N=2, H=4, W=4, stream=None)
    for change, msg in (({'flow': None}, "ofk_track: NULL pointer"), ({'nz': None}, "ofk_track: NULL pointer"),
                        ({'pts': None}, "ofk_track: NULL pointer"), ({'out': None}, "ofk_track: NULL pointer"),
                        ({'errors': None}, "ofk_track: NULL pointer"), ({'ref': ord('x')}, "ref must be 's' or 't'"),
                        ({'pts_dtype': lib.U8}, "pts_dtype must be"), ({'pts_dtype': 7}, "pts_dtype must be"),
                        ({'arith': lib.I32}, "arith must be"), ({'arith': lib.F32}, "float32 arithmetic needs"),
                        ({'arith': lib.F32, 'pts_dtype': lib.I32, 'ref': t}, "float32 arithmetic needs"),
                        ({'arith': lib.F32, 'pts_dtype': lib.F32, 'exact': 1}, "float32 arithmetic needs"),
                        ({'N': -1}, "bad shape"), ({'P': -1}, "bad shape"), ({'H': -4}, "bad shape"),
                        ({'W': 0}, "bad shape"), ({'ref': t, 'H': 1}, "mesh route needs"),
                        ({'exact': 1, 'W': 1}, "mesh route needs"),
                        ({'ref': t, 'status': 16}, "ref 't' status needs status_plane")):
        args = dict(good, **change)
        with pytest.raises(lib.OflibCudaError, match=msg):
            lib.call('ofk_track', *args.values())


EXPECTED_MESSAGES = [
    # (pts, int_out, get_valid_status, s_exact_mode) -> the exception Flow.track raised before the checks were shared
    (([[1.0, 2.0]], None, None, None), TypeError, "Error tracking points: Pts needs to be a numpy array"),
    ((np.zeros(4), None, None, None), ValueError, "Error tracking points: Pts needs to have shape N-2"),
    ((np.zeros((4, 3)), None, None, None), ValueError, "Error tracking points: Pts needs to have shape N-2"),
    ((np.zeros((4, 2)), 1, None, None), TypeError, "Error tracking points: Int_out needs to be a boolean"),
    ((np.zeros((4, 2)), None, None, 'yes'), TypeError, "Error tracking points: S_exact_mode needs to be a boolean"),
    ((np.zeros((4, 2)), None, 'test', None), TypeError, "Error tracking points: Get_tracked needs to be a boolean"),
    (([[1.0, 2.0]], 1, 'test', None), TypeError, "Error tracking points: Get_tracked needs to be a boolean"),
]


@pytest.mark.parametrize('args,exc,msg', EXPECTED_MESSAGES)
def test_flow_track_and_batch_share_the_argument_checks(lib, args, exc, msg):
    """Flow.track, track_pts' checks and FlowBatch.track raise the same types and messages, before any device work."""
    from oflibnumpy_b200.flow import Flow
    from oflibnumpy_b200.validation import validate_track_args
    with pytest.raises(exc) as e:
        validate_track_args(*args)
    assert str(e.value) == msg
    with pytest.raises(exc) as e:
        Flow.__new__(Flow).track(*args)
    assert str(e.value) == msg
    if not (msg.endswith("shape N-2")):
        with pytest.raises(exc) as e:
            fake_batch().track(*args)
        assert str(e.value) == msg


def test_batch_checks_shape_and_dtype(lib):
    fb = fake_batch(n=3)
    for pts in (np.zeros((2, 4, 2)), np.zeros((3, 4, 3)), np.zeros(6), np.zeros((1, 3, 4, 2))):
        with pytest.raises(ValueError) as e:
            fb.track(pts)
        assert str(e.value) == "Error tracking points: Pts needs to have shape (3,P,2) or (P,2)"
    for ref in ('s', 't'):
        for dt in (bool, np.complex64, object):
            with pytest.raises(TypeError) as e:
                fake_batch(ref=ref).track(np.zeros((4, 2), dt))
            assert str(e.value) == "Error tracking points: Pts numpy array needs to have a float or int dtype"


def test_range_tests_and_lowest_frame(lib):
    from oflibnumpy_b200.batch import _raise_track_error, _track_range_fails
    h, w = 10, 20
    inside = np.array([[0, 0], [9, 19], [4.5, 7.25]])
    assert not _track_range_fails(inside, True, False, True, h, w)
    assert _track_range_fails(np.array([[9.01, 0]]), True, False, False, h, w)
    assert _track_range_fails(np.array([[np.nan, 0]]), True, False, False, h, w)
    assert not _track_range_fails(np.array([[-10, -20], [9, 19]]), True, True, True, h, w)
    assert _track_range_fails(np.array([[10, 0]]), True, True, False, h, w)
    assert _track_range_fails(np.array([[0, -21]], np.int16), True, True, False, h, w)
    assert not _track_range_fails(np.array([[50.0, -3.0]]), False, False, False, h, w)   # mesh route: no raise
    assert _track_range_fails(np.array([[9.5, 0]]), False, False, True, h, w)            # rounds to 10
    assert not _track_range_fails(np.array([[9.49, -20.5]]), False, False, True, h, w)   # 9, -20 (half to even)
    _raise_track_error(np.zeros(4, np.int32), h, w)
    with pytest.raises(IndexError, match="frame 2 index outside"):
        _raise_track_error(np.array([0, 0, 2, 1], np.int32), h, w)
    with pytest.raises(IndexError, match="^Some points are outside of the data area.$"):
        _raise_track_error(np.array([0, 5, 2, 1], np.int32), h, w)
    with pytest.raises(IndexError, match="frame 3 for the valid status"):
        _raise_track_error(np.array([0, 0, 0, 4], np.int32), h, w)


# ------------------------------------------------------------------------------------------------------------- GPU
def swirl(h, w, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[:h, :w].astype(np.float32)
    a, b = rng.uniform(0.3, 0.9, 2) * min(h, w) / 4
    v = np.stack([4 * np.sin(xx / a + seed) * np.cos(yy / b) + 0.002 * (xx - w / 2),
                  3 * np.cos(xx / b + 1) * np.sin(yy / a) - 0.003 * (yy - h / 2)], -1)
    return (v * scale).astype(np.float32)


def make_batch(of, h, w, n, ref, seed=0):
    """Swirls at several scales, a rotation about the centre, and one frame whose vectors all lie below the 1e-3
    threshold (frame 1); masks with ~2 % holes."""
    from oflibnumpy_b200.ops import from_transforms
    rng = np.random.default_rng(seed)
    frames = [swirl(h, w, 1), rng.uniform(-5e-4, 5e-4, (h, w, 2)).astype(np.float32),
              from_transforms([['rotation', w / 2, h / 2, 3.0]], (h, w), ref), swirl(h, w, 2, 0.2),
              swirl(h, w, 3, 2.5), swirl(h, w, 4, 0.7)]
    vecs = np.stack(frames[:n])
    masks = rng.random((n, h, w)) > 0.02
    return vecs, masks


def make_points(h, w, n, p, seed):
    """Float points inside [0,H-1]x[0,W-1], with the borders and corners; integer versions of them also reach the
    negative indices [-H,-1] / [-W,-1] that numpy wraps."""
    rng = np.random.default_rng(seed)
    edge = [[0, 0], [0, w - 1], [h - 1, 0], [h - 1, w - 1], [0, w / 3], [h - 1, w / 2], [h / 2, 0], [h / 3, w - 1],
            [h - 1.5, w - 1.5], [0.5, 0.5]]
    pts = np.concatenate([np.tile(np.array(edge, np.float64), (n, 1, 1)),
                          rng.uniform(0, 1, (n, p, 2)) * [h - 1, w - 1]], 1)
    ints = np.round(pts).astype(np.int64)
    neg = rng.random(ints.shape) < 0.2
    ints[neg] -= np.array([h, w])[np.nonzero(neg)[2]]
    return pts, ints


def as_dtype(fpts, ipts, dt):
    return (fpts if np.issubdtype(dt, np.floating) else ipts).astype(dt)


def expected_frame(of, vecs, ref, masks, i, pts_i, int_out, status, exact):
    return track_reference.track(of.Flow(vecs[i], ref, masks[i]), pts_i, int_out, status, exact)


def check_against_loop(of, vecs, masks, ref, fpts, ipts, zero_frames, shared_cases=(False, True)):
    from oflibnumpy_b200.batch import FlowBatch
    n = len(vecs)
    fb = FlowBatch(vecs, ref, masks)
    for dt in PT_DTYPES:
        for shared in shared_cases:
            pts = as_dtype(fpts, ipts, dt)
            if shared:
                pts = pts[0]
            for exact in (False, True):
                for int_out in (False, True):
                    for status in (False, True):
                        got = fb.track(pts, int_out, status, exact)
                        got_t, got_s = (got[0].numpy(), got[1].numpy()) if status else (got.numpy(), None)
                        wants = [expected_frame(of, vecs, ref, masks, i, pts if shared else pts[i], int_out, status,
                                                exact) for i in range(n)]
                        want_t = [wt[0] if status else wt for wt in wants]
                        odt = next(want_t[i].dtype for i in range(n) if i not in zero_frames)
                        assert got_t.dtype == odt, (ref, dt, shared, exact, int_out, status, got_t.dtype, odt)
                        for i in range(n):
                            wt = want_t[i].astype(odt) if i in zero_frames else want_t[i]
                            assert wt.dtype == odt
                            np.testing.assert_array_equal(got_t[i], wt, err_msg=str((ref, dt, shared, exact, int_out,
                                                                                      status, i)))
                            assert got_t[i].tobytes() == wt.tobytes()
                            if status:
                                assert got_s.dtype == np.uint8
                                np.testing.assert_array_equal(got_s[i].view(bool), wants[i][1])


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
def test_1080p_batch_matches_flow_track(of, ref):
    h, w, n = 1080, 1920, 6
    vecs, masks = make_batch(of, h, w, n, ref)
    fpts, ipts = make_points(h, w, n, 4096, 7)
    check_against_loop(of, vecs, masks, ref, fpts, ipts, zero_frames={1})


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
def test_odd_size_batch_matches_flow_track(of, ref):
    h, w, n = 37, 53, 5
    vecs, masks = make_batch(of, h, w, n, ref, seed=3)
    fpts, ipts = make_points(h, w, n, 300, 11)
    check_against_loop(of, vecs, masks, ref, fpts, ipts, zero_frames={1})


@pytest.mark.gpu
def test_next_rows_golden_in_a_batch(of):
    from oflibnumpy_b200.batch import FlowBatch
    g = load_golden('next_rows')
    vecs, masks = np.stack([g['in_flow']] * 3), np.stack([g['in_mask']] * 3)
    for r in ('s', 't'):
        fb, f = FlowBatch(vecs, r, masks), of.Flow(g['in_flow'], r, g['in_mask'])
        got = fb.track(g['in_pts_f']).numpy()
        got_st = fb.track(g['in_pts_f'], get_valid_status=True)[1].numpy().view(bool)
        got_int = fb.track(g['in_pts_f'], int_out=True).numpy()
        got_i = fb.track(g['in_pts_i']).numpy()
        for i in range(3):
            np.testing.assert_allclose(got[i], g['out_track_f_' + r], rtol=0, atol=1e-3 if r == 't' else 1e-9)
            np.testing.assert_array_equal(got_st[i], g['out_track_status_' + r])
            assert got_int.dtype == g['out_track_int_' + r].dtype
            assert np.abs(got_int[i] - g['out_track_int_' + r]).max() <= (1 if r == 't' else 0)
            np.testing.assert_allclose(got_i[i], g['out_track_ipts_' + r], rtol=0, atol=1e-3)
            assert got[i].tobytes() == track_reference.track(f, g['in_pts_f']).tobytes()
            np.testing.assert_array_equal(got_st[i], track_reference.track(f, g['in_pts_f'], get_valid_status=True)[1])
            assert got_int[i].tobytes() == track_reference.track(f, g['in_pts_f'], int_out=True).tobytes()
            assert got_i[i].tobytes() == track_reference.track(f, g['in_pts_i']).tobytes()
    fs = FlowBatch(np.stack([g['in_flow']] * 3), 's')
    got = fs.track(g['in_pts_f'], s_exact_mode=True).numpy()
    want = track_reference.track(of.Flow(g['in_flow'], 's'), g['in_pts_f'], s_exact_mode=True)
    for i in range(3):
        np.testing.assert_allclose(got[i], g['out_track_exact_s'], rtol=0, atol=1e-3)
        assert got[i].tobytes() == want.tobytes()


def check_flow_track(of, vecs, masks, ref, fpts, ipts):
    """Flow.track of every frame against track_reference, byte for byte, for every point dtype and option. A flow that
    is zero below the threshold hands back the points object itself (rounded with int_out); bool points are tracked as
    float64 on a 't' flow and refused on a non-zero 's' flow."""
    for i in range(len(vecs)):
        f = of.Flow(vecs[i], ref, masks[i])
        zero = R.is_zero_array(vecs[i])
        for dt in PT_DTYPES + (np.bool_,):
            pts = as_dtype(fpts, ipts, dt)[i]
            for exact, int_out, status in itertools.product((False, True), repeat=3):
                what = (ref, i, np.dtype(dt).name, exact, int_out, status)
                if ref == 's' and dt is np.bool_ and not zero:
                    for fn in (f.track, lambda *a: track_reference.track(f, *a)):
                        with pytest.raises(TypeError, match="needs to have a float or int dtype"):
                            fn(pts, int_out, status, exact)
                    continue
                got = f.track(pts, int_out, status, exact)
                want = track_reference.track(f, pts, int_out, status, exact)
                if status:
                    (got, got_s), (want, want_s) = got, want
                    assert got_s.dtype == want_s.dtype == np.bool_, what
                    np.testing.assert_array_equal(got_s, want_s, err_msg=str(what))
                assert (got is pts) == (want is pts) == (zero and not int_out), what
                assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, want.dtype)
                assert got.tobytes() == want.tobytes(), what


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
@pytest.mark.parametrize('size', [(1080, 1920, 6, 4096), (37, 53, 5, 300)], ids=['1080p', '37x53'])
def test_flow_track_matches_the_reference(of, ref, size):
    h, w, n, p = size
    vecs, masks = make_batch(of, h, w, n, ref, seed=h)
    fpts, ipts = make_points(h, w, n, p, 7)
    check_flow_track(of, vecs, masks, ref, fpts, ipts)


@pytest.mark.gpu
def test_device_points_give_the_bytes_of_host_points(of):
    import torch
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    h, w, n = 120, 160, 4
    for ref in ('s', 't'):
        vecs, masks = make_batch(of, h, w, n, ref, seed=5)
        fb = FlowBatch(vecs, ref, masks)
        fpts, ipts = make_points(h, w, n, 500, 13)
        for pts in (fpts, fpts.astype(np.float32), ipts, ipts.astype(np.int32), fpts[0], ipts[2]):
            for kw in ({}, {'int_out': True}, {'get_valid_status': True}, {'s_exact_mode': True}):
                want = fb.track(pts, **kw)
                for dpts in (DeviceArray.from_numpy(pts), torch.as_tensor(pts, device='cuda')):
                    got = fb.track(dpts, **kw)
                    for a, b in zip(got if isinstance(got, tuple) else (got,),
                                    want if isinstance(want, tuple) else (want,)):
                        assert a.dtype == b.dtype and a.shape == b.shape
                        assert a.numpy().tobytes() == b.numpy().tobytes()
        with pytest.raises(TypeError, match="device points need dtype"):
            fb.track(torch.zeros((5, 2), dtype=torch.int16, device='cuda'))


@pytest.mark.gpu
def test_no_points_and_one_frame(of):
    from oflibnumpy_b200.batch import FlowBatch
    h, w = 37, 53
    for ref in ('s', 't'):
        vecs, masks = make_batch(of, h, w, 3, ref, seed=2)
        fb = FlowBatch(vecs, ref, masks)
        for pts in (np.zeros((0, 2)), np.zeros((3, 0, 2), np.int16)):
            out, st = fb.track(pts, get_valid_status=True)
            assert out.shape == (3, 0, 2) and st.shape == (3, 0) and st.dtype == np.uint8
            assert out.dtype == (np.float32 if ref == 's' and pts.dtype == np.int16 else np.float64)
        fpts, ipts = make_points(h, w, 1, 200, 4)
        check_against_loop(of, vecs[:1], masks[:1], ref, fpts, ipts, zero_frames=set(), shared_cases=(False,))


@pytest.mark.gpu
def test_outside_points_raise_like_flow_track(of):
    from oflibnumpy_b200.batch import FlowBatch
    h, w, n = 37, 53, 5
    vecs, masks = make_batch(of, h, w, n, 's', seed=3)            # frame 1 is zero below the threshold
    fb = FlowBatch(vecs, 's', masks)
    fpts, ipts = make_points(h, w, n, 50, 1)
    bad = fpts.copy()
    bad[3, 7] = [-1.0, 3.0]
    with pytest.raises(IndexError) as e:
        fb.track(bad)
    assert str(e.value) == "Some points are outside of the data area."
    with pytest.raises(IndexError):
        fb[3].track(bad[3])
    in_zero = fpts.copy()
    in_zero[1, 7] = [-1.0, 3.0]
    got = fb.track(in_zero).numpy()
    np.testing.assert_array_equal(got[1], fb[1].track(in_zero[1]))
    np.testing.assert_array_equal(got[1], in_zero[1])
    # integer indices: -1 wraps, H raises
    wrap = ipts.copy()
    wrap[:, 0] = [-1, -1]
    got = fb.track(wrap).numpy()
    for i in (0, 2, 3, 4):
        assert got[i].tobytes() == fb[i].track(wrap[i]).tobytes()
    wrap[2, 0] = [h, 0]
    with pytest.raises(IndexError, match="frame 2"):
        fb.track(wrap)
    with pytest.raises(IndexError):
        fb[2].track(wrap[2])
    # status beyond the frame: both refs, host and device points
    for ref, kw in (('s', {'s_exact_mode': True}), ('t', {})):
        fr = FlowBatch(vecs, ref, masks)
        st = fpts.copy()
        st[0, 3] = [h - 0.4, 2.0]                                   # rounds to row H
        with pytest.raises(IndexError, match="frame 0 for the valid status"):
            fr.track(st, get_valid_status=True, **kw)
        with pytest.raises(IndexError):
            fr[0].track(st[0], get_valid_status=True, **kw)
        with pytest.raises(IndexError, match="frame 0 for the valid status"):
            fr.track(of.device.DeviceArray.from_numpy(st), get_valid_status=True, **kw)
        fr.track(st, **kw)                                           # no status: no raise
    # several bad frames: the lowest one is reported, whatever its kind of error
    many = ipts.copy()
    many[4, 0] = [0, w]
    many[2, 5] = [-h - 1, 0]
    many[3, 1] = [h + 5, 0]
    with pytest.raises(IndexError, match="frame 2 index"):
        fb.track(many)
    many_f = fpts.copy()
    many_f[4, 0] = [0, w + 0.5]
    many_f[2, 5] = [h, 0]
    with pytest.raises(IndexError) as e:
        fb.track(many_f)
    assert str(e.value) == "Some points are outside of the data area."
    with pytest.raises(IndexError, match="frame 2 for the valid status"):
        fb.track(many_f, get_valid_status=True, s_exact_mode=True)


@pytest.mark.gpu
def test_launch_count_does_not_grow_with_the_batch(of):
    from oflibnumpy_b200.batch import FlowBatch
    h, w = 60, 84
    vecs, masks = make_batch(of, h, w, 2, 's', seed=9)
    fpts, ipts = make_points(h, w, 1, 100, 2)

    def launches(fb, pts, **kw):
        fb.track(pts, **kw)                                          # warm-up
        before = of._lib.call('ofk_rt_launch_count')
        fb.track(pts, **kw)
        return of._lib.call('ofk_rt_launch_count') - before

    for ref, pts, kw in (('s', fpts[0], {}), ('s', ipts[0], {}), ('s', fpts[0], {'get_valid_status': True}),
                         ('s', fpts[0], {'s_exact_mode': True}), ('s', ipts[0], {'int_out': True}),
                         ('t', fpts[0], {}), ('t', ipts[0], {'int_out': True})):
        small = FlowBatch(vecs, ref, masks)
        big = FlowBatch(np.concatenate([vecs] * 32), ref, np.concatenate([masks] * 32))
        assert launches(small, pts, **kw) == launches(big, pts, **kw), (ref, kw)


@pytest.mark.gpu
def test_host_points_inside_the_frame_do_not_synchronise(of, monkeypatch):
    """Host points that pass the range tests: no download, no synchronisation, no read-back of the error words."""
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    h, w = 60, 84
    fpts, ipts = make_points(h, w, 3, 100, 2)
    vecs, masks = make_batch(of, h, w, 3, 's', seed=4)
    batches = {r: FlowBatch(vecs, r, masks) for r in ('s', 't')}
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
    for pts in (fpts, ipts, fpts[0], ipts.astype(np.int16)):
        results.append(batches['s'].track(pts, int_out=True, get_valid_status=True))
        results.append(batches['s'].track(pts, s_exact_mode=True))
        results.append(batches['t'].track(pts))
    monkeypatch.undo()
    assert len(results) == 12
