"""Accumulation of clips of flows to their keyframe: FlowBatch.accumulate (ofk_accumulate). Every result frame must equal,
vectors and mask byte for byte, the loop of Flow.combine_with(., 3, thresholded) it replaces: ref 's' the left fold
``acc = F[0]; acc = acc.combine_with(F[k], 3)``, ref 't' the right fold ``acc = F[L-1]; acc = F[j].combine_with(acc,
3)``, with the early exits at every step, including a composed state that is zero by cancellation."""
import numpy as np
import pytest

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


def oracle_fold(frames, ref, thresholded):
    """The fold as a loop over oracle.flowref.combine: one result per input frame, in the input's order."""
    out = [None] * len(frames)
    if ref == 's':
        acc = out[0] = frames[0]
        for k in range(1, len(frames)):
            acc = out[k] = R.combine(acc, frames[k], 3, thresholded)
    else:
        acc = out[-1] = frames[-1]
        for j in range(len(frames) - 2, -1, -1):
            acc = out[j] = R.combine(frames[j], acc, 3, thresholded)
    return out


def translation(h, w, u, v):
    return np.broadcast_to(np.array([u, v], np.float32), (h, w, 2)).copy()


# ------------------------------------------------------------------------------------------------------------- CPU
def test_bad_arguments_are_rejected_without_a_gpu(lib):
    """ofk_accumulate checks every argument before a stream or the device is touched."""
    good = dict(flow=16, mask=16, ref=ord('s'), thr=0.0, S=2, L=3, H=4, W=4, cum=1, out=16, out_mask=16, ws=16,
                ws_bytes=1 << 20, stream=None)
    for change, msg in (({'flow': None}, "NULL pointer"), ({'mask': None}, "NULL pointer"),
                        ({'out': None}, "NULL pointer"), ({'out_mask': None}, "NULL pointer"),
                        ({'ws': None}, "NULL pointer"), ({'ref': ord('x')}, "ref must be 's' or 't'"),
                        ({'thr': -1.0}, "thr must be >= 0"), ({'thr': float('nan')}, "thr must be >= 0"),
                        ({'S': -1}, "bad shape"), ({'L': 0}, "bad shape"), ({'H': 0}, "bad shape"),
                        ({'W': -2}, "bad shape"), ({'W': 32768}, "bad shape"), ({'H': 40000}, "bad shape"),
                        ({'S': 256, 'L': 256}, "exceeds 65535 frames"), ({'S': 1 << 30, 'L': 1 << 30}, "exceeds"),
                        ({'flow': 20}, "8-byte aligned"), ({'out': 12}, "8-byte aligned"),
                        ({'ws': 18}, "ws must be 4-byte aligned"), ({'ws_bytes': 511}, "workspace too small")):
        args = dict(good, **change)
        with pytest.raises(lib.OflibCudaError, match="ofk_accumulate: .*" + msg):
            lib.call('ofk_accumulate', *args.values())


def test_workspace_size(lib):
    ws = lambda s, l: lib.call('ofk_accumulate_workspace', s, l)
    assert ws(2, 3) == 512                      # two int32 flag arrays of S*L, each rounded up to 256 bytes
    assert ws(16, 40) == 2 * 2560
    assert ws(1, 65535) == 2 * 262144
    assert ws(0, 5) == 0
    assert ws(-1, 5) == 0 and ws(2, 0) == 0 and ws(2, 65535) == 0


@pytest.mark.parametrize('args,exc,msg', [
    ((None, 1, False, 4), TypeError, "Error accumulating flows: Cumulative needs to be a boolean"),
    ((None, True, None, 4), TypeError, "Error accumulating flows: Thresholded needs to be a boolean"),
    ((3, True, False, 4), ValueError, "Error accumulating flows: Clip_length needs to be a positive integer that "
                                      "divides the batch size 4, not 3"),
    ((0, True, False, 4), ValueError, "Error accumulating flows: Clip_length needs to be a positive integer that "
                                      "divides the batch size 4, not 0"),
    ((2.0, True, False, 4), ValueError, "Error accumulating flows: Clip_length needs to be a positive integer that "
                                        "divides the batch size 4, not 2.0"),
    ((True, True, False, 4), ValueError, "Error accumulating flows: Clip_length needs to be a positive integer that "
                                         "divides the batch size 4, not True"),
])
def test_argument_messages(lib, args, exc, msg):
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    from oflibnumpy_b200.validation import validate_accumulate_args
    with pytest.raises(exc) as e:
        validate_accumulate_args(*args)
    assert str(e.value) == msg
    fake = FlowBatch._wrap(DeviceArray(0, (4, 3, 5, 2), np.float32), 's', DeviceArray(0, (4, 3, 5), np.uint8))
    with pytest.raises(exc) as e:
        fake.accumulate(args[0], args[1], args[2])
    assert str(e.value) == msg


def test_argument_defaults(lib):
    from oflibnumpy_b200.validation import validate_accumulate_args
    assert validate_accumulate_args(None, True, False, 12) == 12
    assert validate_accumulate_args(4, False, True, 12) == 4
    assert validate_accumulate_args(np.int64(3), True, False, 12) == 3
    assert validate_accumulate_args(None, True, False, 0) == 1
    assert validate_accumulate_args(5, True, False, 0) == 5


def test_oracle_fold_takes_the_exits():
    """The test's own fold reproduces both exits and the restart after a cancelled state (returned objects)."""
    h, w = 10, 12
    rng = np.random.default_rng(0)
    zero = R.make(np.zeros((h, w, 2), np.float32), 's')
    a = R.make(rng.uniform(-2, 2, (h, w, 2)).astype(np.float32), 's')
    b = R.make(rng.uniform(-2, 2, (h, w, 2)).astype(np.float32), 's')
    out = oracle_fold([zero, a, zero, b], 's', False)
    assert out[0] is zero and out[1] is a and out[2] is a          # restart from a, then pass-through of the zero
    np.testing.assert_array_equal(out[3].vecs, R.combine(a, b, 3).vecs)
    # +(3,2) then -(3,2): the composite is zero on its valid pixels (pixels that sampled outside lose their mask)
    mask = rng.random((h, w)) > 0.1
    fwd = R.make(translation(h, w, 3, 2), 's', mask)
    fwd.vecs[~mask] = 7                                            # non-zero vectors on invalid pixels
    back = R.make(translation(h, w, -3, -2), 's')
    out = oracle_fold([fwd, back, b, a], 's', False)
    assert R.is_zero(out[1], thresholded=False) and not out[1].mask.all()
    assert out[2] is b                                             # restart after the cancelled state
    np.testing.assert_array_equal(out[3].vecs, R.combine(b, a, 3).vecs)
    # 't' walks backwards: D_3 = a, B_2 zero -> pass, then B_1 = fwd composes, B_0 = zero passes
    out = oracle_fold([zero, fwd, zero, a], 't', False)
    assert out[3] is a and out[2] is a and out[0] is out[1]
    np.testing.assert_array_equal(out[1].vecs, R.combine(fwd, a, 3).vecs)
    # a cancellation that exists only below the threshold
    near = R.make(translation(h, w, -3 + 4e-4, -2), 's')
    assert not R.is_zero(oracle_fold([fwd, near], 's', False)[1], thresholded=False)
    assert oracle_fold([fwd, near, b], 's', True)[2] is b


# ------------------------------------------------------------------------------------------------------------- GPU
def swirl(h, w, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[:h, :w].astype(np.float32)
    a, b = rng.uniform(0.3, 0.9, 2) * min(h, w) / 4
    v = np.stack([4 * np.sin(xx / a + seed) * np.cos(yy / b) + 0.002 * (xx - w / 2),
                  3 * np.cos(xx / b + 1) * np.sin(yy / a) - 0.003 * (yy - h / 2)], -1)
    return (v * scale).astype(np.float32)


def make_clips(h, w, s, ref, seed=0):
    """S clips of 6 frames: swirls at several scales, a rotation about the centre, motion that leaves the frame and a
    frame below the 1e-3 threshold (zero only when thresholded); masks with ~2 % holes."""
    from oflibnumpy_b200.ops import from_transforms
    rng = np.random.default_rng(seed)
    frames = []
    for c in range(s):
        clip = [swirl(h, w, 1 + c), from_transforms([['rotation', w / 2, h / 2, 3.0 + c]], (h, w), ref),
                swirl(h, w, 2 + c, 0.2), translation(h, w, w / 9 + c, -h / 7),
                rng.uniform(-5e-4, 5e-4, (h, w, 2)).astype(np.float32), swirl(h, w, 4 + c, 2.5)]
        frames += clip[c % 2:] + clip[:c % 2]                  # the clips differ in order too
    vecs = np.stack(frames).astype(np.float32)
    masks = rng.random(vecs.shape[:3]) > 0.02
    return vecs, masks


def loop_fold(of, vecs, masks, ref, clip, thresholded):
    """The combine_with loop per clip, results in the cumulative layout (numpy vecs, bool masks)."""
    fb = of.FlowBatch(vecs, ref, masks)
    ov, om = np.empty_like(vecs), np.empty(vecs.shape[:3], bool)
    for s in range(len(vecs) // clip):
        f = [fb[s * clip + k] for k in range(clip)]
        order = range(clip) if ref == 's' else range(clip - 1, -1, -1)
        acc = None
        for k in order:
            if acc is None:
                acc = f[k]
            elif ref == 's':
                acc = acc.combine_with(f[k], 3, thresholded)
            else:
                acc = f[k].combine_with(acc, 3, thresholded)
            ov[s * clip + k], om[s * clip + k] = acc.vecs, acc.mask
    return ov, om


def pick_final(arr, clip, ref):
    return arr[clip - 1::clip] if ref == 's' else arr[0::clip]


def check(of, vecs, masks, ref, clip, thresholded, cumulative, want=None):
    got = of.FlowBatch(vecs, ref, masks).accumulate(clip, cumulative, thresholded)
    gv, gm = got.numpy()
    assert got.ref == ref
    wv, wm = loop_fold(of, vecs, masks, ref, clip, thresholded) if want is None else want
    if not cumulative:
        wv, wm = pick_final(wv, clip, ref), pick_final(wm, clip, ref)
    assert gv.shape == wv.shape and gm.shape == wm.shape
    for i in range(len(wv)):
        tag = (ref, clip, thresholded, cumulative, i)
        np.testing.assert_array_equal(gm[i], wm[i], err_msg=str(tag))
        np.testing.assert_array_equal(gv[i], wv[i], err_msg=str(tag))
        assert gv[i].tobytes() == wv[i].tobytes(), tag
    return gv, gm


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
def test_1080p_matches_the_combine_with_loop(of, ref):
    h, w = 1080, 1920
    vecs, masks = make_clips(h, w, 2, ref)
    for thresholded in (False, True):
        want = loop_fold(of, vecs, masks, ref, 6, thresholded)
        for cumulative in (True, False):
            check(of, vecs, masks, ref, 6, thresholded, cumulative, want)


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
def test_small_frames_match_the_loop_and_the_oracle(of, ref):
    """37 x 53: the loop takes the non-TMA composition kernels; the oracle fold agrees value for value."""
    h, w = 37, 53
    vecs, masks = make_clips(h, w, 2, ref, seed=1)
    for thresholded in (False, True):
        for cumulative in (True, False):
            gv, gm = check(of, vecs, masks, ref, 6, thresholded, cumulative)
            want = []
            for s in range(2):
                want += oracle_fold([R.make(vecs[s * 6 + k], ref, masks[s * 6 + k]) for k in range(6)], ref,
                                    thresholded)
            if not cumulative:
                want = want[5::6] if ref == 's' else want[0::6]
            for i, f in enumerate(want):
                np.testing.assert_array_equal(gm[i], f.mask)
                np.testing.assert_array_equal(gv[i], f.vecs)


def exit_clips(h, w, rng):
    """Clips that exercise the exits: zero inputs at the start, in the middle and at the end, an all-zero clip,
    alternating translations +-(3, 2) that cancel several times, one cancellation that exists only at the threshold.
    Invalid pixels carry large non-zero vectors, so that a missed exit shows in the vectors."""
    z = np.zeros((h, w, 2), np.float32)
    fwd, back = translation(h, w, 3, 2), translation(h, w, -3, -2)
    near = translation(h, w, -3 + 4e-4, -2)
    sw = [swirl(h, w, 10 + i) for i in range(4)]
    clips = [[z, sw[0], sw[1], sw[2], sw[3], sw[0]],             # zero at the start
             [sw[0], z, sw[1], z, sw[2], z],                      # zero in the middle and at the end
             [z] * 6,                                             # all zero
             [fwd, back] * 3,                                     # cancels twice before the last step, both refs
             [z, fwd, back, sw[1], sw[2], sw[0]],                 # 's': restart, then a cancellation in the middle
             [fwd, near, sw[2], sw[0], sw[1], sw[3]],             # 's': cancels only when thresholded
             [sw[1], sw[2], sw[3], sw[0], fwd, near],             # 't': cancels only when thresholded
             [back, fwd] * 3]
    vecs = np.stack([f for c in clips for f in c]).astype(np.float32)
    masks = rng.random(vecs.shape[:3]) > 0.05
    masks[12:18] = True                                  # the all-zero clip: valid everywhere
    noise = rng.uniform(5, 9, vecs.shape).astype(np.float32)
    vecs[~masks] = noise[~masks]
    return vecs, masks


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
def test_exits_and_cancellation(of, ref):
    h, w = 48, 64
    vecs, masks = exit_clips(h, w, np.random.default_rng(2))
    for thresholded in (False, True):
        for cumulative in (True, False):
            check(of, vecs, masks, ref, 6, thresholded, cumulative)
    # the cancellations really happen: the loop restarts from the next input
    fb = of.FlowBatch(vecs, ref, masks)
    assert fb[18].combine_with(fb[19], 3).is_zero(thresholded=False)
    assert fb[22].combine_with(fb[23], 3).is_zero(thresholded=False)
    near = fb[30].combine_with(fb[31], 3) if ref == 's' else fb[40].combine_with(fb[41], 3)
    assert near.is_zero(thresholded=True) and not near.is_zero(thresholded=False)


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
def test_one_clip_needs_the_repair(of, ref):
    """Only the middle clip of three cancels; the others take the walk alone. 1080p, so the walk's interior path and
    the repair's frame passes both run at full size."""
    h, w = 1080, 1920
    rng = np.random.default_rng(5)
    sw = [swirl(h, w, 20 + i) for i in range(5)]
    fwd, back = translation(h, w, 3, 2), translation(h, w, -3, -2)
    vecs = np.stack([sw[0], sw[1], sw[2], sw[3], fwd, back, fwd, sw[4], sw[3], sw[2], sw[1], sw[0]])
    masks = rng.random(vecs.shape[:3]) > 0.02
    vecs[~masks] = 6.5
    for cumulative in (True, False):
        check(of, vecs, masks, ref, 4, False, cumulative)


@pytest.mark.gpu
def test_clips_equal_each_clip_alone(of):
    h, w = 64, 96
    vecs, masks = make_clips(h, w, 4, 's', seed=3)
    for ref in ('s', 't'):
        for cumulative in (True, False):
            whole = of.FlowBatch(vecs, ref, masks).accumulate(6, cumulative)
            wv, wm = whole.numpy()
            per = 6 if cumulative else 1
            for s in range(4):
                one = of.FlowBatch(vecs[s * 6:(s + 1) * 6], ref, masks[s * 6:(s + 1) * 6]).accumulate(
                    None, cumulative)
                ov, om = one.numpy()
                assert wv[s * per:(s + 1) * per].tobytes() == ov.tobytes()
                assert np.array_equal(wm[s * per:(s + 1) * per], om)


@pytest.mark.gpu
def test_length_one_and_empty_batches(of):
    h, w = 20, 30
    vecs, masks = make_clips(h, w, 1, 't', seed=4)
    for ref in ('s', 't'):
        fb = of.FlowBatch(vecs, ref, masks)
        for cumulative in (True, False):
            res = fb.accumulate(1, cumulative)
            v, m = res.numpy()
            assert v.tobytes() == vecs.tobytes() and np.array_equal(m, masks)
            assert res.vecs.ptr != fb.vecs.ptr and res.masks.ptr != fb.masks.ptr      # copies, not aliases
        empty = of.FlowBatch(np.zeros((0, h, w, 2), np.float32), ref).accumulate()
        assert len(empty) == 0 and empty.shape == (h, w) and empty.ref == ref
        assert len(of.FlowBatch(np.zeros((0, h, w, 2), np.float32), ref).accumulate(3, False)) == 0


@pytest.mark.gpu
def test_final_only_equals_the_last_step(of):
    h, w = 50, 70
    vecs, masks = make_clips(h, w, 3, 's', seed=6)
    for ref in ('s', 't'):
        for thresholded in (False, True):
            fb = of.FlowBatch(vecs, ref, masks)
            cv, cm = fb.accumulate(6, True, thresholded).numpy()
            fv, fm = fb.accumulate(6, False, thresholded).numpy()
            assert fv.tobytes() == pick_final(cv, 6, ref).tobytes()
            assert np.array_equal(fm, pick_final(cm, 6, ref))


@pytest.mark.gpu
def test_batches_beyond_4_gib(of):
    """260 x 1080p flows (4.3 GB of vectors): the last clip lies beyond 2^32 bytes and must equal the same clip alone."""
    from oflibnumpy_b200 import _lib, _ops
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    h, w, s, clip = 1080, 1920, 4, 65
    n = s * clip
    rng = np.random.default_rng(7)
    mats = np.stack([R.matrix_from_transforms([['rotation', w / 2, h / 2, rng.uniform(-2, 2)],
                                               ['translation', rng.uniform(-3, 3), rng.uniform(-3, 3)]])
                     for _ in range(n)])
    v = _ops.from_matrix(DeviceArray.from_numpy(mats), (h, w), 1.0)
    m = DeviceArray.empty((n, h, w), np.uint8)
    _lib.call('ofk_rt_memset', m.ptr, 1, m.nbytes, of.device.current_stream())
    assert v.nbytes > (1 << 32)
    fb = FlowBatch._wrap(v, 's', m)
    last = FlowBatch._wrap(v.frames(n - clip, n), 's', m.frames(n - clip, n))
    for ref in ('s', 't'):
        fb.ref = last.ref = ref
        fin = fb.accumulate(clip, False)
        alone = last.accumulate(None, False)
        assert fin.vecs.frames(s - 1, s).numpy().tobytes() == alone.vecs.numpy().tobytes()
        assert np.array_equal(fin.masks.frames(s - 1, s).numpy(), alone.masks.numpy())
        del fin
        cum = fb.accumulate(clip, True)
        alone = last.accumulate(None, True)
        for k in (0, clip // 2, clip - 1):
            i = n - clip + k
            assert cum.vecs.frames(i, i + 1).numpy().tobytes() == alone.vecs.frames(k, k + 1).numpy().tobytes()
            assert np.array_equal(cum.masks.frames(i, i + 1).numpy(), alone.masks.frames(k, k + 1).numpy())
        del cum


@pytest.mark.gpu
def test_launch_count_does_not_depend_on_the_shape_of_the_batch(of):
    from oflibnumpy_b200 import _lib
    h, w = 20, 24
    rng = np.random.default_rng(8)

    def launches(s, clip, ref, cumulative):
        vecs = rng.uniform(-2, 2, (s * clip, h, w, 2)).astype(np.float32)
        fb = of.FlowBatch(vecs, ref, rng.random((s * clip, h, w)) > 0.1)
        fb.accumulate(clip, cumulative)                                  # warm-up
        before = _lib.call('ofk_rt_launch_count')
        fb.accumulate(clip, cumulative)
        return _lib.call('ofk_rt_launch_count') - before

    for ref in ('s', 't'):
        for cumulative in (True, False):
            assert launches(2, 3, ref, cumulative) == launches(16, 40, ref, cumulative), (ref, cumulative)


@pytest.mark.gpu
def test_no_read_back_or_synchronisation(of, monkeypatch):
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.device import DeviceArray
    h, w = 40, 56
    vecs, masks = exit_clips(h, w, np.random.default_rng(9))          # includes clips that need the repair
    batches = {r: of.FlowBatch(vecs, r, masks) for r in ('s', 't')}
    of.device.set_stream(None)
    real_call = _lib.call

    def no_sync(name, *args):
        assert name not in ('ofk_rt_memcpy_d2h', 'ofk_rt_stream_sync', 'ofk_rt_device_sync', 'ofk_rt_event_sync'), name
        return real_call(name, *args)

    def no_numpy(self, out=None):
        raise AssertionError("DeviceArray.numpy called")

    results = []
    monkeypatch.setattr(_lib, 'call', no_sync)
    monkeypatch.setattr(DeviceArray, 'numpy', no_numpy)
    for r in ('s', 't'):
        for cumulative in (True, False):
            results.append(batches[r].accumulate(6, cumulative, True))
    monkeypatch.undo()
    assert len(results) == 4
    want = loop_fold(of, vecs, masks, 't', 6, True)
    assert results[3].vecs.numpy().tobytes() == pick_final(want[0], 6, 't').tobytes()
