"""FlowBatch.accumulate(fold=) / ofk_accumulate_fold: either fold for either ref. Every result frame must equal, vectors
and mask byte for byte, the loop of Flow.combine_with(., 3, thresholded) of its fold: 'left' ``acc = F[0]; acc =
acc.combine_with(F[k], 3)``, 'right' ``acc = F[L-1]; acc = F[j].combine_with(acc, 3)``, with the early exits at every
step, including a composed state that is zero by cancellation. ('t', 'left') and ('s', 'right') are the combinations
that sample the running composite and run one launch per step; the walked ones are tested in test_accumulate_batch."""
import numpy as np
import pytest

from oracle import flowref as R
from test_accumulate_batch import exit_clips, lib, make_clips, of, pick_final, swirl, translation  # noqa: F401

SAMPLED = [('t', 'left'), ('s', 'right')]


def oracle_fold(frames, thresholded, fold):
    """The fold as a loop over oracle.flowref.combine: one result per input frame, in the input's order."""
    out = [None] * len(frames)
    if fold == 'left':
        acc = out[0] = frames[0]
        for k in range(1, len(frames)):
            acc = out[k] = R.combine(acc, frames[k], 3, thresholded)
    else:
        acc = out[-1] = frames[-1]
        for j in range(len(frames) - 2, -1, -1):
            acc = out[j] = R.combine(frames[j], acc, 3, thresholded)
    return out


def final_of(arr, clip, fold):
    return pick_final(arr, clip, 's' if fold == 'left' else 't')


# ------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('ref,fold', [('s', ord('l')), ('s', ord('r')), ('t', ord('l')), ('t', ord('r'))])
def test_bad_arguments_are_rejected_without_a_gpu(lib, ref, fold):
    """ofk_accumulate_fold checks every argument before a stream or the device is touched."""
    sampled = (ref == 't') == (fold == ord('l'))
    good = dict(flow=16, mask=16, ref=ord(ref), fold=fold, thr=0.0, S=2, L=3, H=4, W=4, cum=0, out=16, out_mask=16,
                ws=16, ws_bytes=1 << 20, stream=None)
    for change, msg in (({'flow': None}, "NULL pointer"), ({'mask': None}, "NULL pointer"),
                        ({'out': None}, "NULL pointer"), ({'out_mask': None}, "NULL pointer"),
                        ({'ws': None}, "NULL pointer"), ({'ref': ord('x')}, "ref must be 's' or 't'"),
                        ({'fold': ord('x')}, "fold must be 'l' or 'r'"), ({'fold': 0}, "fold must be 'l' or 'r'"),
                        ({'thr': -1.0}, "thr must be >= 0"), ({'thr': float('nan')}, "thr must be >= 0"),
                        ({'S': -1}, "bad shape"), ({'L': 0}, "bad shape"), ({'H': 0}, "bad shape"),
                        ({'W': -2}, "bad shape"), ({'W': 32768}, "bad shape"), ({'H': 40000}, "bad shape"),
                        ({'S': 256, 'L': 256}, "exceeds 65535 frames"), ({'S': 1 << 30, 'L': 1 << 30}, "exceeds"),
                        ({'flow': 20}, "8-byte aligned"), ({'out': 12}, "8-byte aligned"),
                        ({'ws': 18}, "ws must be [48]-byte aligned"),
                        ({'ws_bytes': 1023 if sampled else 511}, "workspace too small")):
        args = dict(good, **change)
        with pytest.raises(lib.OflibCudaError, match="ofk_accumulate_fold: .*" + msg):
            lib.call('ofk_accumulate_fold', *args.values())
    if sampled:      # the frame buffer of the sampled folds needs 8-byte alignment
        with pytest.raises(lib.OflibCudaError, match="ws must be 8-byte aligned"):
            lib.call('ofk_accumulate_fold', *dict(good, ws=20).values())


def test_workspace_size(lib):
    ws = lambda ref, fold, s, l, h, w, cum: lib.call('ofk_accumulate_fold_workspace', ord(ref), ord(fold), s, l, h,
                                                     w, cum)
    for s, l in ((2, 3), (16, 40), (1, 65535), (0, 5)):
        for h, w, cum in ((4, 4, 0), (1080, 1920, 1), (1080, 1920, 0)):
            # the walked folds: ofk_accumulate's two int32 flag arrays of S*L, whatever the frame size
            assert ws('s', 'l', s, l, h, w, cum) == ws('t', 'r', s, l, h, w, cum) == \
                lib.call('ofk_accumulate_workspace', s, l)
            if cum:
                assert ws('t', 'l', s, l, h, w, cum) == ws('s', 'r', s, l, h, w, cum) == \
                    lib.call('ofk_accumulate_workspace', s, l)
    # the sampled folds, final-only: the flags plus one S-frame buffer (vectors, then mask), each rounded up to 256
    assert ws('t', 'l', 2, 3, 4, 4, 0) == ws('s', 'r', 2, 3, 4, 4, 0) == 512 + 256 + 256
    assert ws('t', 'l', 32, 8, 1080, 1920, 0) == 2 * 1024 + 32 * 1080 * 1920 * 9
    assert ws('s', 'r', 3, 5, 37, 53, 0) == 2 * 256 + 47104 + 5888       # 3*37*53 = 5883 px
    assert ws('t', 'l', 0, 5, 37, 53, 0) == 0
    for bad in (('x', 'l', 2, 3, 4, 4, 0), ('s', 'x', 2, 3, 4, 4, 0), ('t', 'l', -1, 3, 4, 4, 0),
                ('t', 'l', 2, 0, 4, 4, 0), ('s', 'r', 2, 65535, 4, 4, 1), ('t', 'l', 2, 3, 0, 4, 0),
                ('s', 'r', 2, 3, 4, 32768, 0), ('s', 'l', 2, 3, 32768, 4, 1)):
        assert ws(*bad) == 0, bad


@pytest.mark.parametrize('fold', ['up', 'Left', 'l', '', 1, True, b'left', ['left']])
def test_fold_messages(lib, fold):
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    from oflibnumpy_b200.validation import validate_accumulate_args
    msg = "Error accumulating flows: Fold needs to be 'left' or 'right', not {!r}".format(fold)
    with pytest.raises(ValueError) as e:
        validate_accumulate_args(None, True, False, 4, fold=fold)
    assert str(e.value) == msg
    for ref in ('s', 't'):
        fake = FlowBatch._wrap(DeviceArray(0, (4, 3, 5, 2), np.float32), ref, DeviceArray(0, (4, 3, 5), np.uint8))
        with pytest.raises(ValueError) as e:
            fake.accumulate(2, fold=fold)
        assert str(e.value) == msg


def test_fold_defaults(lib):
    from oflibnumpy_b200.validation import validate_accumulate_args
    for fold in (None, 'left', 'right'):
        assert validate_accumulate_args(None, True, False, 12, fold=fold) == 12
        assert validate_accumulate_args(4, False, True, 12, fold=fold) == 4


@pytest.mark.parametrize('ref', ['s', 't'])
def test_oracle_fold_takes_the_exits(ref):
    """The test's own fold reproduces both exits and the restart after a cancelled state, for either fold (returned
    objects)."""
    h, w = 10, 12
    rng = np.random.default_rng(0)
    zero = R.make(np.zeros((h, w, 2), np.float32), ref)
    a = R.make(rng.uniform(-2, 2, (h, w, 2)).astype(np.float32), ref)
    b = R.make(rng.uniform(-2, 2, (h, w, 2)).astype(np.float32), ref)
    # left fold: state zero -> restart, else input zero -> pass
    out = oracle_fold([zero, a, zero, b], False, 'left')
    assert out[0] is zero and out[1] is a and out[2] is a
    np.testing.assert_array_equal(out[3].vecs, R.combine(a, b, 3).vecs)
    # right fold: input zero -> pass, else state zero -> restart
    out = oracle_fold([b, zero, a, zero], False, 'right')
    assert out[3] is zero and out[2] is a and out[1] is a
    np.testing.assert_array_equal(out[0].vecs, R.combine(b, a, 3).vecs)
    # +(3,2) then -(3,2): zero on its valid pixels (pixels that sampled outside lose their mask)
    mask = rng.random((h, w)) > 0.1
    fwd = R.make(translation(h, w, 3, 2), ref, mask)
    fwd.vecs[~mask] = 7                                            # non-zero vectors on invalid pixels
    back = R.make(translation(h, w, -3, -2), ref)
    out = oracle_fold([fwd, back, b, a], False, 'left')
    assert R.is_zero(out[1], thresholded=False) and not out[1].mask.all()
    assert out[2] is b                                             # restart after the cancelled state
    np.testing.assert_array_equal(out[3].vecs, R.combine(b, a, 3).vecs)
    out = oracle_fold([a, b, fwd, back], False, 'right')
    assert out[3] is back and R.is_zero(out[2], thresholded=False) and not out[2].mask.all()
    assert out[1] is b                                             # restart after the cancelled state
    np.testing.assert_array_equal(out[0].vecs, R.combine(a, b, 3).vecs)
    # a cancellation that exists only below the threshold
    near = R.make(translation(h, w, -3 + 4e-4, -2), ref)
    assert not R.is_zero(oracle_fold([fwd, near], False, 'left')[1], thresholded=False)
    assert oracle_fold([fwd, near, b], True, 'left')[2] is b
    assert not R.is_zero(oracle_fold([fwd, near], False, 'right')[0], thresholded=False)
    assert oracle_fold([b, fwd, near], True, 'right')[0] is b


# ------------------------------------------------------------------------------------------------------------- GPU
def loop_fold(of, vecs, masks, ref, clip, thresholded, fold):
    """The combine_with loop of the fold per clip, results in the cumulative layout (numpy vecs, bool masks)."""
    fb = of.FlowBatch(vecs, ref, masks)
    ov, om = np.empty_like(vecs), np.empty(vecs.shape[:3], bool)
    for s in range(len(vecs) // clip):
        f = [fb[s * clip + k] for k in range(clip)]
        order = range(clip) if fold == 'left' else range(clip - 1, -1, -1)
        acc = None
        for k in order:
            if acc is None:
                acc = f[k]
            elif fold == 'left':
                acc = acc.combine_with(f[k], 3, thresholded)
            else:
                acc = f[k].combine_with(acc, 3, thresholded)
            ov[s * clip + k], om[s * clip + k] = acc.vecs, acc.mask
    return ov, om


def check(of, vecs, masks, ref, fold, clip, thresholded, cumulative, want=None):
    got = of.FlowBatch(vecs, ref, masks).accumulate(clip, cumulative, thresholded, fold=fold)
    gv, gm = got.numpy()
    assert got.ref == ref
    wv, wm = loop_fold(of, vecs, masks, ref, clip, thresholded, fold) if want is None else want
    if not cumulative:
        wv, wm = final_of(wv, clip, fold), final_of(wm, clip, fold)
    assert gv.shape == wv.shape and gm.shape == wm.shape
    for i in range(len(wv)):
        tag = (ref, fold, clip, thresholded, cumulative, i)
        np.testing.assert_array_equal(gm[i], wm[i], err_msg=str(tag))
        assert gv[i].tobytes() == wv[i].tobytes(), tag
    return gv, gm


@pytest.mark.gpu
@pytest.mark.parametrize('ref,fold', SAMPLED)
def test_1080p_matches_the_combine_with_loop(of, ref, fold):
    h, w = 1080, 1920
    vecs, masks = make_clips(h, w, 2, ref)
    for thresholded in (False, True):
        want = loop_fold(of, vecs, masks, ref, 6, thresholded, fold)
        for cumulative in (True, False):
            check(of, vecs, masks, ref, fold, 6, thresholded, cumulative, want)


@pytest.mark.gpu
@pytest.mark.parametrize('ref,fold', SAMPLED)
def test_small_frames_match_the_loop_and_the_oracle(of, ref, fold):
    """37 x 53: the loop takes the non-TMA composition kernels; the oracle fold agrees value for value."""
    h, w = 37, 53
    vecs, masks = make_clips(h, w, 2, ref, seed=1)
    for thresholded in (False, True):
        for cumulative in (True, False):
            gv, gm = check(of, vecs, masks, ref, fold, 6, thresholded, cumulative)
            want = []
            for s in range(2):
                want += oracle_fold([R.make(vecs[s * 6 + k], ref, masks[s * 6 + k]) for k in range(6)], thresholded,
                                    fold)
            if not cumulative:
                want = final_of(want, 6, fold)
            for i, f in enumerate(want):
                np.testing.assert_array_equal(gm[i], f.mask)
                np.testing.assert_array_equal(gv[i], f.vecs)


def fold_exit_clips(h, w, rng):
    """exit_clips plus two clips with a cancellation that exists only at the threshold in the middle of the clip, after
    a restart: [fwd, near] met by the right fold after a zero tail, and by the left fold after a zero head."""
    vecs, masks = exit_clips(h, w, rng)
    z = np.zeros((h, w, 2), np.float32)
    fwd, near = translation(h, w, 3, 2), translation(h, w, -3 + 4e-4, -2)
    extra = np.stack([swirl(h, w, 30), swirl(h, w, 31), fwd, near, z, z,
                      z, z, fwd, near, swirl(h, w, 32), swirl(h, w, 33)]).astype(np.float32)
    emask = rng.random(extra.shape[:3]) > 0.05
    extra[~emask] = rng.uniform(5, 9, extra.shape).astype(np.float32)[~emask]
    return np.concatenate([vecs, extra]), np.concatenate([masks, emask])


@pytest.mark.gpu
@pytest.mark.parametrize('ref,fold', SAMPLED)
def test_exits_and_cancellation(of, ref, fold):
    h, w = 48, 64
    vecs, masks = fold_exit_clips(h, w, np.random.default_rng(2))
    for thresholded in (False, True):
        for cumulative in (True, False):
            check(of, vecs, masks, ref, fold, 6, thresholded, cumulative)
    # the cancellations really happen where this fold meets them: (state, input) pairs of the left fold, (input,
    # state) pairs of the right fold, each followed by a restart from the next input
    fb = of.FlowBatch(vecs, ref, masks)
    pairs = [(18, 19), (20, 21), (22, 23), (25, 26), (42, 43)] if fold == 'left' else \
        [(22, 23), (20, 21), (18, 19), (46, 47)]
    for a, b in pairs:
        assert fb[a].combine_with(fb[b], 3).is_zero(thresholded=False), (a, b)
    near = [(30, 31), (56, 57)] if fold == 'left' else [(40, 41), (50, 51)]
    for a, b in near:
        res = fb[a].combine_with(fb[b], 3)
        assert res.is_zero(thresholded=True) and not res.is_zero(thresholded=False), (a, b)


@pytest.mark.gpu
def test_explicit_default_fold_is_the_default(of):
    h, w = 64, 96
    vecs, masks = make_clips(h, w, 2, 's', seed=3)
    for ref, fold in (('s', 'left'), ('t', 'right')):
        fb = of.FlowBatch(vecs, ref, masks)
        for cumulative in (True, False):
            for thresholded in (False, True):
                a = fb.accumulate(6, cumulative, thresholded).numpy()
                b = fb.accumulate(6, cumulative, thresholded, fold=fold).numpy()
                assert a[0].tobytes() == b[0].tobytes() and np.array_equal(a[1], b[1])


@pytest.mark.gpu
@pytest.mark.parametrize('ref,fold', SAMPLED)
def test_clips_equal_each_clip_alone(of, ref, fold):
    h, w = 64, 96
    vecs, masks = make_clips(h, w, 4, ref, seed=3)
    for cumulative in (True, False):
        wv, wm = of.FlowBatch(vecs, ref, masks).accumulate(6, cumulative, fold=fold).numpy()
        per = 6 if cumulative else 1
        for s in range(4):
            ov, om = of.FlowBatch(vecs[s * 6:(s + 1) * 6], ref, masks[s * 6:(s + 1) * 6]).accumulate(
                None, cumulative, fold=fold).numpy()
            assert wv[s * per:(s + 1) * per].tobytes() == ov.tobytes()
            assert np.array_equal(wm[s * per:(s + 1) * per], om)


@pytest.mark.gpu
@pytest.mark.parametrize('ref,fold', SAMPLED)
def test_length_one_and_empty_batches(of, ref, fold):
    h, w = 20, 30
    vecs, masks = make_clips(h, w, 1, ref, seed=4)
    fb = of.FlowBatch(vecs, ref, masks)
    for cumulative in (True, False):
        res = fb.accumulate(1, cumulative, fold=fold)
        v, m = res.numpy()
        assert v.tobytes() == vecs.tobytes() and np.array_equal(m, masks)
        assert res.vecs.ptr != fb.vecs.ptr and res.masks.ptr != fb.masks.ptr          # copies, not aliases
    empty = of.FlowBatch(np.zeros((0, h, w, 2), np.float32), ref).accumulate(fold=fold)
    assert len(empty) == 0 and empty.shape == (h, w) and empty.ref == ref
    assert len(of.FlowBatch(np.zeros((0, h, w, 2), np.float32), ref).accumulate(3, False, fold=fold)) == 0


@pytest.mark.gpu
@pytest.mark.parametrize('ref,fold', SAMPLED)
def test_final_only_equals_the_last_step(of, ref, fold):
    """Clip lengths 2 to 6 (the final-only steps alternate between two buffers), and at L = 2 a last step that passes
    the state through (a zero input) or restarts (a zero state), next to one that composes."""
    h, w = 50, 70
    vecs, masks = make_clips(h, w, 2, ref, seed=6)
    z = np.zeros((h, w, 2), np.float32)
    a, b = swirl(h, w, 40), swirl(h, w, 41)
    pairs = [a, z, z, a, a, b] if fold == 'left' else [z, a, a, z, a, b]     # pass, restart, compose
    for v, m, clip in [(vecs, masks, l) for l in (2, 3, 4, 6)] + [(np.stack(pairs), np.ones((6, h, w), bool), 2)]:
        fb = of.FlowBatch(v, ref, m)
        for thresholded in (False, True):
            cv, cm = fb.accumulate(clip, True, thresholded, fold=fold).numpy()
            fv, fm = fb.accumulate(clip, False, thresholded, fold=fold).numpy()
            assert fv.tobytes() == final_of(cv, clip, fold).tobytes(), clip
            assert np.array_equal(fm, final_of(cm, clip, fold)), clip
    assert fv[0].tobytes() == fv[1].tobytes() == a.tobytes() and fm[:2].all()


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
    for ref, fold in SAMPLED:
        fb.ref = last.ref = ref
        fin = fb.accumulate(clip, False, fold=fold)
        alone = last.accumulate(None, False, fold=fold)
        assert fin.vecs.frames(s - 1, s).numpy().tobytes() == alone.vecs.numpy().tobytes()
        assert np.array_equal(fin.masks.frames(s - 1, s).numpy(), alone.masks.numpy())
        del fin
        cum = fb.accumulate(clip, True, fold=fold)
        alone = last.accumulate(None, True, fold=fold)
        for k in (0, clip // 2, clip - 1):
            i = n - clip + k
            assert cum.vecs.frames(i, i + 1).numpy().tobytes() == alone.vecs.frames(k, k + 1).numpy().tobytes()
            assert np.array_equal(cum.masks.frames(i, i + 1).numpy(), alone.masks.frames(k, k + 1).numpy())
        del cum


@pytest.mark.gpu
def test_launch_count_is_one_per_step(of):
    from oflibnumpy_b200 import _lib
    rng = np.random.default_rng(8)

    def launches(s, clip, h, w, ref, fold, cumulative):
        vecs = rng.uniform(-2, 2, (s * clip, h, w, 2)).astype(np.float32)
        fb = of.FlowBatch(vecs, ref, rng.random((s * clip, h, w)) > 0.1)
        fb.accumulate(clip, cumulative, fold=fold)                           # warm-up
        before = _lib.call('ofk_rt_launch_count')
        fb.accumulate(clip, cumulative, fold=fold)
        return _lib.call('ofk_rt_launch_count') - before

    for ref, fold in SAMPLED:
        for cumulative in (True, False):
            tag = (ref, fold, cumulative)
            base = launches(2, 3, 20, 24, ref, fold, cumulative)
            assert launches(16, 3, 70, 40, ref, fold, cumulative) == base, tag
            assert launches(3, 4, 20, 24, ref, fold, cumulative) == base + 1, tag
            assert launches(1, 40, 33, 17, ref, fold, cumulative) == base + 37, tag


@pytest.mark.gpu
def test_no_read_back_or_synchronisation(of, monkeypatch):
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.device import DeviceArray
    h, w = 40, 56
    vecs, masks = fold_exit_clips(h, w, np.random.default_rng(9))
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
    for ref, fold in SAMPLED:
        for cumulative in (True, False):
            results.append(batches[ref].accumulate(6, cumulative, True, fold=fold))
    monkeypatch.undo()
    assert len(results) == 4
    want = loop_fold(of, vecs, masks, 's', 6, True, 'right')
    assert results[3].vecs.numpy().tobytes() == final_of(want[0], 6, 'right').tobytes()
