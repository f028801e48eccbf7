"""Batched flow visualisation: FlowBatch.visualise (ofk_visualise_batch) and batch.visualise_flows_host
(ofh_visualise). Frame i of every result must equal Flow(vecs[i], ref, masks[i]).visualise(...) byte for byte, with the
default range of each frame (99th percentile, else maximum, else 1) resolved on the device."""
import numpy as np
import pytest

import golden_inputs as gi
from conftest import load_golden
from oracle import flowref as R
from test_oracle_golden import VIS_VARIANTS


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


def same(got, want):
    assert got.dtype == want.dtype == np.uint8, (got.dtype, want.dtype)
    assert got.shape == want.shape, (got.shape, want.shape)
    np.testing.assert_array_equal(got, want)


def variants():
    return [(key.split('_')[0], kw) for key, kw in VIS_VARIANTS]


def field(h, w, seed, scale=1.0):
    """A smooth swirl with noise, different for every seed."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[:h, :w].astype(np.float32)
    a, b = rng.uniform(20, 60, 2)
    v = np.stack([8 * np.sin(xx / a + seed) * np.cos(yy / b) + 0.002 * (xx - w / 2),
                  6 * np.cos(xx / b + 1) * np.sin(yy / a) - 0.003 * (yy - h / 2)], -1)
    v += rng.standard_normal((h, w, 2)) * 0.05
    return (v * scale).astype(np.float32)


def batch_1080p(n=6):
    """Frames with different content: swirls at several scales, a sparse frame (99th percentile 0, maximum > 0) and a
    frame whose vectors all lie below the threshold (range 1)."""
    h, w = 1080, 1920
    rng = np.random.default_rng(21)
    frames = [field(h, w, 1), field(h, w, 2, 0.1), field(h, w, 3, 25.0)]
    sparse = np.zeros((h, w, 2), np.float32)
    idx = rng.integers(0, h * w, 200)
    sparse.reshape(-1, 2)[idx] = rng.standard_normal((200, 2)).astype(np.float32) * 4
    frames.append(sparse)
    frames.append((rng.standard_normal((h, w, 2)) * 1e-4).astype(np.float32))
    frames.append(field(h, w, 4, 3.0))
    vecs = np.stack(frames[:n])
    masks = rng.random((n, h, w)) > 0.02
    return vecs, masks


# ------------------------------------------------------------------------------------------------------------- CPU
def test_bad_arguments_are_rejected_without_a_gpu(lib):
    """ofh_visualise / ofk_visualise_batch check their arguments before a device, a stream or the ring is touched."""
    nan = float('nan')
    for args, msg in (((None, None, 1e-3, 1, 0, 0, 0.0, 16, 1, 4, 4, 0), "ofh_visualise: bad arguments"),
                      ((16, None, 1e-3, 3, 0, 0, 0.0, 16, 1, 4, 4, 0), "ofh_visualise: mode must be"),
                      ((16, None, 1e-3, 1, 0, 0, -1.0, 16, 1, 4, 4, 0), "ofh_visualise: range_max must be"),
                      ((16, None, 1e-3, 1, 0, 0, nan, 16, 1, 4, 4, 0), "ofh_visualise: range_max must be")):
        with pytest.raises(lib.OflibCudaError, match=msg):
            lib.call('ofh_visualise', *args)
    for args, msg in (((None, None, 1e-3, 1, 0, 0, 0.0, 16, 1, 4, 4, 16, 1 << 20, None), "NULL pointer"),
                      ((16, None, 1e-3, -1, 0, 0, 0.0, 16, 1, 4, 4, 16, 1 << 20, None), "mode must be"),
                      ((16, None, 1e-3, 1, 0, 0, -2.5, 16, 1, 4, 4, 16, 1 << 20, None), "range_max must be"),
                      ((16, None, 1e-3, 1, 0, 0, nan, 16, 1, 4, 4, 16, 1 << 20, None), "range_max must be"),
                      ((16, None, 1e-3, 1, 0, 0, 0.0, 16, 2, 4, 4, None, 0, None), "workspace too small"),
                      ((16, None, 1e-3, 1, 0, 0, 0.0, 16, 2, 4, 4, 18, 1 << 20, None), "ws must be 4-byte aligned")):
        with pytest.raises(lib.OflibCudaError, match=msg):
            lib.call('ofk_visualise_batch', *args)


def test_workspace_is_n_times_a_per_frame_amount(lib):
    one = lib.call('ofk_visualise_batch_workspace', 1, 1080, 1920)
    assert one >= 1080 * 1920 * 4
    for n in (0, 2, 7, 700):
        assert lib.call('ofk_visualise_batch_workspace', n, 1080, 1920) == n * one
    assert lib.call('ofk_visualise_batch_workspace', 1, 0, 5) == 0


def test_python_callers_share_the_argument_checks(lib):
    """FlowBatch.visualise and visualise_flows_host raise what Flow.visualise raises, before any device work."""
    from oflibnumpy_b200.batch import FlowBatch, visualise_flows_host
    from oflibnumpy_b200.validation import validate_visualise_args
    fb = FlowBatch._wrap(None, 't', None)
    flows = np.zeros((1, 4, 4, 2), np.float32)
    for args, kw, exc in ((('xyz',), {}, ValueError), (('rgb',), {'show_mask': 1}, TypeError),
                          (('rgb',), {'show_mask_borders': 'yes'}, TypeError), (('rgb',), {'range_max': 0}, ValueError),
                          (('rgb',), {'range_max': -3.0}, ValueError), (('rgb',), {'range_max': '2'}, TypeError)):
        with pytest.raises(exc) as want:
            validate_visualise_args(args[0], kw.get('show_mask'), kw.get('show_mask_borders'), kw.get('range_max'))
        with pytest.raises(exc) as got:
            fb.visualise(*args, **kw)
        assert str(got.value) == str(want.value)
        with pytest.raises(exc) as got:
            visualise_flows_host(flows, *args, **kw)
        assert str(got.value) == str(want.value)
    with pytest.raises(ValueError, match="Mode needs to be either"):       # an unhashable mode, as the reference
        validate_visualise_args(['rgb'], None, None, None)
    with pytest.raises(ValueError, match="out needs to be"):
        visualise_flows_host(flows, 'rgb', out=np.empty((1, 4, 4, 3), np.float32))


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_golden_frames_in_one_batch(of):
    """The swirl (99th percentile > 0), sparse (percentile 0, maximum > 0) and zero (range 1) frames of the reference's
    own outputs, stacked into one batch: every variant, bit for bit."""
    from oflibnumpy_b200.batch import FlowBatch
    g = load_golden('visualise')
    names = ('swirl', 'sparse', 'zero')
    vecs = np.stack([g['in_' + n] for n in names])
    fb = FlowBatch(vecs, 't', np.stack([g['in_mask']] * 3))
    for key, kw in VIS_VARIANTS:
        got = fb.visualise(key.split('_')[0], **kw).numpy()
        for i, n in enumerate(names):
            same(got[i], g['out_%s_%s' % (n, key)])


@pytest.mark.gpu
def test_1080p_batch_equals_flow_visualise_and_oracle(of):
    from oflibnumpy_b200.batch import FlowBatch
    vecs, masks = batch_1080p()
    fb = FlowBatch(vecs, 's', masks)
    for mode, kw in variants():
        got = fb.visualise(mode, **kw).numpy()
        for i in range(len(vecs)):
            want = R.visualise(R.make(vecs[i], 's', masks[i]), mode, **kw)
            same(got[i], want)
            same(of.Flow(vecs[i], 's', masks[i]).visualise(mode, **kw), want)


@pytest.mark.gpu
def test_odd_shapes(of):
    """Shapes whose rows do not fill whole 8-pixel groups, frames of one row or column, and single frames from 1x1 to
    4K, where the device's plan of numpy.percentile(mag, 99) (float32 virtual index and lerp) must match numpy's."""
    from oflibnumpy_b200.batch import FlowBatch
    rng = np.random.default_rng(7)
    for (h, w) in ((1, 1), (1, 37), (29, 1), (37, 53), (5, 7), (9, 30), (13, 17)):
        for n in (1, 5):
            vecs = np.stack([field(h, w, 10 + i, 0.5 + i) for i in range(n)])
            masks = rng.random((n, h, w)) > 0.2
            fb = FlowBatch(vecs, 't', masks)
            for mode, kw in variants():
                got = fb.visualise(mode, **kw).numpy()
                for i in range(n):
                    same(got[i], R.visualise(R.make(vecs[i], 't', masks[i]), mode, **kw))
    shapes = [(1, 1), (1, 2), (1, 3), (1, 7), (10, 10), (1, 101), (10, 100), (45, 64), (48, 60), (216, 192),
              (1080, 1920), (2160, 3840)]
    for k, (h, w) in enumerate(shapes):
        v = field(h, w, 40 + k, (1e-3, 1.0, 300.0)[k % 3] * 4)
        if h * w > 10:
            v.reshape(-1, 2)[rng.integers(0, h * w, h * w // 3)] = 0
        m = rng.random((h, w)) > 0.05
        got = FlowBatch(v[None], 't', m[None]).visualise('rgb', show_mask=True).numpy()[0]
        same(got, R.visualise(R.make(v, 't', m), 'rgb', show_mask=True))


@pytest.mark.gpu
def test_launches_do_not_grow_with_the_batch(of):
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.batch import FlowBatch
    lib = _lib.load()
    counts = {}
    for n in (2, 64):
        fb = FlowBatch(np.stack([field(60, 80, i) for i in range(n)]), 't')
        for rng_max in (None, 4.0):
            fb.visualise('bgr', range_max=rng_max)          # warm-up: allocations, module load
            before = lib.ofk_rt_launch_count()
            out = fb.visualise('bgr', range_max=rng_max)
            counts[(n, rng_max)] = lib.ofk_rt_launch_count() - before
            assert out.shape == (n, 60, 80, 3)
    assert counts[(2, None)] == counts[(64, None)]
    assert counts[(2, 4.0)] == counts[(64, 4.0)] == 1


@pytest.mark.gpu
def test_more_frames_than_grid_y_holds(of):
    """70000 small frames with the default range: more frames than a grid's y dimension holds (65535), one call with the
    same launch count as any other batch. Frames across the batch equal the same frames visualised alone, and the
    library stays usable afterwards."""
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.batch import FlowBatch
    n, h, w = 70000, 4, 6
    rng = np.random.default_rng(11)
    vecs = (rng.standard_normal((n, h, w, 2)) * rng.uniform(0.01, 5, (n, 1, 1, 1))).astype(np.float32)
    vecs[rng.integers(0, n, 50)] = 0
    masks = rng.random((n, h, w)) > 0.1
    fb = FlowBatch(vecs, 't', masks)
    lib = _lib.load()
    before = lib.ofk_rt_launch_count()
    got = fb.visualise('rgb', show_mask_borders=True).numpy()
    assert lib.ofk_rt_launch_count() - before == 7
    for i in [0, 1, 65534, 65535, 65536, n - 1] + [int(k) for k in rng.integers(0, n, 20)]:
        same(got[i], R.visualise(R.make(vecs[i], 't', masks[i]), 'rgb', show_mask_borders=True))
    same(fb[5].visualise('hsv'), R.visualise(R.make(vecs[5], 't', masks[5]), 'hsv'))


@pytest.mark.gpu
def test_outputs_beyond_4_gib(of):
    """700 frames at 1080p (4.35 GB of output): first, middle and last frames equal the same frames visualised alone
    (64-bit offsets in the colourise kernel and in the per-frame selection records)."""
    from oflibnumpy_b200 import _lib, _ops
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    h, w, n = 1080, 1920, 700
    rng = np.random.default_rng(3)
    st = of.device.current_stream()
    mats = np.stack([np.linalg.pinv(R.matrix_from_transforms(gi.cfg4_transforms(9000 + i))) for i in range(n)])
    v = _ops.from_matrix(DeviceArray.from_numpy(mats), (h, w), -1.0)
    m = DeviceArray.empty((n, h, w), np.uint8)
    _lib.call('ofk_rt_memset', m.ptr, 1, m.nbytes, st)
    check = (0, n // 2 + 7, n - 1)
    for i in check:
        mk = (rng.random((1, h, w)) > 0.03).astype(np.uint8)
        _lib.call('ofk_rt_memcpy_h2d', m.frames(i, i + 1).ptr, mk.ctypes.data, mk.nbytes, st)
        of.device.synchronize()
    fb = FlowBatch._wrap(v, 't', m)
    for mode, kw in (('rgb', {'show_mask_borders': True}), ('hsv', {'show_mask': True, 'range_max': 9.0})):
        out = fb.visualise(mode, **kw)
        assert out.nbytes > (1 << 32)
        for i in check:
            one = FlowBatch._wrap(v.frames(i, i + 1), 't', m.frames(i, i + 1)).visualise(mode, **kw).numpy()
            same(out.frames(i, i + 1).numpy(), one)
        del out


@pytest.mark.gpu
def test_host_entry_equals_device_batch(of):
    """visualise_flows_host against FlowBatch.visualise: pageable and pinned buffers, with and without masks, one frame
    per ring chunk (1080p) and several frames per chunk with a short last chunk (13 frames of 540x960: chunks of 6 or
    8 frames), caller-supplied out."""
    from oflibnumpy_b200 import device
    from oflibnumpy_b200.batch import FlowBatch, visualise_flows_host
    vecs, masks = batch_1080p(4)
    small = np.stack([field(540, 960, 60 + i, 0.3 * (i + 1)) for i in range(13)])
    small_masks = np.random.default_rng(9).random(small.shape[:3]) > 0.1
    keep = []
    for v, m in ((vecs, masks), (small, small_masks)):
        pv, hv = device.pinned_empty(v.shape, np.float32)
        pv[...] = v
        pm, hm = device.pinned_empty(m.shape, np.bool_)
        pm[...] = m
        keep += [hv, hm]
        for mode, kw in (('rgb', {'show_mask': True, 'show_mask_borders': True}), ('hsv', {}),
                         ('bgr', {'range_max': 3.5})):
            for use_mask in (False, True):
                want = FlowBatch(v, 't', m if use_mask else None).visualise(mode, **kw).numpy()
                same(visualise_flows_host(v, mode, m if use_mask else None, **kw), want)
                po, ho = device.pinned_empty(want.shape, np.uint8)
                got = visualise_flows_host(pv, mode, pm if use_mask else None, out=po, **kw)
                assert got is po
                same(po, want)
                del ho
    out = np.zeros(small.shape[:3] + (3,), np.uint8)
    assert visualise_flows_host(small, 'bgr', small_masks, out=out) is out
    same(out, FlowBatch(small, 't', small_masks).visualise('bgr').numpy())
