"""The source-referenced resampling (`forward_s`: Flow.apply with ref 's', same-reference invert, switch_ref, combine
modes 1 and 2, the 's'-side valid areas) against scipy.interpolate.griddata itself, through oracle/flowref.py, which runs
the reference's own griddata sequence.

Inputs are chosen where the resampler can go wrong: fields that fold (occlusion bands, a sine fold, two overlapping
bands, a mirrored frame), stretched cells (zoom 1.7-3, and a zoom whose cell size crosses 2 px, so both raster branches
meet), shrinking cells (zoom-out 0.4), a smooth non-affine field (hull pockets), a translation that moves most of the
frame out; frame sizes around the 64 x 16 raster tile and tiny frames; masks from none to 25 % removed and a rectangle
touching the border; C = 1..5 and uint8 / int16 / float64 targets. No field is a similarity transform, so no cell is
co-circular and the Delaunay triangulation is unique (the flip-tolerance tests of test_gpu_forward_s.py cover those).

The bar:
  * validity masks are bit-exact;
  * float values satisfy |dev - ref| <= 2^-20 * max|payload| of the frame, at every pixel;
  * integer payloads are exact, except where the float64 value lies within one float32 ulp of a .5 tie (+-1: the
    interpolated value is stored as float32 before it is rounded, the documented float32 round trip);
  * float64 payloads are compared with the interpolation of their float32 values (the same round trip).

The CPU half runs the same fields through the host build of the algorithm (tests/hostsim/forward_hostsim.cpp) against
griddata, so that the triangulation of folding frames is pinned without a GPU. Inputs griddata rejects (a single row or
column, fewer than three kept points, only collinear kept points: QhullError) are pinned to what the library does
instead: the pixels that coincide with a kept point take its value, all others are 0 / invalid (DESIGN.md section 11).
"""
import numpy as np
import pytest
from scipy.spatial import QhullError

from oracle import flowref as R
from test_forward_hostsim import sim  # noqa: F401  (the host build of the algorithm, compiled once per module)

REL = 2.0 ** -20


# ------------------------------------------------------------------------------------------------------------ fields
def _grid(h, w):
    y, x = np.mgrid[:h, :w].astype(np.float64)
    return y, x


def f_shear(h, w):
    y, x = _grid(h, w)
    return np.dstack([0.137 * x + 0.31 * y + 0.41, -0.171 * x + 0.0613 * y + 0.23])


def f_zoom(h, w):                      # x 2.3 / y 1.7 with a little shear: stretched cells, 4-9 candidate pixels
    y, x = _grid(h, w)
    return np.dstack([1.3 * (x - w / 2) + 0.11 * y, 0.7 * (y - h / 2) + 0.07 * x])


def f_zoom_grad(h, w):                 # cell width 1 -> 3.2 px across the frame: both raster branches side by side
    y, x = _grid(h, w)
    return np.dstack([1.1 * x * x / w + 0.013 * y, 0.021 * x + 0.17 * y])


def f_zoom_out(h, w):                  # x 0.4 / y 0.45: several cells per pixel
    y, x = _grid(h, w)
    return np.dstack([-0.6 * (x - w / 2) + 0.07 * y, -0.55 * (y - h / 2) + 0.03 * x])


def f_smooth(h, w):                    # curved frame border: hull pockets
    y, x = _grid(h, w)
    return np.dstack([2.5 * np.sin(y / 7 + 0.3) + 0.3 + 0.05 * x, 1.7 * np.cos(x / 11) + 0.02 * y])


def f_translate(h, w):                 # most of the displaced grid leaves the frame
    y, x = _grid(h, w)
    return np.dstack([0.8 * w + 0.37 + 0.013 * y, 0.21 + 0.007 * x - 0.011 * y])


def f_band(h, w):                      # an occlusion band moving 6 px over a slightly sheared background
    y, x = _grid(h, w)
    band = (x > 0.4 * w) & (x < 0.65 * w)
    return np.dstack([np.where(band, 6.0, 0.3) + 0.02 * y + 0.013 * x, 0.1 + 0.01 * x + 0.017 * y])


def f_sin(h, w):                       # a field folded by 6 sin(x / 3)
    y, x = _grid(h, w)
    return np.dstack([6 * np.sin(x / 3.0) + 0.05 * y, 0.2 * np.cos(y / 5) + 0.031 * x + 0.3 * np.sin(x / 7)])


def f_two_bands(h, w):                 # two bands moving over each other
    y, x = _grid(h, w)
    b1 = (x > 0.2 * w) & (x < 0.5 * w)
    b2 = (x > 0.45 * w) & (x < 0.75 * w) & (y > 0.3 * h)
    return np.dstack([0.3 + 0.02 * y + np.where(b1, 7.0, 0.0) - np.where(b2, 5.0, 0.0),
                      0.1 + 0.01 * x + np.where(b2, 3.0, 0.0) - 0.013 * y])


def f_mirror(h, w):                    # every cell negatively oriented, nothing overlaps
    y, x = _grid(h, w)
    return np.dstack([(w - 1 - 2 * x) + 0.13 * y, 0.07 * x - 0.1 * y])


FIELDS = {'shear': f_shear, 'zoom': f_zoom, 'zoom_grad': f_zoom_grad, 'zoom_out': f_zoom_out, 'smooth': f_smooth,
          'translate': f_translate, 'band': f_band, 'sin': f_sin, 'two_bands': f_two_bands, 'mirror': f_mirror}
FOLDING = ('band', 'sin', 'two_bands', 'mirror')
SHAPES = [(16, 63), (16, 64), (16, 65), (15, 129), (17, 64), (2, 2), (3, 5), (37, 53)]


def field(name, h, w):
    return FIELDS[name](h, w).astype(np.float32)


def make_mask(kind, h, w, seed=0):
    rng = np.random.default_rng(seed + h * 1000 + w)
    if kind == 'none':
        return None
    if kind == 'true':
        return np.ones((h, w), bool)
    if kind == 'rect':
        m = np.ones((h, w), bool)
        m[: max(1, h // 3), w // 4: max(w // 4 + 1, w // 2)] = False
        return m
    return rng.random((h, w)) >= {'m2': 0.02, 'm5': 0.05, 'm25': 0.25}[kind]


def image(h, w, c, seed=1):
    rng = np.random.default_rng(seed)
    return (rng.random((h, w, c)) * 200 - 50).astype(np.float32)


def frame_bound(payload):
    return REL * max(float(np.abs(np.asarray(payload, np.float64)).max()), 1e-30)


def assert_masks(got, want, what):
    bad = got != want
    assert not bad.any(), '%s: %d of %d mask pixels differ' % (what, int(bad.sum()), bad.size)


def assert_float(got, want, payload, what):
    err = np.abs(np.asarray(got, np.float64) - np.asarray(want, np.float64))
    bound = frame_bound(payload)
    assert err.max() <= bound, '%s: value error %g > %g at %d pixels' % (what, err.max(), bound,
                                                                         int((err > bound).sum()))


def assert_int(got, exact_ref, what):
    """exact_ref: the float64 interpolation before rounding"""
    got = np.asarray(got, np.float64)
    want = np.round(exact_ref)
    # the payload goes through float32 after interpolation: a value within a float32 ulp of a .5 tie can land on it
    tie = np.abs(np.abs(exact_ref - np.floor(exact_ref)) - 0.5) <= np.spacing(np.abs(exact_ref).astype(np.float32))
    err = np.abs(got - want)
    assert (err[~tie] == 0).all(), '%s: %d integer values differ' % (what, int((err[~tie] != 0).sum()))
    assert (err[tie] <= 1).all(), what


def griddata_ok(vecs, mask):
    """False where griddata raises (QhullError) for these points."""
    try:
        R.warp_array(vecs, np.ones(vecs.shape[:2] + (1,)), 's', mask)
        return True
    except QhullError:
        return False


# ------------------------------------------------------------------------------------------------------- CPU half
BIG = (375, 1242)
HOST_CASES = [(n, s) for n in sorted(FIELDS) for s in SHAPES] + [
    ('band', BIG), ('sin', BIG), ('smooth', BIG), ('zoom_grad', BIG)]


@pytest.mark.parametrize('name,shape', HOST_CASES, ids=lambda v: '%dx%d' % v if isinstance(v, tuple) else v)
def test_host_build_against_griddata(sim, name, shape):  # noqa: F811
    """The host build of the algorithm against griddata on every field and shape, with point masks of every kind and
    a payload mask: apply of a float32 image with its valid area, and the flow payload of invert."""
    h, w = shape
    v = field(name, h, w)
    big = h * w > 100000
    kinds = ('none', 'm5') if big else ('none', 'true', 'm2', 'm5', 'm25', 'rect')
    img = image(h, w, 3)
    folded_seen = False
    for kind in kinds:
        m = make_mask(kind, h, w)
        fm = np.ones((h, w), bool) if m is None else m
        if not griddata_ok(v, fm):
            continue
        for cm in ((True, False) if m is not None else (True,)):
            rf = R.make(v, 's', fm)
            want_v, want_m = R.apply(rf, img, return_valid_area=True, consider_mask=cm)
            got_v, got_m = sim(img, v, 1.0, fm, fm if cm else None)
            folded_seen |= bool(sim.stats[10])
            what = '%s %dx%d %s cm=%s' % (name, h, w, kind, cm)
            assert_masks(got_m, want_m, what)
            assert_float(got_v, want_v, img, what)
            if big:
                continue
            inv = R.invert(rf)
            got_v, got_m = sim(-v, v, 1.0, fm, fm if cm else None)
            if cm:
                assert_masks(got_m, inv.mask, 'invert ' + what)
                assert_float(got_v, inv.vecs, v, 'invert ' + what)
    if name in ('band', 'sin', 'two_bands') and min(h, w) >= 15:
        assert folded_seen, 'the field did not fold'


def test_folded_frames_are_triangulated_as_a_whole(sim):  # noqa: F811
    """Every folding field folds (the frame is triangulated as a whole), no other field does."""
    for name in FIELDS:
        v = field(name, 37, 53)
        sim(v, v)
        assert bool(sim.stats[10]) == (name in FOLDING), name
        assert sim.stats[3] == 0


def degenerate_cases():
    yield 'row', np.full((1, 9, 2), 0.37, np.float32), None
    yield 'column', np.full((7, 1, 2), -0.21, np.float32), None
    yield 'pixel', np.full((1, 1, 2), 0.0, np.float32) + np.float32(0.5), None
    v = f_shear(9, 11).astype(np.float32)
    m = np.zeros((9, 11), bool)
    m[4, 3] = m[2, 7] = True
    yield 'two_points', v, m
    m = np.zeros((9, 11), bool)
    m[5, :] = True
    yield 'one_row_kept', np.zeros((9, 11, 2), np.float32) + np.float32(0.25), m
    yield 'none_kept', v, np.zeros((9, 11), bool)
    # integer displacements: kept points land on pixels and give them their values
    shift = np.zeros((1, 9, 2), np.float32)
    shift[..., 0] = 1.0
    yield 'row_shifted', shift, None
    shift = np.zeros((7, 1, 2), np.float32)
    shift[..., 1] = -2.0
    yield 'column_shifted', shift, None
    shift = np.zeros((9, 11, 2), np.float32)
    shift[..., 0], shift[..., 1] = 2.0, -1.0
    m = np.zeros((9, 11), bool)
    m[2, 1] = m[4, 5] = m[6, 9] = True
    yield 'three_collinear_shifted', shift, m


def degenerate_expected(v, m, payload):
    """What the library does where griddata raises: pixels that coincide with a kept point take its value, all
    others are 0 / invalid."""
    h, w = v.shape[:2]
    out = np.zeros(payload.shape, np.float32)
    valid = np.zeros((h, w), bool)
    ys, xs = np.nonzero(np.ones((h, w), bool) if m is None else m)
    for y, x in zip(ys, xs):
        py = y + np.float64(v[y, x, 1])
        px = x + np.float64(v[y, x, 0])
        if py == int(py) and px == int(px) and 0 <= py < h and 0 <= px < w:
            out[int(py), int(px)] = payload[y, x]
            valid[int(py), int(px)] = True
    return out, valid


@pytest.mark.parametrize('case', [c[0] for c in degenerate_cases()])
def test_degenerate_input_is_pinned(sim, case):  # noqa: F811
    """griddata raises QhullError on these; the library resamples them as stated in DESIGN.md section 11."""
    v, m = [(c[1], c[2]) for c in degenerate_cases() if c[0] == case][0]
    h, w = v.shape[:2]
    img = image(h, w, 2)
    with pytest.raises((QhullError, ValueError)):        # ValueError: no points at all
        R.warp_array(v, img, 's', m)
    got_v, got_m = sim(img, v, 1.0, None, m)
    want_v, want_m = degenerate_expected(v, m, img)
    assert want_m.any() == case.endswith('_shifted')
    assert_masks(got_m, want_m, case)
    np.testing.assert_array_equal(got_v, want_v)


# ------------------------------------------------------------------------------------------------------- GPU half
@pytest.fixture(scope='module')
def of():
    import oflibnumpy_b200 as of
    of.device.require_gpu()
    return of


@pytest.fixture
def no_failed_walks(of):
    """A device test: no point-location walk may hit its step limit (counter 8 of ofk_rt_path_count) -- such a pixel
    would be left 0 / invalid."""
    before = of._lib.call('ofk_rt_path_count', 8)
    yield
    assert of._lib.call('ofk_rt_path_count', 8) == before


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
@pytest.mark.parametrize('shape', SHAPES, ids=lambda s: '%dx%d' % s)
@pytest.mark.parametrize('name', sorted(FIELDS))
def test_apply_against_griddata(of, name, shape):
    """Flow.apply (ref 's') of float32 images with C = 1, 3, 4, 5, of uint8 / int16 / float64 images and of a flow,
    with the valid area, every point mask, consider_mask True and False and a payload mask."""
    h, w = shape
    v = field(name, h, w)
    rng = np.random.default_rng(h * 7 + w)
    for kind in ('none', 'true', 'm2', 'm5', 'm25', 'rect'):
        m = make_mask(kind, h, w)
        fm = np.ones((h, w), bool) if m is None else m
        if not griddata_ok(v, fm):
            continue
        f, rf = of.Flow(v, 's', m), R.make(v, 's', fm)
        for cm in (True, False):
            what = '%s %dx%d %s cm=%s' % (name, h, w, kind, cm)
            for c in (1, 3, 4, 5):
                img = image(h, w, c, seed=c)
                tm = rng.random((h, w)) > 0.1 if c == 4 else None       # a payload mask
                got_v, got_m = f.apply(img, target_mask=tm, return_valid_area=True, consider_mask=cm)
                want_v, want_m = R.apply(rf, img, target_mask=tm, return_valid_area=True, consider_mask=cm)
                assert_masks(got_m, want_m, 'C=%d %s' % (c, what))
                assert_float(got_v, want_v, img, 'C=%d %s' % (c, what))
            if kind not in ('none', 'm5'):
                continue
            for dt, lo, hi in ((np.uint8, 0, 256), (np.int16, -32768, 32768)):
                img = rng.integers(lo, hi, (h, w, 3)).astype(dt)
                got_v, got_m = f.apply(img, return_valid_area=True, consider_mask=cm)
                want_v, want_m = R.apply(rf, img, return_valid_area=True, consider_mask=cm)
                exact = R.warp_array(v, img.astype(np.float64), 's', fm if cm else None)
                assert got_v.dtype == dt
                assert_masks(got_m, want_m, '%s %s' % (dt.__name__, what))
                assert_int(got_v, exact, '%s %s' % (dt.__name__, what))
            img64 = rng.random((h, w, 2)) * 1e3 - 300
            got_v, got_m = f.apply(img64, return_valid_area=True, consider_mask=cm)
            want_v, want_m = R.apply(rf, img64.astype(np.float32), return_valid_area=True, consider_mask=cm)
            assert got_v.dtype == np.float64
            assert_masks(got_m, want_m, 'float64 ' + what)
            assert_float(got_v, want_v, img64.astype(np.float32), 'float64 ' + what)
            # a flow payload (the flow algebra's path)
            tgt = of.Flow(image(h, w, 2, seed=9), 't', rng.random((h, w)) > 0.05)
            rt = R.make(tgt.vecs, 't', tgt.mask)
            got = f.apply(tgt, consider_mask=cm)
            want = R.apply(rf, rt, consider_mask=cm)
            assert_masks(got.mask, want.mask, 'flow ' + what)
            assert_float(got.vecs, want.vecs, tgt.vecs, 'flow ' + what)


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
@pytest.mark.parametrize('name', sorted(FIELDS))
@pytest.mark.parametrize('kind', ['none', 'm5', 'rect'])
def test_apply_flow_without_valid_area_against_griddata(of, name, kind):
    """of.apply_flow(flow, img, 's', mask): no validity plane is asked for, the resampler tracks coverage in its own
    workspace plane -- pixels found by the per-pixel search (every pixel of a folding frame, bridged holes of a masked
    one) must keep their values."""
    h, w = 37, 53
    v = field(name, h, w)
    m = make_mask(kind, h, w)
    img = image(h, w, 3)
    got = of.apply_flow(v, img, 's', m)
    want = R.warp_array(v, img, 's', m)
    assert_float(got, want, img, '%s %s' % (name, kind))
    img8 = np.random.default_rng(5).integers(0, 256, (h, w)).astype(np.uint8)
    got = of.apply_flow(v, img8, 's', m)
    assert_int(got, R.warp_array(v, img8.astype(np.float64), 's', m), 'uint8 %s %s' % (name, kind))


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
@pytest.mark.parametrize('shape', SHAPES, ids=lambda s: '%dx%d' % s)
@pytest.mark.parametrize('name', sorted(FIELDS))
def test_invert_switch_valid_areas_against_griddata(of, name, shape):
    """Same-reference invert, switch_ref both ways, valid_target ('s') and valid_source ('t'), with and without a
    point mask."""
    h, w = shape
    v = field(name, h, w)
    for kind in ('none', 'm5', 'rect'):
        m = make_mask(kind, h, w)
        fm = np.ones((h, w), bool) if m is None else m
        if not griddata_ok(v, fm) or not griddata_ok(-v, fm):
            continue
        what = '%s %dx%d %s' % (name, h, w, kind)
        fs, ft = of.Flow(v, 's', m), of.Flow(v, 't', m)
        rs, rt = R.make(v, 's', fm), R.make(v, 't', fm)
        for got, want, tag in ((fs.invert(), R.invert(rs), 'invert s'), (ft.invert(), R.invert(rt), 'invert t'),
                               (fs.switch_ref(), R.switch_ref(rs), 'switch s'),
                               (ft.switch_ref(), R.switch_ref(rt), 'switch t')):
            assert got.ref == want.ref
            assert_masks(got.mask, want.mask, tag + ' ' + what)
            assert_float(got.vecs, want.vecs, v, tag + ' ' + what)
        for cm in (True, False):
            assert_masks(fs.valid_target(cm), R.valid_target(rs, cm), 'valid_target %s cm=%s' % (what, cm))
            assert_masks(ft.valid_source(cm), R.valid_source(rt, cm), 'valid_source %s cm=%s' % (what, cm))


def _chain_xfail(mode, ref, name, why):
    return pytest.param(mode, ref, name, marks=pytest.mark.xfail(strict=True, reason=why))


_T_CHAIN = ('mode 1 of ref t chains five resamplings, two of them cv2.remap-style warps that quantise positions to '
            '1/32 px: the reference itself moves by 0.38 when its intermediate flow moves by 2^-22 relative, so no '
            'resampler within the 2^-20 bar can match it to that bar (DESIGN.md section 11)')
_T_MESH = ('mode 2 of ref t samples the mesh of the cells (mesh_sample_kernel): its fixed-point walk towards the source '
           'cell diverges where the flow stretches by more than 1 (the zoom), and it has no hull pockets (the smooth '
           'field) (DESIGN.md section 11)')
COMBINE_CASES = [(m, r, n) for m in (1, 2) for r in ('s', 't')
                 for n in ('shear', 'zoom', 'smooth', 'band', 'sin', 'mirror')
                 if (m, r, n) not in ((1, 't', 'smooth'), (1, 't', 'mirror'), (2, 't', 'zoom'), (2, 't', 'smooth'))] + [
    _chain_xfail(1, 't', 'smooth', _T_CHAIN), _chain_xfail(1, 't', 'mirror', _T_CHAIN),
    _chain_xfail(2, 't', 'zoom', _T_MESH), _chain_xfail(2, 't', 'smooth', _T_MESH)]


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
@pytest.mark.parametrize('mode,ref,name', COMBINE_CASES)
def test_combine_modes_1_2_against_griddata(of, mode, ref, name):
    """combine_with modes 1 and 2 for both references, on fields the golden files lack (no similarity transforms)."""
    h, w = 37, 53
    a = field(name, h, w)
    b = (f_shear(h, w) * 0.7 + f_smooth(h, w) * 0.3).astype(np.float32)
    ma = make_mask('m2', h, w, seed=3)
    fa, fb = of.Flow(a, ref, ma), of.Flow(b, ref)
    ra, rb = R.make(a, ref, ma), R.make(b, ref)
    if mode == 2 and ref == 't' and name in FOLDING:
        pytest.skip('mode 2 ref t samples the mesh of the cells (test_mesh_sampling_on_folding_fields)')
    got, want = fa.combine_with(fb, mode), R.combine(ra, rb, mode)
    assert_masks(got.mask, want.mask, 'mode %d %s %s' % (mode, ref, name))
    assert_float(got.vecs, want.vecs, np.concatenate([a, b]), 'mode %d %s %s' % (mode, ref, name))


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
@pytest.mark.parametrize('name', ['zoom', 'smooth', 'band', 'mirror'])
@pytest.mark.parametrize('cut', [True, False])
def test_padding_against_griddata(of, name, cut):
    """apply with padding: the flow is edge-padded for 's' and the target is the padded size; cut True and False."""
    h, w = 37, 53
    pad = [3, 2, 4, 1]
    v = field(name, h, w)
    m = make_mask('m5', h, w)
    img = image(h + 5, w + 5, 3)
    tm = np.random.default_rng(4).random((h + 5, w + 5)) > 0.1
    got_v, got_m = of.Flow(v, 's', m).apply(img, target_mask=tm.copy(), return_valid_area=True, padding=pad, cut=cut)
    want_v, want_m = R.apply(R.make(v, 's', m), img, target_mask=tm.copy(), return_valid_area=True, padding=pad,
                             cut=cut)
    assert_masks(got_m, want_m, '%s cut=%s' % (name, cut))
    assert_float(got_v, want_v, img, '%s cut=%s' % (name, cut))


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
@pytest.mark.parametrize('shape', [(37, 53), (375, 1242)], ids=lambda s: '%dx%d' % s)
def test_batch_of_mixed_frames_against_griddata(of, shape):
    """FlowBatch.apply on one batch holding every kind of field (folding and not) with different point masks: the
    frames share one launch and each one is the griddata answer."""
    h, w = shape
    names = sorted(FIELDS) if h * w < 100000 else ['shear', 'smooth', 'band', 'sin', 'translate', 'zoom_grad']
    vecs = np.stack([field(n, h, w) for n in names])
    masks = np.stack([make_mask(k, h, w, seed=i) if k != 'none' else np.ones((h, w), bool)
                      for i, k in enumerate(['none', 'm2', 'm5', 'true', 'rect'] * 2)][:len(names)])
    imgs = np.stack([image(h, w, 3, seed=i) for i in range(len(names))])
    fb = of.FlowBatch(vecs, 's', masks)
    got_v, got_m = fb.apply(imgs, return_valid_area=True)
    got_v, got_m = got_v.numpy(), got_m.numpy().view(bool)
    inv = fb.invert()
    inv_v, inv_m = inv.vecs.numpy(), inv.masks.numpy().view(bool)
    for i, n in enumerate(names):
        rf = R.make(vecs[i], 's', masks[i])
        want_v, want_m = R.apply(rf, imgs[i], return_valid_area=True)
        assert_masks(got_m[i], want_m, 'batch %s' % n)
        assert_float(got_v[i], want_v, imgs[i], 'batch %s' % n)
        want = R.invert(rf)
        assert_masks(inv_m[i], want.mask, 'batch invert %s' % n)
        assert_float(inv_v[i], want.vecs, vecs[i], 'batch invert %s' % n)


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
@pytest.mark.parametrize('name', ['band', 'sin', 'two_bands'])
def test_folding_1080p_frame_against_griddata(of, name):
    """One 1080p folding frame, with 2 % of the points removed."""
    h, w = 1080, 1920
    v = field(name, h, w)
    m = make_mask('m2', h, w)
    img = image(h, w, 1)
    got_v, got_m = of.Flow(v, 's', m).apply(img, return_valid_area=True)
    want_v, want_m = R.apply(R.make(v, 's', m), img, return_valid_area=True)
    assert_masks(got_m, want_m, name)
    assert_float(got_v, want_v, img, name)


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
@pytest.mark.parametrize('case', [c[0] for c in degenerate_cases()])
def test_degenerate_input_on_the_device(of, case):
    """The inputs griddata rejects give on the device what the host build gives (test_degenerate_input_is_pinned)."""
    v, m = [(c[1], c[2]) for c in degenerate_cases() if c[0] == case][0]
    h, w = v.shape[:2]
    img = image(h, w, 2)
    want_v, want_m = degenerate_expected(v, m, img)
    got_v, got_m = of.Flow(v, 's', m).apply(img, return_valid_area=True)
    assert_masks(got_m, want_m, case)
    np.testing.assert_array_equal(got_v, want_v)


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
def test_one_stream_gives_the_same_bytes(of, tmp_path):
    """OFK_FWD_OVERLAP=0 (everything on the caller's stream) gives the same bytes as the side stream on the fields and
    shapes of this file."""
    import os
    import subprocess
    import sys
    script = tmp_path / 'dump.py'
    script.write_text(
        'import sys, numpy as np\n'
        'sys.path[:0] = %r\n'
        'import test_forward_griddata as T\n'
        'import oflibnumpy_b200 as of\n'
        'out = []\n'
        'for shape in T.SHAPES:\n'
        '    for name in sorted(T.FIELDS):\n'
        '        v = T.field(name, *shape)\n'
        '        for kind in ("none", "m5"):\n'
        '            m = T.make_mask(kind, *shape)\n'
        '            r, vm = of.Flow(v, "s", m).apply(T.image(shape[0], shape[1], 3), return_valid_area=True)\n'
        '            out += [r.tobytes(), vm.tobytes()]\n'
        'sys.stdout.buffer.write(b"".join(out))\n' % [os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                     os.path.dirname(os.path.abspath(__file__))])
    runs = []
    for val in ('1', '0'):
        env = dict(os.environ, OFK_FWD_OVERLAP=val)
        runs.append(subprocess.run([sys.executable, str(script)], env=env, check=True,
                                   stdout=subprocess.PIPE).stdout)
    assert len(runs[0]) > 0 and runs[0] == runs[1]


@pytest.mark.gpu
@pytest.mark.usefixtures('no_failed_walks')
@pytest.mark.xfail(strict=True, reason='mesh sampling (combine mode 2 ref t, Flow.track ref t) still uses the mesh of '
                                       'the cells on folding fields (DESIGN.md section 11)')
@pytest.mark.parametrize('entry', ['combine2_t', 'track_t'])
def test_mesh_sampling_on_folding_fields(of, entry):
    h, w = 37, 53
    a = field('sin', h, w)
    if entry == 'combine2_t':
        b = field('shear', h, w)
        got, want = of.Flow(a, 't').combine_with(of.Flow(b, 't'), 2), R.combine(R.make(a, 't'), R.make(b, 't'), 2)
        assert_masks(got.mask, want.mask, entry)
        assert_float(got.vecs, want.vecs, np.concatenate([a, b]), entry)
    else:
        rng = np.random.default_rng(2)
        pts = np.stack([rng.random(500) * (h - 1), rng.random(500) * (w - 1)], -1)
        got = of.Flow(a, 't').track(pts)
        want = R.track(R.make(a, 't'), pts)
        assert_float(got, want, pts, entry)
