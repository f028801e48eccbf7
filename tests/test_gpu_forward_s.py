"""GPU parity of the source-referenced path (forward resampling, invert / switch_ref, combine modes 1 and 2, track,
resize) against outputs of the unmodified reference (tests/golden), through the public API -> ctypes -> C ABI.

The bar: validity masks bit-exact, flow and warped values within 1e-3 on valid pixels -- including `consider_mask=True`
with removed points (holes bridged as Qhull bridges them) and the pockets between the displaced frame border and its
convex hull, at the full size of configuration 3 (436x1024). The one documented exception: cells of the displaced
grid whose corners are co-circular to within rounding (pure similarity transforms) have no unique Delaunay diagonal and
Qhull's pick is an artefact of its facet merging. There the reference is compared against BOTH diagonals (test hook
ofk_forward_s_set_flip_tol, in-circle determinant within +-1e-7); it only matters for payloads that are not affine
across the cell (images; validity around masked points with consider_mask=False).
"""
import numpy as np
import pytest

import golden_inputs as gi
from conftest import load_golden
from oracle import flowref as R

pytestmark = pytest.mark.gpu
TOL = 1e-3
FLIP_TOL = 1e-7


@pytest.fixture(scope='module')
def of():
    import oflibnumpy_b200 as of
    of.device.require_gpu()
    return of


@pytest.fixture(autouse=True)
def no_failed_searches(of):
    """Every test: no point-location walk may hit its step limit (counter 8 of ofk_rt_path_count)."""
    before = of._lib.call('ofk_rt_path_count', 8)
    yield
    assert of._lib.call('ofk_rt_path_count', 8) == before


class flipped(object):
    """Context: co-circular cells take their other diagonal."""

    def __init__(self, of):
        self.of = of

    def __enter__(self):
        self.of._lib.call('ofk_forward_s_set_flip_tol', FLIP_TOL)

    def __exit__(self, *exc):
        self.of._lib.call('ofk_forward_s_set_flip_tol', 0.0)
        return False


def close_on_valid(got_v, got_m, want_v, want_m, tol=TOL):
    both = got_m & want_m
    assert both.any()
    err = np.abs(got_v.astype(np.float64) - want_v.astype(np.float64))[both]
    assert err.max() <= tol, err.max()


def check_flow(g, key, fl):
    want_v, want_m = g['out_' + key + '_vecs'], g['out_' + key + '_mask']
    assert fl.ref == str(g['out_' + key + '_ref'])
    diff = fl.mask != want_m
    assert not diff.any(), '%s: %d mask mismatches' % (key, int(diff.sum()))
    close_on_valid(fl.vecs, fl.mask, want_v, want_m)


def test_affine_field_bit_exact_masks(of):
    g = load_golden('forward')
    fs, ft = of.Flow(g['in_aff'], 's'), of.Flow(g['in_aff'], 't')
    check_flow(g, 'invert_ss_aff', fs.invert())
    check_flow(g, 'invert_tt_aff', ft.invert())
    check_flow(g, 'invert_st_aff', fs.invert('t'))
    check_flow(g, 'invert_ts_aff', ft.invert('s'))
    check_flow(g, 'switch_s_aff', fs.switch_ref())
    check_flow(g, 'switch_t_aff', ft.switch_ref())
    np.testing.assert_array_equal(fs.valid_target(), g['out_valid_target_s_aff'])
    np.testing.assert_array_equal(ft.valid_source(), g['out_valid_source_t_aff'])
    np.testing.assert_array_equal(fs.valid_source(), g['out_valid_source_s_aff'])
    np.testing.assert_array_equal(ft.valid_target(), g['out_valid_target_t_aff'])
    # functional wrappers
    np.testing.assert_allclose(of.invert_flow(g['in_aff'], 's')[g['out_invert_ss_aff_mask']],
                               g['out_invert_ss_aff_vecs'][g['out_invert_ss_aff_mask']], rtol=0, atol=TOL)
    np.testing.assert_allclose(of.switch_flow_ref(g['in_aff'], 't')[g['out_switch_t_aff_mask']],
                               g['out_switch_t_aff_vecs'][g['out_switch_t_aff_mask']], rtol=0, atol=TOL)
    np.testing.assert_array_equal(of.valid_target(g['in_aff'], 's'), g['out_valid_target_s_aff'])


def test_smooth_field_values_and_hull_pockets(of):
    """Non-affine field: the displaced border is curved, Qhull fills the pockets up to the convex hull with long
    triangles between border points -- masks and values have to match there too."""
    g = load_golden('forward')
    fs, ft = of.Flow(g['in_smooth'], 's'), of.Flow(g['in_smooth'], 't')
    pockets_before = of._lib.call('ofk_rt_path_count', 6)
    check_flow(g, 'invert_ss_smooth', fs.invert())
    check_flow(g, 'invert_tt_smooth', ft.invert())
    check_flow(g, 'switch_s_smooth', fs.switch_ref())
    check_flow(g, 'switch_t_smooth', ft.switch_ref())
    assert of._lib.call('ofk_rt_path_count', 6) > pockets_before          # pocket pixels were located, not dropped
    np.testing.assert_array_equal(fs.valid_target(), g['out_valid_target_s_smooth'])
    np.testing.assert_array_equal(ft.valid_source(), g['out_valid_source_t_smooth'])
    # image payload: on a non-degenerate field the Delaunay triangulation is unique, values agree everywhere
    w, m = fs.apply(g['in_img_f32c3'], return_valid_area=True)
    np.testing.assert_array_equal(m, g['out_applyva_s_f32c3_smooth_valid'])
    close_on_valid(w, m[..., None] & np.ones(3, bool), g['out_applyva_s_f32c3_smooth'],
                   g['out_applyva_s_f32c3_smooth_valid'][..., None] & np.ones(3, bool))
    np.testing.assert_allclose(fs.apply(g['in_img_f32c3']), g['out_apply_s_f32c3_smooth'], rtol=0, atol=TOL)
    w8 = fs.apply(g['in_img_u8c3'])
    assert np.abs(w8.astype(int) - g['out_apply_s_u8c3_smooth'].astype(int)).max() <= 1      # rounding of x.5 ties


def test_image_payload_on_cocircular_cells_matches_one_of_the_two_diagonals(of):
    """Pure rotations leave ~8 % of the cells co-circular to within 1e-10 (in-circle determinant): Qhull's diagonal
    there is an artefact of its merge order. Every value of the reference equals the interpolation along one of the
    two diagonals of its cell; masks agree everywhere."""
    g = load_golden('forward')
    fs = of.Flow(g['in_aff'], 's')
    w, m = fs.apply(g['in_img_f32c3'], return_valid_area=True)
    with flipped(of):
        w2, m2 = fs.apply(g['in_img_f32c3'], return_valid_area=True)
    np.testing.assert_array_equal(m, g['out_applyva_s_f32c3_aff_valid'])
    np.testing.assert_array_equal(m2, m)
    want = g['out_applyva_s_f32c3_aff']
    err = np.minimum(np.abs(w - want).max(axis=-1), np.abs(w2 - want).max(axis=-1))[m]
    assert err.max() <= TOL
    assert (np.abs(w - want).max(axis=-1)[m] <= TOL).mean() >= 0.9


def test_reference_7x7_golden_masks_s_side(of):
    """tests/test_flow_class.py:852-980 of the reference, the cases resampled in 's' direction -- including
    consider_mask=True, where the reference triangulates the remaining points only and the hull of those becomes
    valid (docs/usage.rst:353-361 of the reference)."""
    g = load_golden('small_masks')
    fs, ft = of.Flow(g['in_vecs_s'], 's'), of.Flow(g['in_vecs_t'], 't')
    fsm, ftm = of.Flow(g['in_vecs_s'], 's', g['in_mask_s']), of.Flow(g['in_vecs_t'], 't', g['in_mask_t'])
    np.testing.assert_array_equal(fs.valid_target(), g['out_vt_s'])
    np.testing.assert_array_equal(ft.valid_source(), g['out_vs_t'])
    np.testing.assert_array_equal(fsm.valid_target(False), g['out_vt_s_masked'])
    np.testing.assert_array_equal(ftm.valid_source(False), g['out_vs_t_masked'])
    np.testing.assert_array_equal(fsm.valid_target(), g['out_vt_s_masked_cm'])
    np.testing.assert_array_equal(ftm.valid_source(), g['out_vs_t_masked_cm'])


def test_masked_points_are_bridged_like_the_reference(of):
    g = load_golden('forward')
    for pair in ('aff', 'smooth'):
        fsm = of.Flow(g['in_' + pair], 's', g['in_mask'])
        np.testing.assert_array_equal(fsm.valid_target(), g['out_valid_target_s_masked_cm_' + pair])
        got = fsm.valid_target(consider_mask=False)
        if pair == 'smooth':
            np.testing.assert_array_equal(got, g['out_valid_target_s_masked_nocm_' + pair])
            check_flow(g, 'invert_ss_masked_nocm_' + pair, fsm.apply(-fsm, consider_mask=False))
        else:
            with flipped(of):
                got2 = fsm.valid_target(consider_mask=False)
            want = g['out_valid_target_s_masked_nocm_' + pair]
            assert ((got == want) | (got2 == want)).all()


def unpack(bits, shape):
    return np.unpackbits(bits)[:shape[0] * shape[1]].reshape(shape).astype(bool)


def near_removed_points(flow, sign, mask, radius=1):
    """Pixels within `radius` of the displaced position of a removed point: the region a bridged hole can cover."""
    h, w = mask.shape
    yy, xx = np.nonzero(~mask)
    px = np.rint(xx + sign * flow[yy, xx, 0]).astype(int)
    py = np.rint(yy + sign * flow[yy, xx, 1]).astype(int)
    out = np.zeros((h, w), bool)
    for dy in range(-radius, radius + 1):
        for dx in range(-radius, radius + 1):
            x, y = px + dx, py + dy
            ok = (x >= 0) & (x < w) & (y >= 0) & (y < h)
            out[y[ok], x[ok]] = True
    return out


@pytest.mark.parametrize('pair', ['smooth', 'aff'])
@pytest.mark.parametrize('tag', ['full', 'm5'])
def test_cfg3_full_size_against_reference(of, pair, tag):
    """Configuration 3 of BASELINE.json as written (436x1024): Flow.apply 's' of a float32 x3 image, invert() s->s and
    t->t, switch_ref both ways and the 's'-resampled valid areas, with full masks and with 5 % of the points masked
    (consider_mask=True, the default, and False) -- against tests/golden/cfg3_full.npz from the unmodified reference.
    Masks are complete (bit-packed) in the fixture, values are kept at a seeded subset of pixels."""
    g = load_golden('cfg3_full')
    inp = gi.cfg3_full()
    v = inp[pair]
    h, w = v.shape[:2]
    idx = gi.sample_pixels(h, w, frac=0.02, band=2)
    m = None if tag == 'full' else inp['mask']
    k = pair + '_' + tag
    fs, ft = of.Flow(v, 's', m), of.Flow(v, 't', m)
    report = {}

    def check_mask(name, got, key, got_alt=None):
        want = unpack(g[key], (h, w))
        bad = got != want if got_alt is None else (got != want) & (got_alt != want)
        report[name] = int(bad.sum())
        assert not bad.any(), '%s %s: %d mask mismatches' % (name, k, int(bad.sum()))
        return want

    def check_vals(name, got, want_s, valid, got_alt=None):
        c = got.shape[-1]
        err = np.abs(got.reshape(-1, c)[idx].astype(np.float64) - want_s).max(-1)
        if got_alt is not None:
            err = np.minimum(err, np.abs(got_alt.reshape(-1, c)[idx].astype(np.float64) - want_s).max(-1))
        sel = valid.ravel()[idx]
        assert sel.mean() > 0.3
        assert err[sel].max() <= TOL, '%s %s: value error %g' % (name, k, err[sel].max())

    img = inp['img_f32c3']
    wimg, va = fs.apply(img, return_valid_area=True)
    if pair == 'smooth':
        want = check_mask('apply', va, 'out_applyva_%s_validbits' % k)
        check_vals('apply', wimg, g['out_applyva_%s_img_s' % k], want)
    else:
        with flipped(of):
            wimg2, va2 = fs.apply(img, return_valid_area=True)
        want = check_mask('apply', va, 'out_applyva_%s_validbits' % k)
        np.testing.assert_array_equal(va2, va)
        # a bridged hole on the rotation is a ring of co-circular points (no unique triangulation either): image
        # values there are pinned on the non-degenerate field only; flows (affine payloads) are pinned everywhere
        sel = want if m is None else want & ~near_removed_points(v, 1.0, m)
        check_vals('apply', wimg, g['out_applyva_%s_img_s' % k], sel, wimg2)
    for name, fl in (('invert_ss', fs.invert()), ('invert_tt', ft.invert()), ('switch_s', fs.switch_ref()),
                     ('switch_t', ft.switch_ref())):
        assert fl.ref == str(g['out_%s_%s_ref' % (name, k)])
        want = check_mask(name, fl.mask, 'out_%s_%s_maskbits' % (name, k))
        check_vals(name, fl.vecs, g['out_%s_%s_vecs_s' % (name, k)], want)
    check_mask('valid_target_s', fs.valid_target(), 'out_valid_target_s_%s_bits' % k)
    check_mask('valid_source_t', ft.valid_source(), 'out_valid_source_t_%s_bits' % k)
    if m is not None:
        got = fs.valid_target(consider_mask=False)
        inv = fs.apply(-fs, consider_mask=False)
        if pair == 'smooth':
            check_mask('valid_target_s nocm', got, 'out_valid_target_s_%s_nocm_bits' % k)
            want = check_mask('invert_ss nocm', inv.mask, 'out_invert_ss_%s_nocm_maskbits' % k)
        else:
            with flipped(of):
                got2 = fs.valid_target(consider_mask=False)
                inv2 = fs.apply(-fs, consider_mask=False)
            check_mask('valid_target_s nocm', got, 'out_valid_target_s_%s_nocm_bits' % k, got2)
            want = check_mask('invert_ss nocm', inv.mask, 'out_invert_ss_%s_nocm_maskbits' % k, inv2.mask)
        check_vals('invert_ss nocm', inv.vecs, g['out_invert_ss_%s_nocm_vecs_s' % k], want & inv.mask)
    print('cfg3', k, 'mask mismatches:', report)


def test_combine_modes_1_and_2(of):
    g = load_golden('combine12')
    for r in ('s', 't'):
        f1, f2, f3 = (of.Flow(g['in_f%d_%s' % (i, r)], r) for i in (1, 2, 3))
        check_flow(g, 'm1_' + r, f2.combine_with(f3, 1))
        check_flow(g, 'm2_' + r, f1.combine_with(f3, 2))
        check_flow(g, 'm3_' + r, f1.combine_with(f2, 3))
        np.testing.assert_allclose(of.combine_flows(g['in_f1_' + r], g['in_f3_' + r], 2, r)[g['out_m2_%s_mask' % r]],
                                   g['out_m2_%s_vecs' % r][g['out_m2_%s_mask' % r]], rtol=0, atol=TOL)


def test_combine_against_analytic_composition(of):
    """The reference's own criterion (tests/test_flow_class.py:1020-1057): combined flows equal the flow of the
    composed transforms within 5e-2 on the valid area, all modes, both references."""
    shape = (96, 96)
    transforms = [['rotation', 47.5, 47.5, -30], ['scaling', 20, 20, 0.8]]
    for ref in ('s', 't'):
        f1 = of.Flow.from_transforms(transforms[0:1], shape, ref)
        f2 = of.Flow.from_transforms(transforms[1:2], shape, ref)
        f3 = of.Flow.from_transforms(transforms, shape, ref)
        for mode, (a, b, want) in ((1, (f2, f3, f1)), (2, (f1, f3, f2)), (3, (f1, f2, f3))):
            got = a.combine_with(b, mode)
            assert isinstance(got, of.Flow) and got.ref == ref
            comb = got.mask & want.mask
            assert comb.mean() > 0.2
            np.testing.assert_allclose(got.vecs[comb], want.vecs[comb], atol=5e-2)


def test_switch_ref_and_invert_against_analytic(of):
    """tests/test_flow_class.py:509-573 of the reference: rtol = atol = 1e-3 against the analytic opposite flows."""
    shape = (128, 128)
    tr = [['rotation', 64, 64, 30]]
    tr_inv = [['rotation', 64, 64, -30]]
    f_s, f_t = of.Flow.from_transforms(tr, shape, 's'), of.Flow.from_transforms(tr, shape, 't')
    b_s, b_t = of.Flow.from_transforms(tr_inv, shape, 's'), of.Flow.from_transforms(tr_inv, shape, 't')
    for got, want in ((f_s.switch_ref(), f_t), (f_t.switch_ref(), f_s), (f_s.invert(), b_s), (f_t.invert(), b_t),
                      (f_s.invert('t'), b_t), (f_t.invert('s'), b_s)):
        assert got.ref == want.ref
        np.testing.assert_allclose(got.vecs[got.mask], want.vecs[got.mask], rtol=1e-3, atol=1e-3)
    z = of.Flow.zero(shape, 's')
    assert z.switch_ref().ref == 't' and z.switch_ref(mode='invalid').ref == 't'
    with pytest.raises(ValueError):
        z.switch_ref('test')


def test_identity_and_integer_translation_exact(of):
    """tests/test_utils.py:277-283 of the reference demands exact equality with an integer shift, both refs."""
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (40, 53, 3), dtype=np.uint8)
    imgf = rng.random((40, 53)).astype(np.float32)
    for ref in ('s', 't'):
        for sh in ((0, 0), (10, 0), (0, -7), (4, 9)):
            flow = np.zeros((40, 53, 2), np.float32)
            flow[..., 0], flow[..., 1] = sh
            for im in (img, imgf):
                got = of.apply_flow(flow, im, ref)
                want = R.warp_array(flow, im, ref)
                np.testing.assert_array_equal(got, want)


def test_next_rows_track_resize_padding(of):
    g = load_golden('next_rows')
    for r in ('s', 't'):
        f = of.Flow(g['in_flow'], r, g['in_mask'])
        np.testing.assert_allclose(f.track(g['in_pts_f']), g['out_track_f_' + r], rtol=0, atol=1e-3 if r == 't' else 1e-9)
        pts, st = f.track(g['in_pts_f'], get_valid_status=True)
        np.testing.assert_array_equal(st, g['out_track_status_' + r])
        got_int = f.track(g['in_pts_f'], int_out=True)
        assert got_int.dtype == g['out_track_int_' + r].dtype
        assert np.abs(got_int - g['out_track_int_' + r]).max() <= (1 if r == 't' else 0)
        np.testing.assert_allclose(f.track(g['in_pts_i']), g['out_track_ipts_' + r], rtol=0, atol=1e-3)
        for j, sc in enumerate(gi.RESIZE_SCALES):
            rz = f.resize(sc)
            want_v, want_m = g['out_resize_%d_%s_vecs' % (j, r)], g['out_resize_%d_%s_mask' % (j, r)]
            assert rz.vecs.shape == want_v.shape
            np.testing.assert_array_equal(rz.vecs, want_v)
            np.testing.assert_array_equal(rz.mask, want_m)
            np.testing.assert_array_equal(of.resize_flow(g['in_flow'], sc), want_v)
        assert f.get_padding() == list(g['out_padding_' + r])
    fs = of.Flow(g['in_flow'], 's')
    np.testing.assert_allclose(fs.track(g['in_pts_f'], s_exact_mode=True), g['out_track_exact_s'], rtol=0, atol=1e-3)
    np.testing.assert_allclose(of.track_pts(g['in_flow'], 's', g['in_pts_f']), g['out_track_f_s'], rtol=0, atol=1e-9)
    with pytest.raises(IndexError):
        fs.track(np.array([[-1.0, 3.0]]))
    with pytest.raises(TypeError):
        fs.track(g['in_pts_f'], True, get_valid_status='test')
    # the reference's own known answers (tests/test_utils.py:543-571): rotation 30 deg about the origin
    f_s = of.from_transforms([['rotation', 0, 0, 30]], (512, 512), 's')
    f_t = of.from_transforms([['rotation', 0, 0, 30]], (512, 512), 't')
    pts = np.array([[20.5, 10.5], [8.3, 7.2], [120.4, 160.2]])
    desired = np.array([[12.5035207776, 19.343266740], [3.58801085141, 10.385382907], [24.1694586156, 198.93726969]])
    np.testing.assert_allclose(of.track_pts(f_s, 's', pts), desired, atol=1e-1, rtol=1e-2)
    np.testing.assert_allclose(of.track_pts(f_s, 's', pts, s_exact_mode=True), desired, atol=1e-5)
    np.testing.assert_allclose(of.track_pts(f_t, 't', pts), desired, atol=1e-5, rtol=1e-6)
    got = of.track_pts(f_t, 't', pts, int_out=True)
    np.testing.assert_array_equal(got, np.round(desired))
    assert np.issubdtype(got.dtype, np.integer)
    f = of.from_transforms([['translation', 10, 20]], (512, 512), 's')
    np.testing.assert_array_equal(of.track_pts(f, 's', np.array([[20, 10], [8, 7]])), [[40, 20], [28, 17]])


def test_point_mask_that_removes_nothing_takes_the_unmasked_path(of):
    """Flow.apply / invert hand the flow's mask to ofk_forward_s as `consider_mask`; a frame whose mask is all true is
    recognised on the device and processed like one without a point mask (hull pockets triangulated arc by arc):
    bit-identical outputs, in a batch that mixes both kinds of frames."""
    from oflibnumpy_b200 import _lib, _ops
    from oflibnumpy_b200.device import DeviceArray
    h, w = 200, 320
    rng = np.random.default_rng(11)
    flows = np.stack([gi.smooth_field(h, w), gi.smooth_field(h, w) * 0.5, gi.smooth_field(h, w)]).astype(np.float32)
    masks = np.ones((3, h, w), bool)
    masks[1] = rng.random((h, w)) > 0.03
    pay = rng.random((3, h, w, 2)).astype(np.float32)
    d_f, d_p = DeviceArray.from_numpy(flows), DeviceArray.from_numpy(pay)
    d_m = DeviceArray.from_numpy(masks.view(np.uint8))
    o1, m1 = _ops.forward_s(d_f, 1.0, d_p, d_m, d_m)
    # frames 0 and 2 alone, without any point mask
    sel = np.ascontiguousarray(flows[[0, 2]])
    o2, m2 = _ops.forward_s(DeviceArray.from_numpy(sel), 1.0, DeviceArray.from_numpy(np.ascontiguousarray(pay[[0, 2]])),
                            None, None)
    o1, m1, o2, m2 = o1.numpy(), m1.numpy(), o2.numpy(), m2.numpy()
    assert np.array_equal(m1[[0, 2]], m2) and np.array_equal(o1[[0, 2]], o2)
    assert m2.any() and not m2.all()
    # the masked frame in the middle equals the same frame processed alone
    o3, m3 = _ops.forward_s(DeviceArray.from_numpy(flows[1:2]), 1.0, DeviceArray.from_numpy(pay[1:2]),
                            DeviceArray.from_numpy(masks[1:2].view(np.uint8)),
                            DeviceArray.from_numpy(masks[1:2].view(np.uint8)))
    assert np.array_equal(m1[1:2], m3.numpy()) and np.array_equal(o1[1:2], o3.numpy())


def test_forward_s_is_deterministic(of):
    """Pockets are shared between the warps of a CTA and holes between threads in whatever order the scheduler picks:
    the result may not depend on it."""
    g = load_golden('forward')
    v = g['in_smooth']
    fs = of.Flow(v, 's', g['in_mask'])
    first = fs.apply(g['in_img_f32c3'], return_valid_area=True)
    for _ in range(5):
        again = fs.apply(g['in_img_f32c3'], return_valid_area=True)
        assert np.array_equal(first[0], again[0]) and np.array_equal(first[1], again[1])


def _rotated_frame_mask(h, w, angle):
    yy, xx = np.mgrid[:h, :w].astype(np.float64)
    a = np.deg2rad(angle)
    u = (xx - w / 2) * np.cos(a) + (yy - h / 2) * np.sin(a)
    t = -(xx - w / 2) * np.sin(a) + (yy - h / 2) * np.cos(a)
    return (np.abs(u) < 0.42 * w) & (np.abs(t) < 0.38 * h)


def test_enumerated_triangles_equal_the_per_pixel_search_on_the_device(of):
    """The passes that triangulate explicitly -- hull pockets along the frame border or along the traced boundary of a
    mask that a forward pass left behind (a rotated frame with staircase edges), small faces of removed points -- give
    what the per-pixel search through the Delaunay triangulation of the boundary sites gives when they are switched off
    (ofk_forward_s_set_disable): same masks, values equal to rounding. One batch mixes all kinds of frames."""
    from oflibnumpy_b200 import _lib, _ops
    from oflibnumpy_b200.device import DeviceArray
    h, w = 240, 352
    rng = np.random.default_rng(21)
    base = gi.smooth_field(h, w).astype(np.float32)
    flows = np.stack([base, base * 0.5, base, base * 0.7, base * 0.3])
    masks = np.ones((5, h, w), bool)
    masks[1] = rng.random((h, w)) > 0.03
    masks[2] = _rotated_frame_mask(h, w, 7.0)
    masks[3] = _rotated_frame_mask(h, w, 31.0)
    masks[4] = rng.random((h, w)) > 0.15
    yy, xx = np.mgrid[:h, :w].astype(np.float32)
    pay = np.stack([np.stack([xx, yy, rng.random((h, w)).astype(np.float32) * 255], -1)] * 5)
    d_f, d_p = DeviceArray.from_numpy(flows), DeviceArray.from_numpy(np.ascontiguousarray(pay))
    d_m = DeviceArray.from_numpy(masks.view(np.uint8))
    before = [_lib.call('ofk_rt_path_count', k) for k in (6, 8)]
    o1, m1 = _ops.forward_s(d_f, 1.0, d_p, d_m, d_m)
    o1, m1 = o1.numpy(), m1.numpy()
    enumerated = _lib.call('ofk_rt_path_count', 6) - before[0]
    _lib.call('ofk_forward_s_set_disable', 4 | 8 | 16)
    try:
        o2, m2 = _ops.forward_s(d_f, 1.0, d_p, d_m, d_m)
        o2, m2 = o2.numpy(), m2.numpy()
    finally:
        _lib.call('ofk_forward_s_set_disable', 0)
    assert enumerated > 1000
    assert _lib.call('ofk_rt_path_count', 8) == before[1]
    for n in range(5):
        assert np.array_equal(m1[n], m2[n]), 'frame %d: %d mask mismatches' % (n, int((m1[n] != m2[n]).sum()))
        assert np.abs(o1[n] - o2[n])[m1[n] != 0].max() <= 1e-3, 'frame %d' % n
        assert m1[n].any() and not m1[n].all()


_OVERLAP_CODE = r'''
import hashlib, sys, threading
import numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import golden_inputs as gi
import oflibnumpy_b200 as of
from oflibnumpy_b200.device import Stream
h, w, n = 270, 480, 6
rng = np.random.default_rng(5)
flows = np.stack([np.asarray(of.from_transforms(gi.cfg4_transforms(i), (h, w), 's')) for i in range(n)])
flows[1] = gi.smooth_field(h, w)                       # curved border: hull pockets
yy, xx = np.mgrid[:h, :w].astype(np.float32)
flows[2, ..., 0] = 60 * np.sin(xx / 9)                 # folds: redone by the order-independent resolve
flows[3] = 0                                           # zero flow: passed through
masks = rng.random((n, h, w)) > 0.03
masks[4] = True
dig = hashlib.sha256()
def run(tag):
    fb = of.FlowBatch(flows, 's', masks)
    for res in (fb.invert(), fb.switch_ref()):
        v, m = res.numpy()
        dig.update(np.ascontiguousarray(m).tobytes()); dig.update(np.ascontiguousarray(v).tobytes())
run('main')
# two host threads enqueue ofk_forward_s on two streams at once (C ABI, explicit streams): the shared side stream
# serialises their chains
from oflibnumpy_b200 import _lib
from oflibnumpy_b200.device import DeviceArray
d_fl = DeviceArray.from_numpy(flows)
d_pm = DeviceArray.from_numpy(masks.view(np.uint8))
wsb = _lib.call('ofk_forward_s_workspace', n, h, w)
bufs = [(DeviceArray.empty((n, h, w, 2), np.float32), DeviceArray.empty((n, h, w), np.uint8),
         DeviceArray.empty((wsb,), np.uint8), Stream()) for _ in range(2)]
of.device.synchronize()
def worker(k):
    o_v, o_m, ws, st = bufs[k]
    for _ in range(3):
        _lib.call('ofk_forward_s', d_fl.ptr, 2, d_fl.ptr, 1.0, d_pm.ptr, d_pm.ptr, o_v.ptr, o_m.ptr, _lib.RULE_STRICT, n, h,
                  w, ws.ptr, wsb, st.handle)
    st.synchronize()
ts = [threading.Thread(target=worker, args=(k,)) for k in range(2)]
[t.start() for t in ts]; [t.join() for t in ts]
out = [hashlib.sha256(b[1].numpy().tobytes() + b[0].numpy().tobytes()).hexdigest() for b in bufs]
assert out[0] == out[1]
print('DIGEST', dig.hexdigest(), out[0])
'''


def test_side_stream_overlap_gives_the_same_bytes():
    """ofk_forward_s runs its site / hull chain on a side stream beside the raster kernel (fork / join with events).
    The result must be byte-identical to everything on one stream (OFK_FWD_OVERLAP=0, read once per process): batch with
    a curved field, a folding frame, a zero-flow frame and removed points; and two host threads on two streams."""
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    code = _OVERLAP_CODE % (os.path.dirname(here), here)
    digests = []
    for env_extra in ({}, {'OFK_FWD_OVERLAP': '0'}):
        res = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, **env_extra), capture_output=True,
                             text=True, timeout=900)
        assert res.returncode == 0, res.stdout + res.stderr
        digests.append([l for l in res.stdout.splitlines() if l.startswith('DIGEST')][0])
    assert digests[0] == digests[1]
