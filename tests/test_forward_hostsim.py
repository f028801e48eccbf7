"""CPU check of the forward-resampling ALGORITHM (oflibnumpy_b200/csrc/forward_geom.cuh + forward_irregular.cuh, the
header code the CUDA kernels execute) against outputs of the unmodified reference at the full size of configuration 3
(436x1024, tests/golden/cfg3_full.npz) and on the reference's own 7x7 golden masks.

The headers are compiled for the host by tests/hostsim/forward_hostsim.cpp into a scratch directory (test infrastructure;
the package cannot load it). What is asserted is the stated bar: validity masks bit-exact, values within 1e-3 -- including
`consider_mask=True` with 5 % of the points removed (holes bridged like Qhull does) and the pockets between the
displaced frame border and its convex hull. The one documented exception are cells whose corners are co-circular to
within rounding (pure similarity transforms): Qhull's diagonal there is arbitrary, so the reference is compared against
BOTH diagonals of those cells (in-circle determinant within +-1e-7), everywhere else against the one answer.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import golden_inputs as gi
from conftest import load_golden, ROOT

TOL = 1e-3
FLIP_TOL = 1e-7


@pytest.fixture(scope='module')
def sim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp('hostsim') / 'fwd_hostsim.so')
    src = os.path.join(ROOT, 'tests', 'hostsim', 'forward_hostsim.cpp')
    subprocess.check_call(['g++', '-O2', '-ffp-contract=off', '-shared', '-fPIC', '-o', so, src])
    lib = C.CDLL(so)

    def ptr(a):
        return None if a is None else a.ctypes.data_as(C.c_void_p)

    def run(payload, flow, sign=1.0, payload_mask=None, point_mask=None, strict=True, flip=0.0, flags=1):
        h, w = flow.shape[:2]
        pay = None if payload is None else np.ascontiguousarray(payload, np.float32)
        c = 0 if pay is None else pay.shape[2]
        out = np.zeros((h, w, max(c, 1)), np.float32)
        om = np.zeros((h, w), np.uint8)
        stats = np.zeros(12, np.int64)
        pm = None if payload_mask is None else np.ascontiguousarray(payload_mask).view(np.uint8)
        pt = None if point_mask is None else np.ascontiguousarray(point_mask).view(np.uint8)
        fl = np.ascontiguousarray(flow, np.float32)
        lib.fwd_hostsim(ptr(pay), c, ptr(fl), C.c_float(sign), ptr(pm), ptr(pt), ptr(out), ptr(om), int(strict), h, w,
                        flags, C.c_double(flip), ptr(stats))
        run.stats = stats
        assert stats[3] == 0, "point-location walks that did not terminate"
        assert stats[5] == 0 or stats[10] == 1, "folded cells left to the mesh of the cells"
        assert stats[6] == 0, "pixels produced by more than one triangle: the fill rule is broken"
        return out[..., :c], om.astype(bool)
    return run


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


def check(name, got, got_alt, want_vals_s, want_mask, idx, exact, skip_values=None):
    """got / got_alt: (values, mask) of the production diagonal rule and of the flipped co-circular cells."""
    (v, m), (v2, m2) = got, got_alt
    if exact:
        assert np.array_equal(m, want_mask), '%s: %d mask mismatches' % (name, int((m != want_mask).sum()))
    else:
        ok = (m == want_mask) | (m2 == want_mask)
        assert ok.all(), '%s: %d mask pixels match neither diagonal' % (name, int((~ok).sum()))
    if want_vals_s is None:
        return
    c = v.shape[-1]
    a = v.reshape(-1, c)[idx].astype(np.float64)
    b = v2.reshape(-1, c)[idx].astype(np.float64)
    valid = want_mask.ravel()[idx] & m.ravel()[idx]
    if skip_values is not None:
        valid &= ~skip_values.ravel()[idx]
    assert valid.mean() > 0.3
    err_a = np.abs(a - want_vals_s).max(-1)
    err_b = np.abs(b - want_vals_s).max(-1)
    if exact:
        assert err_a[valid].max() <= TOL, '%s: value error %g' % (name, err_a[valid].max())
    else:
        assert np.minimum(err_a, err_b)[valid].max() <= TOL, '%s: %g' % (name, np.minimum(err_a, err_b)[valid].max())


def both(sim, *args, **kw):
    return sim(*args, **kw), sim(*args, flip=FLIP_TOL, **kw)


@pytest.mark.slow
@pytest.mark.parametrize('pair', ['smooth', 'aff'])
@pytest.mark.parametrize('tag', ['full', 'm5'])
def test_cfg3_full_size_against_reference(sim, pair, tag):
    g = load_golden('cfg3_full')
    inp = gi.cfg3_full()
    v = inp[pair]
    h, w = v.shape[:2]
    idx = gi.sample_pixels(h, w, frac=0.02, band=2)
    m = None if tag == 'full' else inp['mask']
    k = pair + '_' + tag
    # on the non-degenerate field the Delaunay triangulation is unique: everything has to match the one answer; on
    # the rotation, values of a non-affine payload (the image) depend on the diagonal of co-circular cells
    def mask_of(key):
        return unpack(g[key], (h, w))
    img = inp['img_f32c3']
    # a bridged hole on the rotation is a ring of co-circular points (its Delaunay triangulation is not unique either):
    # image values there are only pinned on the non-degenerate field; flows (affine payloads) are pinned everywhere
    skip = near_removed_points(v, 1.0, m) if (pair == 'aff' and m is not None) else None
    check('apply ' + k, *both(sim, img, v, 1.0, m, m), g['out_applyva_%s_img_s' % k], mask_of('out_applyva_%s_validbits' % k),
          idx, exact=(pair == 'smooth'), skip_values=skip)
    for name, payload, sign in (('invert_ss', -v, 1.0), ('invert_tt', -v, -1.0), ('switch_s', v, 1.0),
                                ('switch_t', v, -1.0)):
        # reference algebra (flow_class.py:697-753): invert s->s = self.apply(-self); invert t->t = (-self as 's')
        # .apply(itself); switch s->t = self.apply(self); switch t->s = (-f).apply(f) with f = self relabelled 's'
        check(name + ' ' + k, *both(sim, payload, v, sign, m, m), g['out_%s_%s_vecs_s' % (name, k)],
              mask_of('out_%s_%s_maskbits' % (name, k)), idx, exact=True)
    ones = None if m is None else m
    check('valid_target_s ' + k, *both(sim, None, v, 1.0, ones, m), None, mask_of('out_valid_target_s_%s_bits' % k), idx,
          exact=True)
    check('valid_source_t ' + k, *both(sim, None, v, -1.0, ones, m), None, mask_of('out_valid_source_t_%s_bits' % k), idx,
          exact=True)
    if m is not None:
        # consider_mask=False: every point stays, the payload mask carries the holes; which pixels around a hole are
        # valid depends on the diagonal of the cells there -> exact on the unique triangulation, either diagonal on
        # co-circular cells
        check('valid_target_s nocm ' + k, *both(sim, None, v, 1.0, m, None), None,
              mask_of('out_valid_target_s_%s_nocm_bits' % k), idx, exact=(pair == 'smooth'))
        check('invert_ss nocm ' + k, *both(sim, -v, v, 1.0, m, None), g['out_invert_ss_%s_nocm_vecs_s' % k],
              mask_of('out_invert_ss_%s_nocm_maskbits' % k), idx, exact=(pair == 'smooth'))


def test_reference_7x7_golden_masks(sim):
    """tests/test_flow_class.py:852-980 of the reference incl. the `consider_mask=True` cases where Qhull bridges the
    removed points with long triangles (the hull of the remaining points becomes valid)."""
    g = load_golden('small_masks')
    vs, vt, ms, mt = g['in_vecs_s'], g['in_vecs_t'], g['in_mask_s'], g['in_mask_t']
    assert np.array_equal(sim(None, vs, 1.0, None, None)[1], g['out_vt_s'])
    assert np.array_equal(sim(None, vt, -1.0, None, None)[1], g['out_vs_t'])
    assert np.array_equal(sim(None, vs, 1.0, ms, None)[1], g['out_vt_s_masked'])
    assert np.array_equal(sim(None, vt, -1.0, mt, None)[1], g['out_vs_t_masked'])
    assert np.array_equal(sim(None, vs, 1.0, ms, ms)[1], g['out_vt_s_masked_cm'])
    assert np.array_equal(sim(None, vt, -1.0, mt, mt)[1], g['out_vs_t_masked_cm'])


def test_small_forward_goldens(sim):
    g = load_golden('forward')
    for pair in ('aff', 'smooth'):
        v = g['in_' + pair]
        vals, m = sim(-v, v)
        assert np.array_equal(m, g['out_invert_ss_%s_mask' % pair])
        assert np.abs(vals - g['out_invert_ss_%s_vecs' % pair])[m].max() <= TOL
        vals, m = sim(g['in_img_f32c3'], v)
        assert np.array_equal(m, g['out_applyva_s_f32c3_%s_valid' % pair])
        mk = g['in_mask']
        assert np.array_equal(sim(None, v, 1.0, mk, mk)[1], g['out_valid_target_s_masked_cm_' + pair])


def test_integer_translation_and_exact_hull_edges(sim):
    """Pixels exactly on the hull (tests/test_utils.py:277-283 of the reference demands equality with an integer
    shift) are inside; the search treats the hull inclusively."""
    rng = np.random.default_rng(5)
    img = rng.random((23, 31, 1)).astype(np.float32)
    for dx, dy in ((0, 0), (4, 0), (0, -3), (5, 7)):
        flow = np.zeros((23, 31, 2), np.float32)
        flow[..., 0], flow[..., 1] = dx, dy
        vals, m = sim(img, flow)
        want = np.zeros_like(img)
        wm = np.zeros((23, 31), bool)
        ys, xs = slice(max(dy, 0), 23 + min(dy, 0)), slice(max(dx, 0), 31 + min(dx, 0))
        yt, xt = slice(max(-dy, 0), 23 + min(-dy, 0)), slice(max(-dx, 0), 31 + min(-dx, 0))
        want[ys, xs] = img[yt, xt]
        wm[ys, xs] = True
        assert np.array_equal(m, wm)
        assert np.array_equal(vals, want)


@pytest.mark.slow
@pytest.mark.parametrize('masked', [False, True])
def test_enumerated_triangles_equal_the_per_pixel_search(sim, masked):
    """Hull pockets (frames without removed points) and the small faces left by removed points are triangulated
    explicitly and rasterised; flags 4 / 8 switch that off, so that every pixel outside the intact cells is located by
    the walk through the Delaunay triangulation of the boundary sites instead. Both are the same triangulation: masks
    identical, values equal to rounding (the weights come out of different but equivalent expressions)."""
    inp = gi.cfg3_full()
    v, img = inp['smooth'], inp['img_f32c3']
    m = inp['mask'] if masked else None
    a_v, a_m = sim(img, v, 1.0, m, m)
    produced = int(sim.stats[1])
    b_v, b_m = sim(img, v, 1.0, m, m, flags=1 | 4 | 8 | 16)
    assert produced > 1000 and int(sim.stats[1]) >= produced      # the search path now finds all of them itself
    assert np.array_equal(a_m, b_m)
    assert np.abs(a_v - b_v)[a_m].max() <= 1e-4


@pytest.mark.parametrize('density', [0.02, 0.06, 0.12, 0.25])
def test_enumerated_faces_equal_the_search_on_random_masks(sim, density):
    """The same equivalence over masks of growing density (faces merge, pinch, surround islands of intact cells and
    single points, reach the frame border): whatever hole_loop() accepts has to be a simple polygon without anything
    inside, everything else has to be left to the search."""
    h, w = 150, 220
    for seed in range(3):
        rng = np.random.default_rng(100 + seed)
        v = (gi.smooth_field(h, w) * 0.6).astype(np.float32)
        m = rng.random((h, w)) > density
        yy, xx = np.mgrid[:h, :w].astype(np.float32)
        pay = np.stack([xx, yy, rng.random((h, w)).astype(np.float32) * 255], -1)
        a_v, a_m = sim(pay, v, 1.0, m, m)
        faces = int(sim.stats[8])
        b_v, b_m = sim(pay, v, 1.0, m, m, flags=1 | 4 | 8 | 16)
        assert faces > 20
        assert np.array_equal(a_m, b_m)
        assert np.abs(a_v - b_v)[a_m].max() <= 1e-3


@pytest.mark.parametrize('angle', [4.0, 17.0, 45.0])
def test_pockets_of_a_mask_left_by_a_forward_pass(sim, angle):
    """A forward pass leaves a mask that is valid inside the hull of the resampled points -- a rotated frame with
    staircase edges -- and the next pass of a chain (switch_ref, modes 1 / 2) uses it as its point mask. The boundary of
    such a mask is traced (trace_outer_loop) and the pockets between the staircase and its hull are triangulated like
    those of the frame border: same result as the per-pixel search (flag 16 switches the tracing off)."""
    h, w = 160, 240
    yy, xx = np.mgrid[:h, :w].astype(np.float64)
    a = np.deg2rad(angle)
    u = (xx - w / 2) * np.cos(a) + (yy - h / 2) * np.sin(a)
    t = -(xx - w / 2) * np.sin(a) + (yy - h / 2) * np.cos(a)
    m = (np.abs(u) < 0.42 * w) & (np.abs(t) < 0.38 * h)
    rng = np.random.default_rng(int(angle))
    v = (gi.smooth_field(h, w) * 0.5).astype(np.float32)
    pay = np.stack([xx, yy, rng.random((h, w)) * 255], -1).astype(np.float32)
    a_v, a_m = sim(pay, v, 1.0, m, m)
    chains = int(sim.stats[9])
    b_v, b_m = sim(pay, v, 1.0, m, m, flags=1 | 16)
    c_v, c_m = sim(pay, v, 1.0, m, m, flags=1 | 4 | 8 | 16)
    assert chains == 1 and int(sim.stats[9]) == 0
    assert np.array_equal(a_m, b_m) and np.array_equal(a_m, c_m)
    assert np.abs(a_v - b_v)[a_m].max() <= 1e-3 and np.abs(a_v - c_v)[a_m].max() <= 1e-3
    assert a_m.sum() > 0.3 * h * w
