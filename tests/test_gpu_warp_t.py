"""GPU parity: the CUDA target-referenced path (through the Python shim -> ctypes -> C ABI) against outputs of the
unmodified reference (tests/golden) and against the CPU oracle on the same seeded inputs.

Bar (BASELINE.json north_star): valid masks bit-exact; flow / warped values within 1e-3 on valid pixels. The kernels
restate cv2.remap's arithmetic operation by operation, so on this path the tests additionally demand bit-exact values.
"""
import hashlib
import json
import os

import numpy as np
import pytest

import golden_inputs as gi
from conftest import load_golden
from oracle import flowref as R

pytestmark = pytest.mark.gpu

TOL = 1e-3  # px / intensity, north_star tolerance


@pytest.fixture(scope='module')
def of():
    import oflibnumpy_b200 as of
    of.device.require_gpu()
    return of


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def same(got, want):
    assert got.dtype == want.dtype, (got.dtype, want.dtype)
    assert got.shape == want.shape, (got.shape, want.shape)
    if np.issubdtype(want.dtype, np.floating):
        assert np.abs(got.astype(np.float64) - want.astype(np.float64)).max() <= TOL
    np.testing.assert_array_equal(got, want)


def flow_same(g, prefix, f):
    same(f.mask, g['out_' + prefix + '_mask'])
    assert f.ref == str(g['out_' + prefix + '_ref'])
    same(f.vecs, g['out_' + prefix + '_vecs'])


def test_apply_flow_and_flow_apply_all_dtypes(of):
    g = load_golden('warp_t')
    flow, fmask = g['in_flow'], g['in_flow_mask']
    f = of.Flow(flow, 't', fmask)
    f_nomask = of.Flow(flow, 't')
    for name in [k[3:] for k in g if k.startswith('in_img_')]:
        img = g['in_' + name]
        same(of.apply_flow(flow, img, 't'), g['out_applyflow_' + name])
        same(f.apply(img), g['out_apply_' + name])
        if 'err_applyva_' + name in g:
            with pytest.raises(TypeError):
                f.apply(img, return_valid_area=True)
            continue
        w, m = f.apply(img, return_valid_area=True)
        same(w, g['out_applyva_' + name])
        same(m, g['out_applyva_' + name + '_valid'])
        if 'out_applyvatm_' + name in g:
            w, m = f.apply(img, target_mask=g['in_target_mask'], return_valid_area=True)
            same(w, g['out_applyvatm_' + name])
            same(m, g['out_applyvatm_' + name + '_valid'])
            w, m = f_nomask.apply(img, target_mask=g['in_target_mask'], return_valid_area=True)
            same(w, g['out_applyvatm_nofm_' + name])
            same(m, g['out_applyvatm_nofm_' + name + '_valid'])


def test_flow_applied_to_flow_and_valid_areas(of):
    g = load_golden('warp_t')
    f = of.Flow(g['in_flow'], 't', g['in_flow_mask'])
    flow_same(g, 'apply_flowobj', f.apply(of.Flow(g['in_flow2'], 't', g['in_flow2_mask'])))
    flow_same(g, 'apply_flowobj_s', f.apply(of.Flow(g['in_flow2'], 's', g['in_flow2_mask'])))
    same(f.valid_target(), g['out_valid_target'])
    same(of.Flow(g['in_flow'], 's', g['in_flow_mask']).valid_source(), g['out_valid_source_of_s'])
    assert f.get_padding() == list(g['out_get_padding_t'])
    assert of.Flow(g['in_flow'], 's', g['in_flow_mask']).get_padding() == list(g['out_get_padding_s'])


def test_vectorised_and_scalar_paths_agree(of):
    """W % 4 == 0 takes the 4-pixel vector kernel, anything else the scalar kernel: both against the oracle."""
    rng = np.random.default_rng(11)
    for (h, w) in ((37, 64), (37, 66), (64, 128), (5, 4), (1, 1), (3, 257)):
        flow = (rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(12)
        fmask = rng.random((h, w)) > 0.1
        tmask = rng.random((h, w)) > 0.1
        f, fr = of.Flow(flow, 't', fmask), R.make(flow, 't', fmask)
        for dt, c in ((np.uint8, 3), (np.uint8, 1), (np.uint8, 4), (np.uint8, 2), (np.float32, 3), (np.float32, 2),
                      (np.float32, 1), (np.float32, 4), (np.float32, 5), (np.int16, 3), (np.uint16, 1),
                      (np.float64, 3)):
            img = (rng.random((h, w, c)) * 255).astype(dt)
            same(f.apply(img), R.apply(fr, img))
            if dt != np.uint16:
                w1, m1 = f.apply(img, return_valid_area=True)
                w2, m2 = R.apply(fr, img, return_valid_area=True)
                same(w1, w2)
                same(m1, m2)
            w1, m1 = f.apply(img, target_mask=tmask, return_valid_area=True)
            w2, m2 = R.apply(fr, img, target_mask=tmask, return_valid_area=True)
            same(w1, w2)
            same(m1, m2)


def test_padding_and_cut(of):
    g = load_golden('warp_t_padded')
    pad = [int(x) for x in g['in_padding']]
    f = of.Flow(g['in_flow'], 't', g['in_flow_mask'])
    for cut in (True, False):
        tag = 'cut' if cut else 'nocut'
        same(f.apply(g['in_img_u8c3'], padding=pad, cut=cut), g['out_apply_u8_' + tag])
        w, m = f.apply(g['in_img_u8c3'], return_valid_area=True, padding=pad, cut=cut)
        same(w, g['out_applyva_u8_' + tag])
        same(m, g['out_applyva_u8_' + tag + '_valid'])
        w, m = f.apply(g['in_img_f32c3'], target_mask=g['in_target_mask'], return_valid_area=True, padding=pad,
                       cut=cut)
        same(w, g['out_applyvatm_f32_' + tag])
        same(m, g['out_applyvatm_f32_' + tag + '_valid'])
        flow_same(g, 'apply_flowobj_' + tag, f.apply(of.Flow(g['in_big_flow'], 't', g['in_big_flow_mask']),
                                                     padding=pad, cut=cut))
    same(f.pad(pad).vecs, g['out_pad_constant_vecs'])
    same(f.pad(pad).mask, g['out_pad_constant_mask'])
    same(f.pad(pad, 'edge').vecs, g['out_pad_edge_vecs'])
    same(f.pad(pad, 'symmetric').vecs, g['out_pad_symmetric_vecs'])


def test_zero_and_tiny_flows_are_identity(of):
    """The reference returns the target untouched for |v| < 1e-3 (utils.py:215-216); identity taps reproduce it."""
    rng = np.random.default_rng(12)
    h, w = 33, 48
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    imgf = rng.random((h, w, 3)).astype(np.float32)
    tiny = (rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(1.9e-3)
    for flow in (np.zeros((h, w, 2), np.float32), tiny):
        same(of.apply_flow(flow, img, 't'), img)
        same(of.apply_flow(flow, imgf, 't'), imgf)
        wv, m = of.Flow(flow).apply(img, return_valid_area=True)
        same(wv, img)
        assert m.all()
        assert of.Flow(flow).valid_target().all()


def test_combine_mode3_golden(of):
    g = load_golden('combine3')
    for r in ('t', 's'):
        for pair in ('aff', 'smooth'):
            a = of.Flow(g['in_' + pair + '_1'], r, g['in_mask_1'])
            b = of.Flow(g['in_' + pair + '_2'], r, g['in_mask_2'])
            flow_same(g, 'c3_{}_{}'.format(r, pair), a.combine_with(b, 3))
            same(of.combine_flows(g['in_' + pair + '_1'], g['in_' + pair + '_2'], 3, r),
                 g['out_cf3_{}_{}'.format(r, pair)])
        a = of.Flow(g['in_zero_where_valid'], r, g['in_zero_mask'])
        b = of.Flow(g['in_aff_2'], r, g['in_mask_2'])
        res = a.combine_with(b, 3)
        assert res is b                                   # the reference returns the operand itself
        flow_same(g, 'c3_{}_Azero'.format(r), res)
        res = b.combine_with(a, 3)
        assert res is b
        flow_same(g, 'c3_{}_Bzero'.format(r), res)
        a = of.Flow(g['in_tiny'], r, g['in_mask_1'])
        flow_same(g, 'c3_{}_tiny_thr'.format(r), a.combine_with(b, 3, thresholded=True))
        flow_same(g, 'c3_{}_tiny_nothr'.format(r), a.combine_with(b, 3, thresholded=False))


def test_combine_mode3_shapes_vs_oracle(of):
    """Widths that are multiples of 16 take the TMA-staged kernel (box fits: small flows; box does not fit: large
    flows, CTA-uniform fallback), other widths the plain gather kernel; all against the oracle."""
    rng = np.random.default_rng(13)
    for (h, w, amp) in ((40, 64, 10), (41, 67, 10), (2, 4, 10), (1, 1, 10), (96, 160, 10), (96, 160, 60), (64, 48, 3),
                        (33, 16, 200), (70, 130, 25)):
        a = (rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(amp)
        b = (rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(amp)
        am, bm = rng.random((h, w)) > 0.1, rng.random((h, w)) > 0.1
        for r in ('t', 's'):
            got = of.Flow(a, r, am).combine_with(of.Flow(b, r, bm), 3)
            want = R.combine(R.make(a, r, am), R.make(b, r, bm), 3)
            same(got.mask, want.mask)
            same(got.vecs, want.vecs)


def test_zero_test_probe_and_scan(of):
    """The zero tests of the TMA composition path: a sparse probe decides almost every frame, a full scan the rest.
    Frames that are zero except on pixels the probe does not visit must still count as non-zero; frames that are
    non-zero only on invalid pixels must count as zero (the reference tests vecs[mask])."""
    rng = np.random.default_rng(15)
    n, h, w = 6, 64, 96                                     # 6144 px per frame: the probe looks at every 3rd pixel
    a = np.zeros((n, h, w, 2), np.float32)
    b = (rng.random((n, h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(6)
    am, bm = rng.random((n, h, w)) > 0.05, rng.random((n, h, w)) > 0.05
    a[0].reshape(-1, 2)[1] = (0.5, 0)                        # frame 0: one non-zero vector on an unprobed pixel
    am[0].reshape(-1)[1] = True
    a[1].reshape(-1, 2)[4] = (0, -2)                         # frame 1: the only non-zero vector is invalid -> zero
    am[1].reshape(-1)[4] = False
    a[2].reshape(-1, 2)[-1] = (1e-4, 0)                      # frame 2: last pixel, below the threshold
    am[2].reshape(-1)[-1] = True
    a[3] = (rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(6)
    b[4] = 0                                                 # frame 4: B zero, A zero -> B returned
    a[5].reshape(-1, 2)[5000] = (3, 3)
    am[5].reshape(-1)[5000] = True
    for thr, expect_a in ((False, [1, 0, 1, 1, 0, 1]), (True, [1, 0, 0, 1, 0, 1])):
        for r in ('t', 's'):
            res, flags = of.FlowBatch(a, r, am).combine_with(of.FlowBatch(b, r, bm), 3, thresholded=thr,
                                                              return_flags=True)
            fl = flags.numpy()
            assert fl[:, 0].tolist() == expect_a, (thr, r, fl.tolist())
            assert fl[:, 1].tolist() == [1, 1, 1, 1, 0, 1], (thr, r, fl.tolist())
            v, m = res.numpy()
            for i in range(n):
                want = R.combine(R.make(a[i], r, am[i]), R.make(b[i], r, bm[i]), 3, thresholded=thr)
                same(m[i], want.mask)
                same(v[i], want.vecs)


def test_batched_equals_per_frame(of):
    """FlowBatch (one launch for N frames, device-side early exits) == N single-frame calls == oracle."""
    rng = np.random.default_rng(14)
    n, h, w = 5, 36, 64
    a = (rng.random((n, h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(8)
    b = (rng.random((n, h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(8)
    am, bm = rng.random((n, h, w)) > 0.05, rng.random((n, h, w)) > 0.05
    a[1] = 0                         # frame 1: A zero            -> result is B
    b[2][bm[2]] = 0                  # frame 2: B zero where valid -> result is A
    a[3][am[3]] = 0                  # frame 3: both zero         -> result is B (A tested first)
    b[3] = 0
    imgs = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    for r in ('t', 's'):
        fa, fb = of.FlowBatch(a, r, am), of.FlowBatch(b, r, bm)
        res, flags = fa.combine_with(fb, 3, return_flags=True)
        v, m = res.numpy()
        fl = flags.numpy()
        assert fl[1, 0] == 0 and fl[2, 1] == 0 and fl[0].all() and fl[4].all()
        for i in range(n):
            want = R.combine(R.make(a[i], r, am[i]), R.make(b[i], r, bm[i]), 3)
            same(m[i], want.mask)
            same(v[i], want.vecs)
            single = of.Flow(a[i], r, am[i]).combine_with(of.Flow(b[i], r, bm[i]), 3)
            same(single.vecs, want.vecs)
            same(res[i].vecs, want.vecs)
    fa = of.FlowBatch(a, 't', am)
    out, valid = fa.apply(imgs, return_valid_area=True)
    out, valid = out.numpy(), valid.numpy().view(np.bool_)
    for i in range(n):
        w2, m2 = R.apply(R.make(a[i], 't', am[i]), imgs[i], return_valid_area=True)
        same(out[i], w2)
        same(valid[i], m2)
    # host-buffer entry points (ofh_*): same results from numpy buffers
    out_h, valid_h = of.batch.apply_flow_host(a, imgs, flow_masks=am, return_valid_area=True)
    same(out_h, out)
    same(valid_h, valid)
    v_h, m_h = of.batch.combine_flows_host(a, b, 3, 't', am, bm)
    v_d, m_d = of.FlowBatch(a, 't', am).combine_with(of.FlowBatch(b, 't', bm), 3).numpy()
    same(v_h, v_d)
    same(m_h, m_d)


def test_generators_bit_exact(of):
    g = load_golden('generators')
    for i, (kind, arg, shape, r) in enumerate(gi.generator_specs()):
        if kind == 'transforms':
            got = of.from_transforms(arg, shape, r)
            same(of.Flow.from_transforms(arg, shape, r).vecs, g['out_gen_%d' % i])
        else:
            got = of.from_matrix(np.array(arg, dtype=np.float64), shape, r)
        same(got, g['out_gen_%d' % i])
    fb = of.FlowBatch.from_transforms([gi.cfg4_transforms(i) for i in range(3)], (54, 96), 't')
    v, _ = fb.numpy()
    for i in range(3):
        same(v[i], R.from_transforms(gi.cfg4_transforms(i), (54, 96), 't'))


def test_reference_7x7_golden_masks_t_side(of):
    """tests/test_flow_class.py:852-980 of the reference, the cases that sample in 't' direction."""
    g = load_golden('small_masks')
    ft = of.Flow(g['in_vecs_t'], 't')
    fs = of.Flow(g['in_vecs_s'], 's')
    ftm = of.Flow(g['in_vecs_t'], 't', g['in_mask_t'])
    fsm = of.Flow(g['in_vecs_s'], 's', g['in_mask_s'])
    same(ft.valid_target(), g['out_vt_t'])
    same(fs.valid_source(), g['out_vs_s'])
    same(ftm.valid_target(), g['out_vt_t_masked'])
    same(fsm.valid_source(), g['out_vs_s_masked'])
    same(of.Flow.from_transforms([['rotation', 0, 0, 45]], (7, 7), 't').vecs, g['in_vecs_t'])


def test_arithmetic_and_reductions(of):
    rng = np.random.default_rng(15)
    h, w = 30, 52
    a = rng.standard_normal((h, w, 2)).astype(np.float32) * 3
    b = rng.standard_normal((h, w, 2)).astype(np.float32) * 3
    am, bm = rng.random((h, w)) > 0.2, rng.random((h, w)) > 0.2
    fa, fb = of.Flow(a, 't', am), of.Flow(b, 's', bm)
    s = fa + fb
    same(s.vecs, a + b)
    same(s.mask, am & bm)
    assert s.ref == 't'
    d = fa - fb
    same(d.vecs, a - b)
    same((fa + b).vecs, a + b)
    same((fa - b.astype(np.float64)).vecs, (a - b.astype(np.float64)).astype(np.float32))
    same((-fa).vecs, -a)
    same((fa * 2.5).vecs, a * np.float32(2.5))
    same((fa / 3).vecs, a / np.float32(3))
    same((fa * [2, -0.5]).vecs, (a * np.array([2, -0.5])).astype(np.float32))
    same((fa * rng.random((h, w))).mask, am)
    m2 = rng.random((h, w, 2))
    same((fa * m2).vecs, (a * m2).astype(np.float32))
    np.testing.assert_allclose((fa ** 2).vecs, a ** 2, rtol=1e-6)
    with pytest.raises(ValueError):
        fa / 0
    # zero tests (reference: tests/test_flow_class.py:1006-1018, tests/test_utils.py:520-540)
    mask = np.ones((10, 10), bool)
    mask[0, 0] = False
    v = np.zeros((10, 10, 2))
    v[0, 0] = 10
    fz = of.Flow(v, mask=mask)
    assert fz.is_zero() is True and fz.is_zero(masked=True) is True and fz.is_zero(masked=False) is False
    v = np.zeros((10, 10, 2), 'float32')
    assert of.is_zero_flow(v, thresholded=True) and of.is_zero_flow(v, thresholded=False)
    v[:3, :, 0] = 1e-4
    assert of.is_zero_flow(v, thresholded=True) and not of.is_zero_flow(v, thresholded=False)
    v[:3, :, 0] = 1e-2
    assert not of.is_zero_flow(v)
    # points_inside_area (tests/test_utils.py:305-319)
    pts = np.array([[-1, -1], [-1, 0], [0, -1], [0, 0], [9, 20], [9, 19], [10, 19], [4.3, 7.6], [9.4, 19.4],
                    [9.6, 19.4]])
    assert of.points_inside_area(pts, (10, 20)).tolist() == R.points_inside_area(pts, (10, 20)).tolist()
    # cross-reference inversion and slicing
    inv = fa.invert('s')
    same(inv.vecs, -a)
    assert inv.ref == 's'
    cut = fa[3:20, 5:40]
    same(cut.vecs, a[3:20, 5:40])
    same(cut.mask, am[3:20, 5:40])
    same(fa[::2].vecs, a[::2])


def test_host_views_are_live(of):
    """`flow.mask[...] = False` edits the flow in the reference (its arrays are its storage); same here."""
    f = of.Flow.from_transforms([['rotation', 0, 0, 30]], (32, 32), 't')
    f.mask[:, 20:] = False
    assert not f.valid_target()[:, 20:].any()
    f.vecs[...] = 0
    assert f.is_zero(thresholded=False)
    # reading the host views alone does not cost an upload; edits do, once
    g = of.Flow.from_transforms([['rotation', 0, 0, 30]], (32, 32), 't')
    d0 = g._dv
    _ = g.vecs.sum(), g.mask.all()
    g.valid_target()
    assert g._vd() is d0
    g.vecs *= 0.5
    assert g._vd() is not d0
    d1 = g._dv
    g.valid_target()
    assert g._vd() is d1
    with pytest.raises(ValueError):
        g.vecs.fill(0)                                # writers numpy does not let us see fail loudly


def test_constructor_errors(of):
    with pytest.raises(TypeError):
        of.Flow('test')
    with pytest.raises(ValueError):
        of.Flow(np.zeros((10, 10)))
    with pytest.raises(ValueError):
        of.Flow(np.zeros((10, 10, 3)))
    bad = np.zeros((10, 10, 2), np.float32)
    bad[2, 3, 1] = np.nan
    with pytest.raises(ValueError):
        of.Flow(bad)
    with pytest.raises(ValueError):
        of.Flow(bad.astype(np.float64))
    with pytest.raises(ValueError):
        of.Flow(np.zeros((10, 10, 2)), mask=np.ones((10, 11)))
    with pytest.raises(ValueError):
        of.Flow(np.zeros((10, 10, 2)), mask=np.full((10, 10), 2))
    f = of.Flow(np.zeros((10, 10, 2)), 's', np.ones((10, 10)))
    assert f.ref == 's' and f.mask.dtype == bool and f.vecs.dtype == np.float32 and f.shape == (10, 10)
    f2 = of.Flow(np.ones((10, 10, 2)))
    with pytest.raises(ValueError):
        f.combine_with(f2, 3)                # different refs
    with pytest.raises(ValueError):
        f.combine_with(of.Flow(np.ones((10, 10, 2)), 's'), 4)
    with pytest.raises(TypeError):
        f.combine_with(np.ones((10, 10, 2)), 3)
    with pytest.raises(TypeError):
        f2.apply(np.zeros((10, 10)), return_valid_area='test')
    with pytest.raises(ValueError):
        f2.apply(np.zeros((11, 10)))
    with pytest.raises(TypeError):
        f2.apply(np.zeros((10, 10), np.int32))


@pytest.mark.slow
def test_full_size_digests(of):
    """BASELINE.json configurations at full size against SHA-256 digests of the reference's own outputs."""
    dg = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'digests.json')))
    flow, img = gi.cfg1_full()
    assert sha(of.Flow.from_transforms([['rotation', 621, 187.5, 10]], (375, 1242), 't').vecs) == dg['cfg1_flow_sha']
    assert sha(of.apply_flow(flow, img, 't')) == dg['cfg1_apply_flow_u8c3']
    w, m = of.Flow(flow, 't').apply(img, return_valid_area=True)
    assert sha(w) == dg['cfg1_apply_va_u8c3'] and sha(m) == dg['cfg1_apply_va_valid']
    a, am, b, bm = gi.cfg2_full()
    for r in ('t', 's'):
        res = of.Flow(a, r, am).combine_with(of.Flow(b, r, bm), 3)
        assert sha(res.mask) == dg['cfg2_c3_%s_mask' % r]
        assert sha(res.vecs) == dg['cfg2_c3_%s_vecs' % r]
    for idx in (0, 5):
        fa, fam, fb, fbm, img = gi.cfg4_frame(idx)
        w, m = of.Flow(fa, 't', fam).apply(img, return_valid_area=True)
        assert sha(w) == dg['cfg4_f%d_apply_va_u8c3' % idx] and sha(m) == dg['cfg4_f%d_apply_va_valid' % idx]
        res = of.Flow(fa, 't', fam).combine_with(of.Flow(fb, 't', fbm), 3)
        assert sha(res.vecs) == dg['cfg4_f%d_c3_t_vecs' % idx] and sha(res.mask) == dg['cfg4_f%d_c3_t_mask' % idx]
    for r in ('t', 's'):
        assert sha(of.from_transforms(gi.CFG5_TRANSFORMS, gi.CFG5_SHAPE, r)) == dg['cfg5_from_transforms_' + r]
    # cfg 5 chain at 4K, entirely device-resident
    f = of.Flow.from_transforms(gi.CFG5_TRANSFORMS, gi.CFG5_SHAPE, 't')
    g_ = f.invert('s')
    g_ = of.Flow(g_.vecs_device, 't', g_.mask_device)
    acc = f
    for i in range(4):
        acc = acc.combine_with(g_ if i % 2 == 0 else f, 3)
    w, m = acc.apply(gi.cfg5_image(), return_valid_area=True)
    assert sha(acc.vecs) == dg['cfg5_chain_vecs'] and sha(acc.mask) == dg['cfg5_chain_mask']
    assert sha(w) == dg['cfg5_chain_img'] and sha(m) == dg['cfg5_chain_valid']


def test_gather_kernel_fallback_parity():
    """The register-pipelined gather kernel behind ofk_combine3 (what runs for widths that are not multiples of 16)
    forced for every shape with OFK_C3_WS=0 (read once per process), against the oracle."""
    import subprocess
    import sys
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import oflibnumpy_b200 as of
from oracle import flowref as R
rng = np.random.default_rng(21)
for (h, w, amp) in ((40, 64, 10), (96, 160, 10), (96, 160, 60), (64, 48, 3), (33, 16, 200), (70, 128, 25), (130, 96, 6)):
    a = (rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(amp)
    b = (rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(amp)
    am, bm = rng.random((h, w)) > 0.1, rng.random((h, w)) > 0.1
    for r in ('t', 's'):
        got = of.Flow(a, r, am).combine_with(of.Flow(b, r, bm), 3)
        want = R.combine(R.make(a, r, am), R.make(b, r, bm), 3)
        assert np.array_equal(got.mask, want.mask), (h, w, amp, r)
        assert np.array_equal(got.vecs, want.vecs), (h, w, amp, r)
        got = of.combine_flows(a, b, 3, r)
        assert np.array_equal(got, R.combine(R.make(a, r), R.make(b, r), 3).vecs), (h, w, amp, r, 'nomask')
n = 6
a = (rng.random((n, 64, 96, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(8)
b = (rng.random((n, 64, 96, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(8)
am, bm = rng.random((n, 64, 96)) > 0.05, rng.random((n, 64, 96)) > 0.05
a[1] = 0
b[2][bm[2]] = 0
v, m = of.FlowBatch(a, 't', am).combine_with(of.FlowBatch(b, 't', bm), 3).numpy()
for i in range(n):
    want = R.combine(R.make(a[i], 't', am[i]), R.make(b[i], 't', bm[i]), 3)
    assert np.array_equal(m[i], want.mask) and np.array_equal(v[i], want.vecs), i
print("fallback parity ok")
''' % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, OFK_C3_WS='0')
    res = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    assert 'fallback parity ok' in res.stdout


def _smooth_flow(rng, h, w, amp):
    """Affine (rotation / scale / shear / translation) + low-frequency ripple + a little noise: the regime of the TMA
    kernels' box estimate (mostly covered) with pixels that escape it (noise, borders)."""
    yy, xx = np.mgrid[:h, :w].astype(np.float32)
    a = rng.uniform(-0.15, 0.15, 4).astype(np.float32)
    t = rng.uniform(-amp, amp, 2).astype(np.float32)
    u = a[0] * (xx - w / 2) + a[1] * (yy - h / 2) + t[0] + 2 * np.sin(xx / 9 + rng.uniform(0, 6)) * np.cos(yy / 7)
    v = a[2] * (xx - w / 2) + a[3] * (yy - h / 2) + t[1] + 2 * np.cos(xx / 8) * np.sin(yy / 11 + rng.uniform(0, 6))
    f = np.stack([u, v], -1).astype(np.float32)
    f += (rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * np.float32(rng.choice([0, 0.5, 3]))
    if rng.random() < 0.3:                                   # a few wild vectors far outside any box / the frame
        idx = rng.integers(0, h * w, 5)
        f.reshape(-1, 2)[idx] = rng.uniform(-5000, 5000, (5, 2)).astype(np.float32)
    return f


def test_tma_kernels_randomized(of):
    """Randomised shapes (W % 16 == 0, partial tiles in both directions), batches and flow regimes through every
    variant of the warp-specialised TMA kernels -- composition with / without masks, both references; image warp with
    fixed-point / round-half-even arithmetic, no / geometric / resampled validity, with and without a flow mask; a flow
    warped by a flow -- against the oracle, bit for bit, and twice (the kernels are pipelines of asynchronous copies:
    results must not depend on timing)."""
    from oflibnumpy_b200 import _lib
    lib = _lib.load()
    before = [lib.ofk_rt_path_count(k) for k in range(4)]
    rng = np.random.default_rng(77)
    shapes = [(1, 16), (5, 32), (31, 48), (32, 32), (33, 64), (47, 80), (64, 96), (70, 144), (97, 208), (130, 256)]
    for k, (h, w) in enumerate(shapes):
        n = int(rng.integers(1, 4))
        amp = float(rng.choice([1.5, 12, 40]))
        a = np.stack([_smooth_flow(rng, h, w, amp) for _ in range(n)])
        b = np.stack([_smooth_flow(rng, h, w, amp) for _ in range(n)])
        am, bm = rng.random((n, h, w)) > 0.1, rng.random((n, h, w)) > 0.1
        img = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
        for r in ('t', 's'):
            for rep in range(2):
                v, m = of.FlowBatch(a, r, am).combine_with(of.FlowBatch(b, r, bm), 3).numpy()
                for i in range(n):
                    want = R.combine(R.make(a[i], r, am[i]), R.make(b[i], r, bm[i]), 3)
                    same(m[i].view(np.bool_), want.mask)
                    same(v[i], want.vecs)
            got = of.combine_flows(a[0], b[0], 3, r)
            same(got, R.combine(R.make(a[0], r), R.make(b[0], r), 3).vecs)
        for i in range(n):
            fa = of.Flow(a[i], 't', am[i])
            ra = R.make(a[i], 't', am[i])
            for rep in range(2):
                same(fa.apply(img[i]), R.apply(ra, img[i]))                                    # fixed point, no mask
                w1, m1 = fa.apply(img[i], return_valid_area=True)                              # half-even, geometry
                w2, m2 = R.apply(ra, img[i], return_valid_area=True)
                same(w1, w2)
                same(m1, m2)
                w1, m1 = fa.apply(img[i], target_mask=bm[i], return_valid_area=True)           # resampled mask
                w2, m2 = R.apply(ra, img[i], target_mask=bm[i], return_valid_area=True)
                same(w1, w2)
                same(m1, m2)
                w1, m1 = fa.apply(img[i], return_valid_area=True, consider_mask=False)         # no flow mask
                w2, m2 = R.apply(ra, img[i], return_valid_area=True, consider_mask=False)
                same(w1, w2)
                same(m1, m2)
                for chans in (0, 1, 4):                                                        # grey (2-D), 1 and 4 channels
                    im = img[i, ..., 0] if chans == 0 else np.ascontiguousarray(
                        np.concatenate([img[i], img[i][..., :1]], -1)[..., :chans])
                    same(fa.apply(im), R.apply(ra, im))
                    w1, m1 = fa.apply(im, return_valid_area=True)
                    w2, m2 = R.apply(ra, im, return_valid_area=True)
                    same(w1, w2)
                    same(m1, m2)
                    w1, m1 = fa.apply(im, target_mask=bm[i], return_valid_area=True)
                    w2, m2 = R.apply(ra, im, target_mask=bm[i], return_valid_area=True)
                    same(w1, w2)
                    same(m1, m2)
                res = fa.apply(of.Flow(b[i], 't', bm[i]))                                      # flow warped by flow
                want = R.apply(ra, R.make(b[i], 't', bm[i]))
                same(res.mask, want.mask)
                same(res.vecs, want.vecs)
    after = [lib.ofk_rt_path_count(k) for k in range(4)]
    # every call above is eligible for the TMA kernels (W % 16 == 0, pool allocations are 256-byte aligned)
    assert after[0] > before[0] and after[2] > before[2]
    assert after[1] == before[1] and after[3] == before[3], (before, after)


def _rough_flow(rng, h, w, kind):
    """Flows whose 32 x 32 tiles do not fit one 48 x 48 box: motion boundaries and white noise."""
    if kind == 'blocks':
        bs = int(rng.choice([7, 20, 50]))
        by, bx = (h + bs - 1) // bs, (w + bs - 1) // bs
        mot = rng.uniform(-25, 25, (by, bx, 2)).astype(np.float32)
        return np.ascontiguousarray(np.repeat(np.repeat(mot, bs, 0), bs, 1)[:h, :w])
    amp = np.float32(rng.choice([8, 30, 200]))
    return ((rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * (2 * amp)).astype(np.float32)


def test_tma_kernels_discontinuous_and_noisy_flows(of):
    """Motion boundaries and noise: most pixels of a tile lie outside the tile's box and fetch their taps from global
    memory (the out-of-line path of the TMA kernels). Every kernel variant, against the oracle, bit for bit, twice."""
    from oflibnumpy_b200 import _lib
    lib = _lib.load()
    before = [lib.ofk_rt_path_count(k) for k in range(6)]
    rng = np.random.default_rng(4242)
    for (h, w), kind in (((70, 144), 'blocks'), ((97, 208), 'noise'), ((130, 256), 'blocks'), ((64, 96), 'noise')):
        n = 2
        a = np.stack([_rough_flow(rng, h, w, kind) for _ in range(n)])
        b = np.stack([_rough_flow(rng, h, w, kind) for _ in range(n)])
        am, bm = rng.random((n, h, w)) > 0.1, rng.random((n, h, w)) > 0.1
        img = rng.integers(0, 256, (n, h, w, 4), dtype=np.uint8)
        for r in ('t', 's'):
            for rep in range(2):
                v, m = of.FlowBatch(a, r, am).combine_with(of.FlowBatch(b, r, bm), 3).numpy()
                for i in range(n):
                    want = R.combine(R.make(a[i], r, am[i]), R.make(b[i], r, bm[i]), 3)
                    same(m[i].view(np.bool_), want.mask)
                    same(v[i], want.vecs)
            same(of.combine_flows(a[0], b[0], 3, r), R.combine(R.make(a[0], r), R.make(b[0], r), 3).vecs)
        for i in range(n):
            fa, ra = of.Flow(a[i], 't', am[i]), R.make(a[i], 't', am[i])
            for rep in range(2):
                for chans in (0, 1, 3, 4):
                    im = img[i, ..., 0] if chans == 0 else np.ascontiguousarray(img[i, ..., :chans])
                    same(fa.apply(im), R.apply(ra, im))
                    for kw in ({}, {'target_mask': bm[i]}, {'consider_mask': False}):
                        w1, m1 = fa.apply(im, return_valid_area=True, **kw)
                        w2, m2 = R.apply(ra, im, return_valid_area=True, **kw)
                        same(w1, w2)
                        same(m1, m2)
                res = fa.apply(of.Flow(b[i], 't', bm[i]))
                want = R.apply(ra, R.make(b[i], 't', bm[i]))
                same(res.mask, want.mask)
                same(res.vecs, want.vecs)
    after = [lib.ofk_rt_path_count(k) for k in range(6)]
    assert after[0] > before[0] and after[2] > before[2]
    assert after[1] == before[1] and after[3] == before[3], (before, after)
    # ... and inside them, warps did fetch taps from global memory (counters 4 / 5: composition / image kernels)
    assert after[4] > before[4] and after[5] > before[5], (before, after)


_FULL_SIZE_CODE = r'''
import sys, hashlib, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import oflibnumpy_b200 as of
import test_gpu_warp_t as t
rng = np.random.default_rng(99)
h, w, n = 1080, 1920, 3
a = np.stack([t._rough_flow(rng, h, w, k) for k in ('blocks', 'noise', 'blocks')])
b = np.stack([t._rough_flow(rng, h, w, k) for k in ('noise', 'blocks', 'blocks')])
a[2] += t._smooth_flow(rng, h, w, 12)
am, bm = rng.random((n, h, w)) > 0.02, rng.random((n, h, w)) > 0.02
img = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
out = []
for r in ('t', 's'):
    v, m = of.FlowBatch(a, r, am).combine_with(of.FlowBatch(b, r, bm), 3).numpy()
    out += [v, m]
fb = of.FlowBatch(a, 't', am)
res = fb.apply(img, return_valid_area=True)
out += [x.numpy() for x in res]
out += [x.numpy() for x in fb.apply(np.ascontiguousarray(img[..., 0]), target_masks=bm, return_valid_area=True)]
print('DIGEST', hashlib.sha256(b''.join(np.ascontiguousarray(x).tobytes() for x in out)).hexdigest())
'''


def test_full_size_tma_and_gather_kernels_agree_on_rough_flows():
    """Size-independent property at 1080p: the TMA kernels (with their out-of-line global-tap path) and the gather
    kernels are independent implementations of the same arithmetic -- on motion boundaries and noise, where most of a
    tile lies outside its box, their outputs must be byte-identical (composition both references, image warp with
    geometric and resampled validity)."""
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    code = _FULL_SIZE_CODE % (os.path.dirname(here), here)
    digests = []
    for env_extra in ({}, {'OFK_C3_WS': '0', 'OFK_WARP_WS': '0'}):
        res = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, **env_extra), capture_output=True,
                             text=True, timeout=900)
        assert res.returncode == 0, res.stdout + res.stderr
        digests.append([l for l in res.stdout.splitlines() if l.startswith('DIGEST')][0])
    assert digests[0] == digests[1]


def test_tma_kernels_long_pipelines():
    """The same randomised parity suite with the persistent grids capped at 3 CTAs (OFK_WS_MAX_CTAS, read once per
    process): every CTA then walks through dozens of tiles, so the stage rings wrap around and every barrier phase flips
    many times -- the regime of the full-size batches, at test-size cost."""
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import oflibnumpy_b200 as of\n"
            "import test_gpu_warp_t as t\n"
            "t.test_tma_kernels_randomized(of)\n"
            "t.test_tma_kernels_discontinuous_and_noisy_flows(of)\n"
            "t.test_zero_test_probe_and_scan(of)\n"
            "t.test_batched_equals_per_frame(of)\n"
            "print('long pipelines ok')\n") % (os.path.dirname(here), here)
    env = dict(os.environ, OFK_WS_MAX_CTAS='3')
    res = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr
    assert 'long pipelines ok' in res.stdout


def test_combine_flows_integer_shift_over_the_border(of):
    """combine_flows (no masks) with integer-valued flows: sample positions with zero fractions on and beyond the
    right / bottom border. A tap with zero weight never matters, but the tap that carries the whole weight must lie
    inside the frame (found by examples/abi_example.c: the TMA kernel accepted ix >= W when the fraction was 0)."""
    for (h, w) in ((48, 64), (40, 70)):              # TMA kernel / gather kernel
        for (dx, dy) in ((7, -4), (-3, 5), (w, 0), (0, h), (w - 1, h - 1)):
            a = np.zeros((h, w, 2), np.float32)
            a[..., 0], a[..., 1] = dx, dy
            b = -a
            for r in ('t', 's'):
                got = of.Flow(a, r).combine_with(of.Flow(b, r), 3)
                want = R.combine(R.make(a, r), R.make(b, r), 3)
                same(got.mask, want.mask)
                same(got.vecs, want.vecs)
                same(of.combine_flows(a, b, 3, r), want.vecs)


def test_integer_and_half_pixel_shifts_over_the_border(of):
    """Every target-referenced kernel on constant flows whose sample positions have zero or one-half fractions and run
    over each border by less than, exactly, and more than one pixel: the cases where "the tap that carries weight" and
    "the tap that does not" sit on opposite sides of the frame edge."""
    rng = np.random.default_rng(5)
    for (h, w) in ((48, 64), (37, 50)):              # TMA kernels / gather kernels
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        tmask = rng.random((h, w)) > 0.2
        other = of.Flow((rng.random((h, w, 2)).astype(np.float32) - np.float32(0.5)) * 6, 't', rng.random((h, w)) > 0.1)
        ro = R.make(other.vecs, 't', other.mask)
        for (dx, dy) in ((0.5, 0), (-0.5, 0.5), (1, 1), (-1, 0), (w - 1, 0), (w - 0.5, 0), (w, 0), (0, h - 1), (0, h),
                         (-(w - 1), -(h - 1)), (-w, 1.5), (3.5, -(h - 0.5))):
            v = np.zeros((h, w, 2), np.float32)
            v[..., 0], v[..., 1] = dx, dy
            f, rf = of.Flow(v, 't'), R.make(v, 't')
            same(f.valid_target(), R.valid_target(rf))
            same(of.Flow(v, 's').valid_source(), R.valid_source(R.make(v, 's')))
            for im in (img, img[..., 0], np.ascontiguousarray(np.concatenate([img, img[..., :1]], -1))):
                same(f.apply(im), R.apply(rf, im))
                for tm in (None, tmask):
                    w1, m1 = f.apply(im, target_mask=tm, return_valid_area=True)
                    w2, m2 = R.apply(rf, im, target_mask=tm, return_valid_area=True)
                    same(w1, w2)
                    same(m1, m2)
            res, want = f.apply(other), R.apply(rf, ro)
            same(res.mask, want.mask)
            same(res.vecs, want.vecs)


def test_dataset_constructors_decode_on_device(of):
    """Flow.from_kitti / Flow.from_sintel (device decoders ofk_decode_kitti / ofk_decode_sintel_mask) against the
    reference's constructors on the committed sample files."""
    g = load_golden('datasets')
    files = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'files')
    kp, sp, ip = (os.path.join(files, n) for n in ('kitti_sample.png', 'sintel_sample.flo', 'sintel_invalid.png'))
    flow_same(g, 'kitti_valid', of.Flow.from_kitti(kp))
    flow_same(g, 'kitti_novalid', of.Flow.from_kitti(kp, load_valid=False))
    flow_same(g, 'sintel', of.Flow.from_sintel(sp))
    flow_same(g, 'sintel_masked', of.Flow.from_sintel(sp, ip))
    with pytest.raises(TypeError):
        of.Flow.from_kitti(kp, load_valid='yes')
    with pytest.raises(ValueError):
        of.Flow.from_kitti(sp)


def test_visualise_matches_reference_and_oracle(of):
    """Flow.visualise on the device (ofk_visualise_batch of one frame) against the reference's own
    outputs (tests/golden/visualise.npz) and, at 1080p, against the oracle: uint8 images, bit for bit -- hue from the
    same FMA polynomial as cv2.cartToPolar, default range from an exact radix selection of the 99th percentile."""
    from test_oracle_golden import VIS_VARIANTS
    g = load_golden('visualise')
    for name in ('swirl', 'sparse', 'zero'):
        f = of.Flow(g['in_' + name], 't', g['in_mask'])
        for key, kw in VIS_VARIANTS:
            same(f.visualise(key.split('_')[0], **kw), g['out_%s_%s' % (name, key)])
    rng = np.random.default_rng(12)
    h, w = 1080, 1920
    yy, xx = np.mgrid[:h, :w].astype(np.float32)
    v = np.stack([8 * np.sin(xx / 40) * np.cos(yy / 55) + 0.002 * (xx - w / 2),
                  6 * np.cos(xx / 35 + 1) * np.sin(yy / 45) - 0.003 * (yy - h / 2)], -1).astype(np.float32)
    v += rng.standard_normal((h, w, 2)).astype(np.float32) * np.float32(0.05)
    m = rng.random((h, w)) > 0.02
    f, r = of.Flow(v, 's', m), R.make(v, 's', m)
    for key, kw in VIS_VARIANTS:
        same(f.visualise(key.split('_')[0], **kw), R.visualise(r, key.split('_')[0], **kw))
    with pytest.raises(ValueError):
        f.visualise('xyz')
    with pytest.raises(TypeError):
        f.visualise('rgb', show_mask=1)
    with pytest.raises(ValueError):
        f.visualise('rgb', range_max=0)


def test_large_pageable_copies_are_staged_correctly(of):
    """Copies of plain numpy arrays from 4 MB up go through worker threads and pinned pieces (staging.cu): byte-exact
    round trips for sizes around the piece / lane boundaries, source reusable right after the upload returns, and
    ordering against kernels on the same stream."""
    from oflibnumpy_b200.device import DeviceArray
    rng = np.random.default_rng(8)
    mb = 1 << 20
    for nbytes in (mb - 1, mb, mb + 1, 2 * mb + 4097, 4 * mb - 1, 6 * mb - 3, 8 * mb + 1, 16 * mb, 37 * mb + 5, 4 * 2 * mb * 3 + 17):
        a = rng.integers(0, 256, nbytes, dtype=np.uint8)
        keep = a.copy()
        d = DeviceArray.from_numpy(a)
        a[:] = 0                                              # the upload has read its source when it returns
        back = d.numpy()
        assert back.shape == keep.shape and np.array_equal(back, keep), nbytes
    # back-to-back uploads: the pinned pieces of one transfer may still be in flight when the next one starts
    arrays = [rng.integers(0, 256, int(n), dtype=np.uint8) for n in (9 * mb + 7, 20 * mb, 5 * mb + 1, 33 * mb, 6 * mb, 12 * mb)]
    for rep in range(3):
        devs = [DeviceArray.from_numpy(a) for a in arrays]
        for a, d in zip(arrays, devs):
            assert np.array_equal(d.numpy(), a)
    h, w = 1500, 2048                                          # 24.6 MB of vectors: staged both ways around a kernel
    v = rng.standard_normal((h, w, 2)).astype(np.float32)
    f = of.Flow(v, 't')
    g = f + f
    assert np.array_equal(g.vecs, v + v)
    assert np.array_equal((g - f).vecs, (v + v) - v)


def test_functional_api_rejects_non_finite_flows(of):
    """NaN / Inf in a flow array raise ValueError with the reference's message (utils.py:55-56); float32 arrays are
    tested on the device after the upload, other dtypes on the host before the cast (1e300 is finite as float64)."""
    img = np.zeros((64, 64, 3), np.uint8)
    for bad in (np.nan, np.inf, -np.inf):
        f = np.zeros((64, 64, 2), np.float32)
        f[3, 4, 1] = bad
        for fn in (lambda: of.apply_flow(f, img, 't'), lambda: of.is_zero_flow(f), lambda: of.resize_flow(f, 2),
                   lambda: of.apply_flow(f.astype(np.float64), img, 't'), lambda: of.Flow(f)):
            with pytest.raises(ValueError, match="NaN"):
                fn()
    big = np.zeros((64, 64, 2), np.float64)
    big[0, 0, 0] = 1e300                                   # finite before the cast: accepted, as in the reference
    with np.errstate(over='ignore'):
        of.is_zero_flow(big)


def test_rough_full_size_flows_repeat_exactly(of):
    """Regression for a release-before-read race in the out-of-line path of the TMA kernels (a box stage was handed
    back to the producer before the last shared-memory taps of a warp had been read: a handful of wrong pixels in one
    tile row of one launch in five). 1080p motion boundaries + noise, both references and the image warp, 15 launches
    each: the first is compared with the oracle, all must be byte-identical."""
    rng = np.random.default_rng(99)
    h, w, n = 1080, 1920, 2
    a = np.stack([_rough_flow(rng, h, w, k) for k in ('blocks', 'noise')])
    b = np.stack([_rough_flow(rng, h, w, k) for k in ('noise', 'blocks')])
    am, bm = rng.random((n, h, w)) > 0.02, rng.random((n, h, w)) > 0.02
    img = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    first = {}
    for rep in range(15):
        for r in ('t', 's'):
            v, m = of.FlowBatch(a, r, am).combine_with(of.FlowBatch(b, r, bm), 3).numpy()
            if rep == 0:
                for i in range(n):
                    want = R.combine(R.make(a[i], r, am[i]), R.make(b[i], r, bm[i]), 3)
                    same(m[i].view(np.bool_), want.mask)
                    same(v[i], want.vecs)
                first[r] = (v, m)
            else:
                assert np.array_equal(v, first[r][0]) and np.array_equal(m, first[r][1]), (rep, r)
        wi, wm = (x.numpy() for x in of.FlowBatch(a, 't', am).apply(img, return_valid_area=True))
        if rep == 0:
            for i in range(n):
                w2, m2 = R.apply(R.make(a[i], 't', am[i]), img[i], return_valid_area=True)
                same(wi[i], w2)
                same(wm[i].view(np.bool_), m2)
            first['img'] = (wi, wm)
        else:
            assert np.array_equal(wi, first['img'][0]) and np.array_equal(wm, first['img'][1]), rep


def test_batches_beyond_4_gib(of):
    """Maximum sizes: batches whose tensors exceed 2^32 bytes (300 x 1080p flows = 5 GB per operand for the composition,
    700 frames = 11.6 GB of flows and 4.4 GB of images for the warp). Frames at the start, in the middle and at the end
    must equal the same frame processed alone (small offsets): 64-bit addressing in the tensor maps, the tile iterators
    and the global-tap path."""
    from oflibnumpy_b200 import _lib, _ops
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    h, w = 1080, 1920
    rng = np.random.default_rng(3)
    st = of.device.current_stream()

    def flows(n, seed0):
        mats = np.stack([np.linalg.pinv(R.matrix_from_transforms(gi.cfg4_transforms(seed0 + i))) for i in range(n)])
        v = _ops.from_matrix(DeviceArray.from_numpy(mats), (h, w), -1.0)
        m = DeviceArray.empty((n, h, w), np.uint8)
        _lib.call('ofk_rt_memset', m.ptr, 1, m.nbytes, st)
        for i in (0, n // 2 + 7, n - 1):                       # some invalid pixels in the frames that are checked
            mk = (rng.random((1, h, w)) > 0.03).astype(np.uint8)
            fr = m.frames(i, i + 1)
            _lib.call('ofk_rt_memcpy_h2d', fr.ptr, mk.ctypes.data, mk.nbytes, st)
            of.device.synchronize()
        return FlowBatch._wrap(v, 't', m)

    n = 300
    fa, fb = flows(n, 0), flows(n, 5000)
    assert fa.vecs.nbytes > (1 << 32)
    res = fa.combine_with(fb, 3)
    for i in (0, n // 2 + 7, n - 1):
        one = FlowBatch._wrap(fa.vecs.frames(i, i + 1), 't', fa.masks.frames(i, i + 1)).combine_with(
            FlowBatch._wrap(fb.vecs.frames(i, i + 1), 't', fb.masks.frames(i, i + 1)), 3)
        same(res.vecs.frames(i, i + 1).numpy(), one.vecs.numpy())
        same(res.masks.frames(i, i + 1).numpy(), one.masks.numpy())
    del res, fb, fa
    n = 700
    fa = flows(n, 9000)
    imgs = DeviceArray.empty((n, h, w, 3), np.uint8)
    assert imgs.nbytes > (1 << 32)
    pool = rng.integers(0, 256, (4, 1, h, w, 3), dtype=np.uint8)
    for i in range(n):
        fr = imgs.frames(i, i + 1)
        _lib.call('ofk_rt_memcpy_h2d', fr.ptr, pool[i % 4].ctypes.data, pool[i % 4].nbytes, st)
    of.device.synchronize()
    out, valid = fa.apply(imgs, return_valid_area=True)
    for i in (0, n // 2 + 7, n - 1):
        one = FlowBatch._wrap(fa.vecs.frames(i, i + 1), 't', fa.masks.frames(i, i + 1)).apply(imgs.frames(i, i + 1),
                                                                                               return_valid_area=True)
        same(out.frames(i, i + 1).numpy(), one[0].numpy())
        same(valid.frames(i, i + 1).numpy(), one[1].numpy())


def test_host_buffer_api_with_plain_numpy_batches(of):
    """ofh_warp_t / ofh_combine3 on pageable numpy arrays at 1080p: uploads and downloads of the ring go through the
    staged copies (worker threads + pinned pieces), downloads trail the launches by one chunk. Same bytes as the device
    API, flags included."""
    from oflibnumpy_b200.batch import FlowBatch
    rng = np.random.default_rng(17)
    n, h, w = 5, 1080, 1920
    a = np.stack([_smooth_flow(rng, h, w, 20) for _ in range(n)])
    b = np.stack([_smooth_flow(rng, h, w, 20) for _ in range(n)])
    b[3] = 0                                                  # a zero operand: the early-exit flags must come back
    am, bm = rng.random((n, h, w)) > 0.02, rng.random((n, h, w)) > 0.02
    img = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    for rep in range(2):
        wi, wv = of.batch.apply_flow_host(a, img, flow_masks=am, return_valid_area=True)
        d_i, d_v = FlowBatch(a, 't', am).apply(img, return_valid_area=True)
        same(wi, d_i.numpy())
        same(wv.view(np.uint8), d_v.numpy())
        v, m = of.batch.combine_flows_host(a, b, 3, 't', am, bm)
        dv, dm = FlowBatch(a, 't', am).combine_with(FlowBatch(b, 't', bm), 3).numpy()
        same(v, dv)
        same(m.view(np.uint8), dm.view(np.uint8))


def test_host_buffer_apply_combine3_and_flags(of):
    """ofh_apply_combine3 (batch.apply_combine_host) and the flags of ofh_combine3 / ofh_apply_combine3 give the bytes
    of the device API: ref 't' and 's', with and without masks, pageable and pinned buffers, at one frame per chunk
    (1080p: slots are reused, the last download trails) and at several frames per chunk with a short last chunk
    (540x960). The ref 's' image warp samples at p + A[p], i.e. it is FlowBatch(-A, 't').apply."""
    from oflibnumpy_b200 import _lib, _ops
    from oflibnumpy_b200.batch import FlowBatch
    rng = np.random.default_rng(23)
    n, device = 5, of.device.get_device()

    def u8(x):
        return x.view(np.uint8) if x.dtype == np.bool_ else x

    def ptr(x):
        return None if x is None else x.ctypes.data

    def pinned_copy(x, keep):
        if x is None:
            return None
        p, handle = of.device.pinned_empty(x.shape, x.dtype)
        keep.append(handle)
        p[...] = x
        return p

    for h, w in ((1080, 1920), (540, 960)):
        a = np.stack([_smooth_flow(rng, h, w, 20) for _ in range(n)])
        b = np.stack([_smooth_flow(rng, h, w, 20) for _ in range(n)])
        a[1] = 0                                              # zero operands: the early-exit flags must come back
        b[3] = 0
        img = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
        arith, rule = _ops.promoted_rule(img.dtype, False)
        for masked in (True, False):
            am, bm = (rng.random((n, h, w)) > 0.02, rng.random((n, h, w)) > 0.02) if masked else (None, None)
            for r in ('t', 's'):
                d_img, d_valid = FlowBatch(a if r == 't' else -a, 't', am).apply(img, return_valid_area=True)
                res, d_flags = FlowBatch(a, r, am).combine_with(FlowBatch(b, r, bm), 3, return_flags=True)
                want = (d_img.numpy(), d_valid.numpy(), *res.numpy())
                want_flags = d_flags.numpy()
                assert (want_flags[1, 0], want_flags[3, 1]) == (0, 0) and want_flags[0].all()
                for pinned in (False, True):
                    ins, outs, keep = (a, b, img, am, bm), [np.empty_like(x) for x in want], []
                    if pinned:
                        ins, outs = [pinned_copy(x, keep) for x in ins], [pinned_copy(x, keep) for x in outs]
                    got = of.batch.apply_combine_host(ins[0], ins[1], ins[2], r, ins[3], ins[4], out_images=outs[0],
                                                      out_valid=outs[1].view(np.bool_), out=outs[2],
                                                      out_masks=outs[3])
                    for g, x in zip(got, want):
                        same(u8(g), u8(x))
                # flags and outputs of direct calls into plain numpy buffers; out_valid = NULL once
                v, m, flags = np.empty_like(a), np.empty((n, h, w), np.bool_), np.full((n, 2), -1, np.int32)
                _lib.call('ofh_combine3', a.ctypes.data, ptr(am), b.ctypes.data, ptr(bm), ord(r), 0.0, v.ctypes.data,
                          m.ctypes.data, flags.ctypes.data, n, h, w, device)
                for g, x in zip((v, m, flags), want[2:] + (want_flags,)):
                    same(u8(g), u8(x))
                o_img, v, m, flags = np.empty_like(img), np.empty_like(a), np.empty((n, h, w), np.bool_), \
                    np.full((n, 2), -1, np.int32)
                _lib.call('ofh_apply_combine3', img.ctypes.data, _ops.dtype_code(img.dtype), 3, arith, rule,
                          a.ctypes.data, ptr(am), b.ctypes.data, ptr(bm), ord(r), 0.0, o_img.ctypes.data, None,
                          v.ctypes.data, m.ctypes.data, flags.ctypes.data, n, h, w, device)
                for g, x in zip((o_img, v, m, flags), (want[0],) + want[2:] + (want_flags,)):
                    same(u8(g), u8(x))
        _lib.call('ofh_release')                              # the next size starts from a fresh ring


def test_torch_cuda_tensors_pass_through_zero_copy(of):
    """Optional PyTorch interop (north star): torch.cuda tensors are adopted through __cuda_array_interface__ without
    a copy -- as flow vectors / masks of Flow and FlowBatch -- and results are exported the same way."""
    torch = pytest.importorskip('torch')
    if not torch.cuda.is_available():
        pytest.skip('torch sees no GPU')
    h, w = 96, 160
    rng = np.random.default_rng(3)
    vecs = (rng.random((h, w, 2)).astype(np.float32) - 0.5) * 6
    mask = rng.random((h, w)) > 0.1
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    tv = torch.from_numpy(vecs).cuda()
    tm = torch.from_numpy(mask.view(np.uint8)).cuda()
    torch.cuda.synchronize()
    f_t = of.Flow(tv, 't', tm)
    assert f_t.vecs_device.ptr == tv.data_ptr() and f_t.mask_device.ptr == tm.data_ptr()      # adopted, not copied
    f_n = of.Flow(vecs, 't', mask)
    a, va = f_t.apply(img, return_valid_area=True)
    b, vb = f_n.apply(img, return_valid_area=True)
    assert np.array_equal(a, b) and np.array_equal(va, vb)
    c_t, c_n = f_t.combine_with(f_n, 3), f_n.combine_with(f_n, 3)
    assert np.array_equal(c_t.vecs, c_n.vecs) and np.array_equal(c_t.mask, c_n.mask)
    # export: a torch view of the result's device storage, no copy
    out = torch.as_tensor(c_t.vecs_device, device='cuda')
    assert out.data_ptr() == c_t.vecs_device.ptr
    assert np.array_equal(out.cpu().numpy(), c_n.vecs)
    # batch container
    fb = of.FlowBatch(torch.stack([tv, tv]), 't', torch.stack([tm, tm]))
    r = fb.combine_with(fb, 3)
    assert np.array_equal(r.vecs.numpy()[1], c_n.vecs)


def test_matrix_delegates_to_the_reference_on_a_host_copy(of, monkeypatch):
    """Flow.matrix (OpenCV's robust estimators, SURVEY section 2 row 19: out of the hot path) runs on the reference package
    with a host copy of the flow. A stand-in for the package receives the copy (vectors, reference and mask unchanged)
    and the arguments; OpenCV's estimator on that copy, called as the reference's Flow.matrix calls it, recovers the
    generating transform."""
    import sys
    import types
    import cv2
    made, calls = [], []

    class RefFlow:
        def __init__(self, vecs, ref, mask):
            self.vecs, self.ref, self.mask = vecs, ref, mask
            made.append(self)

        def matrix(self, dof, method, masked):
            calls.append(('matrix', dof, method, masked))
            grid = np.stack(np.mgrid[:self.vecs.shape[0], :self.vecs.shape[1]], axis=-1)[..., ::-1]
            src, dst = (grid - self.vecs, grid) if self.ref == 't' else (grid, grid + self.vecs)
            keep = self.mask if masked in (None, True) else np.ones(self.mask.shape, bool)
            est = {4: cv2.estimateAffinePartial2D, 6: cv2.estimateAffine2D}[dof]
            m = est(src[keep].astype(np.float32), dst[keep].astype(np.float32),
                    method={'ransac': cv2.RANSAC, 'lmeds': cv2.LMEDS}[method])[0]
            return np.vstack((m, [0, 0, 1]))

        def visualise_arrows(self, *args):
            calls.append(('visualise_arrows',) + args)
            return np.zeros(self.vecs.shape[:2] + (3,), np.uint8)

    stand_in = types.ModuleType('oflibnumpy')
    stand_in.Flow = RefFlow
    monkeypatch.setitem(sys.modules, 'oflibnumpy', stand_in)
    tr = [['rotation', 30, 20, 12], ['translation', 4.5, -3.0]]
    mask = np.ones((60, 80), bool)
    mask[10:20, 30:50] = False
    f = of.Flow(of.Flow.from_transforms(tr, (60, 80), 's').vecs, 's', mask)
    m = f.matrix(dof=4, method='ransac')
    np.testing.assert_allclose(m, of.matrix_from_transforms(tr), atol=1e-3)
    assert calls[-1] == ('matrix', 4, 'ransac', None)
    copy = made[-1]
    assert copy.ref == 's' and isinstance(copy.vecs, np.ndarray) and isinstance(copy.mask, np.ndarray)
    same(copy.vecs, f.vecs)
    same(copy.mask, mask)
    assert of.get_flow_matrix(f.vecs, 's', dof=6, method='lmeds').shape == (3, 3)
    assert calls[-1] == ('matrix', 6, 'lmeds', False)
    assert f.visualise_arrows(grid_dist=10).shape == (60, 80, 3)
    assert calls[-1] == ('visualise_arrows', 10, None, None, None, None, None, None)
    assert of.visualise_flow(f.vecs, 'bgr').shape == (60, 80, 3)


def test_resampled_mask_where_the_image_box_reaches_beyond_the_estimate(of):
    """The producer sizes the source box of a tile from 16 sampled pixels; pixels between the samples may land anywhere
    inside the (wider) image box. Every such pixel must find its four mask taps inside the mask box as well: with a
    64-byte mask box whose start is rounded down to 16 pixels the right-most 4 pixels of the image box were not
    covered when the first needed pixel sat at 12..15 (mod 16) -- the mask box is 80 wide since. Translations over all
    16 alignments, with outliers placed off the sample grid that push single pixels to both ends of the image box;
    image, resampled validity and geometric validity against the oracle, bit for bit."""
    rng = np.random.default_rng(123)
    h, w = 96, 256
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    tmask = rng.random((h, w)) > 0.3
    fmask = rng.random((h, w)) > 0.05
    ys, xs = np.mgrid[:h, :w]
    off_grid = ~(np.isin(xs % 32, (0, 10, 21, 31)) & np.isin(ys % 32, (0, 10, 21, 31)))
    for shift in range(16):
        for reach in (-13.25, -9.5, 9.5, 13.25):
            f = np.zeros((h, w, 2), np.float32)
            f[..., 0] = -(shift + 0.375)                 # 't' flows sample at x - flow: the box starts at x0 + shift
            f[..., 1] = 0.625
            pick = off_grid & (rng.random((h, w)) < 0.02)
            f[pick, 0] -= np.float32(reach)
            fl, rf = of.Flow(f, 't', fmask), R.make(f, 't', fmask)
            for kw in ({'target_mask': tmask}, {}):
                w1, m1 = fl.apply(img, return_valid_area=True, **kw)
                w2, m2 = R.apply(rf, img, return_valid_area=True, **kw)
                same(w1, w2)
                same(m1, m2)
