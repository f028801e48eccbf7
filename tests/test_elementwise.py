"""The element-wise (streaming) kernels of csrc/elementwise.cu against plain references: get_padding (ofk_extent),
resize (ofk_resize_flow), pad (ofk_pad), windows (ofk_crop), the arithmetic operators (ofk_addsub, ofk_scale,
ofk_scale_array), the zero tests (ofk_nonzero_flags) and points_inside_area.

Every comparison is exact unless a tolerance is written next to it with its reason. The references are the oracle
(oracle/flowref.py), cv2 where the reference calls it, and numpy in the reference's operation order. Float32 results
are compared bit for bit (as uint32) where the reference fixes the sign of zero, by value otherwise."""
import itertools

import numpy as np
import pytest

from oracle import flowref as R

cv2 = pytest.importorskip('cv2')

f32 = np.float32


@pytest.fixture(scope='module')
def of():
    import oflibnumpy_b200 as of
    of.device.require_gpu()
    return of


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


def assert_bits_equal(got, want):
    assert got.shape == want.shape
    bad = bits(got) != bits(want)
    assert not bad.any(), "%d of %d values differ, first at %s: %r vs %r" % (
        bad.sum(), bad.size, np.argwhere(bad)[0], got[bad][0], want[bad][0])


# ============================================================================================================ resize
RESIZE_SCALES = [0.5, (0.5, 0.5), (0.5, 0.25), 2, 3, 1.25, 1 / 3, 0.1, (1.7, 0.3), (0.33, 3.1), 1]
RESIZE_SHAPES = [(1, 9), (9, 1), (3, 3), (5, 7), (37, 53), (120, 77), (1080, 1920)]
RESIZE_CASES = [((1, 1), 2)] + list(itertools.product(RESIZE_SHAPES, RESIZE_SCALES))


def out_size(shape, scale):
    """cv::resize with dsize empty: round-half-even(size * scale) per axis; (fy, fx) as the reference passes them."""
    fy, fx = (scale, scale) if isinstance(scale, (int, float)) else scale
    return int(np.rint(shape[0] * fy)), int(np.rint(shape[1] * fx)), fy, fx


def _coords(n_out, inv_scale):
    """Half-pixel-centre source coordinate in float32, its floor and fraction: OpenCV's ``fx = (float)((dx + 0.5) *
    scale_x - 0.5); sx = cvFloor(fx); fx -= sx``."""
    f = ((np.arange(n_out, dtype=np.float64) + 0.5) * inv_scale - 0.5).astype(f32)
    s = np.floor(f).astype(np.int64)
    return s, (f - s.astype(f32)).astype(f32)


def resize_restated(src, fy, fx):
    """cv2.resize(src, None, fx=fx, fy=fy) (INTER_LINEAR) of a float32 (H, W, C) array, restated in numpy float32 in
    the order of OpenCV's generic code path, which is the arithmetic ofk_resize_flow reproduces:

    * an output of the input's size is a copy;
    * at an inverse scale of exactly 2 on both axes, INTER_LINEAR is INTER_AREA's fast path: ``0 + (((s00 + s01) +
      s10) + s11)`` times 0.25 where the 2x2 block is inside the image; an output whose block the right or bottom
      edge of an odd-sized input cuts, sums the taps it has in the same order (from 0) and divides by their count;
    * otherwise bilinear, horizontal pass then vertical pass, products rounded before the sum. Columns outside
      [0, W-1] are clamped together with their weight (the weight becomes 0); rows outside [0, H-1] have only their
      index clamped and keep the weight, so a border row is ``S*(1-fy) + S*fy``, which is not always S.
    """
    h, w = src.shape[:2]
    ho, wo = int(np.rint(h * fy)), int(np.rint(w * fx))
    if (ho, wo) == (h, w):
        return src.copy()
    sx_, sy_ = 1.0 / fx, 1.0 / fy
    if abs(sx_ - 2.0) < np.finfo(np.float64).eps and abs(sy_ - 2.0) < np.finfo(np.float64).eps:
        ys, xs = 2 * np.arange(ho), 2 * np.arange(wo)
        hx, hy = xs + 1 < w, ys + 1 < h
        x1, y1 = np.where(hx, xs + 1, xs), np.where(hy, ys + 1, ys)
        s00, s01 = src[ys][:, xs], src[ys][:, x1]
        s10, s11 = src[y1][:, xs], src[y1][:, x1]
        full = (f32(0) + (((s00 + s01) + s10) + s11)) * f32(0.25)
        zero = np.zeros_like(s00)
        part = f32(0) + s00
        part = part + np.where(hx[None, :, None], s01, zero)
        part = part + np.where(hy[:, None, None], s10, zero)
        count = (1 + hx[None, :] + hy[:, None]).astype(f32)[..., None]
        return np.where((hx[None, :] & hy[:, None])[..., None], full, part / count).astype(f32)
    s, a1 = _coords(wo, sx_)
    clamp = (s < 0) | (s >= w - 1)
    a1 = np.where(clamp, f32(0), a1).astype(f32)
    s = np.clip(s, 0, w - 1)
    s1 = np.minimum(s + 1, w - 1)
    a0 = (f32(1) - a1).astype(f32)
    hor = src[:, s] * a0[None, :, None] + src[:, s1] * a1[None, :, None]
    t, b1 = _coords(ho, sy_)
    b0 = (f32(1) - b1).astype(f32)
    r0, r1 = np.clip(t, 0, h - 1), np.clip(t + 1, 0, h - 1)
    return (hor[r0] * b0[:, None, None] + hor[r1] * b1[:, None, None]).astype(f32)


def resize_input(shape, seed):
    rng = np.random.default_rng(seed)
    v = (rng.standard_normal(shape + (2,)) * 7).astype(f32)
    v[rng.random(shape) < 0.1] = -0.0                       # signed zeros travel through the blend
    v[rng.random(shape) < 0.05] = 0.0
    return v, rng.random(shape) > 0.3                       # 30 % holes


@pytest.mark.parametrize('shape,scale', RESIZE_CASES)
def test_resize_restatement_is_cv2(shape, scale):
    """The restatement above equals cv2.resize bit for bit on the whole grid: vectors (2 channels) and the float mask
    (1 channel) rounded as the reference rounds it. This pins OpenCV's rules (vertical border weights, the 2x2 area
    branch, the same-size copy) without a GPU.

    OpenCV resizes 1-channel float32 images through a different code path (its IPP build) whose arithmetic is not
    restated: on the mask its float values can differ by an ulp, so the mask is compared after ``np.round``, which is
    all the reference keeps of it."""
    ho, wo, fy, fx = out_size(shape, scale)
    if ho < 1 or wo < 1:
        pytest.skip("empty output: cv2.resize rejects it")
    v, m = resize_input(shape, 1)
    assert_bits_equal(resize_restated(v, fy, fx), cv2.resize(v, None, fx=fx, fy=fy).reshape(ho, wo, 2))
    mf = m.astype(f32)
    np.testing.assert_array_equal(np.round(resize_restated(mf[..., None], fy, fx)[..., 0]),
                                  np.round(cv2.resize(mf, None, fx=fx, fy=fy).reshape(ho, wo)))


def test_resize_restatement_vertical_border_is_not_a_copy():
    """The vertical rule has teeth: at scale 1.25 the first output row (source row -0.1, fy = 0.9) is
    ``S*0.1 + S*0.9`` of source row 0, which differs from the horizontal pass of row 0 alone (what a kernel that
    zeroes fy at the border returns) somewhere."""
    v, _ = resize_input((37, 53), 2)
    out = resize_restated(v, 1.25, 1.25)
    row0 = resize_restated(v[:1], 1, 1.25)[0]
    assert out.shape == (46, 66, 2) and row0.shape == (66, 2)
    assert (bits(out[0]) != bits(row0)).any()
    np.testing.assert_allclose(out[0], row0, rtol=2e-7, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize('shape,scale', RESIZE_CASES)
def test_resize_matches_cv2(of, shape, scale):
    """Flow.resize (vectors and mask) and resize_flow against R.resize (cv2.resize, then the per-axis vector scale),
    bit for bit; an empty output raises ValueError."""
    ho, wo, fy, fx = out_size(shape, scale)
    v, m = resize_input(shape, 3)
    if ho < 1 or wo < 1:
        with pytest.raises(ValueError):
            of.Flow(v, 't', m).resize(scale)
        return
    want = R.resize(R.make(v, 't', m), scale)
    got = of.Flow(v, 't', m).resize(scale)
    assert_bits_equal(got.vecs, want.vecs)
    np.testing.assert_array_equal(got.mask, want.mask)
    assert_bits_equal(of.resize_flow(v, scale), want.vecs)


# ======================================================================================================= get_padding
PAD_SHAPES = [(37, 53), (64, 96), (375, 1242), (1080, 1920)]
TRANSLATIONS = [(3, 0), (-3, 0), (0, 3), (0, -3), (2, 2), (-5, 7)]


def check_padding(of, vecs, ref, mask=None):
    f = of.Flow(vecs, ref, mask)
    assert f.get_padding() == R.get_padding(R.make(vecs, ref, mask))
    assert of.get_flow_padding(vecs, ref) == R.get_padding(R.make(vecs, ref))


@pytest.mark.gpu
@pytest.mark.parametrize('shape', PAD_SHAPES)
@pytest.mark.parametrize('ref', ['t', 's'])
def test_get_padding_integer_translations(of, shape, ref):
    """Integer translations make the extent exactly -0.0 on a whole column or row (x - u == 0): the device min must
    order -0.0 against the negative extents of the other pixels whatever order the warps commit in."""
    for dx, dy in TRANSLATIONS:
        check_padding(of, R.from_transforms([['translation', dx, dy]], shape, ref), ref)


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['t', 's'])
def test_get_padding_rotation_about_origin(of, ref):
    for shape in PAD_SHAPES[:3]:
        for angle in (30, -30, 90, 180):
            check_padding(of, R.from_transforms([['rotation', 0, 0, angle]], shape, ref), ref)


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['t', 's'])
def test_get_padding_zero_border_vectors(of, ref):
    """Vectors zero or below the 1e-3 threshold in column 0 and row 0 (extent -0.0 there), negative extents
    elsewhere; the same field negated (its zeros become -0.0), and explicit -0.0 vectors."""
    rng = np.random.default_rng(5)
    for shape in PAD_SHAPES:
        v = rng.uniform(-9, 9, shape + (2,)).astype(f32)
        v[:, 0] = 0
        v[0, :] = f32(5e-4)
        v[1, 1:] = -6e-4
        check_padding(of, v, ref)
        neg = -of.Flow(v, ref)
        assert (bits(neg.vecs[1:, 0]) == 0x80000000).all()
        check_padding(of, np.array(neg.vecs), ref)
        z = np.full(shape + (2,), -0.0, f32)
        z[shape[0] // 2, shape[1] // 2] = (-2.5, 4.0)
        check_padding(of, z, ref)


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['t', 's'])
def test_get_padding_masked(of, ref):
    """A mask that hides every pixel with a negative extent, one valid pixel, and an empty mask (the reference fails
    on the min of an empty selection with ValueError)."""
    rng = np.random.default_rng(6)
    for shape in PAD_SHAPES[:3]:
        h, w = shape
        v = rng.uniform(-4, 4, shape + (2,)).astype(f32)
        sign = 1 if ref == 't' else -1
        rows, cols = np.mgrid[:h, :w]
        ex, ey = cols - sign * v[..., 0], rows - sign * v[..., 1]
        mask = (ex >= 0) & (ey >= 0)
        check_padding(of, v, ref, mask)
        one = np.zeros(shape, bool)
        one[h // 3, w - 1] = True
        check_padding(of, v, ref, one)
        with pytest.raises(ValueError):
            R.get_padding(R.make(v, ref, np.zeros(shape, bool)))
        with pytest.raises(ValueError):
            of.Flow(v, ref, np.zeros(shape, bool)).get_padding()


@pytest.mark.gpu
def test_extent_batch_of_frames(of):
    """ofk_extent on N = 5 different frames in one launch: each frame's (min ey, max ey, min ex, max ex) equals numpy's
    min / max of the thresholded extents over its valid pixels (+0.0 and -0.0 compare equal)."""
    from oflibnumpy_b200 import _ops
    from oflibnumpy_b200.device import DeviceArray
    rng = np.random.default_rng(7)
    h, w, n = 211, 389, 5
    frames = [R.from_transforms([['translation', 3, -2]], (h, w), 't'),
              R.from_transforms([['rotation', 0, 0, 20]], (h, w), 't'),
              rng.uniform(-50, 50, (h, w, 2)).astype(f32),
              np.full((h, w, 2), -0.0, f32),
              rng.uniform(-2e-3, 2e-3, (h, w, 2)).astype(f32)]
    masks = rng.random((n, h, w)) > 0.2
    masks[3] = True
    vecs = np.stack(frames)
    for sign in (1.0, -1.0):
        got = _ops.extent(DeviceArray.from_numpy(vecs), DeviceArray.from_numpy(masks.view(np.uint8)), sign, 1e-3)
        for k in range(n):
            t = R.threshold(vecs[k]) * f32(sign)
            rows, cols = np.mgrid[:h, :w]
            ex = -(t[..., 0] - cols.astype(f32))
            ey = -(t[..., 1] - rows.astype(f32))
            m = masks[k]
            want = [ey[m].min(), ey[m].max(), ex[m].min(), ex[m].max()]
            np.testing.assert_array_equal(got[k], np.array(want, f32))


# =============================================================================================================== pad
@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['constant', 'edge', 'symmetric'])
def test_pad_matches_numpy(of, mode):
    """Flow.pad against R.pad (np.pad for the vectors, False outside for the mask): no padding, padding larger than
    the frame (symmetric reflects with period 2n), one-row and one-column frames."""
    rng = np.random.default_rng(8)
    for shape in ((1, 1), (1, 7), (6, 1), (5, 4), (37, 53)):
        h, w = shape
        v = rng.standard_normal(shape + (2,)).astype(f32)
        m = rng.random(shape) > 0.3
        for padding in ([0, 0, 0, 0], [1, 2, 3, 4], [h + 3, 2 * h + 1, w + 2, 3 * w], [0, 5 * h, 0, 0],
                        [0, 0, 2 * w + 1, 0]):
            got = of.Flow(v, 't', m).pad(padding, mode)
            want = R.pad(R.make(v, 't', m), padding, mode)
            assert_bits_equal(got.vecs, want.vecs)
            np.testing.assert_array_equal(got.mask, want.mask)


@pytest.mark.gpu
def test_pad_batch_equals_frames(of):
    """ofk_pad on N = 3 frames equals each frame padded alone."""
    from oflibnumpy_b200 import _ops
    from oflibnumpy_b200.device import DeviceArray
    rng = np.random.default_rng(9)
    v = rng.standard_normal((3, 19, 23, 2)).astype(f32)
    m = (rng.random((3, 19, 23)) > 0.3).view(np.uint8)
    for mode in ('constant', 'edge', 'symmetric'):
        padding = [4, 30, 25, 2]
        gv, gm = _ops.pad(DeviceArray.from_numpy(v), DeviceArray.from_numpy(m), padding, mode)
        gv, gm = gv.numpy(), gm.numpy()
        for k in range(3):
            one_v, one_m = _ops.pad(DeviceArray.from_numpy(v[k:k + 1]), DeviceArray.from_numpy(m[k:k + 1]), padding,
                                    mode)
            assert_bits_equal(gv[k], one_v.numpy()[0])
            np.testing.assert_array_equal(gm[k], one_m.numpy()[0])
            want = R.pad(R.make(v[k], 't', m[k]), padding, mode)
            assert_bits_equal(gv[k], want.vecs)
            np.testing.assert_array_equal(gm[k].view(bool), want.mask)


# ============================================================================================================= crop
@pytest.mark.gpu
def test_windows_match_numpy(of):
    """Flow[a:b, c:d] (ofk_crop) at each edge, 1x1, the full frame, and rows wider than 2048 bytes (W > 256 vectors,
    where each block strides along the row); vectors and mask."""
    rng = np.random.default_rng(10)
    for shape in ((9, 13), (40, 700), (3, 2051)):
        h, w = shape
        v = rng.standard_normal(shape + (2,)).astype(f32)
        m = rng.random(shape) > 0.4
        f = of.Flow(v, 't', m)
        wins = [(slice(None), slice(None)), (slice(0, 1), slice(0, 1)), (slice(h - 1, h), slice(w - 1, w)),
                (slice(0, 2), slice(None)), (slice(h - 2, h), slice(None)), (slice(None), slice(0, 3)),
                (slice(None), slice(w - 3, w)), (slice(1, h - 1), slice(1, w - 1)), (slice(h // 2, h // 2 + 1),),
                (slice(None), slice(w // 3, w - 1))]
        for win in wins:
            g = f[win]
            assert g.ref == 't'
            assert_bits_equal(g.vecs, v[win])
            np.testing.assert_array_equal(g.mask, m[win])


# ======================================================================================================= arithmetic
ARITH_SHAPES = [(4, 5), (3, 7), (2, 7), (3, 5), (61, 67), (256, 256)]          # H*W % 4 = 0, 1, 2, 3, 3, 0


def ref_operate(vecs, other, fn):
    """The reference's Flow.__mul__ / __truediv__ / __pow__ (flow_class.py:377-489): ``float(other)`` if that works,
    else a list becomes np.array(list), a size-2 array is broadcast along the channels, an (H,W) array along a new
    channel axis; the result goes through the Flow constructor (finite check, astype float32)."""
    try:
        o = float(other)
    except TypeError:
        o = np.array(other) if isinstance(other, list) else other
        if o.ndim == 1:
            o = o[None, None, :]
        elif o.ndim == 2:
            o = o[..., None]
    with np.errstate(all='ignore'):
        r = fn(vecs, o)
    return R.make(r, 't').vecs


def fields(shape, seed):
    rng = np.random.default_rng(seed)
    a = (rng.standard_normal(shape + (2,)) * 5).astype(f32)
    a.flat[::7] = 0
    a.flat[3::11] = -0.0
    pos = (np.abs(a) + f32(0.125)).astype(f32)
    return rng, a, pos


@pytest.mark.gpu
@pytest.mark.parametrize('shape', ARITH_SHAPES)
def test_add_sub(of, shape):
    """+ and - with a Flow (mask AND) and with float32 / float64 / int16 / int64 arrays (numpy promotion, then the
    constructor's cast to float32; the mask is kept): the addsub float4 body and its tail."""
    rng, a, _ = fields(shape, 11)
    b = (rng.standard_normal(shape + (2,)) * 3).astype(f32)
    am, bm = rng.random(shape) > 0.2, rng.random(shape) > 0.2
    fa, fb = of.Flow(a, 't', am), of.Flow(b, 't', bm)
    for op, rop in ((lambda x, y: x + y, R.add), (lambda x, y: x - y, R.sub)):
        got, want = op(fa, fb), rop(R.make(a, 't', am), R.make(b, 't', bm))
        assert_bits_equal(got.vecs, want.vecs)
        np.testing.assert_array_equal(got.mask, want.mask)
        for arr in (b, b.astype(np.float64) * 1.0000001, (b * 100).astype(np.int16), (b * 1e6).astype(np.int64)):
            got = op(fa, arr)
            assert_bits_equal(got.vecs, R.make(op(a, arr), 't').vecs)
            np.testing.assert_array_equal(got.mask, am)


def scale_operands(shape, rng):
    h, w = shape
    return [3, -1, 0.1, 1e-3, f32(0.3), np.float64(0.3), np.float64(1 / 3), [0.7, -3], [2, 5],
            np.array([0.7, -3.3], f32), np.array([3, -7], np.int16), np.array([3, -7], np.int64),
            rng.uniform(-3, 3, (h, w)).astype(f32), rng.uniform(-3, 3, (h, w)),
            rng.integers(-9, 9, (h, w)).astype(np.int16) | 1,
            rng.uniform(-3, 3, (h, w, 2)).astype(f32), rng.uniform(-3, 3, (h, w, 2))]


@pytest.mark.gpu
@pytest.mark.parametrize('shape', ARITH_SHAPES)
def test_mul_div(of, shape):
    """* and / with python scalars, np.float32 / np.float64 scalars, lists, size-2 arrays of float32 / int16 / int64,
    and (H,W) and (H,W,2) arrays, bit for bit against the reference's numpy expression; the mask is kept."""
    rng, a, _ = fields(shape, 12)
    m = rng.random(shape) > 0.2
    f = of.Flow(a, 's', m)
    for other in scale_operands(shape, rng):
        for op in (lambda x, y: x * y, lambda x, y: x / y):
            got = op(f, other)
            assert got.ref == 's'
            assert_bits_equal(got.vecs, ref_operate(a, other, op))
            np.testing.assert_array_equal(got.mask, m)
    assert_bits_equal((-f).vecs, R.neg(R.make(a, 's', m)).vecs)
    assert_bits_equal(f.invert('t').vecs, R.invert(R.make(a, 's', m), 't').vecs)


@pytest.mark.gpu
def test_non_finite_results_raise(of):
    """Overflow and division by an array containing 0 make the reference's constructor raise ValueError; so must
    the device path."""
    rng, a, _ = fields((5, 7), 13)
    f = of.Flow(a, 't')
    zeros = rng.uniform(1, 2, (5, 7)).astype(f32)
    zeros[2, 3] = 0
    for other, fn in ((1e38, lambda x, y: x * y), (1e300, lambda x, y: x * y), (0, lambda x, y: x / y),
                      (zeros, lambda x, y: x / y), ([1, 0], lambda x, y: x / y), (np.array([0, 1], f32),
                                                                                   lambda x, y: x / y),
                      (-1, lambda x, y: x ** y), (0.5, lambda x, y: x ** y), (40, lambda x, y: x ** y)):
        with pytest.raises(ValueError):
            ref_operate(a, other, fn)
        with pytest.raises(ValueError):
            fn(f, other)
    big = np.full((5, 7, 2), 3e38, f32)
    with pytest.raises(ValueError):
        R.make(big + big, 't')
    with pytest.raises(ValueError):
        of.Flow(big, 't') + of.Flow(big, 't')


@pytest.mark.gpu
@pytest.mark.parametrize('shape', ARITH_SHAPES)
def test_pow_numpy_fast_exponents(of, shape):
    """``vecs ** float(e)`` for e in 2, 0.5, -1, 1, 0: numpy computes square / sqrt / reciprocal / copy / ones, all
    correctly rounded, so the device result is bit-exact (sign of zero included)."""
    _, a, pos = fields(shape, 14)
    for e, base in ((2, a), (2.0, a), (0.5, pos), (-1, pos), (-1.0, -pos), (1, a), (0, a), (np.float32(0.5), pos),
                    (np.float64(2), a)):
        got = of.Flow(base, 't') ** e
        assert_bits_equal(got.vecs, ref_operate(base, e, lambda x, y: x ** y))


POW_ULP_BOUND = 1        # the largest distance measured on a B200 (1000 W power limit) is 1 ulp


def ulp_distance(a, b):
    """Distance in float32 ulps (units in the last place) between finite float32 arrays."""
    ia, ib = bits(a).view(np.int32).astype(np.int64), bits(b).view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, np.int64(-2 ** 31) - ia, ia)
    ib = np.where(ib < 0, np.int64(-2 ** 31) - ib, ib)
    return np.abs(ia - ib)


@pytest.mark.gpu
def test_pow_general_exponents_within_ulp_bound(of):
    """Other scalar exponents and array exponents go to a pow that is not correctly rounded, on the device (CUDA
    powf / pow) as in numpy (whose float32 power depends on its SIMD build). The device result is held to
    POW_ULP_BOUND float32 ulps of float32(float64 pow) of the same operands: a python scalar exponent is rounded to
    float32 first, as numpy does for a float32 array. Both sides are deterministic, so the bound is the largest
    distance measured on a B200: 1 ulp."""
    rng = np.random.default_rng(15)
    shape = (61, 67)
    base = np.exp(rng.uniform(-6, 6, shape + (2,))).astype(f32)
    worst = 0
    for e in (1.7, -2.5, 3, 0.25, 1 / 3, np.array([1.7, 2.0], f32), [2, 3], np.array([0.5, -1.5]),
              rng.uniform(-2, 2, shape).astype(f32), rng.uniform(-2, 2, shape + (2,))):
        got = (of.Flow(base, 't') ** e).vecs
        e64 = e.astype(np.float64) if isinstance(e, np.ndarray) else e if isinstance(e, list) else float(f32(e))
        ex = ref_operate(base.astype(np.float64), e64, lambda x, y: x ** y)
        d = ulp_distance(got, ex)
        worst = max(worst, int(d.max()))
        assert d.max() <= POW_ULP_BOUND, "exponent %r: %d ulp" % (e, d.max())
    print("largest pow distance: %d ulp" % worst)


# ======================================================================================================= zero tests
@pytest.mark.gpu
def test_is_zero_edges(of):
    """is_zero / is_zero_flow against the reference: -0.0 is zero; float32 denormals are not zero unthresholded (the
    library is built without flush-to-zero); exactly +-float32(1e-3) is not below the threshold; vectors that are
    non-zero only under the mask; a single non-zero vector anywhere in a large frame (past the sparse probe)."""
    shape = (375, 1242)
    h, w = shape
    cases = []
    z = np.full(shape + (2,), -0.0, f32)
    cases.append((z, None))
    for val in (np.float32(1e-45), np.float32(-1e-40), f32(1e-3), -f32(1e-3), np.nextafter(f32(1e-3), f32(0)), 7.0):
        for y, x, c in ((0, 0, 0), (h - 1, w - 1, 1), (h // 2, 777, 0), (1, w - 1, 1)):
            v = np.zeros(shape + (2,), f32)
            v[y, x, c] = val
            cases.append((v, None))
            m = np.ones(shape, bool)
            m[y, x] = False
            cases.append((v, m))
    for v, m in cases:
        f = of.Flow(v, 't', m)
        fr = R.make(v, 't', m)
        for thr in (True, False):
            for masked in (True, False):
                assert f.is_zero(thr, masked) == R.is_zero(fr, thr, masked)
            assert of.is_zero_flow(v, thr) == R.is_zero_array(v, thr)


# ============================================================================================== points_inside_area
@pytest.mark.gpu
def test_points_inside_area_half_integers(of):
    """Points at k +- 0.5 next to every border (numpy rounds half to even), NaN and +-1e300, against
    R.points_inside_area."""
    for h, w in ((1, 1), (6, 9), (7, 8)):
        cs = [-1.5, -0.5, -0.49, 0.5, 1.5, h - 1.5, h - 1, h - 0.5, h - 0.51, h + 0.5]
        rs = [-1.5, -0.5, 0.5, w - 1.5, w - 0.5, w - 0.5001, w + 0.5]
        pts = np.array(list(itertools.product(cs, rs)), np.float64)
        np.testing.assert_array_equal(of.points_inside_area(pts, (h, w)), R.points_inside_area(pts, (h, w)))
    pts = np.array([[np.nan, 1], [1, np.nan], [1e300, 1], [-1e300, 1], [1, 1e300], [1, -1e300], [2, 2]])
    with np.errstate(invalid='ignore'):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            want = R.points_inside_area(pts, (5, 5))
    np.testing.assert_array_equal(of.points_inside_area(pts, (5, 5)), want)
    np.testing.assert_array_equal(want, [False] * 6 + [True])
