"""The image warp (ref 't' Flow.apply / FlowBatch.apply / apply_flow_host) against cv2.remap at every dtype cv2.remap
accepts, at payload values where float32 products and sums round, saturate or carry signed zeros, NaN and Inf, and
through every kernel ofk_warp_t dispatches to.

Which kernel a call reaches (csrc/warp_t.cu, ofk_warp_t; "aligned" = payload and out 16-byte aligned, flow 8-byte
aligned; "same frame" = no padding):

    payload                                        | same frame, aligned, H*W*C < 2^30   | otherwise
    -----------------------------------------------+-------------------------------------+----------------
    uint8 C = 1, 3, 4, W % 16 == 0                 | TMA kernel (counter 2)              | warp_t_generic
    uint8 C = 3, W % 16 != 0 (or OFK_WARP_WS=0)    | warp_t_u8x3 (counter 3)             | warp_t_generic
    uint8 C = 1, 4, W % 16 != 0 (or OFK_WARP_WS=0) | warp_t_rows<u8, C, arith> (3)       | warp_t_generic
    float32 C = 2 with target and flow mask        | composition TMA kernel (2) if       | warp_t_generic
      (an image warped like a flow, STRICT rule)   |   W % 16 == 0, else warp_t_rows (3) |
    float32 C = 1..4                               | warp_t_rows<f32, C> (3)             | warp_t_generic
    uint8 C = 2, int16, uint16, float64, f32 C>=5  | warp_t_generic (3)                  | warp_t_generic
    padding (cut or not), any dtype                | warp_t_generic (3)                  |

Counter 3 counts every non-TMA call, so rows / u8x3 / generic are told apart by construction from this table: the
tests pick dtype, C, W, padding and pointer offsets to land on each row. ``valid_target`` runs valid_geom_vec4 when
W % 4 == 0 and its pointers are aligned, else the mask-only warp_t_rows<u8, 0>.

Floats are compared by their bytes (so -0.0 and +0.0 differ), except NaN, which only has to be NaN on both sides.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import load_golden
from oracle import flowref as R
from oracle import remap_q32 as Q

cv2 = pytest.importorskip("cv2")

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DTYPES = [np.uint8, np.int16, np.uint16, np.float32, np.float64]
CHANNELS = [0, 1, 2, 3, 4, 5]          # 0: a 2-D (H, W) target


# ------------------------------------------------------------------------------------------------- the reference
def _remap(payload, flow):
    """cv2.remap(payload (H,W,C), grid - flow) on the float32 map; any C (cv2 returns 2-D arrays for C = 1)."""
    mx, my = Q.backward_map(flow, -1.0)
    out = cv2.remap(payload, np.dstack([mx, my]), None, cv2.INTER_LINEAR)
    return out.reshape(payload.shape), mx, my


def _rule(payload_dtype, mask_is_bool):
    """The promoted dtype of Flow.apply's `payload || mask` (flow_class.py:615,626,644) decides the cv2.remap path that
    samples the payload and the mask rule on the valid-weight sum (remap_q32.valid_weight_sum)."""
    pro = np.result_type(payload_dtype, np.bool_ if mask_is_bool else np.int8)
    if pro == np.uint8:
        return pro, lambda s: s >= 512
    if pro in (np.int16, np.uint16):
        return pro, lambda s: s > 512
    if pro in (np.float32, np.float64):
        return pro, lambda s: s == 1024
    raise TypeError("payload || mask promotes to {}, which cv2.remap rejects".format(pro))


def ref_apply(flow, img, flow_mask=None, target_mask=None, return_valid_area=False, padding=None, cut=True,
              consider_mask=True):
    """``Flow(flow, 't', flow_mask).apply(img, ...)`` (flow_class.py:528-695) on cv2.remap. consider_mask only
    matters for ref 's'."""
    two_d = img.ndim == 2
    payload = img[..., None] if two_d else img
    fh, fw = flow.shape[:2]
    fmask = np.ones((fh, fw), bool) if flow_mask is None else flow_mask.astype(bool)
    tmask = np.ones(payload.shape[:2], bool) if target_mask is None else target_mask
    if return_valid_area:
        pro, rule = _rule(img.dtype, target_mask is not None)
        payload = payload.astype(pro)
    g = flow if padding is None else np.pad(flow, ((padding[0], padding[1]), (padding[2], padding[3]), (0, 0)))
    if R.is_zero_array(g, thresholded=True):      # utils.py:215-216: the target itself, mask included
        warped = payload
        valid = tmask.astype(bool)
    else:
        warped, mx, my = _remap(payload, g)
        valid = rule(Q.valid_weight_sum(tmask, mx, my)) if return_valid_area else None
    if padding is not None and cut:
        win = (slice(padding[0], padding[0] + fh), slice(padding[2], padding[2] + fw))
        warped = warped[win]
        valid = None if valid is None else valid[win]
    if return_valid_area:
        if valid.shape != fmask.shape:
            win = (slice(padding[0], padding[0] + fh), slice(padding[2], padding[2] + fw))
            inner = valid[win] & fmask
            valid = np.zeros_like(valid)
            valid[win] = inner
        else:
            valid = valid & fmask
    warped = warped.astype(img.dtype)
    if two_d:
        warped = warped[..., 0]
    return (warped, valid) if return_valid_area else warped


def same_bits(got, want, what=''):
    got, want = np.asarray(got), np.asarray(want)
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, want.dtype, got.shape, want.shape)
    if np.issubdtype(want.dtype, np.floating):
        gn, wn = np.isnan(got), np.isnan(want)
        assert np.array_equal(gn, wn), (what, 'NaN positions', np.argwhere(gn != wn)[:5])
        u = np.uint32 if want.dtype == np.float32 else np.uint64
        g, w = got.view(u)[~gn], want.view(u)[~wn]
        bad = np.flatnonzero(g != w)
        assert bad.size == 0, (what, bad.size, got[~gn][bad[:5]], want[~wn][bad[:5]])
    else:
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, (what, bad.size, got.ravel()[bad[:5]], want.ravel()[bad[:5]])


# ------------------------------------------------------------------------------------------------- inputs
def payload_sets(rng, dtype, shape):
    """Named payloads of `shape` ([N,] H, W, C) where cv2.remap's arithmetic rounds, saturates, or meets signed zeros,
    subnormals, NaN and Inf."""
    dt = np.dtype(dtype)
    idx = np.indices(shape)
    checker = (idx[-3:].sum(0) % 2).astype(bool)
    xx = idx[-2]
    out = []
    if dt.kind in 'iu':
        lo, hi = np.iinfo(dt).min, np.iinfo(dt).max
        out.append(('uniform', rng.integers(lo, hi, shape, endpoint=True).astype(dt)))
        out.append(('checker', np.where(checker, hi, lo).astype(dt)))
        out.append(('near_limits', rng.choice(np.array([lo, lo + 1, hi - 1, hi], dt), shape)))
        if dt == np.int16:       # runs of -32768 next to 32767: a half-pixel blend is -0.5, a round-half-even tie
            out.append(('tie_runs', np.where((xx // 3) % 2 == 0, -32768, 32767).astype(dt)))
        return out
    mant = lambda: rng.uniform(-1, 1, shape) * (0.5 + 0.5 * rng.random(shape))     # full mantissas, |x| <= 1
    scales = (1e-30, 1.0, 1e30, 3e38) if dt == np.float32 else (1e-300, 1.0, 1e300)
    for s in scales:
        out.append(('mantissa_%g' % s, (mant() * s).astype(dt)))
    if dt == np.float64:     # not representable in float32: a float32 accumulator loses the low bits
        out.append(('one_plus_ulp32', 1 + rng.integers(1, 1 << 12, shape) * 2.0 ** -40))
    out.append(('negzero', np.full(shape, -0.0, dt)))
    out.append(('signed_zeros', np.where(checker, -0.0, 0.0).astype(dt)))
    out.append(('subnormal', (rng.uniform(-1, 1, shape) * (1e-40 if dt == np.float32 else 1e-310)).astype(dt)))
    sp = mant().astype(dt)
    pick = rng.random(shape)
    sp[pick < 0.06] = np.nan
    sp[(pick >= 0.06) & (pick < 0.1)] = np.inf
    sp[(pick >= 0.1) & (pick < 0.14)] = -np.inf
    sp[(pick >= 0.14) & (pick < 0.2)] = -0.0
    out.append(('special', sp))
    return out


def _smooth(rng, h, w):
    from test_gpu_warp_t import _smooth_flow
    return _smooth_flow(rng, h, w, 3.0)


def flow_sets(rng, h, w):
    """Smooth and rough fields, integer / half-pixel shifts over the border, 1/64 ties, zero and sub-threshold."""
    from test_gpu_warp_t import _rough_flow

    def const(dx, dy):
        f = np.zeros((h, w, 2), np.float32)
        f[..., 0], f[..., 1] = dx, dy
        return f
    ties = (rng.integers(-3 * 64, 3 * 64, (h, w, 2)) / 64).astype(np.float32)
    tiny = ((rng.random((h, w, 2)) - 0.5) * 1.9e-3).astype(np.float32)
    return [('smooth', _smooth(rng, h, w)), ('blocks', _rough_flow(rng, h, w, 'blocks')),
            ('noise', _rough_flow(rng, h, w, 'noise')), ('int_shift', const(1, -1)), ('half', const(0.5, 0)),
            ('half_xy', const(-0.5, 0.5)), ('over_right', const(w - 0.5, 0)), ('outside', const(w, 0)),
            ('over_corner', const(-(w - 1), -(h - 1))), ('ties', ties), ('zero', np.zeros((h, w, 2), np.float32)),
            ('tiny', tiny)]


def _img(payload, c):
    return payload[..., 0] if c == 0 else payload


# ------------------------------------------------------------------------------------------------- CPU: the reference
@pytest.mark.parametrize('dtype', DTYPES)
def test_ref_apply_matches_oracle(dtype):
    """ref_apply against oracle.flowref.apply (the reference's own concatenate-and-remap glue) on small inputs."""
    rng = np.random.default_rng(1)
    h, w = 9, 13
    for c in (0, 1, 3, 5):
        for fname, flow in flow_sets(rng, h, w)[:6] + flow_sets(rng, h, w)[-2:]:
            pay = payload_sets(rng, dtype, (h, w, max(c, 1)))[0][1]
            img = _img(pay, c)
            fm = rng.random((h, w)) > 0.2
            tm = rng.random((h, w)) > 0.2
            f = R.make(flow, 't', fm)
            same_bits(ref_apply(flow, img, fm), R.apply(f, img), fname)
            for kw in ({}, {'target_mask': tm}):
                if dtype == np.uint16 and not kw:
                    with pytest.raises(TypeError):
                        ref_apply(flow, img, fm, return_valid_area=True)
                    continue
                wr, vr = ref_apply(flow, img, fm, return_valid_area=True, **kw)
                wo, vo = R.apply(f, img, return_valid_area=True, **kw)
                same_bits(wr, wo, fname)
                same_bits(vr, vo, fname)
            pad = [2, 1, 3, 0]
            big = _img(payload_sets(rng, dtype, (h + 3, w + 3, max(c, 1)))[0][1], c)
            for cut in (True, False):
                same_bits(ref_apply(flow, big, fm, padding=pad, cut=cut), R.apply(f, big, padding=pad, cut=cut))
                bt = rng.random(big.shape[:2]) > 0.2
                wr, vr = ref_apply(flow, big, fm, target_mask=bt, return_valid_area=True, padding=pad, cut=cut)
                wo, vo = R.apply(f, big, target_mask=bt, return_valid_area=True, padding=pad, cut=cut)
                same_bits(wr, wo)
                same_bits(vr, vo)


def test_ref_apply_matches_goldens():
    """ref_apply against the outputs of the unmodified reference stored in the warp_t / warp_t_padded goldens."""
    g = load_golden('warp_t')
    flow, fmask = g['in_flow'], g['in_flow_mask']
    for name in [k[3:] for k in g if k.startswith('in_img_')]:
        img = g['in_' + name]
        same_bits(ref_apply(flow, img, fmask), g['out_apply_' + name], name)
        if 'err_applyva_' + name in g:
            with pytest.raises(TypeError):
                ref_apply(flow, img, fmask, return_valid_area=True)
            continue
        w, m = ref_apply(flow, img, fmask, return_valid_area=True)
        same_bits(w, g['out_applyva_' + name])
        same_bits(m, g['out_applyva_' + name + '_valid'])
        if 'out_applyvatm_' + name in g:
            w, m = ref_apply(flow, img, fmask, target_mask=g['in_target_mask'], return_valid_area=True)
            same_bits(w, g['out_applyvatm_' + name])
            same_bits(m, g['out_applyvatm_' + name + '_valid'])
    g = load_golden('warp_t_padded')
    pad = [int(x) for x in g['in_padding']]
    flow, fmask = g['in_flow'], g['in_flow_mask']
    for cut in (True, False):
        tag = 'cut' if cut else 'nocut'
        same_bits(ref_apply(flow, g['in_img_u8c3'], fmask, padding=pad, cut=cut), g['out_apply_u8_' + tag])
        w, m = ref_apply(flow, g['in_img_u8c3'], fmask, return_valid_area=True, padding=pad, cut=cut)
        same_bits(w, g['out_applyva_u8_' + tag])
        same_bits(m, g['out_applyva_u8_' + tag + '_valid'])
        w, m = ref_apply(flow, g['in_img_f32c3'], fmask, target_mask=g['in_target_mask'], return_valid_area=True,
                         padding=pad, cut=cut)
        same_bits(w, g['out_applyvatm_f32_' + tag])
        same_bits(m, g['out_applyvatm_f32_' + tag + '_valid'])


# ------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope='module')
def of():
    import oflibnumpy_b200 as of
    of.device.require_gpu()
    return of


def _counters():
    from oflibnumpy_b200 import _lib
    lib = _lib.load()
    return np.array([lib.ofk_rt_path_count(k) for k in (2, 3)], np.int64)


def _expect_tma(dtype, c, w, both_masks):
    """Whether a same-frame, aligned call takes a TMA kernel: the uint8 image kernel, or for a float32 x 2 payload with
    a valid area from both a target and a flow mask, the composition kernel without its addition."""
    if w % 16:
        return False
    if np.dtype(dtype) == np.uint8:
        return c in (0, 1, 3, 4)
    return np.dtype(dtype) == np.float32 and c == 2 and both_masks


SHAPES = [(1, 1), (1, 37), (23, 1), (13, 15), (13, 16), (13, 17), (11, 33), (9, 64), (7, 155)]


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
@pytest.mark.parametrize('c', CHANNELS)
def test_payload_values_every_kernel(of, dtype, c):
    """Flow.apply bit for bit against cv2.remap for every payload set, flow set and shape, with no valid area, the
    geometric valid area and a resampled target mask; each call on the kernel the module table names."""
    rng = np.random.default_rng(100 + 7 * c + DTYPES.index(dtype))
    for (h, w) in SHAPES:
        flows = flow_sets(rng, h, w)
        fmask = rng.random((h, w)) > 0.1
        tmask = rng.random((h, w)) > 0.15
        for k, (pname, pay) in enumerate(payload_sets(rng, dtype, (h, w, max(c, 1)))):
            img = _img(pay, c)
            for fname, flow in (flows[k % len(flows)], flows[(k + 5) % len(flows)], flows[4], flows[-2 + k % 2]):
                what = (h, w, pname, fname)
                f = of.Flow(flow, 't', fmask)
                expect = np.zeros(2, np.int64)
                before = _counters()
                same_bits(f.apply(img), ref_apply(flow, img, fmask), what)
                expect[0 if _expect_tma(dtype, c, w, False) else 1] += 1
                for kw in [{'target_mask': tmask}] + ([] if dtype == np.uint16 else [{}]):
                    got = f.apply(img, return_valid_area=True, **kw)
                    want = ref_apply(flow, img, fmask, return_valid_area=True, **kw)
                    same_bits(got[0], want[0], what + ('va', len(kw)))
                    same_bits(got[1], want[1], what + ('valid', len(kw)))
                    expect[0 if _expect_tma(dtype, c, w, bool(kw)) else 1] += 1
                d = _counters() - before
                assert d.tolist() == expect.tolist(), (what, d, expect)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
def test_padding_every_dtype(of, dtype):
    """Padded apply (warp_t_generic with frame offsets), cut and not cut, every dtype, special values included."""
    rng = np.random.default_rng(200 + DTYPES.index(dtype))
    h, w, pad = 19, 33, [3, 2, 5, 1]
    fmask = rng.random((h, w)) > 0.1
    for c in (0, 1, 3, 5):
        flows = flow_sets(rng, h, w)
        for k, (pname, pay) in enumerate(payload_sets(rng, dtype, (h + 5, w + 6, max(c, 1)))):
            img = _img(pay, c)
            tm = rng.random(img.shape[:2]) > 0.15
            for fname, flow in (flows[k % len(flows)], flows[-2]):
                f = of.Flow(flow, 't', fmask)
                for cut in (True, False):
                    what = (c, pname, fname, cut)
                    same_bits(f.apply(img, padding=pad, cut=cut), ref_apply(flow, img, fmask, padding=pad, cut=cut),
                              what)
                    got = f.apply(img, target_mask=tm, return_valid_area=True, padding=pad, cut=cut)
                    want = ref_apply(flow, img, fmask, target_mask=tm, return_valid_area=True, padding=pad, cut=cut)
                    same_bits(got[0], want[0], what)
                    same_bits(got[1], want[1], what)


@pytest.mark.gpu
def test_zero_flow_passes_float_targets_through(of):
    """apply_flow returns its target untouched for a flow that is zero below the threshold (utils.py:215-216): a depth
    map with NaN / Inf / -0.0 comes back byte for byte, also with a valid area, padding, and a flow as the target."""
    rng = np.random.default_rng(3)
    h, w = 24, 40
    for dtype in (np.float32, np.float64):
        depth = rng.uniform(0.5, 20, (h, w)).astype(dtype)
        depth[rng.random((h, w)) < 0.1] = np.nan
        depth[rng.random((h, w)) < 0.05] = np.inf
        depth[rng.random((h, w)) < 0.05] = -0.0
        tm = rng.random((h, w)) > 0.2
        fm = rng.random((h, w)) > 0.2
        for flow in (np.zeros((h, w, 2), np.float32), ((rng.random((h, w, 2)) - 0.5) * 1.9e-3).astype(np.float32)):
            f = of.Flow(flow, 't', fm)
            same_bits(f.apply(depth), depth)
            got, valid = f.apply(depth, target_mask=tm, return_valid_area=True)
            same_bits(got, depth)
            same_bits(valid, tm & fm)
            big = np.pad(depth, ((1, 2), (3, 0)), constant_values=-0.0)
            same_bits(f.apply(big, padding=[1, 2, 3, 0]), depth)
            same_bits(f.apply(big, padding=[1, 2, 3, 0], cut=False), big)
    vecs = np.where(rng.random((h, w, 2)) < 0.5, -0.0, 3.0).astype(np.float32)
    tgt = of.Flow(vecs, 't', rng.random((h, w)) > 0.3)
    res = of.Flow(np.zeros((h, w, 2), np.float32), 't', fm).apply(tgt)
    same_bits(res.vecs, vecs)
    same_bits(res.mask, tgt.mask & fm)


def _da_view(base, offset_elems, shape):
    from oflibnumpy_b200.device import DeviceArray
    return DeviceArray(base.ptr + offset_elems * base.dtype.itemsize, shape, base.dtype, owner=base)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
def test_unaligned_payload_out_and_flow(of, dtype):
    """Payload, output and flow pointers that are not 16-byte aligned (views one element or one pixel into a buffer,
    natural alignment kept) take warp_t_generic and give the bytes of the aligned call."""
    from oflibnumpy_b200 import _lib, _ops
    from oflibnumpy_b200.device import DeviceArray
    rng = np.random.default_rng(4)
    for (h, w, c) in ((13, 16, 1), (13, 16, 3), (13, 17, 4), (9, 64, 2)):
        flow = flow_sets(rng, h, w)[1][1]
        fmask = rng.random((h, w)) > 0.1
        for pname, pay in payload_sets(rng, dtype, (h, w, c))[:2] + payload_sets(rng, dtype, (h, w, c))[-1:]:
            want = ref_apply(flow, pay, fmask)
            n = h * w * c
            for p_off, o_off, f_off in ((1, 0, 0), (c, 0, 0), (0, 1, 0), (0, c, 1), (c, 1, 1)):
                host = np.zeros(n + c + 1, dtype)
                host[p_off:p_off + n] = pay.ravel()
                pbuf = DeviceArray.from_numpy(host)
                p = _da_view(pbuf, p_off, (1, h, w, c))
                obuf = DeviceArray.empty((n + c + 1,), dtype)
                o = _da_view(obuf, o_off, (1, h, w, c))
                fhost = np.zeros((h * w + 1) * 2, np.float32)
                fhost[2 * f_off:2 * f_off + h * w * 2] = flow.ravel()
                fbuf = DeviceArray.from_numpy(fhost)
                fl = _da_view(fbuf, 2 * f_off, (1, h, w, 2))
                vm = DeviceArray.empty((1, h, w), np.uint8)
                fmd = DeviceArray.from_numpy(fmask[None].view(np.uint8))
                before = _counters()
                _lib.call('ofk_warp_t_ex', p.ptr, _ops.dtype_code(dtype), c, _lib.ARITH_NATIVE, fl.ptr, -1.0, None,
                          fmd.ptr, None, o.ptr, vm.ptr, _lib.RULE_STRICT, 1, h, w, h, w, 0, 0, 1, None)
                got = o.numpy()[0]
                same_bits(got, want, (h, w, c, pname, p_off, o_off, f_off))
                assert (_counters() - before).tolist() == [0, 1]


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
def test_batches_with_zero_and_tiny_frames(of, dtype):
    """FlowBatch.apply of N = 4 frames (blockIdx.z frame offsets) equals the per-frame reference; a zero frame and a
    sub-threshold frame return their target byte for byte and the mask that went in."""
    rng = np.random.default_rng(5 + DTYPES.index(dtype))
    n = 4
    for (h, w, c) in ((21, 35, 3), (16, 48, 1), (10, 19, 5)):
        sets = flow_sets(rng, h, w)
        flows = np.stack([sets[0][1], sets[-2][1], sets[-1][1], sets[2][1]])
        pays = payload_sets(rng, dtype, (n, h, w, c))
        imgs = pays[-1][1] if np.dtype(dtype).kind == 'f' else pays[0][1]
        fm = rng.random((n, h, w)) > 0.1
        tm = rng.random((n, h, w)) > 0.15
        fb = of.FlowBatch(flows, 't', fm)
        out = fb.apply(imgs).numpy()
        for i in range(n):
            same_bits(out[i], ref_apply(flows[i], imgs[i], fm[i]), (h, w, c, i))
        for tms in ([None, tm] if dtype != np.uint16 else [tm]):
            got, valid = fb.apply(imgs, target_masks=tms, return_valid_area=True)
            got, valid = got.numpy(), valid.numpy().view(np.bool_)
            for i in range(n):
                want = ref_apply(flows[i], imgs[i], fm[i], target_mask=None if tms is None else tms[i],
                                 return_valid_area=True)
                same_bits(got[i], want[0], (h, w, c, i))
                same_bits(valid[i], want[1], (h, w, c, i))
            for i in (1, 2):
                same_bits(got[i], imgs[i])
                same_bits(valid[i], fm[i] if tms is None else tms[i] & fm[i])
        if dtype == np.uint16:
            with pytest.raises(TypeError):
                fb.apply(imgs, return_valid_area=True)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
def test_host_buffers_match_flowbatch(of, dtype):
    """apply_flow_host (ofh_warp_t's ring) equals FlowBatch.apply byte for byte, pageable and pinned, C = 1, 3, 5 and
    odd widths, zero and sub-threshold frames included; uint16 with a valid area needs a target mask on every entry."""
    rng = np.random.default_rng(6 + DTYPES.index(dtype))
    n, h, w = 5, 17, 31
    for c in (1, 3, 5):
        sets = flow_sets(rng, h, w)
        flows = np.stack([sets[k][1] for k in (0, -2, 1, -1, 2)])
        imgs = payload_sets(rng, dtype, (n, h, w, c))[-1][1]
        fm = rng.random((n, h, w)) > 0.1
        tm = rng.random((n, h, w)) > 0.15
        fb = of.FlowBatch(flows, 't', fm)
        want, want_v = [x.numpy() for x in fb.apply(imgs, target_masks=tm, return_valid_area=True)]
        same_bits(want[1], imgs[1])
        same_bits(want[3], imgs[3])
        got, got_v = of.batch.apply_flow_host(flows, imgs, flow_masks=fm, target_masks=tm, return_valid_area=True)
        same_bits(got, want)
        same_bits(got_v, want_v.view(np.bool_))
        pin, keep = of.device.pinned_empty(imgs.shape, imgs.dtype)
        pin[...] = imgs
        pout, keep2 = of.device.pinned_empty(imgs.shape, imgs.dtype)
        of.batch.apply_flow_host(flows, pin, out=pout)
        same_bits(pout, fb.apply(imgs).numpy())
        if dtype == np.uint16:
            with pytest.raises(TypeError):
                of.batch.apply_flow_host(flows, imgs, flow_masks=fm, return_valid_area=True)
            with pytest.raises(TypeError):
                of.batch.apply_combine_host(flows, flows, imgs)
            with pytest.raises(TypeError):
                of.Flow(flows[0], 't').apply(imgs[0], return_valid_area=True)
        else:
            out_i, out_v, _, _ = of.batch.apply_combine_host(flows, flows, imgs, 't', fm, fm)
            w2, v2 = [x.numpy() for x in fb.apply(imgs, return_valid_area=True)]
            same_bits(out_i, w2)
            same_bits(out_v, v2.view(np.bool_))


@pytest.mark.gpu
def test_host_ring_chunks(of):
    """Chunks of several frames with a short last chunk (7 frames, 3 per chunk), and a frame that is a chunk of its
    own, for a float payload (pass-through flags travel in the ring) and a uint8 one."""
    rng = np.random.default_rng(8)
    for (n, h, w, c, dtype) in ((7, 721, 1283, 3, np.uint8), (7, 361, 1283, 3, np.float32),
                                (2, 1080, 1921, 3, np.float32)):
        from test_gpu_warp_t import _rough_flow
        flows = np.stack([_rough_flow(rng, h, w, 'blocks') for _ in range(n)])
        flows[n // 2] = 0
        if np.dtype(dtype).kind == 'f':
            imgs = rng.standard_normal((n, h, w, c)).astype(dtype)
            imgs[rng.random((n, h, w, c)) < 0.01] = np.nan
        else:
            imgs = rng.integers(0, 256, (n, h, w, c), dtype=np.uint8)
        tm = rng.random((n, h, w)) > 0.1
        fb = of.FlowBatch(flows, 't')
        want, want_v = [x.numpy() for x in fb.apply(imgs, target_masks=tm, return_valid_area=True)]
        same_bits(want[n // 2], imgs[n // 2])
        got, got_v = of.batch.apply_flow_host(flows, imgs, target_masks=tm, return_valid_area=True)
        same_bits(got, want)
        same_bits(got_v, want_v.view(np.bool_))


@pytest.mark.gpu
def test_1080p_every_dtype(of):
    """One 1080p frame per dtype and C = 3 (warp_t_rows for float32, generic for the rest, u8x3 at W = 1919)."""
    rng = np.random.default_rng(9)
    from test_gpu_warp_t import _rough_flow
    for dtype in DTYPES:
        for w in ((1920, 1919) if dtype == np.uint8 else (1920,)):
            h = 1080
            flow = _rough_flow(rng, h, w, 'blocks') + _smooth(rng, h, w)
            pay = payload_sets(rng, dtype, (h, w, 3))
            img = pay[-1][1] if np.dtype(dtype).kind == 'f' else pay[0][1]
            fm = rng.random((h, w)) > 0.05
            f = of.Flow(flow, 't', fm)
            same_bits(f.apply(img), ref_apply(flow, img, fm), (dtype, w))
            tm = rng.random((h, w)) > 0.05
            got = f.apply(img, target_mask=tm, return_valid_area=True)
            want = ref_apply(flow, img, fm, target_mask=tm, return_valid_area=True)
            same_bits(got[0], want[0], (dtype, w))
            same_bits(got[1], want[1], (dtype, w))


@pytest.mark.gpu
@pytest.mark.parametrize('side', [16001, 16400])
def test_frames_at_the_rows_kernel_bound(of, side):
    """uint8 x 4 at 16001^2 (H*W*C just under 2^30: warp_t_rows with its 32-bit frame-local tap offsets) and 16400^2
    (just over: warp_t_generic). W % 16 != 0 keeps the TMA kernel out. A translation by (-2 - 33/64, 1.5) lets the
    first and last rows be checked against cv2.remap on bands of the payload."""
    torch = pytest.importorskip('torch')
    h = w = side
    assert (h * w * 4 < 1 << 30) == (side == 16001)
    dx, dy = -2.515625, 1.5
    g = torch.Generator(device='cuda').manual_seed(10)
    flow = torch.empty((1, h, w, 2), dtype=torch.float32, device='cuda')
    flow[..., 0], flow[..., 1] = dx, dy
    pay = torch.randint(0, 256, (1, h, w, 4), dtype=torch.uint8, device='cuda', generator=g)
    before = _counters()
    out = of.FlowBatch(flow, 't', validate=False).apply(pay)
    torch.cuda.synchronize()
    assert (_counters() - before).tolist() == [0, 1]
    host_out = out.numpy()
    del out
    for y0, y1 in ((0, 40), (h - 40, h)):
        r0, r1 = max(0, y0 - 4), min(h, y1 + 4)
        band = pay[0, r0:r1].cpu().numpy()
        yy, xx = np.mgrid[y0:y1, 0:w].astype(np.float32)
        mx = (np.float32(-dx) + xx).astype(np.float32)
        my = (np.float32(-dy) + yy).astype(np.float32) - np.float32(r0)
        want = cv2.remap(band, np.dstack([mx, my]), None, cv2.INTER_LINEAR)
        same_bits(host_out[0, y0:y1], want, (side, y0))


_WS_CODE = r'''
import sys, hashlib, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import oflibnumpy_b200 as of
from oflibnumpy_b200 import _lib
import test_gpu_warp_t as t
lib = _lib.load()
rng = np.random.default_rng(12)
hsh = hashlib.sha256()
for (hh, ww) in ((40, 64), (33, 160)):
    flow = t._rough_flow(rng, hh, ww, 'blocks') + t._smooth_flow(rng, hh, ww, 3)
    fm, tm = rng.random((hh, ww)) > 0.1, rng.random((hh, ww)) > 0.1
    f = of.Flow(flow, 't', fm)
    for c in (0, 1, 3, 4):
        img = rng.integers(0, 256, (hh, ww, max(c, 1)), dtype=np.uint8)
        img = img[..., 0] if c == 0 else img
        for res in (f.apply(img), *f.apply(img, return_valid_area=True),
                    *f.apply(img, target_mask=tm, return_valid_area=True)):
            hsh.update(np.ascontiguousarray(res).tobytes())
print('PATHS', lib.ofk_rt_path_count(2), lib.ofk_rt_path_count(3))
print('DIGEST', hsh.hexdigest())
'''


@pytest.mark.gpu
def test_warp_ws_off_gives_the_same_bytes():
    """OFK_WARP_WS=0 (read once per process) sends uint8 C = 1, 3, 4 at W % 16 == 0 to warp_t_rows / warp_t_u8x3
    instead of the TMA kernel: both arithmetic modes, same bytes."""
    code = _WS_CODE % (ROOT, HERE)
    outs = []
    for env_extra in ({}, {'OFK_WARP_WS': '0'}):
        res = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, **env_extra), capture_output=True,
                             text=True, timeout=600)
        assert res.returncode == 0, res.stdout + res.stderr
        lines = dict(l.split(' ', 1) for l in res.stdout.splitlines() if l.startswith(('PATHS', 'DIGEST')))
        outs.append(lines)
    tma_on = [int(x) for x in outs[0]['PATHS'].split()]
    tma_off = [int(x) for x in outs[1]['PATHS'].split()]
    assert tma_on[0] > 0 and tma_on[1] == 0, tma_on
    assert tma_off[0] == 0 and tma_off[1] > 0, tma_off
    assert outs[0]['DIGEST'] == outs[1]['DIGEST']


@pytest.mark.gpu
def test_valid_target_vector_and_fallback_paths(of):
    """valid_target through valid_geom_vec4 (W % 4 == 0, aligned) and its fallback (W % 4 != 0, and an unaligned
    mask pointer through ofk_valid_geom_t), against the reference."""
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.device import DeviceArray
    rng = np.random.default_rng(13)
    for (h, w) in ((13, 16), (13, 17), (1, 1), (7, 155), (9, 64)):
        for fname, flow in flow_sets(rng, h, w):
            fm = rng.random((h, w)) > 0.1
            want = R.valid_target(R.make(flow, 't', fm))
            same_bits(of.Flow(flow, 't', fm).valid_target(), want, (h, w, fname))
            mbuf = DeviceArray.from_numpy(np.concatenate([[1], fm.ravel().view(np.uint8)]).astype(np.uint8))
            m = _da_view(mbuf, 1, (1, h, w))
            fl = DeviceArray.from_numpy(flow[None])
            out = DeviceArray.empty((1, h, w), np.uint8)
            _lib.call('ofk_valid_geom_t', fl.ptr, -1.0, m.ptr, out.ptr, 1, h, w, None)
            same_bits(out.numpy()[0].view(np.bool_), want, (h, w, fname, 'unaligned mask'))
