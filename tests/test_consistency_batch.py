"""Forward-backward consistency check: FlowBatch.consistent_with / Flow.consistent_with (ofk_consistency). For every
pixel p, with w = self[p] and s = Q(other, p + sign*w) (the cv2.remap sample of the mode-3 composition), in float32
with every operation rounded on its own:

    valid = self_mask[p] & strict(other_mask at the taps);  consistent = valid & (|w + s|^2 < a1 (|w|^2 + |s|^2) + a2)

(w + s, valid) is the composition self.combine_with(other, 3) for ref 's' and other.combine_with(self, 3) for ref 't'.
The test's own oracle restates this on oracle/remap_q32; the GPU output must equal it byte for byte."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import flowref as R
from oracle import remap_q32 as Q

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALPHAS = [(None, None), (0.0, 0.0), (0.05, 2.0), (0.01, 1e4)]
SIZES = [(1080, 1920), (64, 96), (37, 53), (375, 1242)]
MASKS = [None, 0.05, 0.5]


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


# ---------------------------------------------------------------------------------------------------------- oracle
def oracle(fw, fm, bw, bm, ref, a1=None, a2=None):
    """One frame: fw, bw (H,W,2) float32, fm, bm (H,W) bool or None. Returns (consistent, valid, r, s) with r = w + s
    and s the sampled backward flow, (H,W,2) float32."""
    h, w = fw.shape[:2]
    a1 = np.float32(0.01 if a1 is None else a1)
    a2 = np.float32(0.5 if a2 is None else a2)
    fm = np.ones((h, w), bool) if fm is None else fm
    bm = np.ones((h, w), bool) if bm is None else bm
    mx, my = Q.backward_map(fw, 1.0 if ref == 's' else -1.0)
    ix, iy, a, b = Q.quantise_coords(mx, my)
    weights = Q.float_weights(a, b)
    s = np.zeros((h, w, 2), np.float32)
    for k, (dy, dx) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
        yy, xx = iy + dy, ix + dx
        inside = (yy >= 0) & (yy < h) & (xx >= 0) & (xx < w)
        tap = np.where(inside[..., None], bw[np.clip(yy, 0, h - 1), np.clip(xx, 0, w - 1)], np.float32(0))
        s = tap * weights[k][..., None] if k == 0 else s + tap * weights[k][..., None]
    valid = fm & (Q.valid_weight_sum(bm, mx, my) == 1024)
    r = fw + s
    lhs = r[..., 0] * r[..., 0] + r[..., 1] * r[..., 1]
    ww = fw[..., 0] * fw[..., 0] + fw[..., 1] * fw[..., 1]
    ss = s[..., 0] * s[..., 0] + s[..., 1] * s[..., 1]
    rhs = a1 * (ww + ss) + a2
    assert lhs.dtype == rhs.dtype == np.float32
    return valid & (lhs < rhs), valid, r, s


def smooth_pair(h, w, n, ref, seed):
    """Forward flows of smooth per-frame transforms and noisy approximations of their inverses."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    fw, bw = [], []
    for _ in range(n):
        th, tx, ty = rng.uniform(-0.03, 0.03), rng.uniform(-6, 6), rng.uniform(-6, 6)
        c, s_ = np.cos(th), np.sin(th)
        u = (c - 1) * (xx - w / 2) - s_ * (yy - h / 2) + tx
        v = s_ * (xx - w / 2) + (c - 1) * (yy - h / 2) + ty
        f = np.stack([u, v], -1).astype(np.float32)
        fw.append(f)
        bw.append((-f + rng.normal(0, 0.6, f.shape)).astype(np.float32))
    return np.stack(fw), np.stack(bw)


def rough_pair(h, w, n, ref, seed):
    """Noise and motion boundaries every 50 px: tiles whose boxes do not cover their taps (counter 4 moves)."""
    rng = np.random.default_rng(seed)
    fw = rng.uniform(-4, 4, (n, h, w, 2)).astype(np.float32)
    yy, xx = np.mgrid[0:h, 0:w]
    jump = (((xx // 50) + (yy // 50)) % 2 == 1)
    fw[:, jump] += np.float32(60)
    bw = (-fw + rng.normal(0, 1.0, fw.shape)).astype(np.float32)
    bw[:, rng.random((h, w)) < 0.1] *= np.float32(-1)
    return fw, bw


def make_masks(n, h, w, frac, seed):
    if frac is None:
        return None, None
    rng = np.random.default_rng(seed)
    return rng.random((n, h, w)) >= frac, rng.random((n, h, w)) >= frac


def squares(h, w, ref):
    """Three squares moving by (+10, 0) px over a static background: sq1 inside the frame, sq2 leaving on the right,
    sq3 entering on the left. Returns (forward, backward) flows of reference ref, and the expected (consistent,
    valid)."""
    f1 = [(slice(30, 50), 40, 60), (slice(60, 75), w - 12, w), (slice(90, 100), -5, 5)]   # rows, x0, x1 in frame 1
    fwd, bwd = np.zeros((h, w, 2), np.float32), np.zeros((h, w, 2), np.float32)
    for rows, x0, x1 in f1:
        frame1 = slice(max(x0, 0), min(x1, w))
        frame2 = slice(max(x0 + 10, 0), min(x1 + 10, w))
        if ref == 's':          # forward on frame 1's grid, backward on frame 2's grid
            fwd[rows, frame1, 0] = 10
            bwd[rows, frame2, 0] = -10
        else:                   # forward on frame 2's grid, backward on frame 1's grid
            fwd[rows, frame2, 0] = 10
            bwd[rows, frame1, 0] = -10
    cons, valid = np.ones((h, w), bool), np.ones((h, w), bool)
    if ref == 's':
        cons[30:50, 60:70] = False                    # background of frame 1 that sq1 covers in frame 2
        cons[90:100, 5:15] = False                    # ... and that sq3 covers
        valid[60:75, w - 10:w] = False                # sq2 pixels that leave the frame
    else:
        cons[30:50, 40:50] = False                    # background of frame 2 that sq1 uncovers
        cons[60:75, w - 12:w - 2] = False             # ... that sq2 uncovers
        cons[90:100, 0:5] = False                     # ... that sq3 uncovers
        valid[90:100, 5:10] = False                   # sq3 pixels that come from outside frame 1
    return fwd, bwd, cons & valid, valid


# ------------------------------------------------------------------------------------------------------------- CPU
def test_bad_arguments_are_rejected_without_a_gpu(lib):
    """ofk_consistency checks every argument before a stream or the device is touched."""
    good = dict(F=16, Fm=16, G=16, Gm=16, ref=ord('s'), a1=0.01, a2=0.5, out=16, out_valid=16, N=2, H=4, W=4,
                stream=None)
    for change, msg in (({'F': None}, "NULL pointer"), ({'G': None}, "NULL pointer"), ({'out': None}, "NULL pointer"),
                        ({'Fm': None}, "Fm and Gm must both be given or both be NULL"),
                        ({'Gm': None}, "Fm and Gm must both be given or both be NULL"),
                        ({'ref': ord('x')}, "ref must be 's' or 't'"), ({'ref': 0}, "ref must be 's' or 't'"),
                        ({'a1': -1.0}, "alpha1 and alpha2 must be finite and >= 0"),
                        ({'a2': -1e-30}, "alpha1 and alpha2 must be finite and >= 0"),
                        ({'a1': float('nan')}, "alpha1 and alpha2 must be finite and >= 0"),
                        ({'a2': float('inf')}, "alpha1 and alpha2 must be finite and >= 0"),
                        ({'N': -1}, "bad shape"), ({'H': 0}, "bad shape"), ({'W': -2}, "bad shape"),
                        ({'W': 32768}, "bad shape"), ({'H': 40000}, "bad shape"),
                        ({'N': 65536}, "exceeds 65535 frames"),
                        ({'F': 20}, "F and G must be 8-byte aligned"), ({'G': 12}, "F and G must be 8-byte aligned")):
        args = dict(good, **change)
        with pytest.raises(lib.OflibCudaError, match="ofk_consistency: .*" + msg):
            lib.call('ofk_consistency', *args.values())
    # N = 0 passes the checks and does nothing, also without a device
    lib.call('ofk_consistency', *dict(good, N=0).values())
    lib.call('ofk_consistency', *dict(good, N=0, Fm=None, Gm=None, out_valid=None).values())


def fakes(ref='t', n=4, h=3, w=5):
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    from oflibnumpy_b200.flow import Flow
    batch = FlowBatch._wrap(DeviceArray(0, (n, h, w, 2), np.float32), ref, DeviceArray(0, (n, h, w), np.uint8))
    flow = Flow._wrap(DeviceArray(0, (1, h, w, 2), np.float32), ref, DeviceArray(0, (1, h, w), np.uint8))
    return batch, flow


@pytest.mark.parametrize('kind', ['batch', 'flow'])
def test_python_messages(lib, kind):
    pre = "Error checking flow consistency: "
    b, f = fakes()
    x = b if kind == 'batch' else f
    name = 'FlowBatch' if kind == 'batch' else 'Flow'
    for other in (f if kind == 'batch' else b, x.vecs if kind == 'batch' else None, 3):
        with pytest.raises(TypeError) as e:
            x.consistent_with(other)
        assert str(e.value) == pre + "Flow need to be of type '{}'".format(name)
    others = [fakes(h=4)[0 if kind == 'batch' else 1], fakes(w=6)[0 if kind == 'batch' else 1]]
    if kind == 'batch':
        others.append(fakes(n=3)[0])
    for other in others:
        with pytest.raises(ValueError) as e:
            x.consistent_with(other)
        assert str(e.value) == pre + "Flow fields need to have the same shape"
    with pytest.raises(ValueError) as e:
        x.consistent_with(fakes('s')[0 if kind == 'batch' else 1])
    assert str(e.value) == pre + "Flow fields need to have the same reference"
    for bad in (-1, -1e-9, float('nan'), float('inf'), -float('inf'), 1e39, True, False, np.bool_(True), '0.1',
                [0.1], 1j, np.float64(-2)):
        for k, kw in ((1, 'alpha_1'), (2, 'alpha_2')):
            with pytest.raises(ValueError) as e:
                x.consistent_with(x, **{kw: bad})
            assert str(e.value) == pre + "Alpha_{} needs to be a non-negative finite number, not {!r}".format(k, bad)
    for bad in (1, 0, 'yes', np.bool_(True)):
        with pytest.raises(TypeError) as e:
            x.consistent_with(x, return_valid_area=bad)
        assert str(e.value) == pre + "Return_valid_area needs to be a boolean"


def test_validation_defaults_and_accepted_numbers(lib):
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.validation import validate_consistency_args
    b, _ = fakes()
    assert validate_consistency_args(b, b, None, None, False, FlowBatch) == (0.01, 0.5)
    for a in (0, 2, 0.25, np.float32(0.5), np.float64(3), np.int64(7), 3.4e38):
        assert validate_consistency_args(b, b, a, a, True, FlowBatch) == (float(a), float(a))


@pytest.mark.parametrize('ref', ['s', 't'])
@pytest.mark.parametrize('kind', ['smooth', 'rough'])
def test_oracle_is_the_composition(monkeypatch, ref, kind):
    """The oracle's (w + s, valid) are oracle.flowref.combine's vectors and mask on non-zero pairs, with the operand
    order of the contract."""
    monkeypatch.setattr(R, 'REMAP_IMPL', 'q32')
    h, w = 37, 53
    fw, bw = (smooth_pair if kind == 'smooth' else rough_pair)(h, w, 1, ref, 3)
    fm, bm = make_masks(1, h, w, 0.05, 4)
    _, valid, r, s = oracle(fw[0], fm[0], bw[0], bm[0], ref)
    F, G = R.make(fw[0], ref, fm[0]), R.make(bw[0], ref, bm[0])
    comp = R.combine(F, G, 3) if ref == 's' else R.combine(G, F, 3)
    assert comp.vecs.tobytes() == r.tobytes()
    np.testing.assert_array_equal(comp.mask, valid)
    # s is the warp of the backward flow: invert('t').apply for 's', apply for 't'
    warped = R.apply(R.invert(F, 't') if ref == 's' else F, bw[0])
    assert np.asarray(warped, np.float32).tobytes() == s.tobytes()


@pytest.mark.parametrize('ref', ['s', 't'])
def test_oracle_moving_squares(ref):
    fwd, bwd, want_c, want_v = squares(120, 160, ref)
    c, v, _, _ = oracle(fwd, None, bwd, None, ref)
    np.testing.assert_array_equal(v, want_v)
    np.testing.assert_array_equal(c, want_c)
    assert (want_v & ~want_c).sum() > 0


# ------------------------------------------------------------------------------------------------------------- GPU
def gpu_case(of, fw, bw, fm, bm, ref, alphas, valid=True):
    F, G = of.FlowBatch(fw, ref, fm), of.FlowBatch(bw, ref, bm)
    a1, a2 = alphas
    c, v = F.consistent_with(G, a1, a2, return_valid_area=True)
    return c.numpy(), v.numpy()


def check_against_oracle(got_c, got_v, fw, bw, fm, bm, ref, a1, a2, tag):
    for i in range(len(fw)):
        c, v, _, _ = oracle(fw[i], None if fm is None else fm[i], bw[i], None if bm is None else bm[i], ref, a1, a2)
        np.testing.assert_array_equal(got_v[i], v.view(np.uint8), err_msg=str(tag + (i, 'valid')))
        np.testing.assert_array_equal(got_c[i], c.view(np.uint8), err_msg=str(tag + (i, 'consistent')))


def parity_inputs():
    for (h, w) in SIZES:
        n = 2 if h * w > 1e6 else 3
        for kind in ('smooth', 'rough'):
            for frac in MASKS:
                yield h, w, n, kind, frac


def build_case(h, w, n, kind, frac, ref):
    seed = h * 7 + w + (1 if kind == 'rough' else 0) + (0 if frac is None else int(frac * 100)) + ord(ref)
    fw, bw = (smooth_pair if kind == 'smooth' else rough_pair)(h, w, n, ref, seed)
    fm, bm = make_masks(n, h, w, frac, seed + 1)
    return fw, bw, fm, bm


def all_outputs(of):
    """Both outputs of every parity case (in order), as one dict of arrays."""
    out = {}
    for ref in ('s', 't'):
        for h, w, n, kind, frac in parity_inputs():
            fw, bw, fm, bm = build_case(h, w, n, kind, frac, ref)
            for k, al in enumerate(ALPHAS):
                c, v = gpu_case(of, fw, bw, fm, bm, ref, al)
                key = '{}_{}x{}_{}_{}_{}'.format(ref, h, w, kind, frac, k)
                out[key + '_c'], out[key + '_v'] = c, v
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
def test_parity_with_the_oracle(of, ref):
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.device import DeviceArray
    mixed_before = _lib.call('ofk_rt_path_count', 4)
    for h, w, n, kind, frac in parity_inputs():
        fw, bw, fm, bm = build_case(h, w, n, kind, frac, ref)
        for al in ALPHAS:
            tma_before = [_lib.call('ofk_rt_path_count', k) for k in (12, 13)]
            c, v = gpu_case(of, fw, bw, fm, bm, ref, al)
            after = [_lib.call('ofk_rt_path_count', k) for k in (12, 13)]
            want = [1, 0] if w % 16 == 0 else [0, 1]
            assert [a - b for a, b in zip(after, tma_before)] == want, (h, w)
            check_against_oracle(c, v, fw, bw, fm, bm, ref, al[0], al[1], (ref, h, w, kind, frac, al))
        if frac is None:
            # NULL masks at the C level are all-valid masks
            Fd, Gd = DeviceArray.from_numpy(fw), DeviceArray.from_numpy(bw)
            from oflibnumpy_b200 import _ops
            c2, v2 = _ops.consistency(Fd, None, Gd, None, ref, 0.01, 0.5, True)
            c1, v1 = gpu_case(of, fw, bw, None, None, ref, (None, None))
            np.testing.assert_array_equal(c2.numpy(), c1)
            np.testing.assert_array_equal(v2.numpy(), v1)
            c3, _ = _ops.consistency(Fd, None, Gd, None, ref, 0.01, 0.5, False)
            np.testing.assert_array_equal(c3.numpy(), c1)
    # the rough inputs sent warps of the TMA kernel to the global-tap path
    assert _lib.call('ofk_rt_path_count', 4) > mixed_before


@pytest.mark.gpu
def test_gather_kernel_gives_the_same_bytes(of, tmp_path):
    """OFK_C3_WS=0 forces the rows kernel: every output of the parity cases is identical."""
    path = str(tmp_path / 'rows.npz')
    code = ("import sys, numpy as np; sys.path[:0] = [{root!r}, {tests!r}]; import oflibnumpy_b200 as of; "
            "import test_consistency_batch as T; from oflibnumpy_b200 import _lib; of.device.require_gpu(); "
            "out = T.all_outputs(of); np.savez({path!r}, **out); "
            "print(_lib.call('ofk_rt_path_count', 12), _lib.call('ofk_rt_path_count', 13), len(out) // 2)"
            ).format(root=ROOT, tests=os.path.join(ROOT, 'tests'), path=path)
    env = dict(os.environ, OFK_C3_WS='0')
    res = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=1800)
    assert res.returncode == 0, res.stderr[-3000:]
    tma, rows, cases = (int(x) for x in res.stdout.split()[-3:])
    assert tma == 0 and rows == cases
    rows_out = np.load(path)
    here = all_outputs(of)
    assert sorted(here) == sorted(rows_out.files)
    for k in here:
        np.testing.assert_array_equal(here[k], rows_out[k], err_msg=k)


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
@pytest.mark.parametrize('hw', [(1080, 1920), (37, 53)])
def test_agrees_with_combine_with_and_apply(of, ref, hw):
    h, w = hw
    fw, bw = rough_pair(h, w, 2, ref, 11)
    fm, bm = make_masks(2, h, w, 0.05, 12)
    F, G = of.FlowBatch(fw, ref, fm), of.FlowBatch(bw, ref, bm)
    c, v = (x.numpy() for x in F.consistent_with(G, return_valid_area=True))
    comp = F.combine_with(G, 3) if ref == 's' else G.combine_with(F, 3)
    rv, rm = comp.numpy()
    np.testing.assert_array_equal(v, rm.view(np.uint8))
    s = (F.invert('t') if ref == 's' else F).apply(bw).numpy()
    lhs = rv[..., 0] * rv[..., 0] + rv[..., 1] * rv[..., 1]
    rhs = np.float32(0.01) * ((fw[..., 0] * fw[..., 0] + fw[..., 1] * fw[..., 1]) +
                              (s[..., 0] * s[..., 0] + s[..., 1] * s[..., 1])) + np.float32(0.5)
    np.testing.assert_array_equal(c, (rm & (lhs < rhs)).view(np.uint8))
    np.testing.assert_array_equal(rv, fw + s)


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
@pytest.mark.parametrize('w', [160, 157])
def test_moving_squares(of, ref, w):
    fwd, bwd, want_c, want_v = squares(120, w, ref)
    c, v = of.Flow(fwd, ref).consistent_with(of.Flow(bwd, ref), return_valid_area=True)
    assert c.dtype == v.dtype == np.bool_ and c.shape == v.shape == (120, w)
    np.testing.assert_array_equal(v, want_v)
    np.testing.assert_array_equal(c, want_c)
    np.testing.assert_array_equal(of.Flow(fwd, ref).consistent_with(of.Flow(bwd, ref)), want_c)


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
def test_exact_inverse_pairs_and_zero_flows(of, ref):
    h, w = 240, 320
    fwd = [[['rotation', 150, 100, 7]], [['translation', 12, -5]], [['rotation', 30, 200, -3], ['translation', 2, 3]]]
    bwd = [[['rotation', 150, 100, -7]], [['translation', -12, 5]], [['translation', -2, -3], ['rotation', 30, 200, 3]]]
    F, G = of.FlowBatch.from_transforms(fwd, (h, w), ref), of.FlowBatch.from_transforms(bwd, (h, w), ref)
    c, v = (x.numpy() for x in F.consistent_with(G, return_valid_area=True))
    assert v.sum() > 0.5 * v.size
    np.testing.assert_array_equal(c, v)
    zero = of.FlowBatch(np.zeros((2, h, w, 2), np.float32), ref, np.random.default_rng(0).random((2, h, w)) > 0.3)
    c, v = (x.numpy() for x in zero.consistent_with(zero, return_valid_area=True))
    np.testing.assert_array_equal(c, v)
    np.testing.assert_array_equal(v, zero.masks.numpy())
    c = zero.consistent_with(zero, 0, 0).numpy()
    assert not c.any()


@pytest.mark.gpu
@pytest.mark.parametrize('ref', ['s', 't'])
def test_batches_frames_and_slices(of, ref):
    h, w = 64, 96
    fw, bw = rough_pair(h, w, 7, ref, 21)
    fm, bm = make_masks(7, h, w, 0.05, 22)
    F, G = of.FlowBatch(fw, ref, fm), of.FlowBatch(bw, ref, bm)
    c, v = (x.numpy() for x in F.consistent_with(G, 0.05, 2.0, return_valid_area=True))
    for i in range(7):
        fc, fv = F[i].consistent_with(G[i], 0.05, 2.0, return_valid_area=True)
        np.testing.assert_array_equal(c[i], fc.view(np.uint8))
        np.testing.assert_array_equal(v[i], fv.view(np.uint8))
        alone = of.FlowBatch(fw[i:i + 1], ref, fm[i:i + 1]).consistent_with(of.FlowBatch(bw[i:i + 1], ref, bm[i:i + 1]),
                                                                            0.05, 2.0)
        np.testing.assert_array_equal(c[i:i + 1], alone.numpy())
    for start, stop in ((1, 4), (3, 7), (5, 6)):      # offset views: mask bases not 16-byte aligned for odd starts
        sc = F[start:stop].consistent_with(G[start:stop], 0.05, 2.0).numpy()
        np.testing.assert_array_equal(sc, c[start:stop])
    e = F[2:2].consistent_with(G[2:2], return_valid_area=True)
    assert e[0].shape == e[1].shape == (0, h, w) and e[0].dtype == np.uint8


@pytest.mark.gpu
def test_one_launch_and_no_read_back(of, monkeypatch):
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.device import DeviceArray
    rng = np.random.default_rng(5)
    for n in (2, 64):
        for h, w in ((64, 96), (37, 53)):
            for ref in ('s', 't'):
                F = of.FlowBatch(rng.uniform(-3, 3, (n, h, w, 2)).astype(np.float32), ref, rng.random((n, h, w)) > .1)
                G = of.FlowBatch(rng.uniform(-3, 3, (n, h, w, 2)).astype(np.float32), ref, rng.random((n, h, w)) > .1)
                F.consistent_with(G)
                before = _lib.call('ofk_rt_launch_count')
                F.consistent_with(G, return_valid_area=True)
                assert _lib.call('ofk_rt_launch_count') - before == 1, (n, h, w, ref)
                before = _lib.call('ofk_rt_launch_count')
                F[0:0].consistent_with(G[0:0])
                assert _lib.call('ofk_rt_launch_count') == before
    real_call = _lib.call

    def no_sync(name, *args):
        assert name not in ('ofk_rt_memcpy_d2h', 'ofk_rt_stream_sync', 'ofk_rt_device_sync', 'ofk_rt_event_sync'), name
        return real_call(name, *args)

    def no_numpy(self, out=None):
        raise AssertionError("DeviceArray.numpy called")

    monkeypatch.setattr(_lib, 'call', no_sync)
    monkeypatch.setattr(DeviceArray, 'numpy', no_numpy)
    res = F.consistent_with(G, return_valid_area=True)
    monkeypatch.undo()
    assert res[0].shape == (64, 37, 53)
