"""Flow error metrics: FlowBatch.evaluate / Flow.evaluate / evaluate_flows_host (ofk_evaluate, ofh_evaluate). For every
pixel, with (ue, ve) the estimate and (ug, vg) the truth, in float32 with every operation rounded on its own:

    du = ue - ug;  dv = ve - vg;  d2 = du*du + dv*dv;  epe = sqrt(d2);  mg = sqrt(ug*ug + vg*vg)
    fl = epe > 3 & epe / mg > 0.05;  out_k = epe > k;  band = 0 if mg < 10, 1 if mg < 40, else 2
    cz = ue*vg - ve*ug;  cr = sqrt(d2 + cz*cz);  dot = (1 + ue*ug) + ve*vg;  ae = atan2(cr, dot) * 57.29578

over the pixels est_mask & truth_mask & region. The numpy oracle below restates this; the EPE map must equal it byte
for byte, the counts exactly, the EPE sums within 1e-12 of math.fsum and the AE sums within 1e-6 (atan2f is not
correctly rounded on either side)."""
import math
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [(1080, 1920), (375, 1242), (436, 1024), (64, 96), (37, 53)]
MASKS = [None, 0.05, 0.5]
KITTI = os.path.join(ROOT, 'tests', 'golden', 'files', 'kitti_sample.png')


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
def oracle(est, truth):
    """Per-pixel (epe, ae, fl, band) of float32 arrays (..., 2)."""
    with np.errstate(over='ignore', invalid='ignore', divide='ignore'):
        ue, ve, ug, vg = est[..., 0], est[..., 1], truth[..., 0], truth[..., 1]
        du, dv = ue - ug, ve - vg
        d2 = du * du + dv * dv
        epe = np.sqrt(d2)
        mg = np.sqrt(ug * ug + vg * vg)
        fl = (epe > np.float32(3)) & (epe / mg > np.float32(0.05))
        cz = ue * vg - ve * ug
        cr = np.sqrt(d2 + cz * cz)
        dot = (np.float32(1) + ue * ug) + ve * vg
        ae = np.arctan2(cr, dot) * np.float32(57.29578)
        band = np.where(mg < np.float32(10), 0, np.where(mg < np.float32(40), 1, 2))
    assert epe.dtype == ae.dtype == np.float32
    return epe, ae, fl, band


def oracle_rows(est, truth, ev):
    """Rows of one frame: counts (8,) int64 and sums (5,) float64 by math.fsum."""
    epe, ae, fl, band = oracle(est, truth)
    ev = ev.astype(bool)
    sel = [ev, ev & fl, ev & (epe > 1), ev & (epe > 3), ev & (epe > 5), ev & (band == 0), ev & (band == 1),
           ev & (band == 2)]
    counts = np.array([s.sum() for s in sel], np.int64)
    sums = np.array([math.fsum(epe[ev].astype(np.float64)), math.fsum(ae[ev].astype(np.float64))] +
                    [math.fsum(epe[s].astype(np.float64)) for s in sel[5:]])
    return counts, sums


def close(got, want, rel):
    """|got - want| <= rel * |want|, with NaN = NaN and inf = inf."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    same = (got == want) | (np.isnan(got) & np.isnan(want))
    with np.errstate(invalid='ignore'):
        return bool(np.all(same | (np.abs(got - want) <= rel * np.abs(want))))


def smooth_pair(n, h, w, seed):
    """Truth: a smooth transform per frame; estimate: the truth plus low-amplitude noise."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    truth = []
    for _ in range(n):
        th, k, tx, ty = rng.uniform(-0.05, 0.05), rng.uniform(0.9, 1.1), rng.uniform(-20, 20), rng.uniform(-20, 20)
        c, s = k * np.cos(th), k * np.sin(th)
        u = (c - 1) * (xx - w / 2) - s * (yy - h / 2) + tx
        v = s * (xx - w / 2) + (c - 1) * (yy - h / 2) + ty
        truth.append(np.stack([u, v], -1))
    truth = np.stack(truth).astype(np.float32)
    est = (truth + rng.normal(0, 0.8, truth.shape)).astype(np.float32)
    return est, truth


def rough_pair(n, h, w, seed):
    """Motion boundaries every 40 px in the truth, blocks of large errors, exact copies, zero truth, and estimates off
    by exactly 3 px (the Fl and out_3 edges)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    truth = rng.uniform(-3, 3, (n, h, w, 2)).astype(np.float32)
    truth[:, ((xx // 40) + (yy // 40)) % 2 == 1] += np.float32(45)
    truth[:, (xx // 10) % 3 == 1] += np.float32([15, -12])
    est = (truth + rng.normal(0, 2.0, truth.shape)).astype(np.float32)
    est[:, (xx // 17) % 5 == 0] += rng.uniform(-80, 80, 2).astype(np.float32)
    est[:, (yy % 7) == 0] = truth[:, (yy % 7) == 0]
    zero = (xx % 11) == 3
    truth[:, zero] = 0
    edge = (xx % 13) == 5
    truth[:, edge] = np.round(truth[:, edge])
    est[:, edge] = truth[:, edge] + np.float32([3, 0])
    return est, truth


def make_masks(n, h, w, frac, where, seed):
    """(est_mask, truth_mask, region) with density frac of False where asked, else None."""
    if frac is None:
        return None, None, None
    rng = np.random.default_rng(seed)
    return tuple(rng.random((n, h, w)) >= frac if where in ('all', k) else None for k in ('est', 'truth', 'region'))


# ------------------------------------------------------------------------------------------------------------- CPU
def fakes(ref='t', n=4, h=3, w=5):
    from oflibnumpy_b200.batch import FlowBatch
    from oflibnumpy_b200.device import DeviceArray
    from oflibnumpy_b200.flow import Flow
    batch = FlowBatch._wrap(DeviceArray(0, (n, h, w, 2), np.float32), ref, DeviceArray(0, (n, h, w), np.uint8))
    flow = Flow._wrap(DeviceArray(0, (1, h, w, 2), np.float32), ref, DeviceArray(0, (1, h, w), np.uint8))
    return batch, flow


@pytest.mark.parametrize('kind', ['batch', 'flow'])
def test_python_messages(lib, kind):
    pre = "Error evaluating flow: "
    b, f = fakes()
    x = b if kind == 'batch' else f
    name = 'FlowBatch' if kind == 'batch' else 'Flow'
    for other in (f if kind == 'batch' else b, x.vecs if kind == 'batch' else None, 3):
        with pytest.raises(TypeError) as e:
            x.evaluate(other)
        assert str(e.value) == pre + "Truth needs to be of type '{}'".format(name)
    others = [fakes(h=4)[0 if kind == 'batch' else 1], fakes(w=6)[0 if kind == 'batch' else 1]]
    if kind == 'batch':
        others.append(fakes(n=3)[0])
    for other in others:
        with pytest.raises(ValueError) as e:
            x.evaluate(other)
        assert str(e.value) == pre + "Flow fields need to have the same shape"
    with pytest.raises(ValueError) as e:
        x.evaluate(fakes('s')[0 if kind == 'batch' else 1])
    assert str(e.value) == pre + "Flow fields need to have the same reference"
    shape = (4, 3, 5) if kind == 'batch' else (3, 5)
    for bad in (np.ones(shape[1:] if kind == 'batch' else (1,) + shape, bool), np.ones(shape, np.float32),
                np.ones(shape, np.int64), np.ones(shape[:-1] + (6,), bool)):
        with pytest.raises(ValueError) as e:
            x.evaluate(x, region=bad)
        assert str(e.value) == pre + "Region needs shape {} and dtype bool or uint8".format(shape)
    with pytest.raises(ValueError) as e:
        x.evaluate(x, region=np.full(shape, 2, np.uint8))
    assert str(e.value) == pre + "Region values must be 0 or 1"
    with pytest.raises(TypeError) as e:
        x.evaluate(x, region=[[1]])
    assert str(e.value) == pre + "Region needs to be a numpy or device array"
    if kind == 'batch':
        for bad in (1, 0, 'yes', None, np.bool_(True)):
            with pytest.raises(TypeError) as e:
                x.evaluate(x, return_epe=bad)
            assert str(e.value) == pre + "Return_epe needs to be a boolean"


def test_c_arguments_are_checked_without_a_gpu(lib):
    """ofk_evaluate / ofh_evaluate check every argument before a stream or the device is touched."""
    ws = lib.call('ofk_evaluate_workspace', 2, 4, 4)
    assert ws == 2 * 72
    assert lib.call('ofk_evaluate_workspace', 3, 1080, 1920) == 3 * 254 * 72
    assert lib.call('ofk_evaluate_workspace', 1, 37, 53) == 72
    for args in ((-1, 4, 4), (65536, 4, 4), (1, 0, 4), (1, 4, -1), (1, 46341, 46341)):
        assert lib.call('ofk_evaluate_workspace', *args) == 0
    good = dict(est=16, em=None, truth=16, tm=None, rg=None, epe=None, counts=16, sums=16, N=2, H=4, W=4, ws=16,
                ws_bytes=ws, stream=None)
    for change, msg in (({'est': None}, "NULL pointer"), ({'truth': None}, "NULL pointer"),
                        ({'counts': None}, "NULL pointer"), ({'sums': None}, "NULL pointer"),
                        ({'N': -1}, "bad shape"), ({'H': 0}, "bad shape"), ({'W': -2}, "bad shape"),
                        ({'N': 65536}, "exceeds 65535 frames"), ({'H': 46341, 'W': 46341}, "fewer than 2\\^31"),
                        ({'est': 20}, "est and truth must be 8-byte aligned"),
                        ({'truth': 12}, "est and truth must be 8-byte aligned"),
                        ({'counts': 20}, "counts and sums must be 8-byte aligned"),
                        ({'epe': 18}, "epe must be 4-byte aligned"),
                        ({'ws': None}, "workspace needs 144 bytes"), ({'ws_bytes': ws - 1}, "workspace needs"),
                        ({'ws': 20}, "workspace needs")):
        args = dict(good, **change)
        with pytest.raises(lib.OflibCudaError, match="ofk_evaluate: .*" + msg):
            lib.call('ofk_evaluate', *args.values())
    lib.call('ofk_evaluate', *dict(good, N=0, ws=None, ws_bytes=0).values())   # nothing to do, also without a device
    host = dict(good)
    del host['ws'], host['ws_bytes'], host['stream']
    host['device'] = 0
    for change, msg in (({'est': None}, "bad arguments"), ({'sums': None}, "bad arguments"),
                        ({'W': 0}, "bad arguments"), ({'N': 65536}, "exceeds 65535 frames")):
        with pytest.raises(lib.OflibCudaError, match="ofh_evaluate: .*" + msg):
            lib.call('ofh_evaluate', *dict(host, **change).values())


def test_host_entry_checks_shapes(lib):
    from oflibnumpy_b200.batch import evaluate_flows_host
    a = np.zeros((2, 3, 4, 2), np.float32)
    with pytest.raises(ValueError, match="estimates and truths need the same shape"):
        evaluate_flows_host(a, a[:1])
    with pytest.raises(ValueError, match="Regions need shape \\(2, 3, 4\\)"):
        evaluate_flows_host(a, a, regions=np.ones((2, 3, 5), bool))
    with pytest.raises(ValueError, match="out_epe needs to be"):
        evaluate_flows_host(a, a, out_epe=np.zeros((2, 3, 4), np.float64))


def test_oracle_hand_cases():
    f = np.float32
    # a pure translation error: EPE is its length
    truth = np.array([[[2.5, -1.0], [0.0, 0.0], [7.0, 3.0]]], f)
    est = truth + f([3, 4])
    epe, ae, _, _ = oracle(est, truth)
    assert np.all(epe == 5)
    # (1, 0) against (0, 1): the vectors (1, 0, 1) and (0, 1, 1) make 60 degrees
    epe, ae, _, _ = oracle(f([[1, 0]]), f([[0, 1]]))
    assert abs(float(ae[0]) - 60.0) < 1e-4 and epe[0] == f(math.sqrt(2))
    # identical flows: 0 exactly, for any truth
    t = np.random.default_rng(0).uniform(-300, 300, (1000, 2)).astype(f)
    epe, ae, fl, _ = oracle(t, t)
    assert not epe.any() and not ae.any() and not fl.any()
    # Fl at mg = 0: any EPE above 3 counts (epe / 0 = inf), 3 itself does not
    epe, _, fl, band = oracle(f([[3.5, 0], [3, 0], [0, 0]]), f([[0, 0], [0, 0], [0, 0]]))
    assert fl.tolist() == [True, False, False] and band.tolist() == [0, 0, 0]
    # Fl at epe = 3 exactly with a small truth: not an outlier (3 > 3 is false); just above with a large truth: the
    # relative test decides (3.5 / 100 < 0.05)
    epe, _, fl, band = oracle(f([[13, 0], [103.5, 0], [20, 4]]), f([[10, 0], [100, 0], [20, 0]]))
    assert epe.tolist() == [3, 3.5, 4] and fl.tolist() == [False, False, True] and band.tolist() == [1, 2, 1]
    # squares that overflow float32 give inf, as float32 arithmetic does
    epe, ae, fl, band = oracle(f([[3e38, 0], [2e19, 2e19], [1e30, 0]]), f([[-3e38, 0], [0, 0], [1e30, 0]]))
    assert np.isinf(epe[0]) and np.isinf(epe[1]) and epe[2] == 0
    assert band.tolist() == [2, 0, 2] and fl.tolist() == [False, True, False]
    assert ae[0] == np.float32(135) and ae[2] == 0          # atan2(inf, -inf), and atan2(0, inf)


def test_oracle_rows_and_summary():
    from oflibnumpy_b200.batch import FlowErrors
    f = np.float32
    truth = f([[[0, 0], [5, 0], [20, 0], [50, 0]]])
    est = truth + f([[[2, 0], [0, 4], [0, 0], [6, 8]]])
    ev = np.array([[True, True, False, True]])
    counts, sums = oracle_rows(est, truth, ev)
    assert counts.tolist() == [3, 2, 3, 2, 1, 2, 0, 1]
    np.testing.assert_array_equal(sums[[0, 2, 3, 4]], [16, 6, 0, 10])
    rows = FlowErrors(np.stack([counts, np.zeros(8, np.int64)]), np.stack([sums, np.zeros(5)]))
    s = rows.summary()
    assert s['pixels'] == 3 and s['epe'] == 16 / 3 and s['fl'] == 2 / 3 and s['out5'] == 1 / 3
    assert s['s0-10'] == 3 and math.isnan(s['s10-40']) and s['s40+'] == 10 and s['ae'] == sums[1] / 3
    assert set(s) == {'epe', 'ae', 'fl', 'out1', 'out3', 'out5', 's0-10', 's10-40', 's40+', 'pixels'}
    # two frames are weighted by their pixels and added in frame order
    c2 = np.array([[10, 1, 2, 3, 4, 10, 0, 0], [30, 3, 4, 5, 6, 0, 30, 0]], np.int64)
    s2 = np.array([[10.0, 1.0, 10.0, 0, 0], [0.1, 2.0, 0, 0.1, 0]])
    s = FlowErrors(c2, s2).summary()
    assert s['pixels'] == 40 and s['epe'] == (10.0 + 0.1) / 40 and s['fl'] == 0.1 and math.isnan(s['s40+'])
    empty = FlowErrors(np.zeros((0, 8), np.int64), np.zeros((0, 5))).summary()
    assert empty['pixels'] == 0 and all(math.isnan(v) for k, v in empty.items() if k != 'pixels')


# ------------------------------------------------------------------------------------------------------------- GPU
def check_rows(counts, sums, est, truth, ev, tag):
    for i in range(len(est)):
        wc, ws = oracle_rows(est[i], truth[i], ev[i])
        np.testing.assert_array_equal(counts[i], wc, err_msg=str(tag + (i,)))
        assert close(sums[i, [0, 2, 3, 4]], ws[[0, 2, 3, 4]], 1e-12), (tag, i, sums[i], ws)
        assert close(sums[i, 1], ws[1], 1e-6), (tag, i, sums[i, 1], ws[1])


def evaluated(n, h, w, em, tm, rg):
    ev = np.ones((n, h, w), bool)
    for m in (em, tm, rg):
        if m is not None:
            ev &= m
    return ev


def parity_cases():
    for h, w in SIZES:
        n = 2 if h * w > 1e6 else 5
        for kind in ('smooth', 'rough'):
            yield h, w, n, kind, None, None
            for frac in MASKS[1:]:
                for where in ('est', 'truth', 'region', 'all'):
                    yield h, w, n, kind, frac, where


@pytest.mark.gpu
def test_parity_with_the_oracle(of):
    for h, w, n, kind, frac, where in parity_cases():
        seed = h * 3 + w + (7 if kind == 'rough' else 0)
        est, truth = (smooth_pair if kind == 'smooth' else rough_pair)(n, h, w, seed)
        em, tm, rg = make_masks(n, h, w, frac, where, seed + int(100 * (frac or 0)) + len(where or ''))
        res = of.FlowBatch(est, 't', em).evaluate(of.FlowBatch(truth, 't', tm), region=rg, return_epe=True)
        counts, sums, epe = res.numpy()
        assert counts.dtype == np.int64 and counts.shape == (n, 8) and sums.dtype == np.float64 and \
            sums.shape == (n, 5) and epe.dtype == np.float32 and epe.shape == (n, h, w)
        tag = (h, w, kind, frac, where)
        assert epe.tobytes() == oracle(est, truth)[0].tobytes(), tag
        check_rows(counts, sums, est, truth, evaluated(n, h, w, em, tm, rg), tag)
        if frac == 0.5 and where == 'all':
            assert counts[:, 0].min() > 0 and counts[:, 0].max() < 0.2 * h * w
        if kind == 'rough' and frac is None:      # the rough fields reach every count
            assert (counts[:, 1:] > 0).all(), counts


@pytest.mark.gpu
def test_extreme_values(of):
    """Zero truth, EPE exactly 3, perfect estimates and inputs whose squares overflow, at both kernel paths."""
    f = np.float32
    for h, w in ((37, 53), (64, 96)):
        n = 4
        rng = np.random.default_rng(h)
        base = rng.uniform(-50, 50, (n, h, w, 2)).astype(f)
        truth, est = base.copy(), base.copy()
        est[:, ::3] += f([3e38, -2e30])
        truth[:, ::3] = f([-3e38, 1e20])                            # du overflows; mg overflows
        truth[:, 1::5, ::2] = 0                                     # mg = 0
        est[:, 1::5, ::2] = f([0, 3])                               # epe exactly 3 on zero truth
        truth[:, 2::5, 1::2] = f([1e-30, 1e19])
        est[:, 2::5, 1::2] = f([-1e-30, -1e19])
        res = of.FlowBatch(est, 's').evaluate(of.FlowBatch(truth, 's'), return_epe=True)
        counts, sums, epe = res.numpy()
        assert epe.tobytes() == oracle(est, truth)[0].tobytes()
        assert np.isinf(epe).any()
        check_rows(counts, sums, est, truth, np.ones((n, h, w), bool), (h, w))
        # a perfect estimate: no error at all, AE exactly 0
        perfect = of.FlowBatch(base, 's').evaluate(of.FlowBatch(base, 's')).numpy()
        assert not perfect[1].any() and (perfect[0][:, 0] == h * w).all() and not perfect[0][:, 1:5].any()


@pytest.mark.gpu
@pytest.mark.parametrize('hw', [(37, 53), (64, 96), (375, 1242)])
def test_rows_do_not_depend_on_the_batch(of, hw):
    """Frame i alone, at other positions of larger batches, as a slice, in a second call and through the host ring
    (pageable and pinned buffers): identical rows and maps. 37 x 53 is odd, so frames at n % 4 != 0 take the scalar
    loads and the others the vector loads; slices at odd starts move every base off 16 bytes."""
    from oflibnumpy_b200 import device
    from oflibnumpy_b200.batch import evaluate_flows_host
    h, w = hw
    n = 9
    est, truth = rough_pair(n, h, w, 5)
    em, tm, rg = make_masks(n, h, w, 0.05, 'all', 6)
    E, T = of.FlowBatch(est, 't', em), of.FlowBatch(truth, 't', tm)
    counts, sums, epe = E.evaluate(T, rg, return_epe=True).numpy()
    again = E.evaluate(T, rg, return_epe=True).numpy()
    assert all(a.tobytes() == b.tobytes() for a, b in zip((counts, sums, epe), again))
    for i in range(n):
        alone = of.FlowBatch(est[i:i + 1], 't', em[i:i + 1]).evaluate(of.FlowBatch(truth[i:i + 1], 't', tm[i:i + 1]),
                                                                      rg[i:i + 1], return_epe=True).numpy()
        assert all(a.tobytes() == b[i:i + 1].tobytes() for a, b in zip(alone, (counts, sums, epe))), i
        # frame i at position 3 of a larger batch
        order = [j for j in range(n) if j != i]
        order.insert(3, i)
        moved = of.FlowBatch(est[order], 't', em[order]).evaluate(of.FlowBatch(truth[order], 't', tm[order]),
                                                                  rg[order], return_epe=True).numpy()
        assert all(a[3].tobytes() == b[i].tobytes() for a, b in zip(moved, (counts, sums, epe))), i
    for start, stop in ((1, 4), (3, 8), (5, 6), (0, 9)):
        part = E[start:stop].evaluate(T[start:stop], rg[start:stop], return_epe=True).numpy()
        assert all(a.tobytes() == b[start:stop].tobytes() for a, b in zip(part, (counts, sums, epe))), (start, stop)
    host = evaluate_flows_host(est, truth, em, tm, rg, out_epe=np.empty((n, h, w), np.float32))
    assert all(a.tobytes() == b.tobytes() for a, b in zip(host, (counts, sums, epe)))
    keep = []
    pinned = []
    for arr in (est, truth, em, tm, rg):
        p, k = device.pinned_empty(arr.shape, arr.dtype)
        p[...] = arr
        pinned.append(p)
        keep.append(k)
    out, k = device.pinned_empty((n, h, w), np.float32)
    keep.append(k)
    host = evaluate_flows_host(*pinned, out_epe=out)
    assert all(a.tobytes() == b.tobytes() for a, b in zip(host, (counts, sums, epe)))
    rows = evaluate_flows_host(est, truth, em, tm, rg)
    assert len(rows) == 2 and rows[0].tobytes() == counts.tobytes() and rows[1].tobytes() == sums.tobytes()


@pytest.mark.gpu
def test_host_ring_chunks(of, monkeypatch):
    """More frames than one chunk of the ring holds: rows come back to the right frames."""
    from oflibnumpy_b200.batch import evaluate_flows_host
    h, w, n = 436, 1024, 40                 # 7.6 MB per frame of traffic: several chunks
    est, truth = smooth_pair(n, h, w, 8)
    rg = make_masks(n, h, w, 0.5, 'region', 9)[2]
    counts, sums = evaluate_flows_host(est, truth, regions=rg)
    dc, ds = of.FlowBatch(est).evaluate(of.FlowBatch(truth), rg).numpy()
    assert counts.tobytes() == dc.tobytes() and sums.tobytes() == ds.tobytes()
    check_rows(counts[::13], sums[::13], est[::13], truth[::13], rg[::13], ('host',))


@pytest.mark.gpu
def test_flow_evaluate_and_refs(of):
    h, w = 64, 96
    est, truth = rough_pair(3, h, w, 12)
    em, tm, rg = make_masks(3, h, w, 0.05, 'all', 13)
    for i in range(3):
        got = of.Flow(est[i], 't', em[i]).evaluate(of.Flow(truth[i], 't', tm[i]), region=rg[i])
        want = of.FlowBatch(est[i:i + 1], 't', em[i:i + 1]).evaluate(of.FlowBatch(truth[i:i + 1], 't', tm[i:i + 1]),
                                                                     rg[i:i + 1]).summary()
        assert got == want
        assert got['pixels'] == int((em[i] & tm[i] & rg[i]).sum())
    # both refs give the same rows, and the region may be a device array
    from oflibnumpy_b200.device import DeviceArray
    rows = {}
    for ref in ('s', 't'):
        rows[ref] = of.FlowBatch(est, ref, em).evaluate(of.FlowBatch(truth, ref, tm), DeviceArray.from_numpy(rg),
                                                        return_epe=True).numpy()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(rows['s'], rows['t']))
    flow_dev = of.Flow(est[0], 's').evaluate(of.Flow(truth[0], 's'), region=DeviceArray.from_numpy(rg[0]))
    assert flow_dev == of.Flow(est[0], 's').evaluate(of.Flow(truth[0], 's'), region=rg[0])


@pytest.mark.gpu
def test_kitti_ground_truth(of):
    """An estimate against the committed KITTI sample counts exactly the file's valid pixels."""
    import cv2
    valid = cv2.imread(KITTI, cv2.IMREAD_UNCHANGED)[..., 0] != 0
    truth = of.Flow.from_kitti(KITTI)
    h, w = truth.shape
    est = of.Flow(truth.vecs + np.float32([1.5, -2.0]), 's')
    s = est.evaluate(truth)
    assert s['pixels'] == int(valid.sum()) and 0 < s['pixels'] < h * w
    assert abs(s['epe'] - 2.5) < 1e-6 and s['out3'] == 0 and s['out1'] == 1
    none = est.evaluate(truth, region=np.zeros((h, w), bool))
    assert none['pixels'] == 0 and math.isnan(none['epe'])


@pytest.mark.gpu
def test_launches_and_no_read_back(of, monkeypatch):
    from oflibnumpy_b200 import _lib
    from oflibnumpy_b200.device import DeviceArray
    rng = np.random.default_rng(5)
    for n in (1, 7, 64):
        for h, w in ((64, 96), (37, 53), (1080, 1920)):
            if n * h * w > 3e7:
                continue
            E = of.FlowBatch(rng.uniform(-3, 3, (n, h, w, 2)).astype(np.float32), 't', rng.random((n, h, w)) > .1)
            T = of.FlowBatch(rng.uniform(-3, 3, (n, h, w, 2)).astype(np.float32), 't')
            for kw in ({}, {'return_epe': True}, {'region': rng.random((n, h, w)) > .5}):
                E.evaluate(T, **kw)
                before = _lib.call('ofk_rt_launch_count')
                E.evaluate(T, **kw)
                assert _lib.call('ofk_rt_launch_count') - before == 2, (n, h, w, kw)
            before = _lib.call('ofk_rt_launch_count')
            res = E[0:0].evaluate(T[0:0], return_epe=True)
            assert _lib.call('ofk_rt_launch_count') == before
            c, s, e = res.numpy()
            assert c.shape == (0, 8) and s.shape == (0, 5) and e.shape == (0, h, w)
    real_call = _lib.call

    def no_sync(name, *args):
        assert name not in ('ofk_rt_memcpy_d2h', 'ofk_rt_stream_sync', 'ofk_rt_device_sync', 'ofk_rt_event_sync'), name
        return real_call(name, *args)

    def no_numpy(self, out=None):
        raise AssertionError("DeviceArray.numpy called")

    monkeypatch.setattr(_lib, 'call', no_sync)
    monkeypatch.setattr(DeviceArray, 'numpy', no_numpy)
    res = E.evaluate(T, return_epe=True)
    monkeypatch.undo()
    assert res.counts.shape == (64, 8)
