"""Transformation matrices fitted on the device: FlowBatch.matrix (ofk_fit_matrix).

The oracle (oracle/matrix_fit.py) restates the device algorithm in numpy and is pinned to OpenCV here, on the CPU: on
the same float32 point pairs, the four frame corners mapped by the oracle's matrix and by cv2's
(estimateAffinePartial2D / estimateAffine2D / findHomography) agree within

    exact fields, every method                : 1e-6 px  (measured max 1.7e-13 for dof 4 / 6, 1.5e-8 for dof 8)
    lms, Gaussian noise + 30 % outliers       : 1e-6 px  (measured max 4.7e-8; deterministic on both sides)
    ransac / lmeds, noise + 30 % outliers     : 0.25 px  (measured max 0.033 dof 4, 0.092 dof 6, 0.028 dof 8: the
                                                          samples differ, so do the inlier sets near the 3 px bound)
    1080p frame, noise + 30 % outliers        : lms 1e-5 px, ransac 0.25 px

Noise is Gaussian with sigma 0.3 px, outliers are uniform within +-20 px, and 2 % of the pixels plus a rectangle are
masked out.

On the GPU the device is pinned to the oracle: the same inlier masks and counts (the same selected hypothesis), and
matrices within rtol 1e-10 for dof 4 and 6 (linear least squares: only the order of the float64 sums differs). dof 8 is
refined by Levenberg-Marquardt from the DLT; its accept / reject decisions and step sizes depend on the last bits of those
sums, so the iterates drift apart slightly: there the matrices agree within rtol 1e-7 and the mapped frame corners within
1e-6 px (measured 2.1e-9 relative on the noisy 120x160 lms frame)."""
import warnings

import numpy as np
import pytest

H8 = np.array([[1.01, 0.02, 3.5], [-0.015, 0.99, -2.0], [2e-5, -1e-5, 1.0]])
A6 = np.array([[1.01, 0.02, 3.5], [-0.015, 0.99, -2.0], [0.0, 0.0, 1.0]])
CASES = [(4, 'ransac'), (4, 'lmeds'), (6, 'ransac'), (6, 'lmeds'), (8, 'lms'), (8, 'ransac'), (8, 'lmeds')]


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


def field(h, w, M, ref, rng, noise=0.0, outliers=0.0, holes=False):
    """Flow (H,W,2) float32 of the transform M (src -> dst) for ref 's' or 't', with Gaussian noise, a share of
    outliers (uniform +-20 px) and, with holes, a masked rectangle and 2 % random invalid pixels."""
    y, x = np.mgrid[:h, :w].astype(np.float64)
    P = np.stack([x, y, np.ones_like(x)], -1)
    Q = P @ (M if ref == 's' else np.linalg.inv(M)).T
    Q = Q[..., :2] / Q[..., 2:]
    vecs = Q - P[..., :2] if ref == 's' else P[..., :2] - Q
    if noise:
        vecs = vecs + rng.normal(0, noise, vecs.shape)
    if outliers:
        o = rng.random((h, w)) < outliers
        vecs[o] += rng.uniform(-20, 20, (int(o.sum()), 2))
    mask = np.ones((h, w), bool)
    if holes:
        mask[h // 4:h // 2, w // 3:w // 2] = False
        mask &= rng.random((h, w)) > 0.02
    return vecs.astype(np.float32), mask


def corners(M, h, w):
    c = np.array([[0, 0, 1], [w - 1, 0, 1], [0, h - 1, 1], [w - 1, h - 1, 1]], np.float64) @ M.T
    return c[:, :2] / c[:, 2:]


def cv2_fit(vecs, mask, ref, dof, method):
    import cv2
    from oracle import matrix_fit as mf
    sx, sy, dx, dy = mf.points(vecs, ref)
    src, dst = np.stack([sx[mask], sy[mask]], -1), np.stack([dx[mask], dy[mask]], -1)
    if dof == 8:
        return cv2.findHomography(src, dst, {'lms': 0, 'ransac': cv2.RANSAC, 'lmeds': cv2.LMEDS}[method])[0]
    est = cv2.estimateAffinePartial2D if dof == 4 else cv2.estimateAffine2D
    return np.vstack([est(src, dst, method={'ransac': cv2.RANSAC, 'lmeds': cv2.LMEDS}[method])[0], [0, 0, 1]])


# ------------------------------------------------------------------------------------------------------------- CPU
def test_bad_arguments_are_rejected_without_a_gpu(lib):
    """ofk_fit_matrix checks every argument before a stream or the device is touched."""
    ws = lib.call('ofk_fit_matrix_workspace', 8, lib.FIT_RANSAC, 16, 2, 4, 4)
    assert ws > 0
    assert lib.call('ofk_fit_matrix_workspace', 5, lib.FIT_RANSAC, 16, 2, 4, 4) == 0
    assert lib.call('ofk_fit_matrix_workspace', 4, lib.FIT_LMS, 16, 2, 4, 4) == 0
    good = dict(flow=256, mask=None, ref=ord('t'), dof=8, method=lib.FIT_RANSAC, K=16, thr=1e-3, masked=1, mats=256,
                inliers=None, counts=None, N=2, H=4, W=4, ws=256, ws_bytes=ws, stream=None)
    for change, msg in (({'flow': None}, "NULL pointer"), ({'mats': None}, "NULL pointer"), ({'ws': None}, "NULL pointer"),
                        ({'ref': ord('x')}, "ref must be 's' or 't'"), ({'dof': 5}, "dof must be 4, 6 or 8"),
                        ({'method': 3}, "method must be"), ({'method': lib.FIT_LMS, 'dof': 6}, "OFK_FIT_LMS needs dof 8"),
                        ({'K': 0}, "hypotheses must be"), ({'K': 65537}, "hypotheses must be"),
                        ({'N': -1}, "bad shape"), ({'N': 65536}, "bad shape"), ({'H': 0}, "bad shape"),
                        ({'W': -3}, "bad shape"), ({'H': 1 << 16, 'W': 1 << 15}, "bad shape"),
                        ({'thr': -1.0}, "thr must be"), ({'flow': 260}, "flow must be 8-byte aligned"),
                        ({'ws': 260}, "ws must be 8-byte aligned"), ({"counts": 258}, "out_mats must be 8-byte and out_counts 4-byte aligned"),
                        ({'ws_bytes': ws - 1}, "workspace too small")):
        args = dict(good, **change)
        with pytest.raises(lib.OflibCudaError, match="ofk_fit_matrix: " + msg):
            lib.call('ofk_fit_matrix', *args.values())


def test_validate_matrix_args():
    from oflibnumpy_b200.validation import validate_matrix_args
    pre = "Error fitting transformation matrix to flow: "
    assert validate_matrix_args(None, None, None, None) == (8, 'ransac', True, 1024)
    assert validate_matrix_args(6, 'lmeds', False, 1) == (6, 'lmeds', False, 1)
    for args, exc, msg in (((5, None, None, None), ValueError, "Dof needs to be 4, 6 or 8"),
                           ((None, 'x', None, None), ValueError, "Method needs to be 'lms', 'ransac', or 'lmeds'"),
                           ((None, None, 1, None), TypeError, "Masked needs to be boolean"),
                           ((None, None, None, 2.0), TypeError, "Hypotheses needs to be an integer"),
                           ((None, None, None, True), TypeError, "Hypotheses needs to be an integer"),
                           ((None, None, None, 0), ValueError, "Hypotheses needs to be between 1 and 65536"),
                           ((None, None, None, 65537), ValueError, "Hypotheses needs to be between 1 and 65536")):
        with pytest.raises(exc) as e:
            validate_matrix_args(*args)
        assert str(e.value) == pre + msg
    for dof in (4, 6):
        with pytest.warns(UserWarning, match="Method 'ransac' used instead"):
            assert validate_matrix_args(dof, 'lms', None, None) == (dof, 'ransac', True, 1024)
    with warnings.catch_warnings():
        warnings.simplefilter('error')
        assert validate_matrix_args(8, 'lms', None, None)[1] == 'lms'


@pytest.mark.parametrize('dof,method', CASES)
@pytest.mark.parametrize('kind', ['exact', 'noisy'])
def test_oracle_matches_cv2(dof, method, kind):
    from oracle import matrix_fit as mf
    rng = np.random.default_rng(dof * 10 + len(method))
    h, w = 120, 160
    for ref in 'st':
        vecs, mask = field(h, w, H8 if dof == 8 else A6, ref, rng,
                           *((0.3, 0.3, True) if kind == 'noisy' else ()))
        m, inl, count = mf.fit_frame(vecs, mask, ref, dof, method)
        assert count == inl.sum() and not inl[~mask].any()
        tol = 1e-6 if kind == 'exact' or method == 'lms' else 0.25
        assert np.abs(corners(m, h, w) - corners(cv2_fit(vecs, mask, ref, dof, method), h, w)).max() < tol
        if dof != 8:
            assert np.array_equal(m[2], [0, 0, 1])
        assert m[2, 2] == 1.0


def test_oracle_matches_cv2_at_1080p():
    from oracle import matrix_fit as mf
    rng = np.random.default_rng(7)
    h, w = 1080, 1920
    vecs, mask = field(h, w, H8, 's', rng, 0.3, 0.3, True)
    for method, K, tol in (('lms', 1024, 1e-5), ('ransac', 16, 0.25)):
        m = mf.fit_frame(vecs, mask, 's', 8, method, K=K)[0]
        assert np.abs(corners(m, h, w) - corners(cv2_fit(vecs, mask, 's', 8, method), h, w)).max() < tol


@pytest.mark.parametrize('ref', ['s', 't'])
def test_oracle_recovers_the_generating_matrix(ref):
    """Fields built like flow_from_matrix (ref 't' from the inverse) give back the matrix for every dof that can
    represent it."""
    from oracle import matrix_fit as mf
    rng = np.random.default_rng(3)
    ang = np.deg2rad(8.0)
    sim = np.array([[1.05 * np.cos(ang), -1.05 * np.sin(ang), 4.0], [1.05 * np.sin(ang), 1.05 * np.cos(ang), -3.0],
                    [0, 0, 1.0]])
    for M, dofs in ((sim, (4, 6, 8)), (A6, (6, 8)), (H8, (8,))):
        vecs, mask = field(90, 130, M, ref, rng)
        for dof in dofs:
            for method in ('ransac', 'lmeds') + (('lms',) if dof == 8 else ()):
                np.testing.assert_allclose(mf.fit_frame(vecs, mask, ref, dof, method, K=128)[0], M, rtol=1e-5,
                                           atol=1e-5 * np.abs(M).max())


# ------------------------------------------------------------------------------------------------------------- GPU
def batch_fields(n, h, w, ref, seed):
    """n frames: exact and noisy homography / affine fields with outliers and mask holes, one sub-threshold frame."""
    rng = np.random.default_rng(seed)
    vs, ms = [], []
    for i in range(n):
        M = (H8, A6)[i % 2].copy()
        M[0, 2] += i
        if i == 2:
            v, m = np.full((h, w, 2), 5e-4, np.float32), np.ones((h, w), bool)
        else:
            v, m = field(h, w, M, ref, rng, *((0.3, 0.3, True) if i % 3 != 0 else ()))
        vs.append(v)
        ms.append(m)
    return np.stack(vs), np.stack(ms)


def assert_matches_oracle(of, vecs, masks, ref, dof, method, masked, K):
    from oracle import matrix_fit as mf
    mats, inl, counts = of.FlowBatch(vecs, ref, masks).matrix(dof, method, masked, hypotheses=K, return_inliers=True)
    om, oi, oc = mf.fit_batch(vecs, masks, ref, dof, method, K, masked)
    assert np.array_equal(inl.numpy().view(bool), oi)
    assert np.array_equal(counts.numpy(), oc)
    om = om.reshape(len(vecs), 9)
    d = mats.numpy().reshape(len(vecs), 9)
    rtol = 1e-7 if dof == 8 else 1e-10
    h, w = vecs.shape[1:3]
    for i in range(len(vecs)):
        np.testing.assert_allclose(d[i], om[i], rtol=rtol, atol=rtol * np.nanmax(np.abs(om[i]), initial=1.0))
        if dof == 8 and np.isfinite(om[i]).all():
            assert np.abs(corners(d[i].reshape(3, 3), h, w) - corners(om[i].reshape(3, 3), h, w)).max() < 1e-6
    return d


@pytest.mark.gpu
@pytest.mark.parametrize('dof,method', CASES)
@pytest.mark.parametrize('ref', ['s', 't'])
@pytest.mark.parametrize('masked', [True, False])
def test_device_matches_oracle(of, dof, method, ref, masked):
    vecs, masks = batch_fields(5, 120, 160, ref, dof + len(method))
    d = assert_matches_oracle(of, vecs, masks, ref, dof, method, masked, 256)
    assert np.array_equal(d[2], np.eye(3).ravel())          # zero below the threshold: identity


@pytest.mark.gpu
@pytest.mark.parametrize('dof,method,ref,masked', [(8, 'ransac', 's', True), (8, 'lms', 't', True),
                                                   (6, 'lmeds', 't', False), (4, 'ransac', 's', False)])
def test_device_matches_oracle_at_1080p(of, dof, method, ref, masked):
    vecs, masks = batch_fields(3, 1080, 1920, ref, 11)
    assert_matches_oracle(of, vecs, masks, ref, dof, method, masked, 16)


@pytest.mark.gpu
@pytest.mark.parametrize('dof,method', [(8, 'ransac'), (8, 'lmeds'), (6, 'lmeds'), (8, 'lms')])
def test_frames_do_not_depend_on_the_batch(of, dof, method):
    """Frame i of a batch equals a batch of one holding frame i, and two calls agree, bit for bit."""
    vecs, masks = batch_fields(5, 120, 160, 't', 5)
    fb = of.FlowBatch(vecs, 't', masks)
    a = [x.numpy() for x in fb.matrix(dof, method, return_inliers=True)]
    b = [x.numpy() for x in fb.matrix(dof, method, return_inliers=True)]
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True) if x.dtype == np.float64 else np.array_equal(x, y)
    for i in range(5):
        one = [x.numpy() for x in of.FlowBatch(vecs[i:i + 1], 't', masks[i:i + 1]).matrix(dof, method,
                                                                                           return_inliers=True)]
        assert np.array_equal(one[0][0].view(np.uint64), a[0][i].view(np.uint64))
        assert np.array_equal(one[1][0], a[1][i]) and one[2][0] == a[2][i]


@pytest.mark.gpu
def test_special_frames(of):
    """Zero flow -> identity. An all-masked frame -> identity too, with masked=True: the reference's zero test
    (is_zero(masked=True)) holds vacuously on a frame without valid pixels and Flow.matrix returns the identity before
    fitting; with masked=False the same frame is fitted. Fewer valid points than the sample, or a single valid row
    (collinear points, dof 6 and 8) -> NaN and count 0. The device agrees with the oracle on every such frame. One
    hypothesis is enough for an exact field."""
    h, w = 40, 50
    rng = np.random.default_rng(2)
    v, _ = field(h, w, A6, 's', rng)
    vecs = np.stack([np.zeros((h, w, 2), np.float32), v, v, v])
    masks = np.ones((4, h, w), bool)
    masks[1] = False
    masks[2] = False
    masks[2, 5, 7] = True                                      # one valid point
    masks[3] = False
    masks[3, 10] = True                                        # one valid row
    for dof in (4, 6, 8):
        for method in ('ransac', 'lmeds') + (('lms',) if dof == 8 else ()):
            mats, inl, counts = of.FlowBatch(vecs, 's', masks).matrix(dof, method, return_inliers=True)
            m, c, i = mats.numpy(), counts.numpy(), inl.numpy()
            assert np.array_equal(m[:2], np.stack([np.eye(3)] * 2)) and (c[:2] == 0).all() and not i[:2].any()
            assert np.isnan(m[2]).all() and c[2] == 0 and not i[2].any()
            if dof == 4:                                       # a similarity fits a row of points
                assert np.isfinite(m[3]).all() and c[3] == w
            else:
                assert np.isnan(m[3]).all() and c[3] == 0 and not i[3].any()
            assert_matches_oracle(of, vecs, masks, 's', dof, method, True, 1024)
            unmasked = of.FlowBatch(vecs, 's', masks).matrix(dof, method, masked=False).numpy()
            assert np.isfinite(unmasked[1:]).all()
    exact = of.FlowBatch(v[None], 's').matrix(6, 'ransac', hypotheses=1).numpy()[0]
    np.testing.assert_allclose(exact, A6, rtol=1e-6, atol=1e-6)
    assert_matches_oracle(of, vecs[1:2], None, 's', 8, 'lmeds', True, 1)


@pytest.mark.gpu
def test_launch_count_does_not_depend_on_n(of):
    from oflibnumpy_b200 import _lib
    rng = np.random.default_rng(4)
    v, m = field(16, 16, H8, 't', rng)
    for dof, method in CASES:
        counts = []
        for n in (2, 64):
            fb = of.FlowBatch(np.repeat(v[None], n, 0), 't', np.repeat(m[None], n, 0))
            fb.matrix(dof, method, hypotheses=32)
            before = _lib.call('ofk_rt_launch_count')
            fb.matrix(dof, method, hypotheses=32, return_inliers=True)
            counts.append(_lib.call('ofk_rt_launch_count') - before)
        assert counts[0] == counts[1], (dof, method, counts)


@pytest.mark.gpu
@pytest.mark.parametrize('h,w', [(200, 300), (300, 300)])
def test_valid_point_counts_around_2_16(of, h, w):
    """M below (60000) and above (90000) 2^16: the sample index (r >> 32) * M >> 32 and the list reach every point."""
    rng = np.random.default_rng(h)
    vecs, masks = zip(*[field(h, w, H8, 's', rng, 0.3, 0.3) for _ in range(2)])
    for dof, method in ((8, 'ransac'), (6, 'lmeds')):
        assert_matches_oracle(of, np.stack(vecs), np.stack(masks), 's', dof, method, True, 64)
