"""numpy restatement of ofk_fit_matrix (csrc/fit_matrix.cu), the device estimator behind FlowBatch.matrix.

The sampling (splitmix64 draws), the minimal solvers and their degeneracy tests run in scalar float64 in the device's
operation order, so the hypotheses are bit-identical; the residuals use the same order elementwise, so the scores, the
selected hypothesis, the inlier masks and the counts are identical too. The refinement uses numpy's reductions and
solvers: only its summation order differs from the device's. Test infrastructure only; the package never imports it.
"""
import math

import numpy as np

SEED = 0x6f666c69625f6669
TRIES = 8
LM_ITERS = 10
FLT_EPSILON = 2.0 ** -23
DBL_EPSILON = 2.0 ** -52
U64 = (1 << 64) - 1


def splitmix64(seed, k, c):
    z = (seed + ((k << 32) | c) * 0x9e3779b97f4a7c15) & U64
    z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & U64
    z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & U64
    return z ^ (z >> 31)


def points(vecs, ref):
    """Float32 (sx, sy, dx, dy) planes of one frame (H,W,2): x = column, y = row."""
    h, w = vecs.shape[:2]
    y, x = np.mgrid[:h, :w].astype(np.float32)
    u, v = vecs[..., 0].astype(np.float32), vecs[..., 1].astype(np.float32)
    if ref == 's':
        return x, y, x + u, y + v
    return x - u, y - v, x, y


def is_nonzero(vecs, mask, thr):
    """ofk_nonzero_flags: some valid component with |c| >= thr (thr > 0), or != 0 (thr == 0)."""
    a = np.abs(vecs[mask] if mask is not None else vecs)
    return bool((a >= thr).any() if thr > 0 else (a != 0).any())


def gauss_solve(A, b):
    """Gaussian elimination with partial pivoting in the device's order (first maximum on ties)."""
    n = len(b)
    A = [list(r) for r in A]
    b = list(b)
    for c in range(n):
        p, best = c, abs(A[c][c])
        for r in range(c + 1, n):
            if abs(A[r][c]) > best:
                best, p = abs(A[r][c]), r
        if not best != 0.0:
            return None
        if p != c:
            A[c], A[p] = A[p], A[c]
            b[c], b[p] = b[p], b[c]
        for r in range(c + 1, n):
            f = A[r][c] / A[c][c]
            for j in range(c + 1, n):
                A[r][j] = A[r][j] - f * A[c][j]
            b[r] = b[r] - f * b[c]
    x = [0.0] * n
    for i in range(n - 1, -1, -1):
        s = b[i]
        for j in range(i + 1, n):
            s = s - A[i][j] * x[j]
        x[i] = s / A[i][i]
    return x if all(math.isfinite(v) for v in x) else None


def collinear(x, y, a, b, c):
    dx1, dy1, dx2, dy2 = x[a] - x[c], y[a] - y[c], x[b] - x[c], y[b] - y[c]
    cr = dx2 * dy1 - dy2 * dx1
    s = ((abs(dx1) + abs(dy1)) + abs(dx2)) + abs(dy2)
    return abs(cr) <= FLT_EPSILON * s


def orient(x, y, a, b, c):
    return (x[b] - x[a]) * (y[c] - y[a]) - (y[b] - y[a]) * (x[c] - x[a])


def minimal_model(dof, sx, sy, dx, dy):
    """The device's minimal solver: 9 floats (row-major, m[8] = 1) or None for a degenerate sample."""
    m = [0.0] * 8 + [1.0]
    if dof == 4:
        ux, uy, vx, vy = sx[1] - sx[0], sy[1] - sy[0], dx[1] - dx[0], dy[1] - dy[0]
        den = ux * ux + uy * uy
        if den == 0.0 or (vx == 0.0 and vy == 0.0):
            return None
        a = (vx * ux + vy * uy) / den
        b = (vy * ux - vx * uy) / den
        m[0], m[1], m[3], m[4] = a, -b, b, a
        m[2] = dx[0] - (a * sx[0] - b * sy[0])
        m[5] = dy[0] - (b * sx[0] + a * sy[0])
        return m if all(math.isfinite(v) for v in (m[0], m[1], m[2], m[5])) else None
    if dof == 6:
        if collinear(sx, sy, 0, 1, 2) or collinear(dx, dy, 0, 1, 2):
            return None
        for r, rhs in enumerate((dx, dy)):
            x = gauss_solve([[sx[i], sy[i], 1.0] for i in range(3)], [rhs[i] for i in range(3)])
            if x is None:
                return None
            m[3 * r:3 * r + 3] = x
        return m
    negative = 0
    for a, b, c in ((0, 1, 2), (1, 2, 3), (0, 2, 3), (0, 1, 3)):
        if collinear(sx, sy, a, b, c) or collinear(dx, dy, a, b, c):
            return None
        negative += orient(sx, sy, a, b, c) * orient(dx, dy, a, b, c) < 0.0
    if negative not in (0, 4):
        return None
    A, b = [], []
    for i in range(4):
        A.append([sx[i], sy[i], 1.0, 0.0, 0.0, 0.0, -(sx[i] * dx[i]), -(sy[i] * dx[i])])
        A.append([0.0, 0.0, 0.0, sx[i], sy[i], 1.0, -(sx[i] * dy[i]), -(sy[i] * dy[i])])
        b += [dx[i], dy[i]]
    x = gauss_solve(A, b)
    return None if x is None else x + [1.0]


def hypotheses(dof, K, sx, sy, dx, dy):
    """K hypotheses of one frame from its valid points (float64 arrays of length M): list of models or None."""
    s, M = dof // 2, len(sx)
    out = []
    for k in range(K):
        idx, c = [], 0
        for _ in range(s):
            for _ in range(TRIES):
                i = ((splitmix64(SEED, k, c) >> 32) * M) >> 32
                c += 1
                if i not in idx:
                    idx.append(i)
                    break
            else:
                break
        if len(idx) < s:
            out.append(None)
            continue
        out.append(minimal_model(dof, [float(sx[i]) for i in idx], [float(sy[i]) for i in idx],
                                 [float(dx[i]) for i in idx], [float(dy[i]) for i in idx]))
    return out


def residuals(models, sx, sy, dx, dy, homog):
    """float32 squared reprojection distances (len(models), M) in the device's order; NaN -> inf."""
    m = np.asarray(models, np.float64)[:, :, None]
    px = m[:, 0] * sx + m[:, 1] * sy + m[:, 2]
    py = m[:, 3] * sx + m[:, 4] * sy + m[:, 5]
    if homog:
        with np.errstate(all='ignore'):
            iw = 1.0 / (m[:, 6] * sx + m[:, 7] * sy + 1.0)
        px, py = px * iw, py * iw
    with np.errstate(all='ignore'):
        ex, ey = px - dx, py - dy
        r = (ex * ex + ey * ey).astype(np.float32)
    r[np.isnan(r)] = np.inf
    return r


def uncentre(hc, cx, cy):
    T = np.array([[1.0, 0.0, -cx], [0.0, 1.0, -cy], [0.0, 0.0, 1.0]])
    Ti = np.array([[1.0, 0.0, cx], [0.0, 1.0, cy], [0.0, 0.0, 1.0]])
    H = Ti @ hc @ T
    return H / H[2, 2]


def _solve(A, b):
    try:
        x = np.linalg.solve(A, b)
    except np.linalg.LinAlgError:
        return None
    return x if np.isfinite(x).all() else None


def _lm_sums(h, X, Y, u, v):
    with np.errstate(all='ignore'):
        iw = 1.0 / (h[6] * X + h[7] * Y + 1.0)
        px, py = (h[0] * X + h[1] * Y + h[2]) * iw, (h[3] * X + h[4] * Y + h[5]) * iw
        z = np.zeros_like(X)
        Jx = np.stack([X * iw, Y * iw, iw, z, z, z, -px * X * iw, -px * Y * iw], 1)
        Jy = np.stack([z, z, z, X * iw, Y * iw, iw, -py * X * iw, -py * Y * iw], 1)
        ex, ey = px - u, py - v
        return Jx.T @ Jx + Jy.T @ Jy, Jx.T @ ex + Jy.T @ ey, float(np.sum(ex * ex + ey * ey))


def refine(dof, X, Y, u, v):
    """Least squares on the inliers in centred coordinates: normal equations (dof 4, 6) or the normalised DLT then
    Levenberg-Marquardt on the forward reprojection error (dof 8). The centred 3x3 matrix, or None if degenerate."""
    n = len(X)
    if dof == 4:
        if n < 2:
            return None
        sR = np.sum(X * X + Y * Y)
        A = np.array([[sR, 0, X.sum(), Y.sum()], [0, sR, -Y.sum(), X.sum()], [X.sum(), -Y.sum(), n, 0],
                      [Y.sum(), X.sum(), 0, n]], np.float64)
        x = _solve(A, np.array([np.sum(X * u + Y * v), np.sum(X * v - Y * u), u.sum(), v.sum()]))
        return None if x is None else np.array([[x[0], -x[1], x[2]], [x[1], x[0], x[3]], [0, 0, 1.0]])
    if dof == 6:
        if n < 3:
            return None
        A = np.array([[np.sum(X * X), np.sum(X * Y), X.sum()], [np.sum(X * Y), np.sum(Y * Y), Y.sum()],
                      [X.sum(), Y.sum(), n]], np.float64)
        r0 = _solve(A, np.array([np.sum(X * u), np.sum(Y * u), u.sum()]))
        r1 = _solve(A, np.array([np.sum(X * v), np.sum(Y * v), v.sum()]))
        return None if r0 is None or r1 is None else np.vstack([r0, r1, [0, 0, 1.0]])
    if n < 4:
        return None
    cen = [X.mean(), Y.mean(), u.mean(), v.mean()]
    mad = [np.sum(np.abs(a - c)) for a, c in zip((X, Y, u, v), cen)]
    if any(abs(s) < DBL_EPSILON for s in mad):
        return None
    scl = [n / s for s in mad]
    Xn, Yn = (X - cen[0]) * scl[0], (Y - cen[1]) * scl[1]
    xn, yn = (u - cen[2]) * scl[2], (v - cen[3]) * scl[3]
    z, o = np.zeros(n), np.ones(n)
    Lx = np.stack([Xn, Yn, o, z, z, z, -xn * Xn, -xn * Yn, -xn], 1)
    Ly = np.stack([z, z, z, Xn, Yn, o, -yn * Xn, -yn * Yn, -yn], 1)
    h0 = np.linalg.eigh(Lx.T @ Lx + Ly.T @ Ly)[1][:, 0].reshape(3, 3)
    norm_src = np.array([[scl[0], 0, -cen[0] * scl[0]], [0, scl[1], -cen[1] * scl[1]], [0, 0, 1]])
    denorm_dst = np.array([[1 / scl[2], 0, cen[2]], [0, 1 / scl[3], cen[3]], [0, 0, 1]])
    hc = denorm_dst @ h0 @ norm_src
    if not hc[2, 2] != 0:
        return None
    cand = (hc / hc[2, 2]).ravel()[:8]
    if not np.isfinite(cand[0]):
        return None
    lam, err, h, jtj, jte = 1e-3, None, None, None, None
    for it in range(LM_ITERS + 1):
        J, g, e = _lm_sums(cand, X, Y, u, v)
        if it == 0 or e < err:
            h, jtj, jte, err = cand, J, g, e
            lam = max(lam * 0.1, 1e-15)
            if it == 0 and not math.isfinite(e):
                return None
        else:
            lam *= 10.0
        if it < LM_ITERS:
            A = jtj.copy()
            A[np.diag_indices(8)] *= 1.0 + lam
            d = _solve(A, -jte)
            cand = h if d is None else h + d
    return np.append(h, 1.0).reshape(3, 3)


def fit_frame(vecs, mask, ref, dof, method, K=1024, masked=True, thr=1e-3):
    """One frame (H,W,2) float32, mask (H,W) bool: (matrix float64 3x3, inliers bool (H,W), count)."""
    h, w = vecs.shape[:2]
    valid = mask.astype(bool) if (masked and mask is not None) else np.ones((h, w), bool)
    eye, none = np.eye(3), np.zeros((h, w), bool)
    nan = np.full((3, 3), np.nan)
    if not is_nonzero(vecs, valid if masked else None, thr):
        return eye, none, 0
    sx, sy, dx, dy = [a.astype(np.float64) for a in points(vecs, ref)]
    flat = np.flatnonzero(valid)
    P = [a.ravel()[flat] for a in (sx, sy, dx, dy)]
    M, s, homog = len(flat), dof // 2, dof == 8
    if M < s:
        return nan, none, 0
    if method == 'lms':
        inl = valid.copy()
    else:
        models = hypotheses(dof, K, *P)
        ok = [i for i, m in enumerate(models) if m is not None]
        if not ok:
            return nan, none, 0
        best, best_score = None, None
        step = max(1, (1 << 22) // M)                        # hypotheses per residual block (bounded memory)
        for c0 in range(0, len(ok), step):
            ks = ok[c0:c0 + step]
            r = residuals([models[k] for k in ks], *P, homog)
            if method == 'ransac':
                sc = -(r <= np.float32(9.0)).sum(1)
            else:
                sc = np.partition(r, M // 2, axis=1)[:, M // 2]
            j = int(np.argmin(sc))
            if best_score is None or sc[j] < best_score:
                best, best_score = ks[j], sc[j]
        if method == 'ransac':
            thr2 = np.float32(9.0)
        else:
            sigma = math.inf
            if M > s:
                sigma = ((2.5 * 1.4826) * (1.0 + 5.0 / (M - s))) * math.sqrt(float(best_score))
            sigma = max(sigma, 0.001)
            thr2 = np.float32(sigma * sigma)
        r = residuals([models[best]], *[a.ravel() for a in (sx, sy, dx, dy)], homog)[0].reshape(h, w)
        inl = valid & (r <= thr2)
    cx, cy = 0.5 * (w - 1), 0.5 * (h - 1)
    X, Y, u, v = sx[inl] - cx, sy[inl] - cy, dx[inl] - cx, dy[inl] - cy
    hc = refine(dof, X, Y, u, v)
    if hc is None:
        return nan, none, 0
    return uncentre(hc, cx, cy), inl, int(inl.sum())


def fit_batch(vecs, masks, ref, dof, method, K=1024, masked=True, thr=1e-3):
    """(N,H,W,2), (N,H,W) -> (matrices (N,3,3), inliers (N,H,W) bool, counts (N,))."""
    res = [fit_frame(vecs[i], None if masks is None else masks[i], ref, dof, method, K, masked, thr)
           for i in range(len(vecs))]
    return np.stack([r[0] for r in res]), np.stack([r[1] for r in res]), np.array([r[2] for r in res], np.int32)
