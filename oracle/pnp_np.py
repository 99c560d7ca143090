"""numpy restatement of the batched GPU PnP (casapose_b200/csrc/pnp.cuh).

TEST INFRASTRUCTURE (see oracle/__init__.py).
The reference's pnp() (/root/reference/casapose/pose_estimation/ransac_voting.py:13-57) is
cv2.solvePnPRansac(EPNP) -> cv2.solvePnP(ITERATIVE) on all points.  OpenCV's RANSAC is randomised, so the GPU
kernel reproduces its structure rather than its bits; this file restates the kernel's algorithm step by step
(candidate subsets, normalised DLT, polar projection, LM) so that GPU-vs-oracle is a tight numerical check,
while tests/test_pnp.py compares both against the reference's actual cv2 sequence (oracle/pose_np.pnp)."""
import itertools

import numpy as np


def _polar(M):
    R = M.copy()
    for _ in range(30):
        Rn = 0.5 * (R + np.linalg.inv(R).T)
        done = np.abs(Rn - R).max() < 1e-15
        R = Rn
        if done:
            break
    return R


PLANAR_RTOL = 1e-10  # pnp.cuh kPnpPlanarRtol


def _reduce(S, Sx, Sy, Sq):
    """dlt_reduce<D>: Schur reduction of the DLT normal equations, rows (h1, h2, h3) of the projection (D = 4) or the
    homography (D = 3); None when a Cholesky pivot of S is not above 1e-14 times its diagonal entry."""
    D = len(S)
    L = np.zeros((D, D))
    for j in range(D):
        d = S[j, j] - L[j, :j] @ L[j, :j]
        if not d > 1e-14 * S[j, j]:
            return None
        L[j, j] = np.sqrt(d)
        for i in range(j + 1, D):
            L[i, j] = (S[i, j] - L[i, :j] @ L[j, :j]) / L[j, j]
    Tx = np.linalg.solve(L.T, np.linalg.solve(L, Sx))
    Ty = np.linalg.solve(L.T, np.linalg.solve(L, Sy))
    M = Sq - Sx @ Tx - Sy @ Ty  # Schur complement on the last row
    M = 0.5 * (M + M.T)
    _, v = np.linalg.eigh(M)
    h3 = v[:, 0]
    return np.stack([Tx @ h3, Ty @ h3, h3])


def _moments(Q, xn):
    x, y = xn[:, 0], xn[:, 1]
    QQ = Q[:, :, None] * Q[:, None, :]
    return QQ.sum(0), (x[:, None, None] * QQ).sum(0), (y[:, None, None] * QQ).sum(0), ((x * x + y * y)[:, None, None] * QQ).sum(0)


def dlt(X, xn):
    c = X.mean(0)
    s = 1.0 / np.sqrt(((X - c) ** 2).sum(1).mean())
    Xs = (X - c) * s
    S = _moments(np.concatenate([Xs, np.ones((len(X), 1))], 1), xn)
    C = S[0][:3, :3]
    n = max((np.cross(C[a], C[b]) for a, b in ((0, 1), (0, 2), (1, 2))), key=lambda v: v @ v)
    flat = C[0] @ np.cross(C[1], C[2]) <= PLANAR_RTOL * np.sqrt(n @ n) * np.trace(C)  # covariance flat to 1e-10
    p = None if flat else _reduce(*S)
    if p is not None:
        M = p[:, :3] * s
        p4 = p[:, 3] - M @ c
    else:  # coplanar points: planar DLT (pnp_dlt's second branch)
        if not (n @ n > 0 and np.isfinite(n @ n)):
            raise np.linalg.LinAlgError("collinear points")
        n = n / np.sqrt(n @ n)
        e1 = np.cross(n, np.eye(3)[int(np.argmin(np.abs(n)))])
        e1 = e1 / np.sqrt(e1 @ e1)
        e2 = np.cross(n, e1)
        h = _reduce(*_moments(np.stack([Xs @ e1, Xs @ e2, np.ones(len(X))], 1), xn))
        if h is None:
            raise np.linalg.LinAlgError("collinear points")
        if h[2, 2] < 0:  # centroid in front of the camera
            h = -h
        a1, a2 = h[:, 0] * s, h[:, 1] * s
        a3 = np.cross(a1, a2) / np.sqrt(np.linalg.norm(a1) * np.linalg.norm(a2))
        M = np.outer(a1, e1) + np.outer(a2, e2) + np.outer(a3, n)
        p4 = h[:, 2] - M @ c
    if np.linalg.det(M) < 0:
        M, p4 = -M, -p4
    sc = np.cbrt(np.linalg.det(M))
    return _polar(M / sc), p4 / sc


def _skew(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])


def _exp(w):
    th = np.linalg.norm(w)
    K = _skew(w)
    if th < 1e-12:
        return np.eye(3) + K + 0.5 * K @ K
    return np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th**2 * K @ K


def lm(X, uv, K4, R, t, iters):
    fx, fy, cx, cy = K4

    def residual(R, t):
        Xc = X @ R.T + t
        return np.stack([fx * Xc[:, 0] / Xc[:, 2] + cx - uv[:, 0], fy * Xc[:, 1] / Xc[:, 2] + cy - uv[:, 1]], 1).ravel(), Xc

    lam = 1e-3
    r, Xc = residual(R, t)
    cost = r @ r
    for _ in range(iters):
        J = np.zeros((2 * len(X), 6))
        RX = X @ R.T
        for i in range(len(X)):
            x, y, z = Xc[i]
            dp = np.array([[fx / z, 0, -fx * x / z**2], [0, fy / z, -fy * y / z**2]])
            J[2 * i : 2 * i + 2, :3] = dp @ (-_skew(RX[i]))
            J[2 * i : 2 * i + 2, 3:] = dp
        H, g = J.T @ J, J.T @ r
        ok, dc, d = False, 0.0, np.zeros(6)
        for _ in range(10):
            try:
                L = np.linalg.cholesky(H + lam * np.diag(np.diag(H)))
            except np.linalg.LinAlgError:
                lam *= 10
                continue
            d = np.linalg.solve(L.T, np.linalg.solve(L, -g))
            R2, t2 = _exp(d[:3]) @ R, t + d[3:]
            r2, Xc2 = residual(R2, t2)
            c2 = r2 @ r2
            if c2 < cost:
                R, t, r, Xc, dc, cost = R2, t2, r2, Xc2, cost - c2, c2
                lam = max(lam / 10, 1e-12)
                ok = True
                break
            lam *= 10
        if not ok or np.abs(d).max() < 1e-12 or dc < 1e-14 * max(cost, 1e-30):
            break
    return R, t


def pnp(points_3d, points_2d, camera_matrix, reproj_px=12.0):
    """[vn,3], [vn,2] (x,y), [3,3] -> [3,4] float32, the algorithm of k_pnp."""
    uv32 = np.asarray(points_2d, np.float32)
    total = uv32.sum(dtype=np.float32)
    # compared in float32 (0.01f), as TensorFlow does; a non-finite keypoint: cv2 returns a NaN translation -> zeros
    if abs(total) < np.float32(0.01) or not np.isfinite(total):
        return np.zeros((3, 4), np.float32)
    X = np.asarray(points_3d, np.float32).astype(np.float64)
    uv = uv32.astype(np.float64)
    K = np.asarray(camera_matrix, np.float32).astype(np.float64)
    K4 = (K[0, 0], K[1, 1], K[0, 2], K[1, 2])
    xn = np.stack([(uv[:, 0] - K4[2]) / K4[0], (uv[:, 1] - K4[3]) / K4[1]], 1)
    n = len(X)
    subsets = [list(range(n))] + [[i for i in range(n) if i != a] for a in range(n)]
    subsets += [[i for i in range(n) if i not in ab] for ab in itertools.combinations(range(n), 2)]
    best = None
    for idx in subsets:
        if len(idx) < 6:
            continue
        with np.errstate(all="ignore"):
            try:
                R, t = dlt(X[idx], xn[idx])
            except np.linalg.LinAlgError:
                continue
            if not (np.isfinite(t).all() and np.isfinite(R).all()):
                continue
            R, t = lm(X[idx], uv[idx], K4, R, t, 5)
            Xc = X @ R.T + t
            e2 = (K4[0] * Xc[:, 0] / Xc[:, 2] + K4[2] - uv[:, 0]) ** 2 + (K4[1] * Xc[:, 1] / Xc[:, 2] + K4[3] - uv[:, 1]) ** 2
        if not (Xc[:, 2] > 0).all():
            continue
        inl = e2 < reproj_px * reproj_px
        cost = float(e2[inl].sum())
        if not np.isfinite(cost):
            continue
        key = (int(inl.sum()), -cost)
        if best is None or key > best[0]:
            best = (key, R, t)
    if best is None:
        return np.zeros((3, 4), np.float32)
    R, t = lm(X, uv, K4, best[1], best[2], 50)
    if not (np.isfinite(t).all() and np.isfinite(R).all()):
        return np.zeros((3, 4), np.float32)
    if t[2] < 0:
        R, t = -R, -t
    return np.concatenate([R, t[:, None]], axis=1).astype(np.float32)
