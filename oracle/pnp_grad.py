"""Gradient oracle for the PnP backward (casa_pnp_backward, DESIGN.md K10): BPnP_fast's implicit-function backward
(/root/reference/casapose/pose_estimation/bpnp_layers.py:138-277, Chen et al., CVPR 2020) restated in torch float64 on
the CPU, in the structure of that code.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The reference source is not vendored here, so this file is pinned by
independent checks in tests/test_pnp_backward.py instead of golden vectors: the closed form J (J^T J)^-1 g, central
finite differences of a float64 Levenberg-Marquardt solve at zero residual, and the invariance of the result to the
rotation parameterisation.

Per object, with y the pose and x the 2-D points (x, y order):
  * the constraint rows f(x, y) = C^T (pi(y) - x) use the coefficients C = -2 dpi/dy evaluated at the forward pose and
    detached (the "fast" variant: no residual-curvature terms);
  * J_fy = df/dy and J_fx = df/dx by autograd, J_yx = -J_fy^-1 J_fx = (J^T J)^-1 J^T, grad_x = J_yx^T grad_y.
Pose forms:
  * 12: [R|t]; y is the left-multiplicative tangent (R <- exp([w]x) R, t <- t + dt) and grad_y comes from autograd
    through that map.  A t_z < 0 flip (-[R|t], ransac_voting.py:53-55) is recognised by det(R) < 0: the un-flipped pose
    is differentiated with the incoming gradient negated.
  * 6: (rvec, tvec); y is the pair itself, through Rodrigues.
Zero gradient for an all-zero pose, for a point at z <= 0 under the differentiated pose or a non-finite J, and for a
numerically singular J^T J (a Cholesky pivot of the diagonally scaled matrix at or below PIVOT_RTOL)."""
import numpy as np
import torch

PIVOT_RTOL = 1e-10  # casapose_b200/csrc/pnp.cuh: kPnpPivotRtol


def rodrigues(r):
    """exp([r]x) for a float64 torch 3-vector, differentiable, with the th -> 0 series."""
    th2 = (r * r).sum()
    o = torch.zeros((), dtype=r.dtype)
    K = torch.stack([torch.stack([o, -r[2], r[1]]), torch.stack([r[2], o, -r[0]]), torch.stack([-r[1], r[0], o])])
    if float(th2.detach()) < 1e-12:
        a, b = 1.0 - th2 / 6.0, 0.5 - th2 / 24.0
    else:
        th = torch.sqrt(th2)
        a, b = torch.sin(th) / th, (1.0 - torch.cos(th)) / th2
    return torch.eye(3, dtype=r.dtype) + a * K + b * (K @ K)


def _project(R, t, X, fx, fy, cx, cy):
    Xc = X @ R.T + t
    return torch.stack([fx * Xc[:, 0] / Xc[:, 2] + cx, fy * Xc[:, 1] / Xc[:, 2] + cy], 1).reshape(-1)


def _singular(H):
    d = torch.sqrt(torch.diagonal(H))
    if not bool((d > 0).all()):
        return True
    L, info = torch.linalg.cholesky_ex(H / d[:, None] / d[None, :])
    return int(info) != 0 or not bool((torch.diagonal(L) ** 2 > PIVOT_RTOL).all())


def _one(X, K, pose, grad, pose_form):
    vn = X.shape[0]
    zero = np.zeros((vn, 2))
    if not pose.any():
        return zero
    X = torch.from_numpy(X)
    fx, fy, cx, cy = float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2])
    pose = torch.from_numpy(pose)
    grad = torch.from_numpy(grad)
    if pose_form == 12:
        P, G = pose.reshape(3, 4), grad.reshape(3, 4)
        if float(torch.linalg.det(P[:, :3])) < 0:
            P, G = -P, -G
        R0, t0 = P[:, :3], P[:, 3]

        def pose_of(y):
            return torch.cat([rodrigues(y[:3]) @ R0, (t0 + y[3:])[:, None]], 1)

        y0 = torch.zeros(6, dtype=torch.float64)
        g_y = torch.autograd.functional.jacobian(lambda y: (pose_of(y) * G).sum(), y0)

        def proj(y):
            return _project(rodrigues(y[:3]) @ R0, t0 + y[3:], X, fx, fy, cx, cy)
    else:
        y0, g_y = pose.reshape(6), grad.reshape(6)

        def proj(y):
            return _project(rodrigues(y[:3]), y[3:], X, fx, fy, cx, cy)

    with torch.no_grad():
        z = (X @ R0.T + t0)[:, 2] if pose_form == 12 else (X @ rodrigues(y0[:3]).T + y0[3:])[:, 2]
    if not bool((z > 0).all()):
        return zero
    x0 = proj(y0).detach()
    C = -2.0 * torch.autograd.functional.jacobian(proj, y0)  # [2vn, 6], detached coefficients
    if not bool(torch.isfinite(C).all()):
        return zero

    def constraint(x, y):  # f(x, y) = C^T (pi(y) - x)
        return C.T @ (proj(y) - x)

    J_fy = torch.autograd.functional.jacobian(lambda y: constraint(x0, y), y0)  # = -2 J^T J
    J_fx = torch.autograd.functional.jacobian(lambda x: constraint(x, y0), x0)  # = 2 J^T
    if _singular(-0.5 * J_fy):
        return zero
    J_yx = -torch.linalg.solve(J_fy, J_fx)  # [6, 2vn]
    return (J_yx.T @ g_y).reshape(vn, 2).numpy()


def pnp_grad(points_3d, camera, poses, grad_poses, pose_form=12):
    """dL/d points2d [n,vn,2] (x,y) float64 for dL/d poses = grad_poses.
    points_3d [n,vn,3]; camera [n,3,3] or [3,3]; poses / grad_poses [n,3,4] (pose_form 12) or [n,6] (pose_form 6)."""
    if pose_form not in (6, 12):
        raise ValueError("pose_form must be 6 or 12")
    X = np.asarray(points_3d, np.float64)
    n = X.shape[0]
    cam = np.broadcast_to(np.asarray(camera, np.float64), (n, 3, 3))
    P = np.asarray(poses, np.float64).reshape(n, pose_form)
    G = np.asarray(grad_poses, np.float64).reshape(n, pose_form)
    return np.stack([_one(X[i], cam[i], P[i], G[i], pose_form) for i in range(n)]) if n else np.zeros((0, X.shape[1], 2))
