"""The reference's BPnP layer (/root/reference/casapose/pose_estimation/bpnp_layers.py:86-135, 278-359).  The forward
is host-side OpenCV like the reference (tf.numpy_function, :322).  The implicit-function-theorem backward of BPnP_fast
(:138-277) is casa_pnp_backward on the GPU: it is routed through torch.autograd when the 2-D points are a CUDA tensor
that requires grad."""
import numpy as np
import torch

from .ransac_voting import PnpGradFn, wants_grad


def pnp(points_3d, points_2d, camera_matrix, init_pose=None):
    """bpnp_layers.py:86-117 -> [6] float32 (rvec, tvec)."""
    import cv2

    assert points_3d.shape[0] == points_2d.shape[0], "points 3D and points 2D must have same number of vertices"
    points_2d = np.expand_dims(points_2d.astype(np.float32), 1)
    points_3d = points_3d.astype(np.float32)
    camera_matrix = camera_matrix.astype(np.float32)
    if init_pose is None:
        _, rvec0, T0, _ = cv2.solvePnPRansac(points_3d, points_2d, camera_matrix, None, flags=cv2.SOLVEPNP_EPNP,
                                             confidence=0.9999, reprojectionError=12)
    else:
        rvec0 = np.array(init_pose[0:3]).reshape([3, 1]).astype(np.float32)
        T0 = np.array(init_pose[3:6]).reshape([3, 1]).astype(np.float32)
    _, r, t = cv2.solvePnP(points_3d, points_2d, camera_matrix, None, flags=cv2.SOLVEPNP_ITERATIVE,
                           useExtrinsicGuess=True, rvec=rvec0, tvec=T0)
    return np.concatenate([r, t], axis=0).astype(np.float32).reshape(6)


def batch_pnp(points, keypoints, camera_matrix, init_pose=None):
    """bpnp_layers.py:129-135."""
    out = np.zeros([len(points), 6], dtype=np.float32)
    for i, pts in enumerate(points):
        out[i] = pnp(keypoints[i], pts, camera_matrix, None if init_pose is None else init_pose[i])
    return out


def rodrigues_batch(rvecs):
    """casapose/utils/geometry_utils.py:206-236, float32."""
    f = np.float32
    rvecs = np.asarray(rvecs, f)
    n = rvecs.shape[0]
    thetas = np.sqrt((rvecs * rvecs).sum(1, keepdims=True)).astype(f)
    with np.errstate(divide="ignore", invalid="ignore"):
        u = rvecs / thetas
    z = np.zeros(n, f)
    Ks = np.stack([np.stack([z, -u[:, 2], u[:, 1]], 1), np.stack([u[:, 2], z, -u[:, 0]], 1),
                   np.stack([-u[:, 1], u[:, 0], z], 1)], 1).astype(f)
    eye = np.broadcast_to(np.eye(3, dtype=f), (n, 3, 3))
    Rs = eye + np.sin(thetas)[..., None] * Ks + (f(1) - np.cos(thetas)[..., None]) * (Ks @ Ks)
    return np.where((thetas == 0)[..., None], eye, Rs).astype(f)


class BPNP_fast:
    """Stand-in for the Keras layer: layer([pts2d, pts3d, K]) -> [n, 6] (rvec, tvec), or [b, oc, 6] for [b, oc, vn, 2]
    points.  pts2d as numpy (or a tensor that needs no gradient) gives the numpy result of the host solve.  pts2d as a
    CUDA tensor that requires grad gives the same values as a float32 torch tensor on that device, whose backward is
    casa_pnp_backward (pose_form 6, BPnP_fast: bpnp_layers.py:138-277).  The gradient w.r.t. pts3d, K and the initial
    pose is not computed."""

    def __init__(self, name):
        self.name = name

    def __call__(self, inputs, **kwargs):
        pts2d, pts3d, K = inputs[:3]
        init = inputs[3] if len(inputs) == 4 else None
        if wants_grad(pts2d):
            return self._differentiable(pts2d, pts3d, K, init)
        return self._solve(pts2d, pts3d, K, init)

    @staticmethod
    def _solve(pts2d, pts3d, K, init):
        pts2d = np.asarray(pts2d, np.float32)
        pts3d = np.asarray(pts3d, np.float32)
        shape2d = pts2d.shape
        if pts2d.ndim == 4:
            pts2d = pts2d.reshape(-1, shape2d[2], 2)
        if pts3d.ndim == 4:
            pts3d = pts3d.reshape(-1, shape2d[2], 3)
        if pts3d.ndim == 2:
            pts3d = np.broadcast_to(pts3d, (pts2d.shape[0],) + pts3d.shape)
        out = batch_pnp(pts2d, pts3d, np.asarray(K, np.float32), None if init is None else np.asarray(init).reshape(-1, 6))
        if len(shape2d) == 4:
            out = out.reshape(-1, shape2d[1], 6)
        return out

    def _differentiable(self, pts2d, pts3d, K, init):
        if not pts2d.is_cuda:
            raise ValueError("BPNP_fast: the gradient runs on the GPU (casa_pnp_backward); pts2d must be a CUDA tensor")

        def host(x):
            return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else x

        dev = pts2d.device
        shape2d = tuple(pts2d.shape)
        vn = shape2d[-2]
        q = pts2d.to(torch.float32).reshape(-1, vn, 2)
        n = q.shape[0]
        p3 = np.asarray(host(pts3d), np.float32)
        p3 = np.broadcast_to(p3, (n, vn, 3)) if p3.ndim == 2 else p3.reshape(-1, vn, 3)[:n]
        p3 = torch.from_numpy(np.ascontiguousarray(p3)).to(dev)
        cam = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(np.asarray(host(K), np.float32), (n, 3, 3)))).to(dev)
        init = None if init is None else host(init)

        def solve(d):
            return torch.from_numpy(self._solve(d.reshape(shape2d).cpu().numpy(), host(pts3d), host(K), init).reshape(n, 6)).to(dev)

        out = PnpGradFn.apply(q, solve, p3, cam, 6)
        return out.reshape(shape2d[0], shape2d[1], 6) if len(shape2d) == 4 else out
