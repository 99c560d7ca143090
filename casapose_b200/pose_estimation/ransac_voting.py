"""Drop-in for the voting entry point of casapose.pose_estimation.ransac_voting.

``ransac_voting_layer_all_masks`` keeps the reference signature
(/root/reference/casapose/pose_estimation/ransac_voting.py:446-463) and output
([b, oc, vn, 2] float32, (x, y) pixels); the body is one call into the sm_100a library.
Additive keyword-only extras (seed, idxs, selection, return_debug, ...) exist for testing."""
import ctypes as C

import torch

from .. import _lib
from .._carrier import as_cuda, as_cuda_f32, current_stream_ptr, ptr

DEBUG_FIELDS = ("tn0", "tn", "rounds", "counts", "win_idx", "hyps", "win_pts", "win_ratio", "ata", "atb",
                "refined", "pix", "pix_off", "stats")


def _params(b, h, w, oc, vn, round_hyp_num, inlier_thresh, confidence, max_iter, min_num, max_num, seed,
            image_offset, pix_capacity, force_exact, vertex_per_class=False):
    return _lib.RansacParams(
        b=b, h=h, w=w, oc=oc, vn=vn, round_hyp_num=int(round_hyp_num), max_iter=int(max_iter),
        inlier_thresh=float(inlier_thresh), confidence=float(confidence), min_num=float(min_num),
        max_num=float(max_num), seed=int(seed) & 0xFFFFFFFFFFFFFFFF, image_offset=int(image_offset),
        pix_capacity=int(pix_capacity), force_exact=int(bool(force_exact)), vertex_per_class=int(bool(vertex_per_class)))


def ransac_voting_layer_all_masks(
    mask,
    vertex,
    round_hyp_num,
    inlier_thresh=0.99,
    confidence=0.99,
    max_iter=20,
    min_num=5,
    max_num=30000,
    *,
    seed=0,
    image_offset=0,
    idxs=None,
    selection=None,
    return_debug=False,
    debug_hyps=False,
    pix_capacity=0,
    force_exact=False,
    seg_scores=False,
    out=None,
):
    """
    :param mask:      [b,h,w,oc]   float32 {0,1}
                      (seg_scores=True: [b,h,w,1+oc] segmentation scores; the one-hot of their arg-max without
                      the background channel is used, pose_evaluation.py:36-51, without materialising it)
    :param vertex:    [b,h,w,vn,2] float32 (dy,dx)   (a [b,h,w,vn*2] tensor is viewed as such;
                      [b,h,w,oc,vn,2] = one field per class, pose_evaluation.py:38-45)
    :param round_hyp_num: hypotheses per round
    :param out:       optional preallocated [b,oc,vn,2] float32 result tensor on the inputs' device
    :return: [b,oc,vn,2] float32 (x,y) — and a dict of intermediates if return_debug
    """
    mask = as_cuda_f32(mask, "mask")
    vertex = as_cuda_f32(vertex, "vertex")
    if mask.dim() != 4:
        raise ValueError("mask must be [b,h,w,oc], got %s" % (tuple(mask.shape),))
    b, h, w, oc = mask.shape
    if seg_scores:
        oc -= 1
        if oc < 1:
            raise ValueError("seg scores need at least one object channel")
    if vertex.dim() == 4:
        vertex = vertex.view(b, h, w, vertex.shape[3] // 2, 2)
    vertex_per_class = vertex.dim() == 6
    if vertex_per_class:
        if tuple(vertex.shape[:4]) != (b, h, w, oc) or vertex.shape[5] != 2:
            raise ValueError("per-class vertex must be [b,h,w,oc,vn,2], got %s" % (tuple(vertex.shape),))
    elif vertex.dim() != 5 or tuple(vertex.shape[:3]) != (b, h, w) or vertex.shape[4] != 2:
        raise ValueError("vertex must be [b,h,w,vn,2] matching mask, got %s" % (tuple(vertex.shape),))
    if vertex.device != mask.device:
        raise ValueError("mask and vertex must be on the same device")
    vn = vertex.shape[-2]
    dev = mask.device
    p = _params(b, h, w, oc, vn, round_hyp_num, inlier_thresh, confidence, max_iter, min_num, max_num, seed,
                image_offset, pix_capacity, force_exact, vertex_per_class)
    hn, mi = p.round_hyp_num, p.max_iter
    if idxs is not None:
        idxs = as_cuda(idxs, torch.int32, "idxs")
        if tuple(idxs.shape) != (b, oc, mi, hn, vn, 2):
            raise ValueError("idxs must be [b,oc,max_iter,hn,vn,2] = %s, got %s" % ((b, oc, mi, hn, vn, 2), tuple(idxs.shape)))
    if selection is not None:
        selection = as_cuda_f32(selection, "selection")
        if tuple(selection.shape) != (b, oc, h, w):
            raise ValueError("selection must be [b,oc,h,w]")
    if out is None:
        out = torch.empty((b, oc, vn, 2), dtype=torch.float32, device=dev)
    else:
        out = as_cuda_f32(out, "out")
        if tuple(out.shape) != (b, oc, vn, 2) or out.device != dev:
            raise ValueError("out must be [b,oc,vn,2] = %s on %s" % ((b, oc, vn, 2), dev))
    dbg_struct = None
    dbg = None
    if return_debug:
        i32, f32 = torch.int32, torch.float32
        cap = pix_capacity if pix_capacity > 0 else h * w
        dbg = {
            "tn0": torch.zeros((b, oc), dtype=i32, device=dev),
            "tn": torch.zeros((b, oc), dtype=i32, device=dev),
            "rounds": torch.zeros((b, oc), dtype=i32, device=dev),
            "counts": torch.zeros((b, oc, mi, hn, vn), dtype=i32, device=dev),
            "win_idx": torch.zeros((b, oc, mi, vn), dtype=i32, device=dev),
            "win_pts": torch.zeros((b, oc, vn, 2), dtype=f32, device=dev),
            "win_ratio": torch.zeros((b, oc, vn), dtype=f32, device=dev),
            "ata": torch.zeros((b, oc, vn, 3), dtype=f32, device=dev),
            "atb": torch.zeros((b, oc, vn, 2), dtype=f32, device=dev),
            "refined": torch.zeros((b, oc), dtype=i32, device=dev),
            "pix": torch.zeros((b, cap), dtype=i32, device=dev),
            "pix_off": torch.zeros((b, oc), dtype=i32, device=dev),
            "stats": torch.zeros((4,), dtype=torch.int64, device=dev),
        }
        if debug_hyps:
            dbg["hyps"] = torch.zeros((b, oc, mi, hn, vn, 2), dtype=f32, device=dev)
        dbg_struct = _lib.RansacDebug(**{k: ptr(dbg.get(k)) for k in DEBUG_FIELDS})
    hdl = _lib.handle(dev.index if dev.index is not None else torch.cuda.current_device(), current_stream_ptr(dev))
    with torch.cuda.device(dev):
        fn = _lib.lib().casa_ransac_vote_seg if seg_scores else _lib.lib().casa_ransac_vote
        rc = fn(
            hdl, C.byref(p), ptr(mask), ptr(vertex), ptr(idxs), ptr(selection), ptr(out),
            C.byref(dbg_struct) if dbg_struct is not None else None, current_stream_ptr(dev))
        if rc == -3 and pix_capacity == 0 and not return_debug:
            # CASA_ERR_WORKSPACE: channels that overlap list a pixel more than once and h*w slots per image are not
            # enough.  The reference treats every channel independently (ransac_voting.py:458-470), so the call is
            # repeated with room for every channel (synchronous calls only: an asynchronous one reports at casa_sync).
            p.pix_capacity = oc * h * w
            rc = fn(hdl, C.byref(p), ptr(mask), ptr(vertex), ptr(idxs), ptr(selection), ptr(out), None,
                    current_stream_ptr(dev))
    _lib.check(rc)
    if return_debug:
        st = C.c_uint32()
        _lib.check(_lib.lib().casa_last_status(hdl, C.byref(st)))
        dbg["status"] = st.value
        return out, dbg
    return out


class PendingHostVote:
    """A host-buffer vote in flight (ransac_voting_layer_all_masks_host(..., wait=False)).  result() blocks until the
    keypoints are in the output tensor and returns it (raises what the synchronous call would have raised); the
    object keeps the input and output buffers alive until then."""

    def __init__(self, hdl, ticket, out, keep):
        self._hdl, self._ticket, self._out, self._keep, self._done = hdl, ticket, out, keep, False

    def result(self):
        if not self._done:
            self._done = True
            rc = _lib.lib().casa_host_wait(self._hdl, self._ticket)
            self._keep = None
            _lib.check(rc)
        return self._out

    def __del__(self):  # the library reads the buffers until the call is done
        if not self._done:
            try:
                self._done = True
                _lib.lib().casa_host_wait(self._hdl, self._ticket)
            except Exception:
                pass


def ransac_voting_layer_all_masks_host(mask, vertex, round_hyp_num, inlier_thresh=0.99, confidence=0.99, max_iter=20,
                                       min_num=5, max_num=30000, *, seed=0, image_offset=0, device=0, out=None, wait=True):
    """Same call with HOST tensors (numpy arrays or CPU torch tensors, ideally pinned): host->device copy,
    voting, device->host copy of the [b,oc,vn,2] result — all inside the library (casa_ransac_vote_host).

    wait=False (casa_ransac_vote_host_async) returns a PendingHostVote at once; up to two such calls run at a time,
    the host packing of one beside the GPU work of the other, and a third call blocks until the oldest has finished.
    The input buffers must not be modified before result() has returned."""
    mask_t = torch.as_tensor(mask)
    vertex_t = torch.as_tensor(vertex)
    if mask_t.is_cuda or vertex_t.is_cuda:
        raise ValueError("host entry point takes CPU buffers")
    if mask_t.dtype != torch.float32 or vertex_t.dtype != torch.float32:
        raise TypeError("mask / vertex must be float32")
    if not (mask_t.is_contiguous() and vertex_t.is_contiguous()):
        raise ValueError("mask / vertex must be C-contiguous")
    if mask_t.dim() != 4:
        raise ValueError("mask must be [b,h,w,oc], got %s" % (tuple(mask_t.shape),))
    b, h, w, oc = mask_t.shape
    if vertex_t.dim() == 4:
        if tuple(vertex_t.shape[:3]) != (b, h, w) or vertex_t.shape[3] % 2:
            raise ValueError("vertex must be [b,h,w,vn*2] matching mask, got %s" % (tuple(vertex_t.shape),))
        vertex_t = vertex_t.view(b, h, w, vertex_t.shape[3] // 2, 2)
    vertex_per_class = vertex_t.dim() == 6
    if vertex_per_class:
        if tuple(vertex_t.shape[:4]) != (b, h, w, oc) or vertex_t.shape[5] != 2:
            raise ValueError("per-class vertex must be [b,h,w,oc,vn,2], got %s" % (tuple(vertex_t.shape),))
    elif vertex_t.dim() != 5 or tuple(vertex_t.shape[:3]) != (b, h, w) or vertex_t.shape[4] != 2:
        raise ValueError("vertex must be [b,h,w,vn,2] matching mask, got %s" % (tuple(vertex_t.shape),))
    vn = vertex_t.shape[-2]
    p = _params(b, h, w, oc, vn, round_hyp_num, inlier_thresh, confidence, max_iter, min_num, max_num, seed,
                image_offset, 0, False, vertex_per_class)
    if out is None:
        out = torch.empty((b, oc, vn, 2), dtype=torch.float32)
    else:
        if not isinstance(out, torch.Tensor) or out.is_cuda or out.dtype != torch.float32 or not out.is_contiguous() \
                or tuple(out.shape) != (b, oc, vn, 2):
            raise ValueError("out must be a contiguous CPU float32 tensor [b,oc,vn,2] = %s" % ((b, oc, vn, 2),))
    hdl = _lib.handle(device)
    if not wait:
        ticket = C.c_int64(-1)
        _lib.check(_lib.lib().casa_ransac_vote_host_async(hdl, C.byref(p), mask_t.data_ptr(), vertex_t.data_ptr(),
                                                          out.data_ptr(), C.byref(ticket)))
        return PendingHostVote(hdl, ticket.value, out, (mask_t, vertex_t))
    rc = _lib.lib().casa_ransac_vote_host(hdl, C.byref(p), mask_t.data_ptr(), vertex_t.data_ptr(), out.data_ptr())
    _lib.check(rc)
    return out


# ------------------------------------------------------------------------------------------------------------
# Post-step on the host: PnP and pose metrics.  The reference leaves TensorFlow here as well
# (tf.numpy_function -> Python -> OpenCV, ransac_voting.py:513), so this part is numpy + the same cv2 calls.
# A batched GPU PnP is a "next" row of SURVEY.md section 8(f).
# ------------------------------------------------------------------------------------------------------------
import math  # noqa: E402

import numpy as np  # noqa: E402


def _np(x, dtype=None):
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().numpy()
    x = np.asarray(x)
    return x.astype(dtype, copy=False) if dtype is not None else x


def pnp(points_3d, points_2d, camera_matrix, method=None):
    """ransac_voting.py:13-57: EPnP-RANSAC initialisation, iterative refinement, [R|t] float32 [3,4]."""
    import cv2

    assert points_3d.shape[0] == points_2d.shape[0], "points 3D and points 2D must have same number of vertices"
    if np.abs(np.sum(points_2d)) < 1e-4:
        return np.zeros([3, 4]).astype(np.float32)
    points_3d = np.expand_dims(points_3d, 0)
    points_2d = np.expand_dims(points_2d, 0)
    points_2d = np.ascontiguousarray(points_2d.astype(np.float64))
    points_3d = np.ascontiguousarray(points_3d.astype(np.float64))
    camera_matrix = camera_matrix.astype(np.float64)
    _, rvec0, T0, _ = cv2.solvePnPRansac(points_3d, points_2d, camera_matrix, None, flags=cv2.SOLVEPNP_EPNP,
                                         confidence=0.9999, reprojectionError=12)
    ret, R_exp, t = cv2.solvePnP(points_3d, points_2d, camera_matrix, None, flags=cv2.SOLVEPNP_ITERATIVE,
                                 useExtrinsicGuess=True, rvec=rvec0, tvec=T0)
    if ret is False or np.isnan(np.sum(t)):
        return np.zeros([3, 4]).astype(np.float32)
    R, _ = cv2.Rodrigues(R_exp)
    if t[2] < 0:
        t *= -1
        R *= -1
    return np.concatenate([R, t], axis=-1).astype(np.float32)


def transform_points_back(points, h_crop, w_crop, sx, sy, dx, dy, angle, scale):
    """transform_points_back_tf (ransac_voting.py:92-121) in float32: undo scale, crop offset, shift and rotation."""
    f = np.float32
    proj = (points.astype(f) / f(scale)).astype(f)
    tm = np.array([[1.0, 0.0, -dx], [0.0, 1.0, -dy], [0.0, 0.0, 1.0]], f)
    cx, cy = f(sx) / f(2.0), f(sy) / f(2.0)
    ang = f(-angle) * f(math.pi / 180)
    a, b = f(np.cos(ang)), f(np.sin(ang))
    c = (f(1.0) - a) * cx - b * cy
    d = b * cx + (f(1.0) - a) * cy
    rm = np.array([[a, b, c], [-b, a, d], [0.0, 0.0, 1.0]], f)
    proj = proj + np.array([w_crop, h_crop], f)
    homog = np.concatenate([proj.T, np.ones([1, points.shape[0]], f)], axis=0)
    new = rm @ (tm @ homog)
    return new[0:2].T.astype(f)


def project(xyz, K, RT):
    """project_tf (ransac_voting.py:173-182), float32."""
    f = np.float32
    xyz_proj = xyz.astype(f) @ RT[:, :3].astype(f).T + RT[:, 3:].astype(f).T
    uvw = xyz_proj @ K.astype(f).T
    with np.errstate(divide="ignore", invalid="ignore"):
        xy = uvw[:, :2] / uvw[:, 2:]
    return xy.astype(f), xyz_proj.astype(f)


def wants_grad(x):
    """True if `x` is a torch tensor that autograd would differentiate here."""
    return isinstance(x, torch.Tensor) and x.requires_grad and torch.is_grad_enabled()


def pnp_backward_cuda(points_3d, camera_matrixes, poses, grad_poses, pose_form):
    """casa_pnp_backward: dL/d points_2d [n,vn,2] (x,y) for dL/d poses = grad_poses, the BPnP_fast gradient
    (bpnp_layers.py:138-277).  points_3d [n,vn,3], camera_matrixes [n,3,3], poses / grad_poses [n,3,4] (pose_form 12,
    [R|t]) or [n,6] (pose_form 6, (rvec, tvec)); all float32 on one CUDA device."""
    p3 = as_cuda_f32(points_3d, "points_3d")
    cam = as_cuda_f32(camera_matrixes, "camera_matrixes")
    poses = as_cuda_f32(poses, "poses")
    grad_poses = as_cuda_f32(grad_poses.contiguous(), "grad_poses")
    n, vn = p3.shape[0], p3.shape[1]
    if tuple(poses.shape) != tuple(grad_poses.shape) or poses.numel() != n * pose_form or tuple(cam.shape) != (n, 3, 3):
        raise ValueError("pnp_backward_cuda: poses / grad_poses must hold %d x %d floats and camera_matrixes be [%d,3,3]"
                         % (n, pose_form, n))
    dev = p3.device
    out = torch.empty((n, vn, 2), dtype=torch.float32, device=dev)
    hdl = _lib.handle(dev.index if dev.index is not None else torch.cuda.current_device(), current_stream_ptr(dev))
    with torch.cuda.device(dev):
        rc = _lib.lib().casa_pnp_backward(hdl, n, vn, ptr(p3), ptr(cam), ptr(poses), int(pose_form), ptr(grad_poses),
                                          ptr(out), current_stream_ptr(dev))
    _lib.check(rc)
    return out


class PnpGradFn(torch.autograd.Function):
    """torch.autograd carrier of a PnP solve whose backward is casa_pnp_backward.  `solve(points_2d)` runs the forward
    (the GPU kernel or the host OpenCV sequence) on the detached points and returns the poses on the points' device;
    PyTorch only routes the gradient."""

    @staticmethod
    def forward(ctx, points_2d, solve, points_3d, camera_matrixes, pose_form):
        poses = solve(points_2d.detach())
        ctx.pose_form = pose_form
        ctx.save_for_backward(points_3d, camera_matrixes, poses)
        return poses

    @staticmethod
    def backward(ctx, grad_poses):
        p3, cam, poses = ctx.saved_tensors
        g = pnp_backward_cuda(p3, cam, poses, grad_poses, ctx.pose_form)
        return g, None, None, None, None


def pnp_cuda(points_2d, points_3d, camera_matrixes, offsets=None):
    """Batched GPU PnP (casa_pnp): points_2d [n,vn,2] (x,y), points_3d [n,vn,3], camera_matrixes [n,3,3],
    offsets [n,10] or None -> poses [n,3,4] float32 on the device of points_2d.  Same guards and sign
    convention as `pnp` / map_offsets / map_pnp (ransac_voting.py:13-57, 487-514).
    If points_2d is a CUDA tensor that requires grad, the poses carry a grad_fn whose backward is casa_pnp_backward
    (BPnP_fast, bpnp_layers.py:138-277); differentiating through `offsets` is not supported (ValueError)."""
    dev = points_2d.device if isinstance(points_2d, torch.Tensor) and points_2d.is_cuda else torch.device("cuda", torch.cuda.current_device())

    def put(x):
        t = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(np.asarray(x, np.float32)))
        return t.to(device=dev, dtype=torch.float32).contiguous()

    grad = wants_grad(points_2d) and points_2d.is_cuda
    if grad and offsets is not None:
        raise ValueError("pnp_cuda: no gradient through the offsets un-mapping; pass offsets=None or detached points")
    p2, p3, cam = put(points_2d), put(points_3d).detach(), put(camera_matrixes).detach()
    off = put(offsets) if offsets is not None else None

    def solve(q):
        n, vn = q.shape[0], q.shape[1]
        out = torch.empty((n, 3, 4), dtype=torch.float32, device=dev)
        hdl = _lib.handle(dev.index if dev.index is not None else torch.cuda.current_device(), current_stream_ptr(dev))
        with torch.cuda.device(dev):
            rc = _lib.lib().casa_pnp(hdl, n, vn, ptr(q), ptr(p3), ptr(cam), ptr(off), ptr(out), current_stream_ptr(dev))
        _lib.check(rc)
        return out

    return PnpGradFn.apply(p2, solve, p3, cam, 12) if grad else solve(p2)


def estimate_poses(points, keypoints, camera_matrixes, valid_points_filter, offsets, pnp_backend="cv2"):
    """ransac_voting.py:525-558.  pnp_backend="cuda" runs the batched GPU PnP (casa_pnp) instead of the
    per-object OpenCV calls of the reference (about 1.4 ms per object on the host).
    :param points:             [b,oc,vn,2]
    :param keypoints:          [b,oc,ic,vn,3]
    :param camera_matrixes:    [b,3,3]
    :param valid_points_filter:[b,oc]
    :param offsets:            [b,10]
    :return: poses [b,oc,3,4] float32, false-positive count per object [oc]
    """
    points = _np(points, np.float32)
    keypoints = _np(keypoints, np.float32)
    camera_matrixes = _np(camera_matrixes, np.float32)
    valid = _np(valid_points_filter)
    offsets = _np(offsets, np.float32)
    b, oc, ic, vn, _ = keypoints.shape
    if pnp_backend == "cuda":
        fp = ((valid == 0) & (points.reshape(b, oc, -1).sum(-1, dtype=np.float32) > 0)).astype(np.float32).sum(axis=0)
        poses = pnp_cuda(points.reshape(b * oc, vn, 2), keypoints[:, :, 0].reshape(b * oc, vn, 3),
                         np.broadcast_to(camera_matrixes[:, None], (b, oc, 3, 3)).reshape(b * oc, 3, 3),
                         np.broadcast_to(offsets[:, None], (b, oc, 10)).reshape(b * oc, 10))
        return poses.cpu().numpy().reshape(b, oc, 3, 4), (fp[0] if oc == 1 else fp)
    if pnp_backend != "cv2":
        raise ValueError("pnp_backend must be 'cv2' or 'cuda'")
    poses = np.zeros((b, oc, 3, 4), np.float32)
    false_positive = np.zeros((b, oc), np.float32)
    for i in range(b):
        o = offsets[i]
        for c in range(oc):
            pts = points[i, c]
            if valid[i, c] == 0 and pts.sum(dtype=np.float32) > 0:  # map_false_positive :517-522
                false_positive[i, c] = 1.0
            if abs(pts.sum(dtype=np.float32)) < 0.01:  # map_offsets :489, map_pnp :510
                continue
            pts = transform_points_back(pts, o[0], o[1], o[8], o[9], o[4], o[5], o[6], o[7])  # :494-504
            if abs(pts.sum(dtype=np.float32)) < 0.01:
                continue
            poses[i, c] = pnp(keypoints[i, c, 0], pts, camera_matrixes[i])  # :513
    fp = false_positive.sum(axis=0)
    return poses, (fp[0] if oc == 1 else fp)  # tf.squeeze(:558)


def _adds_error(A, B):
    """ransac_voting.py:596-610: mean-free closest-point distances in float64."""
    A = A.astype(np.float64)
    B = B.astype(np.float64)
    err = (A * A).sum(1)[:, None] - 2 * (A @ B.T) + (B * B).sum(1)[None, :]
    return np.sqrt(np.abs(err.min(axis=1)) + 1e-5).astype(np.float32)


def map_estimates(pose, pose_gt, object_points_3d, camera_matrix, diameter, valid, count, allowed_error_2d):
    """ransac_voting.py:561-625 -> [err_2d, err_3d, valid_3d, valid_2d, missing, false_positive]."""
    if valid == 0:
        if abs(pose.sum(dtype=np.float32)) > 0.0001:
            return np.array([0, 0, 0, 0, 0, 1], np.float32)
        return np.zeros(6, np.float32)
    if abs(pose.sum(dtype=np.float32)) < 0.0001:
        return np.array([99.9, 999.9, 0.0, 0.0, 1.0, 0.0], np.float32)
    pts = object_points_3d[0][: int(count[0])]
    p2d, p3d = project(pts, camera_matrix, pose)
    t2d, t3d = project(pts, camera_matrix, pose_gt[0])
    err_2d = np.float32(np.sqrt(((t2d - p2d) ** 2).sum(1)).mean())
    if int(count[0]) in (7862, 3417):  # glue and eggbox: ADD-S (:618)
        err_3d = np.float32(_adds_error(t3d, p3d).mean())
    else:
        err_3d = np.float32(np.sqrt(((t3d - p3d) ** 2).sum(1)).mean())
    valid_3d = np.float32(err_3d < np.float32(diameter[0][0]) * np.float32(0.1))
    valid_2d = np.float32(err_2d < allowed_error_2d)
    return np.array([err_2d, err_3d, valid_3d, valid_2d, 0.0, 0.0], np.float32)


def pose_errors_cuda(poses, poses_gt, camera_matrixes, model_points, model_counts, diameters, valid, allowed_error_2d=5.0,
                     obj_model=None):
    """Per-object rows of map_estimates (ransac_voting.py:561-625) on the GPU (casa_pose_errors).
    poses, poses_gt [n,3,4]; camera_matrixes [n,3,3]; model_points [m,maxp,3]; model_counts [m]; diameters [n];
    valid [n]; obj_model [n] or None (object i uses model i % m) -> [n,6] float32 device tensor
    [err_2d, err_3d, valid_3d, valid_2d, missing, false_positive]."""
    dev = poses.device if isinstance(poses, torch.Tensor) and poses.is_cuda else torch.device("cuda", torch.cuda.current_device())

    def put(x, dtype=torch.float32):
        t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.array(x, copy=True))  # also un-broadcasts read-only views
        return t.to(device=dev, dtype=dtype).contiguous()

    po, gt, cam = put(poses).reshape(-1, 3, 4), put(poses_gt).reshape(-1, 3, 4), put(camera_matrixes).reshape(-1, 3, 3)
    pts, cnt = put(model_points), put(model_counts, torch.int32).reshape(-1)
    dia, val = put(diameters).reshape(-1), put(valid, torch.int32).reshape(-1)
    om = put(obj_model, torch.int32).reshape(-1) if obj_model is not None else None
    n, (m, maxp, _) = po.shape[0], pts.shape
    if not (gt.shape[0] == cam.shape[0] == dia.shape[0] == val.shape[0] == n and cnt.shape[0] == m):
        raise ValueError("pose_errors_cuda: inconsistent leading dimensions")
    out = torch.empty((n, 6), dtype=torch.float32, device=dev)
    hdl = _lib.handle(dev.index if dev.index is not None else torch.cuda.current_device(), current_stream_ptr(dev))
    with torch.cuda.device(dev):
        rc = _lib.lib().casa_pose_errors(hdl, n, m, maxp, ptr(po), ptr(gt), ptr(cam), ptr(pts), ptr(cnt), ptr(om), ptr(dia),
                                         ptr(val), float(allowed_error_2d), ptr(out), current_stream_ptr(dev))
    _lib.check(rc)
    return out


def evaluate_poses(poses, poses_gt, points_estimated, object_points_3d, object_points_3d_count, camera_matrixes,
                   diameters, valid_points_filter, allowed_error_2d, backend="numpy"):
    """ransac_voting.py:628-687 -> (err_2d, err_3d, valid_2d, valid_3d, missing_object, valid_points_count,
    false_positive_detection), each summed over the batch -> [oc].  backend="cuda" computes the per-object
    rows with casa_pose_errors (the N x N ADD-S search is the expensive part on the host)."""
    poses = _np(poses, np.float32)
    poses_gt = _np(poses_gt, np.float32)
    object_points_3d = _np(object_points_3d, np.float32)
    counts = _np(object_points_3d_count)
    cams = _np(camera_matrixes, np.float32)
    diameters = _np(diameters, np.float32)
    valid = _np(valid_points_filter)
    b, oc, ic, vn, _ = object_points_3d.shape
    dm = diameters.reshape(-1)  # tf.reshape(diameters, [-1, ic, 1]) (:651); also accept per-object diameters
    if dm.size == b * oc * ic:
        diameters = dm.reshape(b, oc, ic, 1)
    elif dm.size == oc * ic:
        diameters = np.broadcast_to(dm.reshape(1, oc, ic, 1), (b, oc, ic, 1))
    elif dm.size == oc:
        diameters = np.broadcast_to(dm.reshape(1, oc, 1, 1), (b, oc, ic, 1))
    else:
        raise ValueError("diameters must hold b*oc*ic, oc*ic or oc values")
    if backend == "cuda":
        same = all(np.array_equal(object_points_3d[0], object_points_3d[i]) and np.array_equal(counts[0], counts[i])
                   for i in range(1, b)) if object_points_3d.strides[0] != 0 else True
        if same:  # one model table for the whole batch (how :67-72 tiles it): object (i, c) uses model c
            table, cnt_t, om = object_points_3d[0, :, 0], counts.reshape(b, oc, ic)[0, :, 0], None
        else:
            table, cnt_t, om = object_points_3d[:, :, 0].reshape(b * oc, vn, 3), counts.reshape(b, oc, ic)[:, :, 0].reshape(-1), None
        res = pose_errors_cuda(poses.reshape(b * oc, 3, 4), poses_gt.reshape(b, oc, ic, 3, 4)[:, :, 0].reshape(b * oc, 3, 4),
                               np.broadcast_to(cams[:, None], (b, oc, 3, 3)).reshape(b * oc, 3, 3), table, cnt_t,
                               diameters[:, :, 0, 0].reshape(-1), valid.reshape(-1), allowed_error_2d, om)
        s = res.reshape(b, oc, 6).sum(dim=0).cpu().numpy()
        return s[:, 0], s[:, 1], s[:, 3], s[:, 2], s[:, 4], valid.sum(axis=0).astype(np.float32), s[:, 5]
    if backend != "numpy":
        raise ValueError("backend must be 'numpy' or 'cuda'")
    res = np.zeros((b, oc, 6), np.float32)
    for i in range(b):
        for c in range(oc):
            res[i, c] = map_estimates(poses[i, c], poses_gt[i, c], object_points_3d[i, c], cams[i], diameters[i, c],
                                      valid[i, c], counts[i, c], allowed_error_2d)
    s = res.sum(axis=0)
    return s[:, 0], s[:, 1], s[:, 3], s[:, 2], s[:, 4], valid.sum(axis=0).astype(np.float32), s[:, 5]
