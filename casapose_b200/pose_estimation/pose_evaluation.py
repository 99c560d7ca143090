"""Drop-in for casapose.pose_estimation.pose_evaluation (the callers of the voting hot path).

Same names, argument order and outputs as /root/reference/casapose/pose_estimation/pose_evaluation.py.
The pre-step (argmax -> one-hot -> drop background, :36-47) is fused into the voting library
(casa_ransac_vote_seg), the voting itself is the sm_100a path, PnP and the metrics run on the host with
OpenCV exactly like the reference (tf.numpy_function, ransac_voting.py:513)."""
import numpy as np
import torch

from .bpnp_layers import BPNP_fast, rodrigues_batch
from .ransac_voting import PnpGradFn, _np, estimate_poses, evaluate_poses, ransac_voting_layer_all_masks, wants_grad


def _vote_from_scores(output_seg, output_vertex, oc, vc, min_num, **vote_kw):
    """pose_evaluation.py:36-58: one_hot(argmax(seg))[..., 1:], per-class vertex gather, RANSAC voting."""
    b, h, w, c = output_seg.shape
    if oc > 1 and output_vertex.shape[-1] == vc * oc * 2:  # PVNet-style: one field per class (:38-45)
        output_vertex = output_vertex.reshape(b, h, w, oc, vc, 2)
    else:
        output_vertex = output_vertex.reshape(b, h, w, vc, 2)  # :47
    return ransac_voting_layer_all_masks(output_seg, output_vertex, 512, inlier_thresh=0.99, max_iter=20, min_num=min_num,
                                         max_num=30000, seg_scores=True, **vote_kw)  # :50-58


def _objects_available(target_seg, min_num):
    t = target_seg if isinstance(target_seg, torch.Tensor) else torch.as_tensor(np.asarray(target_seg))
    cnt = (t[:, :, :, 1:] != 0).sum(dim=(1, 2))  # tf.math.count_nonzero (:30-32)
    return (cnt > min_num).to(torch.int32).cpu().numpy()  # :33


def _eval_points(evaluation_points, object_points_3d_count, object_points_3d, b, oc, ic):
    if evaluation_points is not None and object_points_3d_count is not None:  # :67-72
        ev = _np(evaluation_points, np.float32)[None, :, None]
        object_points_3d = np.broadcast_to(ev, (b, ev.shape[1], ic) + ev.shape[3:])  # tf.tile (:69), without the copies
        cnt = np.tile(_np(object_points_3d_count)[None], [b, 1, ic])
    else:
        object_points_3d = _np(object_points_3d, np.float32)
        cnt = np.ones([b, oc, ic], dtype=np.int32) * 9  # :74
    return object_points_3d, cnt


def estimate_and_evaluate_poses(output_seg, target_seg, output_vertex, poses_gt, object_points_3d, camera_data,
                                diameters, offsets, evaluation_points=None, object_points_3d_count=None,
                                points_estimated=None, min_num=20, pnp_backend="cv2", metric_backend="numpy", **vote_kw):
    """pose_evaluation.py:11-101 -> ([valid_2d, valid_3d, valid_pose_count, false_positive_mask, err_2d, err_3d,
    missing_object, false_positive_pose], poses [b,oc,3,4], points_estimated [b,oc,vn,2])."""
    b, h, w, c = target_seg.shape
    _, oc, ic, _, _ = poses_gt.shape
    _, _, _, vc, _ = object_points_3d.shape
    objects_available = _objects_available(target_seg, min_num)
    if points_estimated is None:
        points_estimated = _vote_from_scores(output_seg, output_vertex, oc, vc, min_num, **vote_kw)
    else:
        points_estimated = points_estimated * torch.tensor([[[[h, w]]]], dtype=torch.float32, device=points_estimated.device)  # :60
    poses, false_positive_mask = estimate_poses(points_estimated, object_points_3d, camera_data, objects_available, offsets,
                                                pnp_backend=pnp_backend)
    pts3d, cnt = _eval_points(evaluation_points, object_points_3d_count, object_points_3d, b, oc, ic)
    err_2d, err_3d, valid_2d, valid_3d, missing_object, valid_pose_count, false_positive_pose = evaluate_poses(
        poses, poses_gt, points_estimated, pts3d, cnt, camera_data, diameters, objects_available, 5.0,
        backend=metric_backend)  # :76-86
    return ([valid_2d, valid_3d, valid_pose_count, false_positive_mask, err_2d, err_3d, missing_object, false_positive_pose],
            torch.from_numpy(poses), points_estimated)


def evaluate_pose_estimates(points_estimated, poses, poses_gt, target_seg, object_points_3d, camera_data, diameters,
                            evaluation_points=None, object_points_3d_count=None, min_num=20, metric_backend="numpy"):
    """pose_evaluation.py:104-160."""
    b, h, w, c = target_seg.shape
    _, oc, ic, _, _ = poses_gt.shape
    objects_available = _objects_available(target_seg, min_num)
    pts3d, cnt = _eval_points(evaluation_points, object_points_3d_count, object_points_3d, b, oc, ic)
    err_2d, err_3d, valid_2d, valid_3d, missing_object, valid_pose_count, false_positive_pose = evaluate_poses(
        poses, poses_gt, points_estimated, pts3d, cnt, camera_data, diameters, objects_available, 5.0, backend=metric_backend)
    return ([valid_2d, valid_3d, valid_pose_count, np.zeros_like(valid_2d), err_2d, err_3d, missing_object,
             false_positive_pose], poses, points_estimated)


def _host_poses(pts, obj3d, cam):
    """pose_evaluation.py:199-212 before the availability mask: BPNP_fast (OpenCV), Rodrigues, t_z flip -> [n,3,4]."""
    poses6 = BPNP_fast(name="BPNP")([np.ascontiguousarray(pts), obj3d, cam])  # :199
    if not np.isfinite(poses6).all():  # :201-206
        raise FloatingPointError("Tensor had inf or nan values: %r" % (poses6,))
    R = rodrigues_batch(poses6[:, 0:3])  # :208
    T = poses6[:, 3:6][..., None]  # :209
    poses = np.concatenate([R, T], axis=-1)
    return np.where(T[:, 2:3, :] < 0, -poses, poses)  # :212


def poses_pnp(points_estimated, seg_estimated, object_points_3d, camera_data, no_objects, min_num=20, pnp_backend="cv2"):
    """pose_evaluation.py:164-217: LS-layer output (y,x) -> PnP -> [b,oc,1,3,4].  pnp_backend="cuda": casa_pnp.
    If points_estimated is a CUDA tensor that requires grad, the (CPU) result is differentiable w.r.t. it with either
    backend: the backward is casa_pnp_backward on the returned [R|t] (BPnP_fast, bpnp_layers.py:138-277).  The forward
    values are those of the call without grad."""
    b, h, w, _ = seg_estimated.shape
    oc, ic = no_objects, 1
    _, _, _, vc, _ = object_points_3d.shape
    grad = wants_grad(points_estimated)
    if grad and not points_estimated.is_cuda:
        raise ValueError("poses_pnp: the gradient runs on the GPU (casa_pnp_backward); points_estimated must be a CUDA tensor")
    pts = _np(points_estimated, np.float32).reshape(-1, vc, 2)[:, :, ::-1]  # (y,x) -> (x,y) :179
    obj3d = _np(object_points_3d, np.float32).reshape(-1, vc, 3)
    seg = seg_estimated if isinstance(seg_estimated, torch.Tensor) else torch.as_tensor(np.asarray(seg_estimated))
    hot = torch.softmax(seg.float() * 1e6, dim=-1)[:, :, :, 1:]  # :183-185
    count = (hot > 0.1).sum(dim=(1, 2))  # :186-188
    available = (count > min_num).to(torch.float32).reshape(-1, 1, 1).cpu().numpy()  # :190-197
    cam = _np(camera_data, np.float32)[0]
    n = pts.shape[0]
    if grad:  # the same steps as torch ops on the device, so that autograd can route dL/d poses to points_estimated
        dev = points_estimated.device
        q = points_estimated.to(torch.float32).reshape(-1, vc, 2).flip(-1)  # :179
        av = torch.from_numpy(available).to(dev)
    if pnp_backend == "cuda":
        from .ransac_voting import pnp_cuda

        p3 = np.broadcast_to(obj3d, (n,) + obj3d.shape[1:]) if obj3d.shape[0] == n else np.tile(obj3d, (n // obj3d.shape[0], 1, 1))
        if grad:
            return (pnp_cuda(q, p3, np.broadcast_to(cam, (n, 3, 3))) * av).reshape(b, oc, ic, 3, 4).cpu()
        poses = pnp_cuda(np.ascontiguousarray(pts), p3, np.broadcast_to(cam, (n, 3, 3))).cpu().numpy()
        return torch.from_numpy((poses * available).reshape(b, oc, ic, 3, 4).astype(np.float32))
    if pnp_backend != "cv2":
        raise ValueError("pnp_backend must be 'cv2' or 'cuda'")
    if grad:
        p3 = torch.from_numpy(np.ascontiguousarray(obj3d[:n])).to(dev)
        cam_t = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(cam, (n, 3, 3)))).to(dev)

        def solve(d):
            return torch.from_numpy(np.ascontiguousarray(_host_poses(d.cpu().numpy(), obj3d, cam), np.float32)).to(dev)

        return (PnpGradFn.apply(q, solve, p3, cam_t, 12) * av).reshape(b, oc, ic, 3, 4).cpu()
    poses = _host_poses(pts, obj3d, cam)
    poses = poses * available  # :213
    return torch.from_numpy(poses.reshape(b, oc, ic, 3, 4).astype(np.float32))


def pose_estimation(output_seg, target_seg, output_vertex, poses_gt, object_points_3d, camera_data, offsets,
                    points_estimated=None, min_num=20, pnp_backend="cv2", **vote_kw):
    """pose_evaluation.py:222-269 -> poses [b,oc,3,4]."""
    b, h, w, c = target_seg.shape
    _, oc, ic, _, _ = poses_gt.shape
    _, _, _, vc, _ = object_points_3d.shape
    objects_available = np.ones([b, oc])  # :239
    if points_estimated is None:
        points_estimated = _vote_from_scores(output_seg, output_vertex, oc, vc, min_num, **vote_kw)
    else:
        points_estimated = points_estimated * torch.tensor([[[[h, w]]]], dtype=torch.float32, device=points_estimated.device)
    poses, _ = estimate_poses(points_estimated, object_points_3d, camera_data, objects_available, offsets, pnp_backend=pnp_backend)
    return torch.from_numpy(poses)
