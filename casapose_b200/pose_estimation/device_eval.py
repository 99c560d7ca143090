"""Device-resident evaluation loop: voting -> batched PnP -> ADD / ADD-S, one small read-back per batch.

`estimate_and_evaluate_poses` (pose_evaluation.py) keeps the reference's argument list and therefore re-uploads
its constant tables (3-D keypoints, cameras, evaluation meshes) on every call and hands numpy arrays between its
stages like the reference does between TF and OpenCV.  `DeviceEvaluator` is the same computation
(/root/reference/casapose/pose_estimation/pose_evaluation.py:11-101) with the tables uploaded once and every
intermediate left on the GPU: casa_ransac_vote_seg -> casa_pnp -> casa_pose_errors; the per-class sums are one
[oc, 8] read-back.  Same statistics as the drop-in with pnp_backend="cuda", metric_backend="cuda".

The LS-layer path (CoordLSVotingWeighted, what CASAPose's own models use) has the same treatment: `ls_poses` is
poses_pnp (/root/reference/casapose/pose_estimation/pose_evaluation.py:164-217) on the device — the layer's call also
counts the available objects (casa_ls_vote_counts), then casa_pnp — and `evaluate_ls` adds evaluate_pose_estimates
(:104-160) with one [oc, 8] read-back."""
import numpy as np
import torch

from .. import _lib
from .._carrier import current_stream_ptr
from .ransac_voting import pnp_cuda, pose_errors_cuda, ransac_voting_layer_all_masks, wants_grad
from .voting_layers_2d import _LsVoteFn


class DeviceEvaluator:
    def __init__(self, object_points_3d, camera_matrix, diameters, evaluation_points=None, object_points_3d_count=None,
                 min_num=20, allowed_error_2d=5.0, round_hyp_num=512, device=None):
        """object_points_3d [oc,vn,3] keypoints; camera_matrix [3,3]; diameters [oc];
        evaluation_points [oc,P,3] + object_points_3d_count [oc] (mesh vertices for ADD / ADD-S) or None (:67-74)."""
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        f = lambda x: torch.as_tensor(np.ascontiguousarray(np.asarray(x, np.float32))).to(dev)  # noqa: E731
        self.dev = dev
        self.kp3 = f(object_points_3d)
        self.oc, self.vn = self.kp3.shape[0], self.kp3.shape[1]
        self.cam = f(camera_matrix).reshape(3, 3)
        self.diam = f(diameters).reshape(self.oc)
        if evaluation_points is not None and object_points_3d_count is not None:
            self.models = f(evaluation_points)
            self.counts = torch.as_tensor(np.asarray(object_points_3d_count, np.int32).reshape(self.oc)).to(dev)
        else:
            self.models = self.kp3
            self.counts = torch.full((self.oc,), self.vn, dtype=torch.int32, device=dev)
        self.min_num, self.allowed_error_2d, self.hn = min_num, allowed_error_2d, round_hyp_num

    def __call__(self, output_seg, target_seg, output_vertex, poses_gt, offsets=None, **vote_kw):
        """output_seg / target_seg [b,h,w,1+oc], output_vertex [b,h,w,2*vn] (CUDA tensors), poses_gt [b,oc,3,4]
        -> (stats dict of [oc] numpy arrays, poses [b,oc,3,4] CUDA tensor, keypoints [b,oc,vn,2] CUDA tensor)."""
        b, h, w, _ = output_seg.shape
        oc, vn = self.oc, self.vn
        valid = self._valid(target_seg)
        pts = ransac_voting_layer_all_masks(output_seg, output_vertex.reshape(b, h, w, vn, 2), self.hn, inlier_thresh=0.99,
                                            max_iter=20, min_num=self.min_num, max_num=30000, seg_scores=True, **vote_kw)
        n = b * oc
        off = None
        if offsets is not None:
            off = torch.as_tensor(offsets, dtype=torch.float32, device=self.dev).reshape(b, 1, 10).expand(b, oc, 10).reshape(n, 10).contiguous()
        poses = pnp_cuda(pts.reshape(n, vn, 2), self.kp3.unsqueeze(0).expand(b, oc, vn, 3).reshape(n, vn, 3).contiguous(),
                         self.cam.expand(n, 3, 3).contiguous(), off)
        fp_mask = ((valid == 0) & (pts.reshape(b, oc, -1).sum(-1) > 0)).to(torch.float32)  # map_false_positive :517-522
        stats = self._stats(poses, poses_gt, valid, fp_mask)
        return stats, poses.reshape(b, oc, 3, 4), pts

    def _valid(self, target_seg):
        return ((target_seg[..., 1:] != 0).sum(dim=(1, 2)) > self.min_num).to(torch.int32)  # :30-33

    def _stats(self, poses, poses_gt, valid, fp_mask):
        """casa_pose_errors on poses [b*oc,3,4] and the per-class batch sums: the only read-back, [oc, 8]."""
        b, oc = valid.shape
        n = b * oc
        gt = torch.as_tensor(poses_gt, dtype=torch.float32, device=self.dev).reshape(n, 3, 4)
        rows = pose_errors_cuda(poses.reshape(n, 3, 4), gt, self.cam.expand(n, 3, 3).contiguous(), self.models, self.counts,
                                self.diam.unsqueeze(0).expand(b, oc).reshape(n).contiguous(), valid.reshape(n),
                                self.allowed_error_2d).reshape(b, oc, 6)
        packed = torch.cat([rows.sum(dim=0), valid.sum(dim=0, keepdim=True).t().float(), fp_mask.sum(dim=0, keepdim=True).t()], dim=1)
        s = packed.cpu().numpy()
        return {"err_2d": s[:, 0], "err_3d": s[:, 1], "valid_3d": s[:, 2], "valid_2d": s[:, 3], "missing_object": s[:, 4],
                "false_positive_pose": s[:, 5], "valid_pose_count": s[:, 6], "false_positive_mask": s[:, 7]}

    def ls_poses(self, layer, seg, direct, w, check_finite=True):
        """poses_pnp(layer([seg, direct, w]), seg, ..., min_num, pnp_backend="cuda") without leaving the device
        (pose_evaluation.py:164-217): the layer's call with the availability counts, (y,x) -> (x,y), casa_pnp on the
        uploaded keypoints and camera, times (count > min_num).  seg / direct / w as for the layer ([b,h,w,1+oc],
        [b,h,w,2*vn], [b,h,w,vn], one dtype) -> (poses [b,oc,1,3,4], coords [b,oc,vn,2] (y,x)), CUDA tensors.
        Differentiable w.r.t. direct and w (casa_ls_vote_backward, casa_pnp_backward).  check_finite=False: nothing
        waits for the device; a non-finite result or a pixel-list overflow is reported by the handle's casa_sync."""
        oc, vn = self.oc, self.vn
        if layer.num_classes != oc + 1 or layer.num_points != vn:
            raise ValueError("ls_poses: the layer is built for num_classes=%d, num_points=%d; this evaluator needs %d and %d"
                             % (layer.num_classes, layer.num_points, oc + 1, vn))
        if wants_grad(direct) or wants_grad(w):
            coords, hot = _LsVoteFn.apply(layer, seg.detach(), direct, w, True, check_finite)
        else:
            coords, hot = layer._forward(seg, direct, w, False, check_finite, True)
        b = coords.shape[0]
        n = b * oc
        q = coords.reshape(n, vn, 2).flip(-1)  # (y,x) -> (x,y) :179
        poses = pnp_cuda(q, self.kp3.unsqueeze(0).expand(b, oc, vn, 3).reshape(n, vn, 3), self.cam.expand(n, 3, 3))
        available = (hot > self.min_num).to(torch.float32).reshape(n, 1, 1)  # :190-197
        return (poses * available).reshape(b, oc, 1, 3, 4), coords  # :213

    def evaluate_ls(self, layer, seg, direct, w, target_seg, poses_gt, check_finite=True):
        """evaluate_pose_estimates(coords, poses_pnp(...), poses_gt, target_seg, ..., metric_backend="cuda")
        (pose_evaluation.py:104-160) on the device: `ls_poses`, then casa_pose_errors and the batch sums, one [oc, 8]
        read-back.  target_seg [b,h,w,1+oc] CUDA tensor, poses_gt [b,oc,3,4] or [b,oc,1,3,4]
        -> (stats dict of [oc] numpy arrays, poses [b,oc,1,3,4], coords [b,oc,vn,2] (y,x)).
        false_positive_mask is zero, as in evaluate_pose_estimates.  With check_finite=False the handle is
        synchronised (casa_sync) after the read-back, so a non-finite LS result or a pixel-list overflow raises here."""
        poses, coords = self.ls_poses(layer, seg, direct, w, check_finite)
        valid = self._valid(target_seg)
        stats = self._stats(poses.detach(), poses_gt, valid, torch.zeros_like(valid, dtype=torch.float32))
        if not check_finite:
            dev = coords.device
            _lib.sync(dev.index if dev.index is not None else torch.cuda.current_device(), current_stream_ptr(dev))
        return stats, poses, coords
