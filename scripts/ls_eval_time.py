"""The LS evaluation path kept on the device (casa_ls_vote_counts, DeviceEvaluator.ls_poses / evaluate_ls) against the
host round-trips of the drop-ins (poses_pnp, evaluate_pose_estimates).

Synthetic config-1 frames: 16 x 480 x 640, 8 objects, 9 keypoints (seg 9 + direct 18 + conf 9 channels),
CoordLSVotingWeighted with filter_estimates=True.  Variants of one workload are timed in one process and alternated
round by round, so that clock and neighbour drift hit them alike:
  (a) the LS call: casa_ls_vote_typed against casa_ls_vote_counts (check_finite=False), one call at a time and with
      four calls in flight on four lanes; CUDA events around `--steps` calls;
  (b) one evaluation batch: evaluate_ls (check_finite False and True) against layer + poses_pnp + evaluate_pose_estimates
      with the cuda backends, and with the cv2 / numpy backends (`--host-steps` batches);
  (c) one training step: LS forward -> poses -> sum(poses * G) -> backward through ls_poses against the same step
      through poses_pnp(pnp_backend="cuda").
(b) and (c) are synchronous (a read-back ends each), timed with the host clock around batches that end in a device
synchronise.  Prints the card, its power limit and max SM clock (queried, not set), one line per variant, and a JSON
summary.

    python scripts/ls_eval_time.py [--rounds 5 --steps 50 --host-steps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

B, H, W = 16, 480, 640


def smi():
    q = "name,power.limit,clocks.max.sm"
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # the timing does not depend on it
        return "nvidia-smi unavailable: %s" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50, help="calls / batches / steps per variant and round")
    ap.add_argument("--host-steps", type=int, default=3, help="batches per round of the cv2 / numpy variant")
    args = ap.parse_args()

    import numpy as np
    import torch

    from casapose_b200 import _lib, synthetic
    from casapose_b200.pose_estimation import CoordLSVotingWeighted, DeviceEvaluator, evaluate_pose_estimates, poses_pnp

    if not torch.cuda.is_available():
        raise SystemExit("ls_eval_time.py needs a CUDA device")
    if _lib._sources_newer_than_lib():
        _lib.build()
    print("card:", torch.cuda.get_device_name(0), "| nvidia-smi name, power limit, max SM clock:", smi())
    F = np.float32
    ids = synthetic.CONFIG_8_IDS
    oc = len(ids)
    d = synthetic.make_frames(B, H, W, ids, variant="easy", with_logits=True)
    x = [torch.from_numpy(a).cuda() for a in (d["seg_logits"], d["vertex"].reshape(B, H, W, 18), d["conf_logits"])]
    K = synthetic.camera_matrix(H).astype(F)
    cams = np.broadcast_to(K, (B, 3, 3)).copy()
    kp3 = np.broadcast_to(d["keypoints_3d"][None, :, None], (B, oc, 1, 9, 3)).copy()
    target_seg = torch.from_numpy(np.concatenate([(d["labels"] == 0)[..., None].astype(F), d["mask"]], axis=-1)).cuda()
    poses_gt = d["poses_gt"][:, :, None].astype(F)
    poses_gt_dev = torch.from_numpy(poses_gt).cuda()
    diam = np.broadcast_to(d["diameters"][None], (B, oc)).copy()
    layer = CoordLSVotingWeighted("ls", oc + 1, num_points=9, filter_estimates=True)
    ev = DeviceEvaluator(kp3[0, :, 0], cams[0], diam[0])
    G = torch.from_numpy(np.random.default_rng(0).normal(size=(B, oc, 1, 3, 4)).astype(F))
    G_dev = G.cuda()

    # the variants compute the same values
    c0 = layer(x)
    c1, cnt = layer(x, return_counts=True)
    p_dev, _ = ev.ls_poses(layer, *x)
    p_ref = poses_pnp(c0, x[0], kp3, cams, oc, min_num=20, pnp_backend="cuda")
    torch.cuda.synchronize()
    assert torch.equal(c0, c1) and torch.equal(p_dev.cpu(), p_ref)
    print("objects available: %d of %d" % (int((cnt > 20).sum()), B * oc))

    # (a) the LS call
    def ls_call(variant):
        return layer(x, check_finite=False, return_counts=variant == "counts")

    def timed_ls(variant, lanes):
        _lib.set_async(0, lanes)
        for _ in range(2 * max(lanes, 2)):  # every lane's workspace and graph
            ls_call(variant)
        _lib.join(0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            ls_call(variant)
        _lib.join(0)
        e1.record()
        torch.cuda.synchronize()
        _lib.sync(0)
        _lib.set_async(0, 0)
        return e0.elapsed_time(e1) / args.steps

    # (b) one evaluation batch
    def eval_batch(variant):
        if variant == "evaluate_ls":
            return ev.evaluate_ls(layer, *x, target_seg, poses_gt_dev, check_finite=False)[0]
        if variant == "evaluate_ls checked":
            return ev.evaluate_ls(layer, *x, target_seg, poses_gt_dev)[0]
        cuda = variant == "drop-ins cuda"
        coords = layer(x)
        poses = poses_pnp(coords, x[0], kp3, cams, oc, min_num=20, pnp_backend="cuda" if cuda else "cv2")
        return evaluate_pose_estimates(coords, poses[:, :, 0], poses_gt, target_seg, kp3, cams, diam,
                                       metric_backend="cuda" if cuda else "numpy")[0]

    # (c) one training step
    def train_step(variant):
        dd, ww = x[1].clone().requires_grad_(True), x[2].clone().requires_grad_(True)
        if variant == "ls_poses":
            poses, _ = ev.ls_poses(layer, x[0], dd, ww)
            (poses * G_dev).sum().backward()
        else:
            poses = poses_pnp(layer([x[0], dd, ww]), x[0], kp3, cams, oc, min_num=20, pnp_backend="cuda")
            (poses * G).sum().backward()
        return dd.grad, ww.grad

    def timed_host(fn, variant, steps):
        fn(variant)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn(variant)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / steps

    g_dev, g_ref = train_step("ls_poses"), train_step("poses_pnp")
    assert torch.equal(g_dev[0], g_ref[0]) and torch.equal(g_dev[1], g_ref[1])

    workloads = [
        ("(a) ls call, one at a time", ["typed", "counts"], lambda v: timed_ls(v, 1)),
        ("(a) ls call, 4 in flight", ["typed", "counts"], lambda v: timed_ls(v, 4)),
        ("(b) eval batch", ["evaluate_ls", "evaluate_ls checked", "drop-ins cuda", "drop-ins cv2/numpy"],
         lambda v: timed_host(eval_batch, v, args.host_steps if "cv2" in v else args.steps)),
        ("(c) training step", ["ls_poses", "poses_pnp"], lambda v: timed_host(train_step, v, args.steps)),
    ]
    res = {name: {v: [] for v in variants} for name, variants, _ in workloads}
    for r in range(args.rounds):
        for name, variants, run in workloads:
            for v in (variants if r % 2 == 0 else variants[::-1]):
                res[name][v].append(run(v))
    print("after the runs:", smi())
    summary = {}
    for name, variants, _ in workloads:
        for v in variants:
            t = np.array(res[name][v])
            med = float(np.median(t))
            summary.setdefault(name, {})[v] = {"mean_ms": float(t.mean()), "median_ms": med, "min_ms": float(t.min()),
                                               "max_ms": float(t.max()), "batches_per_s": 1e3 / med, "frames_per_s": B * 1e3 / med}
            print("%-28s %-20s ms: mean %8.4f  median %8.4f  min %8.4f  max %8.4f   %9.1f batches/s  %10.1f frames/s"
                  % (name, v, t.mean(), med, t.min(), t.max(), 1e3 / med, B * 1e3 / med))
        s = summary[name]
        base = s[variants[0]]["median_ms"]
        print("%-28s " % name + "   ".join("%s / %s = %.3f" % (variants[0], v, base / s[v]["median_ms"]) for v in variants[1:]))
    print(json.dumps({"card": torch.cuda.get_device_name(0), "smi": smi(), "rounds": args.rounds, "steps": args.steps,
                      "host_steps": args.host_steps, "frames_per_batch": B, "ms": summary}))


if __name__ == "__main__":
    main()
