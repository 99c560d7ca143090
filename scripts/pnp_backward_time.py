"""Times the PnP backward (casa_pnp_backward, DESIGN.md K10) and the training-chain step it completes, with CUDA events,
and prints one JSON object with the card name and its power limit.

  * casa_pnp_backward at n = 128 (16 frames x 8 objects) and n = 4096, both pose forms: per launch from 100 launches
    captured in a CUDA graph (device time), and per call from back-to-back eager calls (includes the host call);
  * the step at 16 x 480x640, 8 objects, 9 keypoints: LS forward + LS backward (casa_ls_vote, casa_ls_vote_backward)
    next to LS forward + casa_pnp + casa_pnp_backward + LS backward, run alternately.

usage: python scripts/pnp_backward_time.py [--iters N] [--steps S] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from casapose_b200 import _lib, synthetic  # noqa: E402
from casapose_b200.pose_estimation import CoordLSVotingWeighted  # noqa: E402
from casapose_b200.pose_estimation.ransac_voting import pnp_backward_cuda, pnp_cuda  # noqa: E402

B, H, W, OC, VN = 16, 480, 640, 8, 9


def card():
    limit = None
    try:
        import pynvml as nv

        nv.nvmlInit()
        limit = nv.nvmlDeviceGetEnforcedPowerLimit(nv.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())) / 1000.0
    except Exception:  # no NVML in this environment: ask nvidia-smi (a read-only query)
        import subprocess

        try:
            q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                                "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
            limit = float(q.stdout.strip().splitlines()[0])
        except Exception as e:  # say so rather than guess
            limit = "unavailable (%s)" % type(e).__name__
    return torch.cuda.get_device_name(), limit


def events_ms(fn, iters, warmup=20):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def backward_inputs(n, form, seed=0):
    rng = np.random.default_rng(seed)
    kp = np.array([synthetic.lm_models()["obj_%06d" % o]["keypoints"] for o in synthetic.CONFIG_8_IDS], np.float32)
    X = kp[np.arange(n) % len(kp)]
    K = synthetic.camera_matrix(H).astype(np.float32)
    uv = np.zeros((n, VN, 2), np.float32)
    for i in range(n):
        R = synthetic._random_rotation(rng)
        t = np.array([rng.uniform(-200, 200), rng.uniform(-150, 150), rng.uniform(600, 1200)])
        c = X[i] @ R.T + t
        p = c @ K.T
        uv[i] = p[:, :2] / p[:, 2:] + rng.normal(scale=0.5, size=(VN, 2))
    p3 = torch.from_numpy(X).cuda()
    cam = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(K, (n, 3, 3)))).cuda()
    poses = pnp_cuda(torch.from_numpy(uv).cuda(), p3, cam)
    if form == 6:  # (rvec, tvec) of the same poses
        from scipy.spatial.transform import Rotation

        P = poses.cpu().numpy()
        r = np.zeros((n, 6), np.float32)
        ok = P.reshape(n, 12).any(1)  # a failed solve stays an all-zero pose
        r[ok] = np.concatenate([Rotation.from_matrix(P[ok, :, :3]).as_rotvec(), P[ok, :, 3]], 1)
        poses = torch.from_numpy(r).cuda()
    grad = torch.from_numpy(rng.normal(size=tuple(poses.shape)).astype(np.float32)).cuda()
    return p3, cam, poses.contiguous(), grad


def time_backward(n, form, iters):
    lib = _lib.lib()
    p3, cam, poses, grad = backward_inputs(n, form)
    out = torch.empty((n, VN, 2), device="cuda")
    side = torch.cuda.Stream()
    hdl = _lib.handle(torch.cuda.current_device(), side.cuda_stream)

    def call():
        rc = lib.casa_pnp_backward(hdl, n, VN, p3.data_ptr(), cam.data_ptr(), poses.data_ptr(), form, grad.data_ptr(),
                                   out.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, lib.casa_last_error()

    with torch.cuda.stream(side):
        eager = events_ms(call, iters)
        launches = C.c_int64()
        lib.casa_last_launches(hdl, C.byref(launches))
        call()
        torch.cuda.synchronize()
        ref = out.clone()
        try:  # no host synchronisation and no allocation inside the call: it can be captured
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                for _ in range(100):
                    call()
            graph = round(events_ms(g.replay, max(iters // 100, 10), warmup=3) / 100 * 1e3, 2)
        except RuntimeError as e:
            graph = "capture failed: %s" % e
        torch.cuda.synchronize()
    assert torch.equal(out, ref) and torch.isfinite(out).all()
    return {"n": n, "pose_form": form, "graph_us_per_launch": graph, "eager_us_per_call": round(eager * 1e3, 2),
            "launches_per_call": launches.value}


def time_chain(steps, rounds=2):
    d = synthetic.make_frames(4, H, W, synthetic.CONFIG_8_IDS, variant="easy", with_logits=True)
    rep = B // 4
    seg = torch.from_numpy(np.tile(d["seg_logits"], (rep, 1, 1, 1))).cuda()
    direct = torch.from_numpy(np.tile(d["vertex"].reshape(4, H, W, 2 * VN), (rep, 1, 1, 1))).cuda()
    conf = torch.from_numpy(np.tile(d["conf_logits"], (rep, 1, 1, 1))).cuda()
    layer = CoordLSVotingWeighted("ls", OC + 1, num_points=VN)
    n = B * OC
    p3 = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(d["keypoints_3d"][None], (B, OC, VN, 3)).reshape(n, VN, 3))).cuda()
    cam = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(d["camera"], (n, 3, 3)))).cuda()
    rng = np.random.default_rng(0)
    g_pts = torch.from_numpy(rng.normal(size=(B, OC, VN, 2)).astype(np.float32)).cuda()
    g_pose = torch.from_numpy(rng.normal(size=(n, 3, 4)).astype(np.float32)).cuda()
    inp = [seg, direct, conf]

    def ls_only():
        out = layer._forward(seg, direct, conf, False, False)
        layer.backward(inp, g_pts)
        return out

    def chain():
        out = layer._forward(seg, direct, conf, False, False)
        poses = pnp_cuda(out.reshape(n, VN, 2).flip(-1), p3, cam)  # (y,x) -> (x,y)
        g = pnp_backward_cuda(p3, cam, poses, g_pose, 12)
        layer.backward(inp, g.flip(-1).reshape(B, OC, VN, 2))
        return poses

    res = {"ls_fwd_bwd_ms": [], "ls_fwd_bwd_pnp_fwd_bwd_ms": []}
    for _ in range(rounds):
        res["ls_fwd_bwd_ms"].append(round(events_ms(ls_only, steps, warmup=5), 4))
        res["ls_fwd_bwd_pnp_fwd_bwd_ms"].append(round(events_ms(chain, steps, warmup=5), 4))
    poses = chain()
    torch.cuda.synchronize()
    assert torch.isfinite(poses).all() and (poses.reshape(n, 12).abs().sum(1) > 0).sum() > n // 2
    fixed = layer._forward(seg, direct, conf, False, False).reshape(n, VN, 2).flip(-1).contiguous()
    res["casa_pnp_ms"] = round(events_ms(lambda: pnp_cuda(fixed, p3, cam), steps, warmup=5), 4)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pnp_backward_time.py needs a CUDA device")
    name, limit = card()
    res = {"gpu": name, "power_limit_w": limit,
           "casa_pnp_backward": [time_backward(n, f, a.iters) for n in (128, 4096) for f in (12, 6)],
           "chain_16x480x640_oc8": time_chain(a.steps)}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
