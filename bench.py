#!/usr/bin/env python
"""Benchmark of the keypoint-voting hot path (BASELINE.json metric: keypoint-voting frames/s).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (ransac_voting_layer_all_masks: mask compaction -> hypothesis
generation -> inlier scoring -> refinement) over one batch of synthetic LM-O-shaped frames.
Workload at every N: BASELINE config 2 per GPU — batch 16, 480x640, 8 objects x 9 keypoints, 512
hypotheses per round (weak scaling: every rank owns its own 16 frames; the [16,8,9,2] keypoints of all
ranks are all-gathered with NCCL inside the timed step).

  value    frames/s, inputs resident in HBM when the timed region starts (CUDA events, max over ranks)
  e2e      frames/s through the host-buffer C-ABI entry point (pinned host -> device copy of mask and
           vertex field, voting, device -> host copy of the keypoints, all inside the timed region), two calls in
           flight (casa_ransac_vote_host_async; every call's keypoints are waited for inside the timed region);
           e2e.one_call_at_a_time is the synchronous call, one behind the other
  roofline the scoring kernel k_score against the FP32 FMA issue rate measured in this same run
           (FFMA micro-kernel of the library); algorithmic work = 11 FLOP per (hypothesis, pixel,
           keypoint) test (SURVEY.md section 8d)
  cpu_baseline  the torch-CPU restatement of the reference (oracle/ransac_voting_torch.py) on a bounded
           sample; `--impl reference` times the same restatement as its own arm.  The reference itself
           (TensorFlow 2.9.1) cannot be installed in this image: every "reference" number here is the
           CPU restatement of the reference, never reference TF.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, OC, VN, HN, BATCH = 480, 640, 8, 9, 512, 16
FLOP_PER_UNIT = 11  # SURVEY.md 8(d)
METRIC = "keypoint-voting frames/s (480x640, 8 obj x 9 kp, 512 hyp)"
# dram__bytes_read.sum + dram__bytes_write.sum of one k_score launch on this workload,
# from profiles/r02_k_score_full.txt (ncu --set full: 53.44 MB read + 0.79 MB written)
K_SCORE_DRAM_BYTES = 54.2e6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="frames per GPU (config 4: global batch); default: the config's")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="BASELINE.json config: 2 (default, the headline), 3 (13 objects, batch 32), 4 (batch 256 sharded: strong scaling), 5 (1080x1920, --hn sweep)")
    ap.add_argument("--hn", type=int, default=None, help="hypotheses per round (config 5 sweep: 128 .. 2048)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--host-calls", type=int, default=2,
                    help="host-buffer calls in flight in the e2e pass (1: synchronous casa_ransac_vote_host; "
                         "2: casa_ransac_vote_host_async, the default)")
    ap.add_argument("--lanes", type=int, default=4, help="calls in flight in the timed region (casa_set_async); 1 = one lane")
    ap.add_argument("--variant", default="easy")
    ap.add_argument("--cpu-sample-frames", type=int, default=None,
                    help="frames of the batch the CPU restatement is timed on (default: 8 for the cpu_baseline leg = about 8 s, 1 per step for --impl reference)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="ransac", choices=["ransac", "ls", "pose"],
                    help="ransac: BASELINE config 2 (the headline); ls: CoordLSVotingWeighted on config-1-shaped tensors")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the keypoints of the last timed step as DIR/keypoints.npy (float32 [b,oc,9,2]; all ranks' "
                         "frames with --gpus > 1), so that two builds can be compared on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "ransac" or args.impl != "ours"):
        ap.error("--dump-outputs writes the keypoints of the voting workload (--workload ransac --impl ours)")
    return args


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
            }
            while not self._halt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.005)
        except Exception as e:  # NVML missing: report it, do not fake numbers
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def mark(self):
        """Start of the timed region: earlier samples (warm-up) are dropped."""
        self.samples = []
        self.reasons = set(r for r in self.reasons if r.startswith("nvml_unavailable"))

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def make_batch(batch, rank, variant):
    """Every rank holds the SAME seeded frames (so the per-GPU work of the weak-scaling run is identical and the
    max-over-ranks time measures the system, not data variance); their global image indices differ, and with
    them the Philox hypothesis streams."""
    from casapose_b200 import synthetic

    return synthetic.make_frames(batch, H, W, synthetic.CONFIG_8_IDS, seed=synthetic.SEED_BASE, variant=variant)


def cpu_restatement(d, frames, steps=1, warmup=0, hn=HN):
    """Times the torch-CPU restatement of the reference on the first `frames` frames; returns (frames/s, info).
    The rate is taken from the MEDIAN pass (BASELINE.md section 3: 2 warm-ups, median of 5)."""
    import torch

    from oracle import ransac_voting_torch as T

    torch.set_num_threads(os.cpu_count() or 1)
    mask = torch.from_numpy(d["mask"][:frames])
    vertex = torch.from_numpy(d["vertex"][:frames])
    times, units = [], 0
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        _, infos = T.ransac_voting_layer_all_masks(mask, vertex, hn, seed=it, return_info=True)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
            units = sum(i["units"] for i in infos)
    med = sorted(times)[len(times) // 2]
    return frames / med, {"seconds_per_step": med, "units_per_step": units, "cores": torch.get_num_threads()}


def run_reference(args):
    """`--impl reference`: the CPU restatement of the reference on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    frames = args.cpu_sample_frames or 1
    d = make_batch(frames, 0, args.variant)
    fps, info = cpu_restatement(d, frames, steps=max(args.steps, 1), warmup=max(args.warmup, 0))
    sample = "%d of the %d frames of one batch per step (all 8 classes, hn=512, same Philox hypothesis indices)" % (frames, args.batch or BATCH)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": info["seconds_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "config 2: keypoint voting only, 480x640, 8 objects x 9 keypoints, 512 hypotheses",
                   "frames_per_step": frames, "note": "CPU restatement of the reference (torch-CPU, materialised [hn,tn,vn] temporaries); TensorFlow 2.9.1 is not installable in this image"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": info["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def run_ls(args):
    """Secondary line: the weighted-LS keypoint layer (SURVEY.md 8a rows B1/B2, HBM-bound) on config-1-shaped
    network outputs [b,480,640,9+18+9], filter_estimates=True, against the measured HBM copy bandwidth."""
    import numpy as np
    import torch

    from casapose_b200 import _lib, synthetic
    from casapose_b200.pose_estimation import CoordLSVotingWeighted
    from oracle import ls_voting_np as OL

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device")
    if _lib._sources_newer_than_lib():
        _lib.build()
    B = args.batch or BATCH
    d = synthetic.make_frames(B, H, W, synthetic.CONFIG_8_IDS, variant=args.variant, with_logits=True)
    seg = torch.from_numpy(d["seg_logits"]).cuda()
    direct = torch.from_numpy(d["vertex"].reshape(B, H, W, 18)).cuda()
    conf = torch.from_numpy(d["conf_logits"]).cuda()
    layer = CoordLSVotingWeighted("ls", OC + 1, num_points=VN, filter_estimates=True)
    lanes = max(1, min(4, args.lanes))
    sampler = ClockSampler(0)
    sampler.start()

    def timed(mode):
        # mode >= 2: that many calls in flight (casa_set_async: consecutive calls rotate over workspaces / streams, so the
        # latency-bound classify / place / component kernels of neighbouring calls overlap); 1: one call at a time
        _lib.set_async(0, mode)
        for _ in range(max(args.warmup, 3, 2 * mode)):  # at least two untimed steps per lane (workspace, graph)
            layer([seg, direct, conf], check_finite=False)
        _lib.join(0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if mode == (lanes if lanes >= 2 else 1):
            sampler.mark()
        e0.record()
        for _ in range(args.steps):
            layer([seg, direct, conf], check_finite=False)
        _lib.join(0)
        e1.record()
        torch.cuda.synchronize()
        _lib.sync(0)
        return e0.elapsed_time(e1) / args.steps

    ms = timed(lanes if lanes >= 2 else 1)
    clocks = sampler.stop()
    ms_one = timed(1) if lanes >= 2 else ms
    _lib.set_async(0, 0)
    layer([seg, direct, conf], check_finite=False)
    torch.cuda.synchronize()
    nl = C.c_int64()
    _lib.check(_lib.lib().casa_last_launches(_lib.handle(0), C.byref(nl)))
    fwd_launches = int(nl.value)
    # backward (casa_ls_vote_backward: forward recomputation + adjoint + one pass over the listed pixels + zero fill)
    gout = torch.randn((B, OC, VN, 2), device="cuda")
    for _ in range(3):
        layer.backward([seg, direct, conf], gout)
    torch.cuda.synchronize()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record()
    for _ in range(args.steps):
        layer.backward([seg, direct, conf], gout)
    b1.record()
    torch.cuda.synchronize()
    bwd_ms = b0.elapsed_time(b1) / args.steps
    alg_bytes = B * H * W * 4 * ((1 + OC) + 2 * VN + VN)  # SURVEY.md 8(d): 44.2 MB per frame at oc = 8
    peak = None
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        src = "MEASURED_PEAKS.json hbm_gbs (copy bandwidth, measured)"
    except Exception:
        peak, src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    achieved = alg_bytes / (ms * 1e-3) / 1e9
    t0 = time.perf_counter()
    OL.coord_ls_voting_weighted(d["seg_logits"][:1], d["vertex"][:1].reshape(1, H, W, 18), d["conf_logits"][:1], filter_estimates=True)
    cpu_s = time.perf_counter() - t0
    print(json.dumps({
        "metric": "weighted-LS keypoint layer frames/s (480x640, 8 obj x 9 kp, filter_estimates)", "value": B / (ms * 1e-3),
        "unit": "frames/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 elementwise, f64 accumulation",
        "data": "synthetic", "config": {"workload": "config 1 shape: [b,480,640,9+18+9] network-output split -> CoordLSVotingWeighted(filter_estimates=True), batch %d" % B,
                                        "l2": "inputs (%.0f MB per step) larger than the 126 MB L2" % (alg_bytes / 1e6),
                                        "calls_in_flight": lanes, "ms_per_step_one_lane": ms_one},
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "CoordLSVotingWeighted (k_ls_classify .. k_ls_solve, %d launches replayed as one CUDA graph)" % fwd_launches, "achieved": achieved,
                     "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": src},
        "cpu_baseline": {"value": 1.0 / cpu_s, "unit": "frames/s", "cores": 1, "kind": "port",
                         "sample": "numpy oracle, 1 frame, %.2f s" % cpu_s},
        "gpu_launches": fwd_launches * args.steps,
        "backward": {"ms_per_step": bwd_ms, "frames_per_s": B / (bwd_ms * 1e-3),
                     "note": "forward recomputation + gradients w.r.t. direct and confidence logits (dense, zero-filled)",
                     "bytes_written": B * H * W * 4 * 3 * VN},
    }))


def run_pose(args):
    """Secondary line: the whole post-network evaluation of a batch (SURVEY.md 8a rows A1-C3 with the 8f rows on the
    GPU): seg arg-max -> voting -> batched PnP -> ADD, device-resident (DeviceEvaluator), one [oc,8] read-back per
    batch inside the timed region; beside it the drop-in with the reference's own host stages (OpenCV PnP, numpy
    metrics) on the same inputs."""
    import numpy as np
    import torch

    from casapose_b200 import _lib, synthetic
    from casapose_b200.pose_estimation import DeviceEvaluator, estimate_and_evaluate_poses

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device")
    if _lib._sources_newer_than_lib():
        _lib.build()
    B = args.batch or BATCH
    d = synthetic.make_frames(B, H, W, synthetic.CONFIG_8_IDS, variant=args.variant, with_logits=True)
    seg = torch.from_numpy(d["seg_logits"]).cuda()
    tgt = torch.from_numpy(np.concatenate([(d["labels"] == 0)[..., None].astype(np.float32), d["mask"]], axis=-1)).cuda()
    vert = torch.from_numpy(d["vertex"].reshape(B, H, W, 2 * VN)).cuda()
    K = synthetic.camera_matrix(H).astype(np.float32)
    offsets = np.zeros((B, 10), np.float32)
    offsets[:, 7], offsets[:, 8], offsets[:, 9] = 1.0, W, H
    gt = d["poses_gt"].astype(np.float32)
    ev = DeviceEvaluator(d["keypoints_3d"], K, d["diameters"])
    for it in range(max(args.warmup, 3)):
        ev(seg, tgt, vert, gt, offsets, seed=it)
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    t0 = time.perf_counter()
    for it in range(args.steps):
        stats, _, _ = ev(seg, tgt, vert, gt, offsets, seed=100 + it)  # ends with the [oc,8] read-back: host-visible result
    dt = (time.perf_counter() - t0) / args.steps
    clocks = sampler.stop()
    kp3 = np.broadcast_to(d["keypoints_3d"][None, :, None], (B, OC, 1, VN, 3)).copy()
    cams = np.broadcast_to(K, (B, 3, 3)).copy()
    diam = np.broadcast_to(d["diameters"][None], (B, OC)).copy()
    n_host = 3
    t0 = time.perf_counter()
    for it in range(n_host):
        s_host, _, _ = estimate_and_evaluate_poses(seg, tgt, vert, gt[:, :, None], kp3, cams, diam, offsets, seed=100 + it)
    dt_host = (time.perf_counter() - t0) / n_host
    print(json.dumps({
        "metric": "post-network pose evaluation frames/s (480x640, 8 obj x 9 kp: voting + PnP + ADD)", "value": B / dt,
        "unit": "frames/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 voting, f64 PnP", "data": "synthetic",
        "config": {"workload": "batch %d: seg logits [b,480,640,9] + vector field -> casa_ransac_vote_seg -> casa_pnp -> casa_pose_errors, wall clock incl. the per-batch read-back" % B},
        "clocks": clocks,
        "host_stages": {"value": B / dt_host, "unit": "frames/s", "ms_per_step": dt_host * 1e3,
                        "note": "same voting kernels, then OpenCV solvePnPRansac + solvePnP and numpy metrics on the host like the reference (drop-in defaults), %d batches" % n_host},
        "valid_3d": [float(x) for x in stats["valid_3d"]], "valid_3d_host_stages": [float(x) for x in np.atleast_1d(s_host[1])],
    }))


CONFIGS = {
    # BASELINE.json configs[1..4] (configs[0] is the reference's CPU case: --impl reference / cpu_baseline)
    2: dict(h=480, w=640, ids="CONFIG_8_IDS", hn=512, batch=16, scaling="weak", gen=16,
            name="config 2: keypoint voting only, batch %(b)d synthetic 480x640 mask + 18-ch vector field, 8 objects x 9 keypoints, %(hn)d hypotheses, per GPU"),
    3: dict(h=480, w=640, ids="CONFIG_13_IDS", hn=512, batch=32, scaling="weak", gen=4,
            name="config 3: config_13 (13 LM-shaped objects) voting, batch %(b)d per GPU, 480x640, %(hn)d hypotheses"),
    4: dict(h=480, w=640, ids="CONFIG_8_IDS", hn=512, batch=256, scaling="strong", gen=8,
            name="config 4: batch 256 synthetic LM-O-shaped frames sharded across the GPUs (%(b)d frames on this rank), NCCL gather of the keypoints, %(hn)d hypotheses"),
    5: dict(h=1080, w=1920, ids="CONFIG_8_IDS", hn=512, batch=4, scaling="weak", gen=1,
            name="config 5: 1080x1920 synthetic fields, 8 objects, %(hn)d hypotheses per round (sweep 128-2048 with --hn), batch %(b)d per GPU, 30000-pixel cap active"),
}


def main():
    args = parse()
    if args.workload == "ls":
        return run_ls(args)
    if args.workload == "pose":
        return run_pose(args)
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from casapose_b200 import _lib, sharding, synthetic
    from casapose_b200.pose_estimation.ransac_voting import (ransac_voting_layer_all_masks,
                                                               ransac_voting_layer_all_masks_host)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the voting path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    distributed = world > 1
    if distributed:
        dist.init_process_group("nccl", device_id=dev)
    if _lib._sources_newer_than_lib():
        if rank == 0:
            _lib.build()
        if distributed:
            dist.barrier()

    cfg = dict(CONFIGS[args.config])
    hn = args.hn or cfg["hn"]
    ids = getattr(synthetic, cfg["ids"])
    h_, w_, oc, vn = cfg["h"], cfg["w"], len(ids), VN
    total_batch = args.batch or cfg["batch"]
    if cfg["scaling"] == "strong":  # a fixed global batch, contiguous image ranges per rank
        start_img, stop_img = sharding.shard_bounds(total_batch, rank, world)
        B = stop_img - start_img
        n_images = total_batch
    else:  # weak: every rank owns its own `batch` frames of a world * batch global batch
        B = total_batch
        n_images = world * B
        start_img = rank * B
    # every rank holds the SAME seeded frames (tiled to its batch) under distinct global image indices, and with them
    # distinct Philox hypothesis streams: the per-GPU work is identical and the max-over-ranks time measures the system
    gen = min(cfg["gen"], B)
    d = synthetic.make_frames(gen, h_, w_, ids, seed=synthetic.SEED_BASE, variant=args.variant)
    reps = (B + gen - 1) // gen
    mask_np = np.tile(d["mask"], (reps, 1, 1, 1))[:B]
    vertex_np = np.tile(d["vertex"], (reps, 1, 1, 1, 1))[:B]
    mask_h = torch.from_numpy(mask_np).pin_memory()
    vertex_h = torch.from_numpy(vertex_np).pin_memory()
    del mask_np, vertex_np
    mask = mask_h.to(dev, non_blocking=True)
    vertex = vertex_h.to(dev, non_blocking=True)
    lib = _lib.lib()
    hdl = _lib.handle(local, torch.cuda.current_stream(dev).cuda_stream)
    in_bytes = mask.numel() * 4 + vertex.numel() * 4

    # The keypoints of a step ([B,oc,9,2], 576 B per frame at oc = 8) are all-gathered with NCCL through the library's
    # own C-ABI gather (casa_allgather_points_overlapped) on a gather stream that waits only for that step's vote,
    # so the exchange overlaps the next step's voting; every gather completes inside the timed region.
    if distributed and cfg["scaling"] == "strong" and total_batch % world:
        raise SystemExit("config 4 needs a batch divisible by the number of GPUs")
    lanes = max(1, min(4, args.lanes))
    gather = sharding.AbiGather((B, oc, vn, 2), dev, world, rank, slots=max(2, 2 * lanes)) if distributed else None
    counter = [0]
    outs = [torch.empty((B, oc, vn, 2), dtype=torch.float32, device=dev) for _ in range(8)]  # results of the calls in flight

    class _Done:
        def __init__(self, v):
            self.v = v

        def wait(self):
            return self.v

    def step(seed):
        i = counter[0]
        counter[0] += 1
        if not distributed:
            return _Done(ransac_voting_layer_all_masks(mask, vertex, hn, seed=seed, image_offset=start_img, out=outs[i % 8]))
        ransac_voting_layer_all_masks(mask, vertex, hn, seed=seed, image_offset=start_img, out=gather.buffer(i))
        return gather.launch(i)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    # --- FP32 peak of this GPU, measured in this run (roofline denominator)
    tf, ms = C.c_double(), C.c_double()
    _lib.check(lib.casa_measure_fp32_peak(hdl, 0, C.byref(tf), C.byref(ms)))
    fp32_peak = tf.value
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        hbm_src = "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"

    # Asynchronous calls: the library enqueues ONE CUDA graph per step (device-driven RANSAC loop) and returns; loop
    # states / statistics / k_score events are collected at the end.  The timed region that gives `value` runs with
    # `lanes` calls in flight (casa_set_async(h, lanes): consecutive votes rotate over that many workspaces / streams, so
    # the latency-bound compaction and refinement kernels of neighbouring steps overlap and the k_score launches run back
    # to back).  k_score's own duration is timed in a second pass of the same K steps on ONE lane, where an event pair
    # around the kernel measures the kernel: with several lanes a launch queues behind the previous lane's k_score and
    # the pair would include that wait.
    stream_ptr = torch.cuda.current_stream(dev).cuda_stream
    sampler = ClockSampler(local)
    sampler.start()  # started before the warm-up so that NVML is initialised when the timed region begins

    def timed_pass(mode, timing, sample, own_sampler=None):
        _lib.check(lib.casa_set_async(hdl, mode))
        _lib.check(lib.casa_set_timing(hdl, 0))
        # at least two untimed steps per lane: a lane builds its workspace and its graph on its first call
        for it in range(max(args.warmup, 3, 2 * mode)):
            step(it).wait()
        if mode >= 2:
            _lib.check(lib.casa_join(hdl, stream_ptr))
        _lib.check(lib.casa_sync(hdl))
        barrier()
        _lib.check(lib.casa_set_timing(hdl, timing))
        sm, sl, st = C.c_double(), C.c_int64(), (C.c_uint64 * 4)()
        nl = C.c_int64()
        lib.casa_last_launches(hdl, C.byref(nl))
        lib.casa_get_timing(hdl, C.byref(sm), C.byref(sl), st)  # drop the warm-up totals
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        if distributed:
            gather.barrier()  # device-side barrier on the compute stream: the ranks enter the timed region together
        if sample:
            sampler.mark()
        if own_sampler is not None:
            own_sampler.mark()
        e0.record()
        pending = None
        for it in range(args.steps):
            nxt = step(1000 + it)
            if pending is not None and it % 16 == 0:
                pending.wait()  # host-side check-point: the gathered keypoints of an earlier step are complete
            pending = nxt
        last = pending.wait()
        if distributed:
            last = last.clone()  # the gather buffers are reused by the next pass
        if mode >= 2:
            _lib.check(lib.casa_join(hdl, stream_ptr))  # the caller's stream waits for every lane
        e1.record()
        barrier()
        clk = sampler.stop() if sample else (own_sampler.stop() if own_sampler is not None else None)
        _lib.check(lib.casa_sync(hdl))
        lib.casa_last_launches(hdl, C.byref(nl))  # asynchronous handle: total over the calls since the last query
        lib.casa_get_timing(hdl, C.byref(sm), C.byref(sl), st)
        _lib.check(lib.casa_set_timing(hdl, 0))
        return dict(ms=e0.elapsed_time(e1), score_ms=sm.value, score_launches=sl.value, launches=nl.value,
                    units=st[0], exact_units=st[1], last=last, clocks=clk)

    main_pass = timed_pass(lanes if lanes >= 2 else 1, 0 if lanes >= 2 else 1, True)
    if args.dump_outputs and rank == 0:
        # written now: the k_score pass below reuses the result buffers
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "keypoints.npy"), main_pass["last"].cpu().numpy())

    def kernel_pass():
        smp = ClockSampler(local)
        smp.start()
        time.sleep(0.05)
        return timed_pass(1, 1, False, own_sampler=smp)

    def throttled(c):
        return bool(c) and (any(r in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap") for r in c["reasons"])
                            or (c["sm_mhz"] and c["sm_max_mhz"] and c["sm_mhz"] < 0.97 * c["sm_max_mhz"]))

    kern_pass = kernel_pass() if lanes >= 2 else main_pass
    kern_repeated = False
    if lanes >= 2 and throttled(kern_pass["clocks"]):  # a clock dip during the kernel pass: measured again, once
        kern_pass = kernel_pass()
        kern_repeated = True
    _lib.check(lib.casa_set_async(hdl, 0))
    clocks = main_pass["clocks"]
    gathered = main_pass["last"]
    score_ms, score_launches = kern_pass["score_ms"], kern_pass["score_launches"]
    launches, units, exact_units = main_pass["launches"], main_pass["units"], main_pass["exact_units"]
    one_lane_ms = kern_pass["ms"] / args.steps
    kern_elapsed_ms = kern_pass["ms"]
    elapsed_ms = main_pass["ms"]
    gather_ok = None
    if distributed:
        # EVERY row of the last step's gathered tensor is checked: each rank recomputes the other ranks' keypoints
        # (same frames, their image offsets, same seed) and compares bit for bit
        last_seed = 1000 + args.steps - 1
        ok = tuple(gathered.shape) == (world * B, oc, vn, 2) and bool(torch.isfinite(gathered).all())
        for r in range(world):
            off_r = (sharding.shard_bounds(total_batch, r, world)[0] if cfg["scaling"] == "strong" else r * B)
            expect = ransac_voting_layer_all_masks(mask, vertex, hn, seed=last_seed, image_offset=off_r)
            ok = ok and bool(torch.equal(gathered[r * B:(r + 1) * B], expect))
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        gather_ok = bool(flag.item())
        t = torch.tensor([elapsed_ms, score_ms, float(units), float(launches), float(exact_units)], device=dev, dtype=torch.float64)
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        elapsed_ms = float(tmax[0].item())
        units_all, launches_all = float(t[2].item()), int(t[3].item())
    else:
        units_all, launches_all = float(units), int(launches)
    value = n_images * args.steps / (elapsed_ms * 1e-3)

    # --- end to end through the host-buffer C-ABI entry point (pinned host buffers)
    e2e = None
    if not args.no_e2e:
        e2e_steps = max(1, min(args.steps, int(2.0e10 / max(in_bytes, 1))))  # about 20 GB over PCIe at most
        outs_h = [torch.empty((B, oc, vn, 2), dtype=torch.float32).pin_memory() for _ in range(args.host_calls + 1)]

        def e2e_pass(in_flight):
            """e2e_steps host-buffer calls, `in_flight` of them at a time (1: the synchronous call; 2: the pipelined
            entry, casa_ransac_vote_host_async — the host packs call i+1 while the GPU finishes call i).  Every call's
            keypoints are waited for inside the timed region; they land in pinned host memory."""
            from collections import deque

            for it in range(2 * in_flight):
                ransac_voting_layer_all_masks_host(mask_h, vertex_h, hn, seed=it, image_offset=start_img, device=local,
                                                   out=outs_h[0], wait=in_flight == 1)
            _lib.sync(local)
            barrier()
            pend = deque()
            t0 = time.perf_counter()
            for it in range(e2e_steps):
                if in_flight == 1:
                    ransac_voting_layer_all_masks_host(mask_h, vertex_h, hn, seed=2000 + it, image_offset=start_img, device=local,
                                                       out=outs_h[0])
                    continue
                if len(pend) == in_flight:
                    pend.popleft().result()
                pend.append(ransac_voting_layer_all_masks_host(mask_h, vertex_h, hn, seed=2000 + it, image_offset=start_img,
                                                               device=local, out=outs_h[it % len(outs_h)], wait=False))
            while pend:
                pend.popleft().result()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if distributed:
                t = torch.tensor([dt], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            return dt

        e2e_one_s = e2e_pass(1)
        e2e_s = e2e_pass(args.host_calls) if args.host_calls > 1 else e2e_one_s
        # context for e2e: pinned host -> device copy bandwidth of this box, and the bytes the host entry point really
        # moves (the whole mask by DMA, the vector field only at masked pixels through mapped reads)
        scratch = torch.empty_like(mask)
        h2d_gbs = 0.0
        for _ in range(3):
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            scratch.copy_(mask_h, non_blocking=True)
            c1.record()
            torch.cuda.synchronize()
            h2d_gbs = max(h2d_gbs, mask_h.numel() * 4 / (c0.elapsed_time(c1) * 1e-3) / 1e9)
        del scratch
        # the host entry splits the batch into image ranges (4 for b >= 8, 2 for b >= 2) whose masks cross PCIe as one
        # host-packed u32 per pixel (6 or more host threads: every range; 4-5 threads: the odd ranges, the even ones as raw
        # floats; fewer: raw floats only — casa_ransac_vote_host); CASA_NO_HOST_PACK=1 moves all raw
        parts = 4 if B >= 8 else (2 if B >= 2 else 1)
        lws = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
        pack_threads = min(12, ((os.cpu_count() or 1) - lws) // lws if lws > 1 else (os.cpu_count() or 1) - 1)  # the library's rule
        packed_imgs = 0 if (os.environ.get("CASA_NO_HOST_PACK") or pack_threads < 4) else (B if pack_threads >= 6 else sum(
            B * (k + 1) // parts - B * k // parts for k in range(parts) if k & 1))
        px = h_ * w_
        moved_bytes = (B - packed_imgs) * px * oc * 4 + packed_imgs * px * 4 + float(mask_h.sum()) * 2 * vn * 4
        e2e = {"value": n_images * e2e_steps / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": in_bytes,
               "d2h_bytes_per_step": B * oc * vn * 2 * 4, "ms_per_step": e2e_s / e2e_steps * 1e3, "steps": e2e_steps,
               "h2d_gbs_measured": h2d_gbs, "bytes_moved_per_step": moved_bytes, "host_packed_images": packed_imgs,
               "pcie_floor_ms": moved_bytes / (h2d_gbs * 1e9) * 1e3 if h2d_gbs else None,
               "host_calls_in_flight": args.host_calls,
               "one_call_at_a_time": {"value": n_images * e2e_steps / e2e_one_s, "ms_per_step": e2e_one_s / e2e_steps * 1e3}}

    if rank == 0:
        sum_tn = float(mask_h.sum())
        # k_score of ROUND 0 of every step is event-timed (a WHILE body cannot hold event nodes).  For single-round frames
        # the statistics' unit count is that launch's; for multi-round frames the units of round 0 are counted from the
        # mask: every job with at least min_num pixels scores tn * vn * hn units (a job above max_num: its expected
        # max_num pixels after the random down-sampling).
        tn_jobs = mask_h.sum(dim=(1, 2)).double()
        tn_round0 = torch.clamp(tn_jobs, max=30000.0) * (tn_jobs >= 5)  # a job above max_num keeps max_num pixels on average (:298)
        units_round0 = float(tn_round0.sum()) * vn * hn * args.steps
        multi_round = units > 1.001 * units_round0
        timed_units = units_round0 if multi_round else units
        achieved = FLOP_PER_UNIT * timed_units / (score_ms * 1e-3) / 1e12 if (score_ms > 0 and timed_units) else None
        # frame-level roofline (SURVEY.md 8d: frame-rate bound = 1 / (t_FP32 + t_HBM), no overlap assumed): algorithmic
        # FLOPs of all rounds at the measured FP32 peak + algorithmic bytes (read-once inputs, keypoints out) at the
        # measured HBM copy bandwidth, against the measured step
        alg_bytes = B * (h_ * w_ * 4 * (oc + 2 * vn) + oc * vn * 8)
        t_fp32_ms = FLOP_PER_UNIT * (units / max(args.steps, 1)) / (fp32_peak * 1e12) * 1e3
        t_hbm_ms = alg_bytes / (hbm_peak * 1e9) * 1e3
        step_ms = elapsed_ms / args.steps
        names = dict(b=B, hn=hn)
        metric = METRIC if args.config == 2 and hn == 512 else \
            "keypoint-voting frames/s (%dx%d, %d obj x %d kp, %d hyp)" % (h_, w_, oc, vn, hn)
        line = {
            "metric": metric, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": cfg["name"] % names,
                "variant": args.variant, "masked_pixels_per_frame": sum_tn / B,
                "units_per_step": units / max(args.steps, 1), "rounds_per_step": score_launches and units and None,
                "units_round0_per_step": units_round0 / max(args.steps, 1),
                "flop_per_unit": FLOP_PER_UNIT,
                "l2": ("inputs (%.0f MB per step) larger than the 126 MB L2, no flush needed" % (in_bytes / 1e6)) if in_bytes > 126e6
                      else "inputs (%.0f MB per step) fit the 126 MB L2: k_score's operands are the compacted lists either way" % (in_bytes / 1e6),
                "parallelism": "images sharded across ranks (same seeded frames on every rank, distinct global image indices), NCCL all-gather of the [b,%d,9,2] keypoints through the C-ABI gather on the library's gather stream, every gathered row verified: %s" % (
                    oc, gather_ok) if distributed else "single GPU",
                "exact_fallback_fraction": exact_units / units if units else None,
                "calls_in_flight": lanes,
                "ms_per_step_one_lane": one_lane_ms,
            },
            "clocks": clocks,
            "gpu_launches": launches_all,
            "roofline": {
                "bound": "fp32", "kernel": "k_score", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                "frac": achieved / fp32_peak if achieved else None,
                "traffic": K_SCORE_DRAM_BYTES if args.config == 2 and B == 16 else None,
                "peak_source": "FFMA micro-kernel of this library measured in this run (MEASURED_PEAKS.json has no FP32 figure); nominal 74.5 TFLOP/s at 1965 MHz",
                "launch_ms": score_ms / score_launches if score_launches else None,
                "launches_timed": score_launches,
                "clocks": kern_pass["clocks"], "repeated_after_clock_dip": kern_repeated,
                "timed_in": ("a second pass of the same %d steps with one call in flight (event pair around the kernel; with %d lanes a "
                             "launch queues behind the previous lane's k_score and the pair would include the wait)" % (args.steps, lanes))
                            if lanes >= 2 else "the timed region itself",
                "share_of_step": score_ms / elapsed_ms if elapsed_ms else None,
                "frame_frac": (t_fp32_ms + t_hbm_ms) / step_ms if step_ms else None,
                "frame_model": {"t_fp32_ms": t_fp32_ms, "t_hbm_ms": t_hbm_ms, "alg_bytes_per_step": alg_bytes,
                                "hbm_peak_gbs": hbm_peak, "hbm_peak_source": hbm_src,
                                "note": "k_score of the first round of every step is event-timed; units and the frame model count all rounds"},
            },
        }
        del line["config"]["rounds_per_step"]
        if e2e is not None:
            line["e2e"] = e2e
        if not args.no_cpu_baseline and args.config == 2:
            cpu_frames = min(args.cpu_sample_frames or 2, B)
            fps, info = cpu_restatement(d, cpu_frames, steps=5, warmup=2, hn=hn)
            line["cpu_baseline"] = {
                "value": fps, "unit": "frames/s", "cores": info["cores"], "kind": "port",
                "sample": "%d of the %d frames of the batch, all %d classes, hn=%d, same Philox hypothesis indices; 2 warm-ups, median of 5 passes of %.1f s (BASELINE.md section 3); CPU restatement of the reference, not reference TF" % (
                    cpu_frames, B, oc, hn, info["seconds_per_step"]),
            }
        print(json.dumps(line))
    if distributed:
        sys.stdout.flush()
        sys.stderr.flush()
        torch.cuda.synchronize()
        gather.close()  # the library's communicator: destroyed before the process group
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
