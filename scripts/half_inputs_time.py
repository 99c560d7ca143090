"""16-bit network outputs read natively against the float32 path and against a .float() conversion in front of it.

Three variants of the same call, timed in one process and alternated round by round so that clock and neighbour
drift hit all three alike:
  (a) f32     float32 inputs (what a float32 network hands over);
  (b) bf16    bfloat16 inputs read natively by the kernels;
  (c) upcast  bfloat16 inputs converted with .float() in front of the float32 call (what a mixed-precision caller had
              to do before the kernels took 16-bit inputs: one more pass over the data and float32 temporaries).
Workloads: the LS layer on config-1-shaped outputs (16 x 480 x 640, seg 9 + direct 18 + conf 9 channels,
filter_estimates=True) with 4 calls in flight and one at a time, and the config-2 seg_scores vote (16 x 480 x 640,
8 objects x 9 keypoints, 512 hypotheses) with 4 calls in flight.  Prints the card, its power limit and SM clocks,
then one line per (workload, variant): mean / median / min over rounds of the ms per call, and a JSON summary.

    python scripts/half_inputs_time.py [--rounds 5 --steps 25]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

B, H, W = 16, 480, 640


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:  # the timing does not depend on it
        return "nvidia-smi unavailable: %s" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=25, help="calls per variant and round")
    args = ap.parse_args()

    import numpy as np
    import torch

    from casapose_b200 import _lib, synthetic
    from casapose_b200.pose_estimation import CoordLSVotingWeighted, ransac_voting_layer_all_masks

    if not torch.cuda.is_available():
        raise SystemExit("half_inputs_time.py needs a CUDA device")
    if _lib._sources_newer_than_lib():
        _lib.build()
    print("card:", torch.cuda.get_device_name(0), "| nvidia-smi name, power limit, SM clock, max SM clock:", smi())
    d = synthetic.make_frames(B, H, W, synthetic.CONFIG_8_IDS, with_logits=True)
    seg = torch.from_numpy(d["seg_logits"]).cuda()
    direct = torch.from_numpy(d["vertex"].reshape(B, H, W, 18)).cuda()
    conf = torch.from_numpy(d["conf_logits"]).cuda()
    vertex = torch.from_numpy(d["vertex"]).cuda()
    ls_in = {"f32": [seg, direct, conf], "bf16": [t.bfloat16() for t in (seg, direct, conf)]}
    vote_in = {"f32": (seg, vertex), "bf16": (seg.bfloat16(), vertex.bfloat16())}
    layer = CoordLSVotingWeighted("ls", 9, num_points=9, filter_estimates=True)

    def ls_call(variant, keep):
        x = ls_in["bf16" if variant == "upcast" else variant]
        if variant == "upcast":
            x = [t.float() for t in x]
            keep.append(x)  # calls in flight read them after the call has returned
        return layer(x, check_finite=False)

    def vote_call(variant, keep):
        m, v = vote_in["bf16" if variant == "upcast" else variant]
        if variant == "upcast":
            m, v = m.float(), v.float()
            keep.append((m, v))
        return ransac_voting_layer_all_masks(m, v, 512, seed=1, seg_scores=True)

    # (b) and (c) compute the same bits; (a) is the float32 network's own input
    for call in (ls_call, vote_call):
        o_b, o_c = call("bf16", []).clone(), call("upcast", []).clone()
        torch.cuda.synchronize()
        assert torch.equal(o_b.view(torch.int32), o_c.view(torch.int32)), call.__name__

    def timed(call, variant, lanes):
        _lib.set_async(0, lanes)
        keep = []
        for _ in range(2 * max(lanes, 2)):  # every lane's workspace and graph
            call(variant, keep)
        _lib.join(0)
        torch.cuda.synchronize()
        keep.clear()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            call(variant, keep)
        _lib.join(0)
        e1.record()
        torch.cuda.synchronize()
        _lib.sync(0)
        _lib.set_async(0, 0)
        return e0.elapsed_time(e1) / args.steps

    workloads = [("ls, 4 in flight", ls_call, 4), ("ls, one at a time", ls_call, 1), ("vote seg_scores, 4 in flight", vote_call, 4)]
    variants = ["f32", "bf16", "upcast"]
    res = {w[0]: {v: [] for v in variants} for w in workloads}
    for r in range(args.rounds):
        for name, call, lanes in workloads:
            order = variants if r % 2 == 0 else variants[::-1]
            for v in order:
                res[name][v].append(timed(call, v, lanes))
    print("after the runs:", smi())
    summary = {}
    for name in res:
        for v in variants:
            t = np.array(res[name][v])
            summary.setdefault(name, {})[v] = {"mean_ms": float(t.mean()), "median_ms": float(np.median(t)), "min_ms": float(t.min()),
                                               "max_ms": float(t.max())}
            print("%-30s %-7s ms per call: mean %.4f  median %.4f  min %.4f  max %.4f  (%d rounds x %d calls)"
                  % (name, v, t.mean(), np.median(t), t.min(), t.max(), args.rounds, args.steps))
        s = summary[name]
        print("%-30s bf16 / f32 = %.3f   bf16 / upcast = %.3f" % (name, s["bf16"]["median_ms"] / s["f32"]["median_ms"],
                                                                 s["bf16"]["median_ms"] / s["upcast"]["median_ms"]))
    print(json.dumps({"card": torch.cuda.get_device_name(0), "smi": smi(), "rounds": args.rounds, "steps": args.steps,
                      "ms_per_call": summary}))


if __name__ == "__main__":
    main()
