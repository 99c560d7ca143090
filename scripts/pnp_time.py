"""Times the batched forward PnP (casa_pnp, DESIGN.md K7) with CUDA events at 128 and 4096 objects, 9 keypoints, on
noisy inputs (0.3 px noise, one object in four with a 40 px outlier) and on noise-free ones, and prints one JSON object
with the card name and its power limit.
With --other LIB it also loads a second build of the library and alternates the two in the same process (A/B).

usage: python scripts/pnp_time.py [--iters N] [--rounds R] [--other path/to/libcasapose_b200.so]"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from casapose_b200 import _lib, synthetic  # noqa: E402
from scripts.pnp_backward_time import card  # noqa: E402


def inputs(n, vn=9, seed=0, noisy=True):
    rng = np.random.default_rng(seed)
    K = synthetic.camera_matrix(480).astype(np.float32)
    p2, p3 = np.zeros((n, vn, 2), np.float32), np.zeros((n, vn, 3), np.float32)
    for i in range(n):
        X = (rng.uniform(-0.5, 0.5, size=(vn, 3)) * 120).astype(np.float32)
        R = synthetic._random_rotation(rng)
        t = np.array([rng.uniform(-150, 150), rng.uniform(-100, 100), rng.uniform(600, 1200)])
        c = X.astype(np.float64) @ R.T + t
        q = c @ K.T
        p2[i] = (q[:, :2] / q[:, 2:]).astype(np.float32) + noisy * rng.normal(scale=0.3, size=(vn, 2)).astype(np.float32)
        if noisy and i % 4 == 3:
            p2[i, rng.integers(vn)] += rng.normal(scale=40, size=2).astype(np.float32)
        p3[i] = X
    cam = np.broadcast_to(K, (n, 3, 3)).copy()
    return [torch.from_numpy(a).cuda() for a in (p2, p3, cam)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--other", default=None)
    a = ap.parse_args()
    libs = {"this": _lib.lib()}
    if a.other:
        o = C.CDLL(os.path.abspath(a.other))
        o.casa_create.argtypes, o.casa_create.restype = [C.c_int, C.POINTER(C.c_void_p)], C.c_int
        o.casa_pnp.argtypes = [C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 6
        o.casa_pnp.restype = C.c_int
        o.casa_destroy.argtypes, o.casa_destroy.restype = [C.c_void_p], C.c_int
        libs["other"] = o
    stream = torch.cuda.current_stream().cuda_stream
    res = {"card": None, "power_limit_w": None, "ms": {}, "equal_outputs": {}}
    res["card"], res["power_limit_w"] = card()
    for n, noisy in ((128, True), (4096, True), (128, False), (4096, False)):
        tag = "n%d%s" % (n, "" if noisy else "_clean")
        p2, p3, cam = inputs(n, noisy=noisy)
        outs = {}
        fns = {}
        handles = []
        for name, lib in libs.items():
            h = C.c_void_p()
            assert lib.casa_create(torch.cuda.current_device(), C.byref(h)) == 0
            handles.append((lib, h))
            out = torch.empty((n, 3, 4), device="cuda")
            outs[name] = out

            def fn(lib=lib, h=h, out=out):
                rc = lib.casa_pnp(h, n, 9, p2.data_ptr(), p3.data_ptr(), cam.data_ptr(), None, out.data_ptr(), stream)
                assert rc == 0
            fns[name] = fn
        for r in range(a.rounds):
            for name, fn in fns.items():
                for _ in range(10):
                    fn()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.iters):
                    fn()
                e1.record()
                e1.synchronize()
                res["ms"].setdefault("%s_%s" % (name, tag), []).append(round(e0.elapsed_time(e1) / a.iters, 4))
        if "other" in outs:
            res["equal_outputs"][tag] = bool(torch.equal(outs["this"], outs["other"]))
        torch.cuda.synchronize()
        for lib, h in handles:
            assert lib.casa_destroy(h) == 0
    print(json.dumps(res))


if __name__ == "__main__":
    main()
