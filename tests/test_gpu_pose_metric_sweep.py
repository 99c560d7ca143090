"""ADD / ADD-S / 2-D errors (casa_pose_errors, pose_metric.cuh K8) across the paths of its three kernels: point counts
at the 256-thread and 1024-point tile edges, ADD-S counts and padding, model tables, ADD-S minima, guards, batch sizes
past the 128-object block of k_pose_finalize and past 65535 objects, and a scratch buffer reused across calls.

Every row is compared with the reference's restatement (oracle/pose_np.evaluate_poses, one object at a time):
the verdict and missing / false-positive columns equal, err_2d and err_3d within rtol 1e-5 and atol 1e-4 (the bar of
tests/test_gpu_pose_metric.py), NaN and inf in the same places.  The verdicts must also follow from the kernel's own errors bit for bit: valid_3d == (err_3d < f32(d) * 0.1f),
valid_2d == (err_2d < allowed_error_2d).  Rows past a model's count are filled with NaN, so a read past it shows.

The pose-sum guards compare |sum of 12 entries| with 1e-4 in float32; the kernel adds sequentially, numpy pairwise, so
the guard poses are built from dyadic entries whose sum is exact in any order.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from casapose_b200 import synthetic  # noqa: E402
from oracle import pose_np as OP  # noqa: E402

pytestmark = pytest.mark.gpu
F = np.float32
SQRT_EPS = F(np.sqrt(1e-5))  # one ADD-S point at distance 0 (ransac_voting.py:609)


# ----------------------------------------------------------------------------------------------- builders
def _models(rng, counts, maxp, ext=(30, 120), centre=0.0):
    pts = np.full((len(counts), maxp, 3), np.nan, F)  # padding: never read
    diam = np.zeros(len(counts), F)
    for c, n in enumerate(counts):
        e = rng.uniform(*ext, size=3)
        pts[c, :n] = (rng.uniform(-0.5, 0.5, size=(n, 3)) * e + centre).astype(F)
        diam[c] = np.linalg.norm(e)
    return pts, np.array(counts, np.int32), diam


def _poses(rng, n, mags=(0.002, 0.02, 0.08), tz=(600, 1200)):
    """Ground truth and estimates perturbed well inside, near and beyond the 0.1 d threshold."""
    gt, est = np.zeros((n, 3, 4), F), np.zeros((n, 3, 4), F)
    for i in range(n):
        R = synthetic._random_rotation(rng)
        t = np.array([rng.uniform(-150, 150), rng.uniform(-100, 100), rng.uniform(*tz)])
        gt[i] = np.concatenate([R, t[:, None]], 1)
        mag = mags[i % len(mags)]
        w = rng.normal(size=3) * mag
        th = np.linalg.norm(w)
        k = w / th
        Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
        dR = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx
        est[i] = np.concatenate([dR @ R, (t + rng.normal(size=3) * mag * 100)[:, None]], 1)
    return gt, est


def _cams(rng, n, distinct=False):
    K = synthetic.camera_matrix(480).astype(F)
    cams = np.broadcast_to(K, (n, 3, 3)).copy()
    if distinct:
        for i in range(n):
            f = rng.uniform(400, 3000)
            cams[i] = [[f, 0, rng.uniform(300, 2000)], [0, f * rng.uniform(0.9, 1.1), rng.uniform(200, 1100)], [0, 0, 1]]
    return cams


# ----------------------------------------------------------------------------------------------- calls and checks
def _rows(est, gt, cams, pts, counts, diam, valid, allowed, obj_model=None):
    from casapose_b200.pose_estimation.ransac_voting import pose_errors_cuda

    return pose_errors_cuda(est, gt, cams, pts, counts, diam, valid, allowed, obj_model).cpu().numpy()


def _ref_row(est, gt, K, pts, cnt, d, valid, allowed):
    o = OP.evaluate_poses(est[None, None], gt[None, None, None], pts[None, None, None], np.array([[[cnt]]]), K[None],
                          np.array([[d]], F), np.array([[valid]]), allowed)
    return np.array([o["err_2d"][0], o["err_3d"][0], o["valid_3d"][0], o["valid_2d"][0], o["missing"][0],
                     o["false_positive"][0]], F)


def _check(rows, est, gt, cams, pts, counts, diam, valid, allowed, obj_model=None, idx=None):
    n, m = len(est), len(counts)
    idx = range(n) if idx is None else idx
    ref = np.zeros((len(idx), 6), F)
    for j, i in enumerate(idx):
        mod = obj_model[i] if obj_model is not None else i % m
        ref[j] = _ref_row(est[i], gt[i], cams[i], pts[mod], min(int(counts[mod]), pts.shape[1]), diam[i], valid[i], allowed)
    got = rows[list(idx)]
    assert np.array_equal(got[:, 2:], ref[:, 2:]), np.nonzero((got[:, 2:] != ref[:, 2:]).any(1))
    # atol: a few float32 ulps of the projected coordinates (~300 px, ~1000 mm), which the kernel (the reference's op
    # order) and numpy's matmul round differently; the small errors are differences of such coordinates
    np.testing.assert_allclose(got[:, :2], ref[:, :2], rtol=1e-5, atol=1e-4, equal_nan=True)
    live = (got[:, 4] == 0) & (np.asarray(valid)[list(idx)] != 0)
    d = np.asarray(diam, F)[list(idx)]
    with np.errstate(invalid="ignore"):
        assert np.array_equal(got[live, 2], (got[live, 1] < d[live] * F(0.1)).astype(F))
        assert np.array_equal(got[live, 3], (got[live, 0] < F(allowed)).astype(F))
    return ref


# ----------------------------------------------------------------------------------------------- cases
@pytest.mark.parametrize("count", [1, 2, 255, 256, 257, 1023, 1024, 1025, 7861, 7863])
def test_add_point_counts(cuda_lib, count):
    rng = np.random.default_rng(count)
    pts, counts, diam = _models(rng, [count], count + 7)
    n = 6
    gt, est = _poses(rng, n)
    allowed = [2.5, 5.0, 10.0][count % 3]
    rows = _rows(est, gt, _cams(rng, n), pts, counts, np.full(n, diam[0]), np.ones(n, np.int32), allowed)
    _check(rows, est, gt, _cams(rng, n), pts, counts, np.full(n, diam[0]), np.ones(n, np.int32), allowed)


@pytest.mark.parametrize("count,maxp", [(3417, 3417), (3417, 7862), (3417, 8192), (7862, 7862), (7862, 8192)])
def test_adds_point_counts_and_padding(cuda_lib, count, maxp):
    rng = np.random.default_rng(count + maxp)
    pts, counts, diam = _models(rng, [count, 700], maxp)
    n = 4
    gt, est = _poses(rng, n)
    cams, dia, val = _cams(rng, n), diam[np.arange(n) % 2], np.ones(n, np.int32)
    rows = _rows(est, gt, cams, pts, counts, dia, val, 5.0)
    _check(rows, est, gt, cams, pts, counts, dia, val, 5.0)


def test_model_tables(cuda_lib):
    rng = np.random.default_rng(1)
    pts, counts, diam = _models(rng, [500, 9, 3417, 1200, 33], 3417)
    n = 12
    gt, est = _poses(rng, n)
    cams, val = _cams(rng, n), np.ones(n, np.int32)
    # m = 1
    rows = _rows(est, gt, cams, pts[:1], counts[:1], np.full(n, diam[0]), val, 5.0)
    _check(rows, est, gt, cams, pts[:1], counts[:1], np.full(n, diam[0]), val, 5.0)
    # obj_model: a permutation with repeats, and m > n through the default obj % m
    om = np.array([4, 2, 2, 0, 3, 1, 4, 4, 2, 0, 1, 3], np.int32)
    rows = _rows(est, gt, cams, pts, counts, diam[om], val, 5.0, om)
    _check(rows, est, gt, cams, pts, counts, diam[om], val, 5.0, om)
    rows = _rows(est[:3], gt[:3], cams[:3], pts, counts, diam[:3], val[:3], 5.0)
    _check(rows, est[:3], gt[:3], cams[:3], pts, counts, diam[:3], val[:3], 5.0)
    rows = _rows(est, gt, cams, pts, counts, diam[np.arange(n) % 5], val, 5.0)
    _check(rows, est, gt, cams, pts, counts, diam[np.arange(n) % 5], val, 5.0)


def test_adds_minima(cuda_lib):
    rng = np.random.default_rng(2)
    pts, counts, diam = _models(rng, [3417, 7862], 7862)
    pts[1, 3000:6000] = pts[1, :3000]  # duplicated points: tied minima
    far, _, _ = _models(rng, [3417], 3417, centre=1e4)  # coordinates around 1e4 mm
    n = 6
    gt, est = _poses(rng, n)
    est[0], est[1] = gt[0], gt[1]  # estimate == ground truth: every point gives exactly f32(sqrt(1e-5))
    cams, val = _cams(rng, n), np.ones(n, np.int32)
    dia = diam[np.arange(n) % 2]
    rows = _rows(est, gt, cams, pts, counts, dia, val, 5.0)
    _check(rows, est, gt, cams, pts, counts, dia, val, 5.0)
    assert rows[0, 1] == SQRT_EPS and rows[1, 1] == SQRT_EPS and rows[0, 0] == 0 and rows[1, 0] == 0
    gt2, est2 = _poses(rng, 3, tz=(12000, 15000))
    rows = _rows(est2, gt2, _cams(rng, 3), far, np.array([3417], np.int32), np.full(3, 200, F), np.ones(3, np.int32), 5.0)
    _check(rows, est2, gt2, _cams(rng, 3), far, np.array([3417], np.int32), np.full(3, 200, F), np.ones(3, np.int32), 5.0)


def test_adds_never_reads_the_scratch_clouds_past_count(cuda_lib):
    """k_adds_min reads the clouds k_pose_project left in the handle's scratch, not model_points, so NaN padding cannot
    show a read past `count` there.  A first call with the same n and maxp (so the same scratch layout) on a
    7862-point model leaves, in the slots past 3417, estimated points that coincide with the second call's
    ground-truth cloud: a read past count in the second call, on a 3417-point model, would find distance 0 there."""
    rng = np.random.default_rng(6)
    maxp = 7862
    B, _, dB = _models(rng, [3417], maxp)
    A, _, dA = _models(rng, [7862], maxp)
    A[0, 3417:6834] = B[0, :3417]
    gt2, _ = _poses(rng, 1)
    est2 = gt2.copy()
    est2[0, 0, 3] += 40.0  # 40 mm off: closest points far from distance 0
    gt1, _ = _poses(rng, 1)
    cams, val = _cams(rng, 1), np.ones(1, np.int32)
    first = _rows(gt2, gt1, cams, A, np.array([7862], np.int32), dA, val, 5.0)  # estimate of call 1 = ground truth of call 2
    _check(first, gt2, gt1, cams, A, np.array([7862], np.int32), dA, val, 5.0)
    rows = _rows(est2, gt2, cams, B, np.array([3417], np.int32), dB, val, 5.0)
    ref = _check(rows, est2, gt2, cams, B, np.array([3417], np.int32), dB, val, 5.0)
    assert ref[0, 1] > 1.0  # the true ADD-S error is far from the f32(sqrt(1e-5)) a stale read would pull towards


def test_guards(cuda_lib):
    rng = np.random.default_rng(3)
    pts, counts, diam = _models(rng, [500, 3417], 3417)
    gt, est = _poses(rng, 14)
    valid = np.ones(14, np.int32)
    h, q = F(2.0 ** -13), F(2.0 ** -14)  # 1.22e-4 (above 1e-4) and 6.1e-5 (under)
    base = np.array([[1, -1, 0.5, 0], [-0.5, 0.25, -0.25, 0], [0, 0, 0, 0]], F)  # dyadic, sums to exactly 0
    for k, s in enumerate([h, -h, q, -q]):
        est[k] = base
        est[k, 2, 3] = s
        valid[k] = 0  # no ground truth: a false positive only if |sum| > 1e-4
        est[4 + k] = est[k]  # with ground truth: missing if |sum| < 1e-4, else scored
    est[8] = base  # non-zero pose whose entries sum to exactly 0: missing, as in the reference
    est[9] = np.concatenate([np.eye(3, dtype=F), np.array([[0], [0], [-pts[1, 0, 2]]], F)], 1)  # point 0 at z = 0 exactly
    est[10, 2, 3] = -300.0  # points behind the camera
    est[11] = gt[11]  # exact estimate
    cams = _cams(rng, 14, distinct=True)
    om = np.array([0, 1] * 7, np.int32)
    rows = _rows(est, gt, cams, pts, counts, diam[om], valid, 5.0, om)
    ref = _check(rows, est, gt, cams, pts, counts, diam[om], valid, 5.0, om)
    assert rows[0].tolist() == [0, 0, 0, 0, 0, 1] and rows[2].tolist() == [0, 0, 0, 0, 0, 0]
    assert rows[4, 4] == 0 and rows[6].tolist() == [F(99.9), F(999.9), 0, 0, 1, 0] and rows[8, 4] == 1
    assert not np.isfinite(ref[9, 0]) and rows[11, 0] == 0


@pytest.mark.parametrize("n", [1, 128, 129])
def test_batch_sizes(cuda_lib, n):
    rng = np.random.default_rng(n)
    pts, counts, diam = _models(rng, [300, 3417, 9], 3417)
    gt, est = _poses(rng, n)
    cams, val = _cams(rng, n, distinct=True), np.ones(n, np.int32)
    val[::7] = 0
    dia = diam[np.arange(n) % 3]
    rows = _rows(est, gt, cams, pts, counts, dia, val, 10.0)
    idx = range(n) if n <= 129 else None
    _check(rows, est, gt, cams, pts, counts, dia, val, 10.0, idx=idx)


def test_more_than_65535_objects(cuda_lib):
    """n = 65536 with maxp = 3417: k_adds_min runs past the 65535 limit of gridDim.y (about 7 GB of scratch)."""
    rng = np.random.default_rng(4)
    n = 65536
    pts, counts, diam = _models(rng, [3417, 200, 64, 9], 3417)
    om = rng.choice(4, n, p=[0.05, 0.35, 0.3, 0.3]).astype(np.int32)  # mostly non-symmetric
    om[-1] = 0  # the last object is symmetric: the one a clamped grid would miss
    gt, est = _poses(rng, n)
    cams, val = _cams(rng, n), np.ones(n, np.int32)
    rows = _rows(est, gt, cams, pts, counts, diam[om], val, 5.0, om)
    idx = sorted(set(rng.choice(n, 40, replace=False).tolist()) | {n - 1} | set(np.nonzero(om == 0)[0][-4:].tolist()))
    ref = _check(rows, est, gt, cams, pts, counts, diam[om], val, 5.0, om, idx=idx)
    np.testing.assert_allclose(rows[idx].sum(0), ref.sum(0), rtol=1e-5)
    # and the same objects in two calls under the limit give the same bits
    half = n // 2
    a = _rows(est[:half], gt[:half], cams[:half], pts, counts, diam[om[:half]], val[:half], 5.0, om[:half])
    b = _rows(est[half:], gt[half:], cams[half:], pts, counts, diam[om[half:]], val[half:], 5.0, om[half:])
    assert np.array_equal(np.concatenate([a, b]).view(np.uint32), rows.view(np.uint32))
    torch.cuda.empty_cache()


def test_scratch_reuse_across_sizes(cuda_lib):
    """One handle, n and maxp going up and then down: each result equals a fresh handle's."""
    from casapose_b200 import _lib
    from casapose_b200._carrier import current_stream_ptr, ptr

    rng = np.random.default_rng(5)
    dev = torch.device("cuda", torch.cuda.current_device())
    st = current_stream_ptr(dev)

    def call(h, n, maxp):
        pts, counts, diam = _models(np.random.default_rng(n + maxp), [min(3417, maxp), 100, maxp], maxp)
        gt, est = _poses(np.random.default_rng(n), n)
        t = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (est, gt, _cams(rng, n), pts)]
        cnt = torch.from_numpy(counts).to(dev)
        dia = torch.from_numpy(diam[np.arange(n) % 3]).to(dev)
        val = torch.ones(n, dtype=torch.int32, device=dev)
        out = torch.full((n, 6), -1.0, device=dev)
        _lib.check(cuda_lib.casa_pose_errors(h, n, 3, maxp, ptr(t[0]), ptr(t[1]), ptr(t[2]), ptr(t[3]), ptr(cnt), C.c_void_p(),
                                             ptr(dia), ptr(val), C.c_float(5.0), ptr(out), st))
        return out.cpu().numpy()

    hp = C.c_void_p()
    _lib.check(cuda_lib.casa_create(dev.index, C.byref(hp)))
    try:
        for n, maxp in [(3, 500), (40, 3417), (200, 7862), (40, 3417), (3, 500), (200, 3417), (7, 7862)]:
            a = call(hp, n, maxp)
            fresh = C.c_void_p()
            _lib.check(cuda_lib.casa_create(dev.index, C.byref(fresh)))
            try:
                b = call(fresh, n, maxp)
            finally:
                _lib.check(cuda_lib.casa_destroy(fresh))
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (n, maxp)
    finally:
        _lib.check(cuda_lib.casa_destroy(hp))
