"""Batched PnP (casa_pnp, pnp.cuh K7) across the paths of its kernel: keypoint counts, batch sizes, per-object cameras
and offsets, outliers, geometry, guards, the t_z < 0 flip and coplanar keypoints.

Every solved case goes through three bars:
  * the kernel against its numpy restatement (oracle/pnp_np.pnp): within 1e-3 on every pose entry (mm and rotation
    entries), the bar of tests/test_pnp.py;
  * the all-point reprojection cost against the reference's cv2 sequence (oracle/pose_np.pnp): the kernel's cost is at
    most cv2's * (1 + 1e-6) + 1e-9.  Where cv2 and the restatement may settle in different minima (planar ambiguity,
    outliers) that is the bar; clean cases also keep tests/test_pnp.py's rule that 95 % agree within 0.05 mm / 1e-4;
  * guard cases give the exact all-zero [3,4], like the oracle and the reference.

The dead guard compares |sum| < 0.01 in float32.  The kernel adds the keypoints sequentially, numpy pairwise and the
reference in TensorFlow's order; these differ in the last bits, about 1e-4 of the threshold.  The guard scenes are
therefore built on a dyadic grid (multiples of 2^-13, partial sums below 2^11), where every order gives the same exact
sum.  0.01 itself is not on such a grid, so these cases are the two grid points around it: 82 * 2^-13 (9.8e-6 above,
alive) and 81 * 2^-13 (1.1e-4 under, dead).  The exact boundary, 0.01f and one ulp under it, is tested on a camera with
a 0.02 px focal length, where every keypoint sits on the 2^-30 grid of 0.01f (`boundary_scene`).

The scene builders are plain numpy; the tests without the gpu marker check on the CPU that each scene is what it
claims (planar after float32 rounding, outliers beyond 12 px, the flip case, exact guard sums), and that the
restatement meets the cost bar against cv2 on the planar and outlier scenes.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from casapose_b200 import synthetic  # noqa: E402
from oracle import pnp_np  # noqa: E402
from oracle import pose_np as OP  # noqa: E402

F = np.float32
GRID = 2.0 ** -13  # dyadic grid of the guard scenes
ALIVE, DEAD = 82 * GRID, 81 * GRID  # the grid points around 0.01: 0.010009765625 and 0.0098876953125
SENTINEL = F(-12345.5)


# ----------------------------------------------------------------------------------------------- scene builders
def _cam(fx=572.4114, fy=573.57043, cx=325.2611, cy=242.04899):
    return np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], F)


def _project(X, R, t, K):
    """float64 projection of float32 model points -> (uv float32 [vn,2], camera-frame points float64)."""
    c = X.astype(np.float64) @ R.T + t
    q = c @ K.astype(np.float64).T
    return (q[:, :2] / q[:, 2:]).astype(F), c


def _small_rotation(rng, deg):
    w = rng.normal(size=3)
    w *= np.deg2rad(deg) / np.linalg.norm(w)
    return pnp_np._exp(w)


def _objects(rng, n, vn, K=None, tz=(600, 1200), ext=(50, 150), noise=0.3, cams=None):
    """n random non-planar keypoint sets seen by a camera each -> p2 [n,vn,2], p3 [n,vn,3], cam [n,3,3], gt [n,3,4]."""
    cam = np.stack([K if K is not None else _cam()] * n) if cams is None else cams
    p2, p3, gt = np.zeros((n, vn, 2), F), np.zeros((n, vn, 3), F), np.zeros((n, 3, 4))
    for i in range(n):
        e = rng.uniform(*ext)
        X = (rng.uniform(-0.5, 0.5, size=(vn, 3)) * e).astype(F)
        R = synthetic._random_rotation(rng)
        z = rng.uniform(*tz)
        # keep the centre inside the middle half of the image
        u0 = rng.uniform(0.25, 0.75) * 2 * cam[i, 0, 2]
        v0 = rng.uniform(0.25, 0.75) * 2 * cam[i, 1, 2]
        t = np.array([(u0 - cam[i, 0, 2]) * z / cam[i, 0, 0], (v0 - cam[i, 1, 2]) * z / cam[i, 1, 1], z])
        uv, _ = _project(X, R, t, cam[i])
        p2[i] = uv + rng.normal(scale=noise, size=(vn, 2)).astype(F) if noise else uv
        p3[i], gt[i] = X, np.concatenate([R, t[:, None]], 1)
    return p2, p3, cam, gt


def _plant(rng, p2, i, idx, lo=20.0, hi=60.0):
    """Moves keypoints idx of object i by lo..hi px in a random direction (outliers beyond the 12 px band)."""
    for k in idx:
        a = rng.uniform(0, 2 * np.pi)
        p2[i, k] += (rng.uniform(lo, hi) * np.array([np.cos(a), np.sin(a)])).astype(F)


def planar_scene(rng, n, vn=9, noise=0.0):
    """Keypoints on a randomly rotated plane (float32 coordinates, so after rounding), at 600..1000 mm."""
    cam = np.stack([_cam()] * n)
    p2, p3, gt = np.zeros((n, vn, 2), F), np.zeros((n, vn, 3), F), np.zeros((n, 3, 4))
    for i in range(n):
        Rp = synthetic._random_rotation(rng)
        X = (np.concatenate([rng.uniform(-60, 60, (vn, 2)), np.zeros((vn, 1))], 1) @ Rp.T + rng.uniform(-20, 20, 3)).astype(F)
        R = synthetic._random_rotation(rng)
        t = np.array([rng.uniform(-100, 100), rng.uniform(-80, 80), rng.uniform(600, 1000)])
        uv, _ = _project(X, R, t, cam[i])
        p2[i] = uv + (rng.normal(scale=noise, size=(vn, 2)).astype(F) if noise else 0)
        p3[i], gt[i] = X, np.concatenate([R, t[:, None]], 1)
    return p2, p3, cam, gt


def thin_scene(rng, depths, vn=9):
    """Keypoints on a plane plus a seeded +-depth (mm) out of it: thin but not planar."""
    n = len(depths)
    cam = np.stack([_cam()] * n)
    p2, p3, gt = np.zeros((n, vn, 2), F), np.zeros((n, vn, 3), F), np.zeros((n, 3, 4))
    for i, d in enumerate(depths):
        Xp = np.concatenate([rng.uniform(-60, 60, (vn, 2)), (rng.choice([-1.0, 1.0], (vn, 1)) * d)], 1)
        X = Xp.astype(F)  # axis-aligned plane: the offset survives float32 rounding
        R = synthetic._random_rotation(rng)
        t = np.array([rng.uniform(-100, 100), rng.uniform(-80, 80), rng.uniform(600, 1000)])
        uv, _ = _project(X, R, t, cam[i])
        p2[i], p3[i], gt[i] = uv + rng.normal(scale=0.3, size=(vn, 2)).astype(F), X, np.concatenate([R, t[:, None]], 1)
    return p2, p3, cam, gt


def flip_scene(rng, n, vn=9):
    """Model points about 1500 mm from the model origin along its z axis, seen from 800 mm with a near-identity
    rotation: every point is in front of the camera, but t_z = 800 - 1500 R_22 < 0."""
    cam = np.stack([_cam()] * n)
    p2, p3, gt = np.zeros((n, vn, 2), F), np.zeros((n, vn, 3), F), np.zeros((n, 3, 4))
    for i in range(n):
        X = (rng.uniform(-50, 50, (vn, 3)) + [0, 0, 1500]).astype(F)
        R = _small_rotation(rng, 20)
        t = np.array([rng.uniform(-80, 80), rng.uniform(-60, 60), 800.0]) - R @ np.array([0, 0, 1500.0])
        uv, _ = _project(X, R, t, cam[i])
        p2[i], p3[i], gt[i] = uv + rng.normal(scale=0.3, size=(vn, 2)).astype(F), X, np.concatenate([R, t[:, None]], 1)
    return p2, p3, cam, gt


def dyadic_scene(rng, target, vn=9):
    """One keypoint set on the 2^-13 grid whose float32 sum is exactly `target` in any order: a camera with its
    principal point at 0 and a small object on the optical axis keep every |coordinate| small, and the last y takes
    up the rest (it may become an outlier, which the leave-one-out candidates absorb)."""
    K = _cam(cx=0.0, cy=0.0)
    X = (rng.uniform(-30, 30, size=(vn, 3))).astype(F)
    uv, _ = _project(X, synthetic._random_rotation(rng), np.array([0.0, 0.0, 900.0]), K)
    uv = (np.round(uv.astype(np.float64) / GRID) * GRID).astype(F)
    uv[-1, 1] = F(target - (uv.astype(np.float64).sum() - float(uv[-1, 1])))
    return uv, X, K


def boundary_scene(rng, target, vn=9):
    """A keypoint set whose float32 sum is exactly `target` (0.01f or one ulp under, either sign) in every order.
    Exactness in every order needs every partial sum below 2^-6 on the 2^-30 grid of 0.01f, so the camera has a focal
    length of 0.02 px and its principal point at 0: the keypoints come in pairs mirrored through the optical axis
    (exact negatives), and the last one sits at (target, 0), the projection of a point 0.5 z off the axis."""
    K = _cam(fx=0.02, fy=0.02, cx=0.0, cy=0.0)
    Xc = np.zeros((vn, 3))
    for k in range((vn - 1) // 2):
        z = rng.uniform(800, 1000)
        a, b = rng.uniform(-0.02, 0.02, 2) * z
        Xc[2 * k], Xc[2 * k + 1] = (a, b, z), (-a, -b, z)
    Xc[-1] = (float(F(target)) / 0.02 * 900.0, 0.0, 900.0)
    uv = (np.round(Xc[:, :2] / Xc[:, 2:] * 0.02 / 2.0 ** -30) * 2.0 ** -30).astype(F)
    uv[1:-1:2] = -uv[0:-1:2]
    uv[-1] = (F(target), F(0))
    R, t = synthetic._random_rotation(rng), np.array([5.0, -3.0, 900.0])
    return uv, ((Xc - t) @ R).astype(F), K


BOUNDARY = [F(0.01), -F(0.01), np.nextafter(F(0.01), F(0)), -np.nextafter(F(0.01), F(0))]


def _seq_sum(a):
    s = F(0)
    for p in a.reshape(-1, 2):
        s = F(s + F(p[0] + p[1]))  # the kernel's order: per point x + y, then the running sum
    return s


# ----------------------------------------------------------------------------------------------- checks
def _cost(P, X, uv, K):
    """All-point squared reprojection cost (px^2) of a [3,4] pose in float64; inf for a zero pose or a point at z <= 0."""
    P = np.asarray(P, np.float64)
    if not P.any():
        return np.inf
    c = X.astype(np.float64) @ P[:, :3].T + P[:, 3]
    if not (c[:, 2] > 0).all():
        return np.inf
    q = c @ K.astype(np.float64).T
    return float(((q[:, :2] / q[:, 2:] - uv.astype(np.float64)) ** 2).sum())


def _close(a, b):
    return np.abs(a[:, 3] - b[:, 3]).max() < 0.05 and np.abs(a[:, :3] - b[:, :3]).max() < 1e-4  # 0.05 mm, 1e-4


def _cost_bar(mine, X, uv, K):
    ref = _cost(OP.pnp(X, uv, K), X, uv, K)
    return _cost(mine, X, uv, K) <= ref * (1 + 1e-6) + 1e-9


def _solve(p2, p3, cam, off=None):
    from casapose_b200.pose_estimation.ransac_voting import pnp_cuda

    return pnp_cuda(torch.from_numpy(np.ascontiguousarray(p2)).cuda(), p3, cam, off).cpu().numpy()


def _check(got, p2, p3, cam, idx=None, cost_bar=True, clean=False):
    idx = range(len(got)) if idx is None else idx
    agree = 0
    for i in idx:
        ref = pnp_np.pnp(p3[i], p2[i], cam[i])
        assert np.abs(got[i] - ref).max() <= 1e-3, (i, got[i], ref)
        if cost_bar:
            assert _cost_bar(got[i], p3[i], p2[i], cam[i]), i
        if clean:
            agree += _close(got[i], OP.pnp(p3[i], p2[i], cam[i]))
    if clean:
        assert agree >= 0.95 * len(idx)


# Seeded objects where the kernel, like its restatement, ends with a larger all-point reprojection cost than cv2: the
# final LM runs on all points from the winning candidate and settles in a different local minimum (with outliers), or
# in the other minimum of the planar two-fold ambiguity (thin or planar sets under 0.3 px noise).  Findings left open
# (DESIGN.md K7); every other object of these scenes meets the cost bar.
KNOWN_MISSES = {
    ("outliers", 9, (2, 5)): (0,),  # different local minimum of the all-point LM (cost 3285 against cv2's 2761)
    ("outliers", 12, (0, 5, 11)): (0,),  # three outliers put every candidate's DLT behind the camera: zeros
    ("thin",): (1,),  # the 10 um set: the other minimum of the planar ambiguity (cost 26.5 against cv2's 2.0)
}


def _cost_bar_except(got, p2, p3, cam, known):
    miss = [i for i in range(len(got)) if not _cost_bar(got[i], p3[i], p2[i], cam[i])]
    assert miss == sorted(known), miss


# ----------------------------------------------------------------------------------------------- builder checks (CPU)
def _flatness(X):
    """pnp_dlt's planarity estimate of a full keypoint set: det C / (largest cross product of two rows of C * tr C), C
    the normalised centred covariance; within a factor 3 of its smallest over its largest eigenvalue."""
    Xd = X.astype(np.float64)
    Xs = (Xd - Xd.mean(0)) / np.sqrt(((Xd - Xd.mean(0)) ** 2).sum(1).mean())
    C = Xs.T @ Xs
    n = max((np.cross(C[a], C[b]) for a, b in ((0, 1), (0, 2), (1, 2))), key=lambda v: v @ v)
    return C[0] @ np.cross(C[1], C[2]) / (np.sqrt(n @ n) * np.trace(C))


@pytest.mark.parametrize("vn", list(range(6, 17)))
def test_planar_scene_is_planar_after_float32_rounding(vn):
    p2, p3, cam, _ = planar_scene(np.random.default_rng(vn), 40, vn=vn)
    pivot_passes = 0
    for X in p3:
        Xd = X.astype(np.float64)
        ev = np.linalg.eigvalsh(np.cov(Xd.T))
        assert ev[0] < 1e-12 * ev[-1]  # rounding leaves the points within ~1e-5 mm of a plane
        assert _flatness(X) <= pnp_np.PLANAR_RTOL  # so the planar branch runs
        Xs = (Xd - Xd.mean(0)) / np.sqrt(((Xd - Xd.mean(0)) ** 2).sum(1).mean())
        S = pnp_np._moments(np.concatenate([Xs, np.ones((len(X), 1))], 1), np.zeros((len(X), 2)))
        pivot_passes += pnp_np._reduce(*S) is not None
    # rounding lifts some pivots above 1e-14: the pivot test alone would send those sets to the singular 4x4 system
    assert vn > 8 or pivot_passes > 0


def test_thin_scene_is_thin_but_takes_the_general_reduction():
    depths = [1e-3, 1e-2, 1e-1, 1.0]
    p2, p3, cam, _ = thin_scene(np.random.default_rng(11), depths)
    for X, d in zip(p3, depths):
        Xd = X.astype(np.float64)
        assert np.allclose(np.abs(Xd[:, 2]), d, rtol=1e-3)
        assert _flatness(X) > pnp_np.PLANAR_RTOL
        Xs = (Xd - Xd.mean(0)) / np.sqrt(((Xd - Xd.mean(0)) ** 2).sum(1).mean())
        S = pnp_np._moments(np.concatenate([Xs, np.ones((len(X), 1))], 1), np.zeros((len(X), 2)))
        assert pnp_np._reduce(*S) is not None


def test_outlier_scenes_plant_outliers_beyond_12_px():
    for vn, idx in _OUTLIER_CASES:
        p2, p3, cam, gt = _outlier_scene(vn, idx)
        for i in range(len(p2)):
            uv, _ = _project(p3[i], gt[i][:, :3], gt[i][:, 3], cam[i])
            e = np.linalg.norm(p2[i].astype(np.float64) - uv, axis=1)
            assert (e[list(idx)] > 12).all() and (np.delete(e, list(idx)) < 3).all()


def test_flip_scene_has_negative_t_z_and_every_point_in_front():
    p2, p3, cam, gt = flip_scene(np.random.default_rng(12), 6)
    for X, P in zip(p3, gt):
        assert P[2, 3] < 0 and ((X.astype(np.float64) @ P[:, :3].T + P[:, 3])[:, 2] > 0).all()


@pytest.mark.parametrize("target", [ALIVE, -ALIVE, DEAD, -DEAD])
def test_guard_sums_are_exact_in_every_order(target):
    rng = np.random.default_rng(13)
    uv, _, _ = dyadic_scene(rng, target)
    flat = uv.reshape(-1)
    assert np.abs(flat).sum() < 2.0 ** 11
    assert _seq_sum(uv) == F(target) and uv.sum(dtype=F) == F(target) and float(uv.astype(np.float64).sum()) == target
    for _ in range(8):
        perm = rng.permutation(flat.size)
        assert flat[perm].sum(dtype=F) == F(target) and _seq_sum(flat[perm]) == F(target)
    assert (abs(F(target)) < F(0.01)) == (abs(target) == DEAD)


@pytest.mark.parametrize("target", BOUNDARY)
def test_boundary_sums_are_exact_in_every_order(target):
    rng = np.random.default_rng(16)
    uv, _, _ = boundary_scene(rng, target)
    flat = uv.reshape(-1)
    assert np.abs(flat).sum() < 2.0 ** -6
    assert _seq_sum(uv) == target and uv.sum(dtype=F) == target and float(uv.astype(np.float64).sum()) == float(target)
    for _ in range(8):
        perm = rng.permutation(flat.size)
        assert flat[perm].sum(dtype=F) == target and _seq_sum(flat[perm]) == target
    assert (abs(target) < F(0.01)) == (abs(target) != F(0.01))


def test_restatement_meets_the_cost_bar_on_planar_and_outlier_scenes():
    for p2, p3, cam, _ in (planar_scene(np.random.default_rng(14), 6), planar_scene(np.random.default_rng(15), 6, noise=0.3),
                           _outlier_scene(9, (7, 8)), _outlier_scene(16, (0, 15))):
        for i in range(len(p2)):
            assert _cost_bar(pnp_np.pnp(p3[i], p2[i], cam[i]), p3[i], p2[i], cam[i]), i


# ----------------------------------------------------------------------------------------------- GPU cases
@pytest.mark.gpu
@pytest.mark.parametrize("vn", list(range(6, 17)))
def test_keypoint_counts(cuda_lib, vn):
    rng = np.random.default_rng(100 + vn)
    p2, p3, cam, _ = _objects(rng, 6, vn)
    if vn >= 7:
        _plant(rng, p2, 5, [rng.integers(vn)])
    got = _solve(p2, p3, cam)
    _check(got, p2, p3, cam)
    _check(got, p2, p3, cam, idx=range(5), cost_bar=False, clean=True)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 5, 127])
def test_batch_sizes_leave_the_rest_of_the_output_alone(cuda_lib, n):
    from casapose_b200 import _lib
    from casapose_b200._carrier import current_stream_ptr, ptr

    vn = 9
    p2, p3, cam, _ = _objects(np.random.default_rng(200 + n), n, vn)
    dev = torch.device("cuda", torch.cuda.current_device())
    t2, t3, tc = (torch.from_numpy(a).to(dev) for a in (p2, p3, cam))
    out = torch.full((n * 12 + 64,), float(SENTINEL), dtype=torch.float32, device=dev)
    hdl = _lib.handle(dev.index, current_stream_ptr(dev))
    rc = cuda_lib.casa_pnp(hdl, n, vn, ptr(t2), ptr(t3), ptr(tc), C.c_void_p(), ptr(out), current_stream_ptr(dev))
    _lib.check(rc)
    res = out.cpu().numpy()
    assert (res[n * 12:] == SENTINEL).all()
    got = res[: n * 12].reshape(n, 3, 4)
    idx = range(n) if n <= 5 else np.random.default_rng(n).choice(n, 16, replace=False)
    _check(got, p2, p3, cam, idx=idx)


@pytest.mark.gpu
def test_large_batch_is_independent_of_batching_and_order(cuda_lib):
    n, vn = 4099, 9
    rng = np.random.default_rng(300)
    p2, p3, cam, _ = _objects(rng, n, vn)
    for i in rng.choice(n, 400, replace=False):
        _plant(rng, p2, i, [rng.integers(vn)])
    a = _solve(p2, p3, cam)
    b = _solve(p2, p3, cam)
    assert np.array_equal(a, b)
    perm = rng.permutation(n)
    c = np.zeros_like(a)
    for lo in range(0, n, 997):
        sl = perm[lo: lo + 997]
        c[sl] = _solve(p2[sl], p3[sl], cam[sl])
    assert np.array_equal(a.view(np.uint32), c.view(np.uint32))
    _check(a, p2, p3, cam, idx=rng.choice(n, 24, replace=False))


def _cameras(rng, n):
    """Distinct cameras: 480p to 4K, fx != fy, principal points off the image centre."""
    cams = np.zeros((n, 3, 3), F)
    for i in range(n):
        w, h = [(640, 480), (1280, 720), (1920, 1080), (3840, 2160)][i % 4]
        f = rng.uniform(0.8, 1.6) * w
        cams[i] = _cam(fx=f, fy=f * rng.uniform(0.9, 1.1), cx=w / 2 + rng.uniform(-0.1, 0.1) * w, cy=h / 2 + rng.uniform(-0.1, 0.1) * h)
    return cams


@pytest.mark.gpu
def test_per_object_cameras(cuda_lib):
    rng = np.random.default_rng(400)
    n = 24
    cams = _cameras(rng, n)
    p2, p3, cam, _ = _objects(rng, n, 9, cams=cams)
    got = _solve(p2, p3, cam)
    _check(got, p2, p3, cam, clean=True)
    # the same objects solved one at a time: no stride mixes cameras
    for i in range(0, n, 5):
        assert np.array_equal(got[i], _solve(p2[i: i + 1], p3[i: i + 1], cam[i: i + 1])[0])


@pytest.mark.gpu
def test_per_object_offsets(cuda_lib):
    from casapose_b200.pose_estimation.ransac_voting import transform_points_back

    rng = np.random.default_rng(500)
    n, vn = 16, 9
    p2, p3, cam, _ = _objects(rng, n, vn)
    angles = [0.0, 90.0, -90.0, 180.0] + list(rng.uniform(-180, 180, n - 4))
    off = np.zeros((n, 10), F)
    raw = np.zeros_like(p2)
    for i in range(n):
        h_crop, w_crop = rng.uniform(0, 80, 2)
        sx, sy = [(640, 480), (800, 600), (1280, 960)][i % 3]
        dx, dy = rng.uniform(-20, 20, 2)
        scale = [0.5, 1.0, 2.0, rng.uniform(0.5, 2.0)][i % 4]
        off[i] = [h_crop, w_crop, 0, 0, dx, dy, angles[i], scale, sx, sy]
        # forward-map p2 so that un-mapping gives it back (up to float32 rounding): inverse of transform_points_back
        ang = np.deg2rad(-angles[i])
        a, b = np.cos(ang), np.sin(ang)
        c, d = (1 - a) * sx / 2 - b * sy / 2, b * sx / 2 + (1 - a) * sy / 2
        u = p2[i].astype(np.float64) - [c, d]
        x1, y1 = a * u[:, 0] - b * u[:, 1], b * u[:, 0] + a * u[:, 1]
        raw[i] = np.stack([(x1 + dx - w_crop) * scale, (y1 + dy - h_crop) * scale], 1).astype(F)
    got = _solve(raw, p3, cam, off)
    back = np.stack([transform_points_back(raw[i], *off[i, [0, 1, 8, 9, 4, 5, 6, 7]]) for i in range(n)])
    assert np.abs(back - p2).max() < 1e-2  # the forward map is right
    _check(got, back, p3, cam)
    for i in range(0, n, 5):  # and no stride mixes offsets
        assert np.array_equal(got[i], _solve(raw[i: i + 1], p3[i: i + 1], cam[i: i + 1], off[i: i + 1])[0])


_OUTLIER_CASES = [(9, ()), (9, (0,)), (9, (8,)), (9, (7, 8)), (9, (0, 8)), (9, (2, 5)), (12, (10, 11)),
                  (16, (0, 15)), (9, (0, 4, 8)), (12, (0, 5, 11))]


def _outlier_scene(vn, idx, n=4):
    rng = np.random.default_rng(600 + 17 * vn + sum(idx) + 100 * len(idx))
    p2, p3, cam, gt = _objects(rng, n, vn, noise=0.3)
    for i in range(n):
        _plant(rng, p2, i, idx)
    return p2, p3, cam, gt


@pytest.mark.gpu
@pytest.mark.parametrize("vn,idx", _OUTLIER_CASES, ids=["vn%d-%s" % (v, "-".join(map(str, i)) or "none") for v, i in _OUTLIER_CASES])
def test_outliers(cuda_lib, vn, idx):
    p2, p3, cam, gt = _outlier_scene(vn, idx)
    got = _solve(p2, p3, cam)
    _check(got, p2, p3, cam, cost_bar=False)
    _cost_bar_except(got, p2, p3, cam, KNOWN_MISSES.get(("outliers", vn, idx), ()))


@pytest.mark.gpu
def test_geometry_far_near_border_thin(cuda_lib):
    rng = np.random.default_rng(700)
    far = _objects(rng, 6, 9, tz=(3000, 5000), ext=(100, 150))
    near = _objects(rng, 6, 9, tz=(190, 210), ext=(40, 60))
    thin = thin_scene(rng, [1e-3, 1e-2, 1e-1, 1.0, 1e-3, 1e-1])
    p2, p3, cam, _ = _objects(rng, 6, 9)
    K = _cam()
    for i in range(6):  # near the image border: centre 20..40 px inside a corner
        R = synthetic._random_rotation(rng)
        z = rng.uniform(900, 1200)
        u0, v0 = [(30, 30), (610, 30), (30, 450), (610, 450), (320, 25), (25, 240)][i]
        X = (rng.uniform(-0.5, 0.5, (9, 3)) * 60).astype(F)
        t = np.array([(u0 - K[0, 2]) * z / K[0, 0], (v0 - K[1, 2]) * z / K[1, 1], z])
        uv, _ = _project(X, R, t, K)
        p2[i], p3[i] = uv + rng.normal(scale=0.3, size=(9, 2)).astype(F), X
    border = (p2, p3, cam, None)
    for name, (q2, q3, qc, _) in (("far", far), ("near", near), ("thin", thin), ("border", border)):
        got = _solve(q2, q3, qc)
        assert got.any(axis=(1, 2)).all(), name
        _check(got, q2, q3, qc, cost_bar=False)
        _cost_bar_except(got, q2, q3, qc, KNOWN_MISSES.get((name,), ()))


@pytest.mark.gpu
def test_guards_give_exact_zeros(cuda_lib):
    from casapose_b200.pose_estimation.ransac_voting import transform_points_back

    rng = np.random.default_rng(800)
    vn = 9
    rows, alive = [], []
    for target in (ALIVE, -ALIVE, DEAD, -DEAD):
        uv, X, K = dyadic_scene(rng, target)
        rows.append((uv, X, K, None))
        alive.append(abs(target) == ALIVE)
    # dead only after un-mapping: angle 0 and scale 1 make it exact; shifts on the grid
    shift = np.array([64.0 - 8.5, 32.0 + 4.25])
    off = np.array([32.0, 64.0, 0, 0, 8.5, -4.25, 0.0, 1.0, 640.0, 480.0], F)
    for target in (DEAD, ALIVE):
        uv, X, K = dyadic_scene(rng, target)
        raw = (uv.astype(np.float64) - shift).astype(F)
        assert abs(float(raw.sum(dtype=F))) > 100 and np.array_equal(transform_points_back(raw, *off[[0, 1, 8, 9, 4, 5, 6, 7]]), uv)
        rows.append((raw, X, K, off))
        alive.append(target == ALIVE)
    rows.append(((np.zeros((vn, 2)) - shift).astype(F), X, K, off))  # every point un-maps to 0
    alive.append(False)
    # a NaN or an inf keypoint: cv2 returns a NaN translation and the reference zeros
    for bad in (np.nan, np.inf, -np.inf):
        p2, p3, cam, _ = _objects(rng, 1, vn)
        p2[0, 4, 1] = bad
        rows.append((p2[0], p3[0], cam[0], None))
        alive.append(False)
    p2 = np.stack([r[0] for r in rows])
    p3 = np.stack([r[1] for r in rows])
    cam = np.stack([r[2] for r in rows])
    offs = np.stack([r[3] if r[3] is not None else np.array([0, 0, 0, 0, 0, 0, 0, 1, 640, 480], F) for r in rows])
    got = _solve(p2, p3, cam, offs)
    for i, (q2, X, K, o) in enumerate(rows):
        o = offs[i]
        back = transform_points_back(q2, *o[[0, 1, 8, 9, 4, 5, 6, 7]])
        ref = pnp_np.pnp(X, back, K) if abs(float(q2.sum(dtype=F))) >= 0.01 or not np.isfinite(q2).all() else np.zeros((3, 4), F)
        # the reference's map_offsets / map_pnp / pnp sequence on the same object
        cv, _ = OP.estimate_poses(q2[None, None], X[None, None, None], K[None], np.ones((1, 1)), o[None])
        if alive[i]:
            assert got[i].any() and np.abs(got[i] - ref).max() <= 1e-3, i
        else:
            assert np.array_equal(got[i], np.zeros((3, 4), F)) and np.array_equal(ref, got[i]), i
            assert np.array_equal(cv[0, 0], got[i]), i


@pytest.mark.gpu
def test_dead_guard_at_exactly_0_01(cuda_lib):
    """|sum| == 0.01f is alive and one ulp under it dead, as TensorFlow's float32 compare decides."""
    rng = np.random.default_rng(850)
    rows = [boundary_scene(rng, t) for t in BOUNDARY]
    got = _solve(np.stack([r[0] for r in rows]), np.stack([r[1] for r in rows]), np.stack([r[2] for r in rows]))
    for i, ((uv, X, K), t) in enumerate(zip(rows, BOUNDARY)):
        ref = pnp_np.pnp(X, uv, K)
        if abs(t) == F(0.01):
            assert got[i].any() and np.abs(got[i] - ref).max() <= 1e-3, i
        else:
            assert np.array_equal(got[i], np.zeros((3, 4), F)) and np.array_equal(ref, got[i]), i
            cv, _ = OP.estimate_poses(uv[None, None], X[None, None, None], K[None], np.ones((1, 1)),
                                      np.array([[0, 0, 0, 0, 0, 0, 0, 1, 640, 480]], F))
            assert np.array_equal(cv[0, 0], got[i]), i


@pytest.mark.gpu
def test_degenerate_geometry_gives_zeros(cuda_lib):
    """Every keypoint behind the camera, and collinear 3-D keypoints: no candidate yields a proper rotation with every
    point in front, so the kernel and its restatement return zeros.  The reference's cv2 sequence returns a pose for
    both (for points behind the camera the improper -[R|t] of its flip), see DESIGN.md K7."""
    rng = np.random.default_rng(900)
    K = _cam()
    p2, p3 = np.zeros((8, 9, 2), F), np.zeros((8, 9, 3), F)
    for i in range(4):
        X = rng.uniform(-60, 60, (9, 3)).astype(F)
        uv, c = _project(X, synthetic._random_rotation(rng), np.array([20.0, -10.0, -800.0]), K)
        assert (c[:, 2] < 0).all()
        p2[i], p3[i] = uv, X
    for i in range(4, 8):
        X = np.outer(rng.uniform(-60, 60, 9), rng.normal(size=3)).astype(F)
        uv, c = _project(X, synthetic._random_rotation(rng), np.array([20.0, -10.0, 800.0]), K)
        p2[i], p3[i] = uv + rng.normal(scale=0.3, size=(9, 2)).astype(F), X
    cam = np.stack([K] * 8)
    got = _solve(p2, p3, cam)
    for i in range(8):
        assert np.array_equal(got[i], np.zeros((3, 4), F)) and np.array_equal(pnp_np.pnp(p3[i], p2[i], K), got[i]), i


@pytest.mark.gpu
def test_negative_t_z_flip(cuda_lib):
    p2, p3, cam, gt = flip_scene(np.random.default_rng(1000), 8)
    got = _solve(p2, p3, cam)
    _check(got, p2, p3, cam, clean=True)
    for i in range(len(got)):
        assert got[i][2, 3] > 0 and np.linalg.det(got[i][:, :3].astype(np.float64)) < 0  # -[R|t], like OP.pnp
        assert np.abs(-got[i][:, :3] - gt[i][:, :3]).max() < 0.05


@pytest.mark.gpu
@pytest.mark.parametrize("vn", list(range(6, 17)))
def test_planar_keypoints_noise_free(cuda_lib, vn):
    p2, p3, cam, gt = planar_scene(np.random.default_rng(1100 + vn), 16, vn=vn)
    got = _solve(p2, p3, cam)
    _check(got, p2, p3, cam)
    for i in range(len(got)):
        rms = np.sqrt(_cost(got[i], p3[i], p2[i], cam[i]) / len(p2[i]))
        assert rms <= 1e-3, (i, rms)
        assert np.abs(got[i][:, 3] - gt[i][:, 3]).max() < 0.05 and np.abs(got[i][:, :3] - gt[i][:, :3]).max() < 1e-4
        cv = OP.pnp(p3[i], p2[i], cam[i])
        if np.sqrt(_cost(cv, p3[i], p2[i], cam[i]) / len(p2[i])) <= 1e-3:  # cv2 sometimes settles in the mirrored minimum
            assert _close(got[i], cv), i


@pytest.mark.gpu
@pytest.mark.parametrize("vn", list(range(6, 17)))
def test_planar_keypoints_with_noise(cuda_lib, vn):
    p2, p3, cam, _ = planar_scene(np.random.default_rng(1200 + vn), 16, vn=vn, noise=0.3)
    got = _solve(p2, p3, cam)
    assert got.any(axis=(1, 2)).all()
    _check(got, p2, p3, cam, cost_bar=False)
    _cost_bar_except(got, p2, p3, cam, KNOWN_MISSES.get(("planar", vn), ()))


@pytest.mark.gpu
def test_input_forms(cuda_lib):
    from casapose_b200.pose_estimation.ransac_voting import pnp_cuda

    p2, p3, cam, _ = _objects(np.random.default_rng(1300), 12, 9)
    base = _solve(p2, p3, cam)
    assert np.array_equal(pnp_cuda(p2, p3, cam).cpu().numpy(), base)  # numpy in
    t64 = pnp_cuda(torch.from_numpy(p2.astype(np.float64)).cuda(), torch.from_numpy(p3.astype(np.float64)),
                   torch.from_numpy(cam.astype(np.float64)).cuda())
    assert np.array_equal(t64.cpu().numpy(), base)  # float64 torch in, values exact in float32
    wide = torch.zeros((12, 9, 5), dtype=torch.float32, device="cuda")
    wide[:, :, 1:3] = torch.from_numpy(p2).cuda()
    view = wide[:, :, 1:3]
    assert not view.is_contiguous()
    assert np.array_equal(pnp_cuda(view, p3, cam).cpu().numpy(), base)
