"""Backward of PnP (casa_pnp_backward, DESIGN.md K10): the BPnP_fast gradient of the pose w.r.t. the 2-D points.

CPU: the gradient oracle (oracle/pnp_grad.py) against the closed form J (J^T J)^-1 g, against central finite differences
of a float64 Levenberg-Marquardt solve at zero residual, across the two pose forms, and under the t_z flip.
GPU: the kernel against the oracle, the three Python call sites through torch.autograd, and the training chain
CoordLSVotingWeighted -> poses_pnp -> loss against the two gradient oracles composed."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from casapose_b200 import synthetic  # noqa: E402
from oracle import ls_voting_np as L  # noqa: E402
from oracle import pnp_grad as PG  # noqa: E402

F = np.float32


def _rotvec(R):
    from scipy.spatial.transform import Rotation

    return Rotation.from_matrix(np.asarray(R, np.float64)).as_rotvec()


def _rotmat(r):
    from scipy.spatial.transform import Rotation

    return Rotation.from_rotvec(r).as_matrix()


def _cases(n, vn=9, seed=0):
    """n objects in the pattern of tests/test_pnp.py: LM keypoints (vn = 9) or random points in a 150 mm box,
    uniformly random rotation, t_z in [600, 1200] mm, the BOP LM camera.  -> X [n,vn,3], K [3,3], [R|t] [n,3,4] (float32)."""
    rng = np.random.default_rng(seed)
    models = synthetic.lm_models()
    K = synthetic.camera_matrix(480).astype(F)
    X = np.zeros((n, vn, 3), F)
    P = np.zeros((n, 3, 4), F)
    for i in range(n):
        if vn == 9:
            X[i] = np.array(models["obj_%06d" % synthetic.CONFIG_13_IDS[i % 13]]["keypoints"], F)
        else:
            X[i] = (rng.uniform(-0.5, 0.5, size=(vn, 3)) * 150).astype(F)
        R = synthetic._random_rotation(rng)
        t = np.array([rng.uniform(-200, 200), rng.uniform(-150, 150), rng.uniform(600, 1200)])
        P[i] = np.concatenate([R, t[:, None]], 1).astype(F)
    return X, K, P


def _project(X, K, R, t):
    c = X @ R.T + t
    uv = c @ K.T
    return uv[:, :2] / uv[:, 2:]


def _closed_form(X, K, P, G):
    """J (J^T J)^-1 g_y with J w.r.t. the left tangent of R and g_w = vee(A - A^T), A = G_R R^T, written out."""
    R, t = P[:, :3].astype(np.float64), P[:, 3].astype(np.float64)
    fx, fy = float(K[0, 0]), float(K[1, 1])
    rows = []
    for Xi in X.astype(np.float64):
        rx = R @ Xi
        x, y, z = rx + t
        for d in (np.array([fx / z, 0, -fx * x / z**2]), np.array([0, fy / z, -fy * y / z**2])):
            rows.append(np.concatenate([np.cross(rx, d), d]))
    J = np.array(rows)
    A = G[:, :3] @ R.T
    g = np.array([A[2, 1] - A[1, 2], A[0, 2] - A[2, 0], A[1, 0] - A[0, 1], *G[:, 3]])
    return (J @ np.linalg.solve(J.T @ J, g)).reshape(-1, 2)


def test_oracle_equals_closed_form():
    X, K, P = _cases(12)
    G = np.random.default_rng(1).normal(size=P.shape)
    got = PG.pnp_grad(X, K, P, G, 12)
    for i in range(len(X)):
        ref = _closed_form(X[i], K, P[i], G[i])
        assert np.abs(got[i] - ref).max() <= 1e-10 * np.abs(ref).max(), i


def test_oracle_equals_finite_differences_of_an_lm_solve_at_zero_residual():
    """At zero residual the fast formula is the exact derivative of the least-squares minimum."""
    from scipy.optimize import least_squares

    X, K, P = _cases(3, seed=2)
    G = np.random.default_rng(3).normal(size=P.shape)
    fx, fy, cx, cy = float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2])
    for i in range(len(X)):
        Xd = X[i].astype(np.float64)
        R0, t0 = P[i, :, :3].astype(np.float64), P[i, :, 3].astype(np.float64)
        uv0 = _project(Xd, K.astype(np.float64), R0, t0)
        y0 = np.concatenate([_rotvec(R0), t0])

        def solve(uv):
            def res(y):
                c = Xd @ _rotmat(y[:3]).T + y[3:]
                return np.stack([fx * c[:, 0] / c[:, 2] + cx - uv[:, 0], fy * c[:, 1] / c[:, 2] + cy - uv[:, 1]], 1).ravel()

            y = least_squares(res, y0, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15).x
            return np.concatenate([_rotmat(y[:3]), y[3:, None]], 1)

        R_star = solve(uv0)  # the LM minimum of the exact projections: the pose itself
        fd = np.zeros_like(uv0)
        eps = 1e-3
        for k in range(uv0.size):
            up, um = uv0.copy(), uv0.copy()
            up.flat[k] += eps
            um.flat[k] -= eps
            fd.flat[k] = ((solve(up) - solve(um)) * G[i]).sum() / (2 * eps)
        ref = PG.pnp_grad(Xd[None], K, R_star[None], G[i][None], 12)[0]
        assert np.abs(fd - ref).max() <= 1e-5 * np.abs(ref).max(), (i, np.abs(fd - ref).max(), np.abs(ref).max())


def test_rvec_form_chained_through_rodrigues_equals_the_rt_form():
    X, K, P = _cases(8, seed=4)
    rng = np.random.default_rng(5)
    G12 = rng.normal(size=P.shape)
    poses6, grads6, poses12 = [], [], []
    for i in range(len(X)):
        r = _rotvec(P[i, :, :3])
        if i == 0:
            r = r / np.linalg.norm(r) * 1e-3  # small angle: the series branches
        if i == 1:
            r = r / np.linalg.norm(r) * 3.1  # close to pi
        y = torch.tensor(np.concatenate([r, P[i, :, 3]]), dtype=torch.float64, requires_grad=True)
        Rt = torch.cat([PG.rodrigues(y[:3]), y[3:, None]], 1)
        (Rt * torch.from_numpy(G12[i])).sum().backward()
        poses6.append(y.detach().numpy())
        grads6.append(y.grad.numpy())
        poses12.append(Rt.detach().numpy())
    a = PG.pnp_grad(X, K, np.array(poses6), np.array(grads6), 6)
    b = PG.pnp_grad(X, K, np.array(poses12), G12, 12)
    assert np.abs(a - b).max() <= 1e-9 * np.abs(b).max()


def test_flipped_pose_gives_the_negated_gradient_and_guards_give_zero():
    X, K, P = _cases(4, seed=6)
    G = np.random.default_rng(7).normal(size=P.shape)
    a = PG.pnp_grad(X, K, P, G, 12)
    b = PG.pnp_grad(X, K, -P, G, 12)
    assert np.abs(a).max() > 0
    assert np.abs(a + b).max() <= 1e-12 * np.abs(a).max()
    Pz = P.copy()
    Pz[0] = 0  # dead object
    Pz[1, :, 3] *= -1  # behind the camera, not flipped (det R > 0)
    Xc = X.copy()
    Xc[2] = np.linspace(0, 1, X.shape[1])[:, None] * np.array([50, -20, 30], F)  # collinear keypoints
    got = PG.pnp_grad(Xc, K, Pz, G, 12)
    assert not got[:3].any() and np.abs(got[3] - a[3]).max() == 0


# ------------------------------------------------------------------------------------------------------------- GPU


def _raw_backward(lib, hdl, X, K, P, G, form):
    n, vn = X.shape[:2]
    t = [torch.from_numpy(np.array(v, F, order="C")).cuda() for v in (X, np.broadcast_to(K, (n, 3, 3)), P, G)]
    out = torch.full((n, vn, 2), float("nan"), device="cuda")
    rc = lib.casa_pnp_backward(hdl, n, vn, *(v.data_ptr() for v in t[:3]), form, t[3].data_ptr(), out.data_ptr(), None)
    assert rc == 0, lib.casa_last_error()
    launches = C.c_int64()
    lib.casa_last_launches(hdl, C.byref(launches))
    torch.cuda.synchronize()
    return out.cpu().numpy(), launches.value


def _per_object_close(got, ref, tol=1e-5):
    for i in range(len(ref)):
        scale = np.abs(ref[i]).max()
        assert np.abs(got[i] - ref[i]).max() <= tol * scale, (i, np.abs(got[i] - ref[i]).max(), scale)


@pytest.mark.gpu
@pytest.mark.parametrize("form", [12, 6])
@pytest.mark.parametrize("vn", [6, 9, 12, 16])
def test_gpu_kernel_matches_oracle(cuda_lib, vn, form):
    from casapose_b200 import _lib

    n = 4 * 9 + 3  # several blocks of 4 objects and a ragged last block
    X, K, P = _cases(n, vn=vn, seed=vn + form)
    rng = np.random.default_rng(vn)
    G = rng.normal(size=P.shape).astype(F)
    P[5] = -P[5]  # flipped (t_z < 0 in the reference's convention, det R < 0)
    P[7] = 0  # dead object
    P[9, :, 3] = -P[9, :, 3]  # behind the camera, det R > 0
    X[11] = (np.linspace(-1, 1, vn)[:, None] * np.array([60, -25, 40])).astype(F)  # collinear keypoints
    if form == 12:
        poses, grads = P, G
    else:
        poses = np.zeros((n, 6), F)
        for i in range(n):
            if P[i].any():
                s = -1.0 if np.linalg.det(P[i, :, :3]) < 0 else 1.0  # the rvec form has no flip
                poses[i] = np.concatenate([_rotvec(s * P[i, :, :3]), s * P[i, :, 3]])
        poses[3, :3] = poses[3, :3] / np.linalg.norm(poses[3, :3]) * 1e-3  # small angle: series branch
        grads = rng.normal(size=(n, 6)).astype(F)
    hdl = _lib.handle(0)
    got, launches = _raw_backward(cuda_lib, hdl, X, K, poses, grads, form)
    assert launches == 1
    assert np.isfinite(got).all()
    ref = PG.pnp_grad(X, K, poses, grads, form)
    for i in (7, 9, 11):
        assert not got[i].any() and not ref[i].any(), i
    assert np.abs(ref).max(axis=(1, 2)).astype(bool).sum() == n - 3
    _per_object_close(got, ref)
    if form == 12:  # the flip: the negated gradient of the un-flipped pose
        un, _ = _raw_backward(cuda_lib, hdl, X[5:6], K, -P[5:6], G[5:6], 12)
        _per_object_close(got[5:6], -un)


@pytest.mark.gpu
def test_gpu_entry_point_validates_and_is_a_noop_for_zero_objects(cuda_lib):
    from casapose_b200 import _lib

    hdl = _lib.handle(0)
    X, K, P = _cases(2)
    t = [torch.from_numpy(np.ascontiguousarray(v, F)).cuda() for v in (X, np.broadcast_to(K, (2, 3, 3)), P, P)]
    out = torch.zeros((2, 9, 2), device="cuda")
    args = [v.data_ptr() for v in t]
    assert cuda_lib.casa_pnp_backward(hdl, 2, 9, args[0], args[1], args[2], 7, args[3], out.data_ptr(), None) == -1
    assert b"pose_form" in cuda_lib.casa_last_error()
    assert cuda_lib.casa_pnp_backward(hdl, 2, 5, args[0], args[1], args[2], 12, args[3], out.data_ptr(), None) == -1
    assert cuda_lib.casa_pnp_backward(hdl, -1, 9, args[0], args[1], args[2], 12, args[3], out.data_ptr(), None) == -1
    assert cuda_lib.casa_pnp_backward(hdl, 2, 9, args[0], args[1], args[2], 12, None, out.data_ptr(), None) == -1
    assert cuda_lib.casa_pnp_backward(hdl, 0, 9, args[0], args[1], args[2], 12, args[3], out.data_ptr(), None) == 0


@pytest.mark.gpu
def test_gpu_pnp_cuda_through_autograd(cuda_lib):
    from casapose_b200.pose_estimation.ransac_voting import pnp_cuda

    n = 10
    X, K, P = _cases(n, seed=11)
    rng = np.random.default_rng(12)
    uv = np.stack([_project(X[i], K, P[i, :, :3], P[i, :, 3]) for i in range(n)]).astype(F)
    uv += rng.normal(scale=0.5, size=uv.shape).astype(F)
    cams = np.broadcast_to(K, (n, 3, 3))
    p2 = torch.from_numpy(uv).cuda().requires_grad_()
    poses = pnp_cuda(p2, X, cams)
    plain = pnp_cuda(p2.detach(), X, cams)
    assert poses.grad_fn is not None and torch.equal(poses.detach(), plain)
    G = torch.from_numpy(rng.normal(size=(n, 3, 4)).astype(F)).cuda()
    (poses * G).sum().backward()
    ref = PG.pnp_grad(X, K, plain.cpu().numpy(), G.cpu().numpy(), 12)
    _per_object_close(p2.grad.cpu().numpy(), ref)
    with pytest.raises(ValueError):
        pnp_cuda(p2, X, cams, np.zeros((n, 10), F))


def _pnp_scene(b=3, h=120, w=160, ids=(1, 5, 6), seed=0):
    """Seeded frames: (y,x) keypoints with noise, seg logits (one object made unavailable), [b,oc,1,vn,3], cameras."""
    d = synthetic.make_frames(b, h, w, ids, variant="easy", with_logits=True)
    rng = np.random.default_rng(seed)
    pts = d["kp2d_gt"][..., ::-1] + rng.normal(scale=0.7, size=d["kp2d_gt"].shape)
    seg = d["seg_logits"].copy()
    seg[1, :, :, 2] = -50.0  # object 1 of image 1 has no pixel: available = 0
    kp3 = np.broadcast_to(d["keypoints_3d"][None, :, None], (b, len(ids), 1, 9, 3)).astype(F)
    cams = np.broadcast_to(d["camera"], (b, 3, 3)).astype(F)
    return np.ascontiguousarray(pts, F), seg, np.ascontiguousarray(kp3), np.ascontiguousarray(cams)


def _poses_pnp_oracle(poses, G, kp3, cam, b, oc):
    """dL/d points_estimated [b,oc,vn,2] (y,x) for L = sum(poses * G), poses = the returned [b,oc,1,3,4]."""
    n = b * oc
    g = PG.pnp_grad(kp3.reshape(n, -1, 3), cam, poses.reshape(n, 12), G.reshape(n, 12), 12)  # (x,y)
    return g.reshape(b, oc, -1, 2)[..., ::-1]


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["cuda", "cv2"])
def test_gpu_poses_pnp_through_autograd(cuda_lib, backend):
    from casapose_b200.pose_estimation import poses_pnp

    pts, seg, kp3, cams = _pnp_scene()
    b, oc = pts.shape[:2]
    pe = torch.from_numpy(pts).cuda().requires_grad_()
    poses = poses_pnp(pe, seg, kp3, cams, oc, pnp_backend=backend)
    plain = poses_pnp(pe.detach(), seg, kp3, cams, oc, pnp_backend=backend)
    assert poses.grad_fn is not None and poses.device.type == "cpu" and poses.dtype == torch.float32
    assert torch.equal(poses.detach(), plain)
    assert not plain[1, 1].any()
    G = torch.from_numpy(np.random.default_rng(1).normal(size=poses.shape).astype(F))
    (poses * G).sum().backward()
    got = pe.grad.cpu().numpy()
    ref = _poses_pnp_oracle(plain.numpy(), G.numpy(), kp3, cams[0], b, oc)
    assert not got[1, 1].any()
    _per_object_close(got.reshape(b * oc, -1, 2), ref.reshape(b * oc, -1, 2))
    with pytest.raises(ValueError):
        poses_pnp(pe.detach().cpu().requires_grad_(), seg, kp3, cams, oc, pnp_backend=backend)


@pytest.mark.gpu
@pytest.mark.parametrize("batched", [False, True])
def test_gpu_bpnp_fast_through_autograd(cuda_lib, batched):
    from casapose_b200.pose_estimation.bpnp_layers import BPNP_fast

    pts, _, kp3, cams = _pnp_scene(seed=3)
    b, oc = pts.shape[:2]
    xy = np.ascontiguousarray(pts[..., ::-1])
    if batched:
        p2, p3 = xy, kp3[:, :, 0]
    else:
        p2, p3 = xy.reshape(b * oc, 9, 2), kp3[:, :, 0].reshape(b * oc, 9, 3)
    layer = BPNP_fast(name="BPNP")
    t2 = torch.from_numpy(np.ascontiguousarray(p2)).cuda().requires_grad_()
    out = layer([t2, p3, cams[0]])
    plain = layer([p2, p3, cams[0]])
    assert out.grad_fn is not None and out.is_cuda and tuple(out.shape) == plain.shape
    assert np.array_equal(out.detach().cpu().numpy(), plain)
    G = np.random.default_rng(4).normal(size=plain.shape).astype(F)
    (out * torch.from_numpy(G).cuda()).sum().backward()
    ref = PG.pnp_grad(p3.reshape(b * oc, 9, 3), cams[0], plain.reshape(-1, 6), G.reshape(-1, 6), 6)
    _per_object_close(t2.grad.cpu().numpy().reshape(b * oc, 9, 2), ref)


def _mask_singular(g, seg, direct, conf, keep_rank_one=(), **kw):
    """Zero the incoming gradient of every (image, class, keypoint) whose 2x2 system is numerically singular
    (a component of a few pixels, an empty class): the derivative of an ill-conditioned pseudo-inverse amplifies
    last-ulp differences by its condition number and is not a meaningful comparison."""
    _, dbg = L.coord_ls_voting_weighted(seg, direct, conf, return_debug=True, **kw)
    sv = np.linalg.svd(dbg["R"], compute_uv=False)  # [b,oc,vn,2]
    bad = ~(sv[..., 1] > 1e-4 * sv[..., 0])
    for k in keep_rank_one:
        bad[:, :, k] &= sv[:, :, k, 1] != 0  # exactly rank one on both sides: the constant-rank formula applies
    g = g.copy()
    g[bad] = 0
    return g


def _check(a, ref, what):
    scale = np.abs(ref).max()
    err = np.abs(a - ref).max()
    assert err <= 2e-4 * scale, "%s: max err %.3g of scale %.3g" % (what, err, scale)
    assert np.array_equal(a != 0, ref != 0) or np.abs(a[(a != 0) != (ref != 0)]).max() <= 1e-6 * scale


@pytest.mark.gpu
def test_gpu_training_chain_from_pose_to_direct_and_confidence(cuda_lib):
    """CoordLSVotingWeighted -> poses_pnp(pnp_backend="cuda") -> sum(poses * G): direct.grad and w.grad against the PnP
    gradient oracle at the GPU's poses composed with the LS-layer gradient oracle."""
    from casapose_b200.pose_estimation import CoordLSVotingWeighted, poses_pnp
    from oracle import ls_voting_grad as LG

    b, h, w, ids = 2, 120, 160, (1, 5, 6)
    d = synthetic.make_frames(b, h, w, ids, variant="easy", with_logits=True)
    seg, direct, conf = d["seg_logits"], d["vertex"].reshape(b, h, w, 18).copy(), d["conf_logits"]
    oc = len(ids)
    kp3 = np.ascontiguousarray(np.broadcast_to(d["keypoints_3d"][None, :, None], (b, oc, 1, 9, 3)), F)
    cams = np.ascontiguousarray(np.broadcast_to(d["camera"], (b, 3, 3)), F)
    # objects with a numerically singular keypoint system get no incoming gradient (the masking of test_ls_backward.py)
    regular = _mask_singular(np.ones((b, oc, 9, 2), F), seg, direct, conf).all(axis=(2, 3))
    layer = CoordLSVotingWeighted("ls", oc + 1)
    ts = torch.from_numpy(seg).cuda()
    td = torch.from_numpy(direct).cuda().requires_grad_()
    tw = torch.from_numpy(conf).cuda().requires_grad_()
    coords = layer([ts, td, tw])
    poses = poses_pnp(coords, ts, kp3, cams, oc, pnp_backend="cuda")
    posed = poses.detach().reshape(b, oc, 12).abs().sum(-1).numpy() > 0
    assert (regular & posed).sum() >= 4
    G = np.random.default_rng(2).normal(size=(b, oc, 1, 3, 4)).astype(F) * (regular & posed)[:, :, None, None, None]
    (poses * torch.from_numpy(G)).sum().backward()
    g_coords = _poses_pnp_oracle(poses.detach().numpy(), G, kp3, d["camera"], b, oc)
    _, rd, rw = LG.ls_vote_with_grads(seg, direct, conf, np.ascontiguousarray(g_coords))
    gd, gw = td.grad.cpu().numpy(), tw.grad.cpu().numpy()
    assert np.isfinite(gd).all() and np.isfinite(gw).all()
    _check(gd, rd, "grad_direct")
    _check(gw, rw, "grad_conf")
