"""The LS path kept on the device: casa_ls_vote_counts (the LS call that also counts poses_pnp's available objects,
pose_evaluation.py:183-190), DeviceEvaluator.ls_poses (poses_pnp on the device) and DeviceEvaluator.evaluate_ls
(evaluate_pose_estimates on the device).

The bars: the counts equal the numpy restatement `hot_counts` (tests/test_oracle_hot_counts.py); every other output of the counting call is bit-identical to
casa_ls_vote_typed's; ls_poses equals poses_pnp(..., pnp_backend="cuda") in value and gradient; evaluate_ls equals
evaluate_pose_estimates(..., metric_backend="cuda"); and neither leaves the device more than the one read-back."""
import ctypes as C
import warnings

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from casapose_b200 import synthetic  # noqa: E402
from oracle import ls_voting_np as L  # noqa: E402

from .test_gpu_ls_sweep import _offset, blocks_scene, overflow_scene  # noqa: E402
from .test_oracle_hot_counts import hot_counts  # noqa: E402

pytestmark = pytest.mark.gpu
F = np.float32
MODES = {"plain": dict(), "filt-sigm": dict(filter_estimates=True, sigmoid_weights=True),
         "filt-second": dict(filter_estimates=True, output_second_largest_component=True)}
TIES = (2, 3, 9, 10, 11)


# ----------------------------------------------------------------------------------------------------------- scenes
def _fields(rng, b, h, w, vn):
    return rng.normal(size=(b, h, w, 2 * vn)).astype(F), rng.normal(size=(b, h, w, vn)).astype(F)


def tie_scene(nc=14, vn=3, seed=11):
    """Two 40 x 60 images, background except a band of one-hot object blocks and one 4 x 6 patch per k in TIES where
    classes 1..k tie exactly at the maximum (hot = 1/k: 1/10 is 0.1f, not above it).  Image 1 has no ties and only
    some classes.  Few enough listed pixels that the first attempt's h*w slots hold them."""
    rng = np.random.default_rng(seed)
    b, h, w = 2, 40, 60
    lab = np.zeros((b, h, w), np.int64)
    lab[0, 30:40] = np.kron(rng.integers(1, nc, size=(1, 6)), np.ones((10, 10), np.int64))
    lab[1, 0:10, 0:30] = 3
    lab[1, 20:30, 30:60] = nc - 1
    seg = rng.uniform(-1, 0, (b, h, w, nc)).astype(F)
    np.put_along_axis(seg, lab[..., None], rng.uniform(1, 2, (b, h, w, 1)).astype(F), -1)
    for j, k in enumerate(TIES):
        patch = seg[0, 2:6, 2 + 10 * j:8 + 10 * j]
        patch[...] = F(-1.0)
        patch[..., 1:k + 1] = F(0.5)
    return (seg,) + _fields(rng, b, h, w, vn)


def random_scene(b=2, h=33, w=47, nc=9, vn=4, seed=12):
    """One-hot logits (three quarters background), and on a fifth of the pixels three random classes with logits of unit
    spread after the 1e6 scale: soft probabilities on both sides of 0.1, at most three listed classes per pixel.  Pixels
    whose hot lies within 1e-6 of 0.1 (where expf and the summation order are not pinned) are made background."""
    rng = np.random.default_rng(seed)
    lab = np.where(rng.random((b, h, w)) < 0.75, 0, rng.integers(1, nc, (b, h, w)))
    seg = rng.uniform(-1, 0, (b, h, w, nc)).astype(F)
    np.put_along_axis(seg, lab[..., None], rng.uniform(1, 2, (b, h, w, 1)).astype(F), -1)
    soft = rng.random((b, h, w)) < 0.2
    rows = np.full((int(soft.sum()), nc), -1.0, F)
    pick = np.argsort(rng.random(rows.shape), axis=1)[:, :3]
    np.put_along_axis(rows, pick, (rng.normal(size=pick.shape) * 1e-6).astype(F), 1)
    seg[soft] = rows
    near = (np.abs(L.hard_softmax_f32(seg) - F(0.1)) < 1e-6).any(-1)
    seg[near] = F(-1.0)
    seg[near, 0] = F(1.0)
    return (seg,) + _fields(rng, b, h, w, vn)


def _blocks(*args, **kw):
    return blocks_scene(*args, **kw)[:3]


SCENES = {  # name -> (builder, overflows the first attempt's lists)
    "nc2-partial-tile": (lambda: _blocks(2, 37, 29, 2, 1, 8, 8, seed=1), False),      # h*w = 1073
    "nc9": (lambda: _blocks(2, 60, 80, 9, 9, 10, 16, seed=2), False),                 # the specialised k_ls_classify<9>
    "nc9-b1": (lambda: _blocks(1, 48, 64, 9, 9, 8, 8, seed=3), False),
    "nc9-b3-absent": (lambda: _blocks(3, 40, 48, 9, 9, 8, 8, seed=4, per_image=3), False),
    "nc14": (lambda: _blocks(2, 24, 44, 14, 16, 6, 11, seed=5), False),
    "nc33": (lambda: _blocks(2, 16, 24, 33, 2, 4, 6, seed=6), False),
    "ties-nc14": (tie_scene, False),
    "random-nc9": (random_scene, False),
    "random-nc14": (lambda: random_scene(nc=14, seed=13), False),
    "overflow-retry": (lambda: overflow_scene()[:3], True),
}


# ---------------------------------------------------------------------------------------------------------- helpers
@pytest.fixture(scope="module")
def Layer(cuda_lib):
    assert torch.cuda.is_available()
    from casapose_b200.pose_estimation import CoordLSVotingWeighted

    return CoordLSVotingWeighted


def _cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _bits(t):
    return t.view(torch.int64 if t.dtype == torch.float64 else torch.int32) if t.is_floating_point() else t


def _same(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _offset_elem(t):
    """A contiguous copy of `t` that starts one element into its allocation."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


def _clear_sticky():
    """casa_sync reports every call since the last one, including synchronous calls that already raised."""
    from casapose_b200 import _lib

    torch.cuda.synchronize()
    try:
        _lib.sync(0)
    except _lib.CasaError:
        pass


def _compare(layer, x, check_finite=True):
    """The counting call against casa_ls_vote_typed: graph-replayed and debug forms, every output bit for bit.
    Returns the counts."""
    want = layer(x, check_finite=check_finite)
    got, cnt = layer(x, check_finite=check_finite, return_counts=True)
    want_d, dbg_w = layer(x, return_debug=True, check_finite=check_finite)
    got_d, cnt_d, dbg_g = layer(x, return_debug=True, check_finite=check_finite, return_counts=True)
    torch.cuda.synchronize()
    assert _same(want, got) and _same(want_d, got_d)
    assert set(dbg_w) == set(dbg_g) and all(_same(dbg_w[k], dbg_g[k]) for k in dbg_w)
    assert cnt.dtype == torch.int32 and cnt.is_cuda and torch.equal(cnt, cnt_d)
    return cnt


# ------------------------------------------------------------------------------------------------ counts and outputs
def test_scenes_deliver_what_they_promise():
    seg, _, _ = tie_scene()
    hot = L.hard_softmax_f32(seg)
    for j, k in enumerate(TIES):
        patch = hot[0, 2:6, 2 + 10 * j:8 + 10 * j, 1:k + 1]
        assert (patch == F(1.0) / F(k)).all(), k
    assert F(1.0) / F(10) == F(0.1) and F(1.0) / F(9) > F(0.1)
    cnt = hot_counts(seg)
    assert (cnt[1] == 0).sum() >= 5  # classes absent from image 1
    for nc in (9, 14):
        seg, _, _ = random_scene(nc=nc)
        hot = L.hard_softmax_f32(seg)[..., 1:]
        assert not (np.abs(hot - F(0.1)) < 1e-6).any()
        assert ((hot > 0.1) & (hot < 0.12)).sum() > 20 and ((hot > 0.08) & (hot < 0.1)).sum() > 20  # both sides of 0.1
    for name, (make, overflows) in SCENES.items():
        seg = make()[0]
        b, h, w, nc = seg.shape
        assert ((L.hard_softmax_f32(seg)[..., 1:] != 0).sum(axis=(1, 2, 3)).max() > h * w) == overflows, name


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("scene", list(SCENES))
def test_counts_equal_the_oracle_and_nothing_else_moves(Layer, scene, mode):
    make, overflows = SCENES[scene]
    seg, direct, conf = make()
    layer = Layer("ls", seg.shape[3], num_points=conf.shape[3], **MODES[mode])
    want = hot_counts(seg)
    x = _cuda(seg, direct, conf)
    for check_finite in ((True,) if overflows else (True, False)):  # an overflow is retried only by the checking call
        cnt = _compare(layer, x, check_finite)
        assert np.array_equal(cnt.cpu().numpy(), want), check_finite
    if not overflows:
        _clear_sticky()
    # seg 4 bytes past alignment: scalar staging in k_ls_classify
    if scene in ("nc9", "nc14", "random-nc9", "ties-nc14"):
        xm = [_offset(t) for t in x]
        assert np.array_equal(_compare(layer, xm).cpu().numpy(), want)


def test_counts_and_outputs_on_four_lanes(Layer):
    """casa_set_async(h, 4), calls in flight on four lanes: after casa_join each call's counts and keypoints are those of
    the synchronous calls."""
    from casapose_b200 import _lib

    scenes = [SCENES[n][0]() for n in ("nc9", "random-nc9", "nc9-b1", "ties-nc14", "nc14", "nc33")]
    layers = [Layer("ls", s[0].shape[3], num_points=s[2].shape[3], filter_estimates=True) for s in scenes]
    inputs = [_cuda(*s) for s in scenes]
    want = [layer(x, return_counts=True) for layer, x in zip(layers, inputs)]
    torch.cuda.synchronize()
    _lib.set_async(0, 4)
    try:
        got = [layer(x, check_finite=False, return_counts=True) for _ in range(2) for layer, x in zip(layers, inputs)]
        _lib.join(0)
        got = [(a.clone(), c.clone()) for a, c in got]
        _lib.sync(0)
    finally:
        _lib.set_async(0, 0)
    torch.cuda.synchronize()
    for i, (a, c) in enumerate(got):
        wa, wc = want[i % len(want)]
        assert _same(wa, a) and torch.equal(wc, c), i
        assert np.array_equal(c.cpu().numpy(), hot_counts(scenes[i % len(scenes)][0])), i


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16], ids=["f16", "bf16"])
@pytest.mark.parametrize("ids", [(1, 5, 6), synthetic.CONFIG_8_IDS], ids=["nc4", "nc9"])
def test_16_bit_counts_equal_the_upcast_call(Layer, dt, ids):
    d = synthetic.make_frames(2, 120, 160, ids, variant="easy", with_logits=True)
    x = [t.to(dt) for t in _cuda(d["seg_logits"], d["vertex"].reshape(2, 120, 160, 18), d["conf_logits"])]
    layer = Layer("ls", len(ids) + 1, num_points=9, filter_estimates=True)
    for xs in (x, [_offset_elem(t) for t in x]):  # one element (2 bytes) past alignment: the scalar staging
        want, wc = layer([t.float() for t in xs], return_counts=True)
        got, gc = layer(xs, return_counts=True)
        torch.cuda.synchronize()
        assert _same(want, got) and torch.equal(wc, gc)
        assert np.array_equal(gc.cpu().numpy(), hot_counts(xs[0].float().cpu().numpy()))


def test_counts_need_a_buffer(Layer):
    from casapose_b200 import _lib
    from casapose_b200._carrier import current_stream_ptr

    seg, direct, conf = SCENES["nc9"][0]()
    b, h, w, nc = seg.shape
    layer = Layer("ls", nc, num_points=9)
    x = _cuda(seg, direct, conf)
    out = torch.empty((b, nc - 1, 9, 2), device="cuda")
    p = layer._params(b, h, w, nc, 9, True)
    hdl = _lib.handle(0, current_stream_ptr(x[0].device))
    rc = _lib.lib().casa_ls_vote_counts(hdl, C.byref(p), 0, *[t.data_ptr() for t in x], out.data_ptr(), None, None,
                                        current_stream_ptr(x[0].device))
    assert rc != 0 and b"hot_counts" in _lib.lib().casa_last_error()


def test_counts_on_the_autograd_path_are_not_differentiable(Layer):
    seg, direct, conf = SCENES["nc9"][0]()
    layer = Layer("ls", seg.shape[3], num_points=9, filter_estimates=True)
    s, d, c = _cuda(seg, direct, conf)
    d.requires_grad_(True)
    coords, cnt = layer([s, d, c], return_counts=True)
    assert coords.requires_grad and not cnt.requires_grad
    assert np.array_equal(cnt.cpu().numpy(), hot_counts(seg))
    g = torch.randn_like(coords)
    (coords * g).sum().backward()
    gd, _ = layer.backward([s, d.detach(), c], g)
    assert torch.equal(d.grad, gd)


# ---------------------------------------------------------------------------------------------------- ls_poses / eval
def _pipeline(b=1, variant="clean"):
    from casapose_b200.pose_estimation import CoordLSVotingWeighted, DeviceEvaluator
    from tests.test_gpu_pipeline import _inputs

    d, cams, offsets, kp3, target_seg, poses_gt, diam = _inputs(b=b, variant=variant)
    h, w = d["seg_logits"].shape[1:3]
    x = _cuda(d["seg_logits"], d["vertex"].reshape(b, h, w, 18), d["conf_logits"])
    layer = CoordLSVotingWeighted("ls", 9, num_points=9, filter_estimates=True)
    ev = DeviceEvaluator(kp3[0, :, 0], cams[0], diam[0])
    return x, layer, ev, cams, kp3, target_seg, poses_gt, diam


@pytest.mark.parametrize("b,variant", [(1, "clean"), (2, "easy")])
def test_ls_poses_equal_poses_pnp_cuda(Layer, b, variant):
    from casapose_b200.pose_estimation import poses_pnp

    x, layer, ev, cams, kp3, *_ = _pipeline(b, variant)
    poses, coords = ev.ls_poses(layer, *x)
    assert poses.is_cuda and coords.is_cuda and tuple(poses.shape) == (b, 8, 1, 3, 4)
    want_c = layer(x)
    want = poses_pnp(want_c, x[0], kp3, cams, 8, min_num=20, pnp_backend="cuda")
    assert torch.equal(coords, want_c) and torch.equal(poses.cpu(), want)
    assert poses.abs().sum() > 0
    with pytest.raises(ValueError):
        ev.ls_poses(Layer("ls", 9, num_points=8), *x)
    with pytest.raises(ValueError):
        ev.ls_poses(Layer("ls", 10, num_points=9), *x)


def test_ls_poses_on_the_golden_inputs(Layer):
    import ast

    from casapose_b200.pose_estimation import DeviceEvaluator
    from oracle import golden_inputs as GI
    from tests.test_golden_oracle import load

    g = load("poses_pnp")
    gen = ast.literal_eval(str(g["gen"]))
    d, cams, offsets, kp3, target_seg, poses_gt, diam = GI.pose_inputs(**gen)
    b, h, w, oc = gen["b"], gen["h"], gen["w"], len(gen["ids"])
    layer = Layer("ls", oc + 1, num_points=9, filter_estimates=True)
    ev = DeviceEvaluator(np.asarray(kp3).reshape(-1, oc, 1, 9, 3)[0, :, 0], np.asarray(cams).reshape(-1, 3, 3)[0],
                         np.ones(oc, F))
    poses, _ = ev.ls_poses(layer, *_cuda(d["seg_logits"], d["vertex"].reshape(b, h, w, 18), d["conf_logits"]))
    poses = poses.cpu().numpy()
    assert np.array_equal(poses.any(axis=(2, 3, 4)), g["poses"].any(axis=(2, 3, 4))), "availability mask differs"
    assert np.abs(poses[..., :3] - g["poses"][..., :3]).max() < 2e-2
    assert np.abs(poses[..., 3] - g["poses"][..., 3]).max() < 5.0


NAMES = ["valid_2d", "valid_3d", "valid_pose_count", "false_positive_mask", "err_2d", "err_3d", "missing_object",
         "false_positive_pose"]
EXACT = ["valid_2d", "valid_3d", "valid_pose_count", "false_positive_mask", "missing_object", "false_positive_pose"]


@pytest.mark.parametrize("b,variant", [(1, "clean"), (2, "easy")])
def test_evaluate_ls_equals_evaluate_pose_estimates(Layer, b, variant):
    from casapose_b200.pose_estimation import evaluate_pose_estimates, poses_pnp

    x, layer, ev, cams, kp3, target_seg, poses_gt, diam = _pipeline(b, variant)
    tgt = torch.from_numpy(target_seg).cuda()
    stats, poses, coords = ev.evaluate_ls(layer, *x, tgt, torch.from_numpy(poses_gt).cuda())
    want_c = layer(x)
    assert torch.equal(coords, want_c)
    ref = {}
    for pnp_backend, metric_backend in (("cuda", "cuda"), ("cv2", "numpy")):
        p = poses_pnp(want_c, x[0], kp3, cams, 8, min_num=20, pnp_backend=pnp_backend)
        s, _, _ = evaluate_pose_estimates(want_c, p[:, :, 0], poses_gt, tgt, kp3, cams, diam, metric_backend=metric_backend)
        ref[pnp_backend] = dict(zip(NAMES, [np.atleast_1d(np.asarray(v, F)) for v in s]))
        if pnp_backend == "cuda":
            assert torch.equal(poses.cpu(), p)
    for n in NAMES:
        got, want = stats[n], ref["cuda"][n]
        if n in EXACT:
            assert np.array_equal(got, want), n
        else:
            assert np.allclose(got, want, rtol=1e-6, atol=1e-5), n
    if variant == "clean":  # the verdicts of the host path (OpenCV PnP, numpy metric); the two PnP solvers agree only
        # within their tolerance, and on the easy scene one valid_2d verdict differs between them
        for n in ("valid_2d", "valid_3d", "valid_pose_count", "missing_object", "false_positive_pose"):
            assert np.array_equal(stats[n], ref["cv2"][n]), n
    assert stats["valid_pose_count"].sum() > 0 and not stats["false_positive_mask"].any()


def test_ls_poses_gradients_equal_the_poses_pnp_chain(Layer):
    from casapose_b200.pose_estimation import poses_pnp

    x, layer, ev, cams, kp3, *_ = _pipeline(2, "easy")
    seg = x[0]
    G = torch.from_numpy(np.random.default_rng(5).normal(size=(2, 8, 1, 3, 4)).astype(F))
    d1, w1 = x[1].clone().requires_grad_(True), x[2].clone().requires_grad_(True)
    poses, coords = ev.ls_poses(layer, seg, d1, w1)
    assert poses.requires_grad and coords.requires_grad
    (poses * G.cuda()).sum().backward()
    d2, w2 = x[1].clone().requires_grad_(True), x[2].clone().requires_grad_(True)
    p2 = poses_pnp(layer([seg, d2, w2]), seg, kp3, cams, 8, min_num=20, pnp_backend="cuda")
    (p2 * G).sum().backward()
    assert torch.equal(poses.detach().cpu(), p2.detach())
    assert torch.equal(d1.grad, d2.grad) and torch.equal(w1.grad, w2.grad)
    assert d1.grad.abs().sum() > 0 and w1.grad.abs().sum() > 0


# ------------------------------------------------------------------------------------------------- no host round-trips
def test_ls_poses_does_not_synchronise(Layer):
    x, layer, ev, *_ = _pipeline(2, "easy")
    ev.ls_poses(layer, *x, check_finite=False)  # first call: graphs and tables built outside the checked window
    _clear_sticky()
    torch.cuda.set_sync_debug_mode("error")
    try:
        poses, coords = ev.ls_poses(layer, *x, check_finite=False)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    want, _ = ev.ls_poses(layer, *x)
    assert torch.equal(poses, want)


def test_evaluate_ls_reads_back_once(Layer):
    x, layer, ev, cams, kp3, target_seg, poses_gt, diam = _pipeline(2, "easy")
    tgt, gt = torch.from_numpy(target_seg).cuda(), torch.from_numpy(poses_gt).cuda()
    want, _, _ = ev.evaluate_ls(layer, *x, tgt, gt)
    _clear_sticky()
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            stats, _, _ = ev.evaluate_ls(layer, *x, tgt, gt, check_finite=False)
        finally:
            torch.cuda.set_sync_debug_mode(0)
    syncs = [str(w.message) for w in caught if "synchroniz" in str(w.message)]
    assert len(syncs) == 1, syncs
    for n in NAMES:
        assert np.array_equal(stats[n], want[n]), n


def test_evaluate_ls_raises_on_a_non_finite_result_without_check_finite(Layer):
    from casapose_b200._lib import CasaError

    x, _, ev, cams, kp3, target_seg, poses_gt, diam = _pipeline(1, "clean")
    layer = Layer("ls", 9, num_points=9)  # no component filter: every listed pixel has a weight
    direct = x[1].clone()
    listed = torch.nonzero(x[0].argmax(-1)[0] == 1)[0]  # a pixel of class 1
    direct[0, int(listed[0]), int(listed[1]), 0] = float("nan")
    _clear_sticky()
    with pytest.raises(CasaError):
        ev.evaluate_ls(layer, x[0], direct, x[2], torch.from_numpy(target_seg).cuda(), torch.from_numpy(poses_gt).cuda(),
                       check_finite=False)
    # the error was reported once: the handle is clean for the next call
    stats, _, _ = ev.evaluate_ls(layer, *x, torch.from_numpy(target_seg).cuda(), torch.from_numpy(poses_gt).cuda(),
                                 check_finite=False)
    assert stats["valid_pose_count"].sum() > 0
