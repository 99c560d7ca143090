"""GPU parity of CoordLSVotingWeighted (K5/K6) against the numpy oracle: keypoints within 1e-3 px, the
float64 sums to 1e-9 relative, the component selection bit-exact."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from casapose_b200 import synthetic  # noqa: E402
from oracle import ls_voting_np as L  # noqa: E402

pytestmark = pytest.mark.gpu
TOL_PX = 1e-3


@pytest.fixture(scope="module")
def Layer(cuda_lib):
    assert torch.cuda.is_available()
    from casapose_b200.pose_estimation import CoordLSVotingWeighted

    return CoordLSVotingWeighted


def _run(Layer, seg, direct, conf, **kw):
    layer = Layer("ls", seg.shape[3], num_points=conf.shape[3], **kw)
    out, dbg = layer([torch.from_numpy(seg).cuda(), torch.from_numpy(direct).cuda(), torch.from_numpy(conf).cuda()],
                     return_debug=True)
    torch.cuda.synchronize()
    ref, rdbg = L.coord_ls_voting_weighted(seg, direct, conf, num_points=conf.shape[3], return_debug=True, **kw)
    sums = dbg["sums"].cpu().numpy()
    R, q = rdbg["R"], rdbg["q"]
    want = np.stack([R[..., 0, 0], R[..., 0, 1], R[..., 1, 1], q[..., 0], q[..., 1]], axis=-1)
    scale = np.abs(want).max() + 1e-30
    assert np.abs(sums - want).max() <= 1e-7 * scale, np.abs(sums - want).max() / scale
    err = float(np.abs(out.cpu().numpy() - ref).max())
    assert err <= TOL_PX, err
    # the forward call proper (no debug outputs) finds the components over horizontal runs (k_cc_runs) instead of the
    # pixel-level union-find the debug call keeps: same component mask, same tiles -> the same bits
    fast = layer([torch.from_numpy(seg).cuda(), torch.from_numpy(direct).cuda(), torch.from_numpy(conf).cuda()])
    torch.cuda.synchronize()
    assert torch.equal(fast, out), float((fast - out).abs().max())
    return out, dbg, ref, rdbg


@pytest.mark.parametrize("filt", [False, True])
@pytest.mark.parametrize("sigm", [False, True])
def test_ls_layer_matches_oracle(Layer, filt, sigm):
    d = synthetic.make_frames(2, 120, 160, (1, 5, 6), variant="easy", with_logits=True)
    _run(Layer, d["seg_logits"], d["vertex"].reshape(2, 120, 160, 18), d["conf_logits"], filter_estimates=filt,
         sigmoid_weights=sigm)


def test_config1_shape_full_resolution(Layer):
    """BASELINE config 1's post-network part: [1,480,640,9+18+9] -> LS layer with filter_estimates=True."""
    d = synthetic.make_frames(1, 480, 640, synthetic.CONFIG_8_IDS, variant="easy", with_logits=True)
    _run(Layer, d["seg_logits"], d["vertex"].reshape(1, 480, 640, 18), d["conf_logits"], filter_estimates=True)


def test_component_selection_quirks(Layer):
    from tests.test_oracle_ls import _scene

    big, small = (5, 25, 8, 30), (30, 36, 40, 50)
    seg, direct, conf = _scene(boxes=(big, small))
    direct[0, 30:36, 40:50, :] = np.array([0.0, 1.0, 1.0, 0.0], np.float32)
    _, dbg, _, _ = _run(Layer, seg, direct, conf, filter_estimates=True)
    assert int(dbg["selected"][0, 0]) == 5 * 56 + 8  # root = first pixel of the big blob
    _, dbg, _, _ = _run(Layer, seg, direct, conf, filter_estimates=True, output_second_largest_component=True)
    assert int(dbg["selected"][0, 0]) == 30 * 56 + 40
    seg3, direct3, conf3 = _scene(boxes=((2, 6, 40, 46), (20, 26, 10, 17)))  # all below 50 px -> label 1
    _, dbg, _, _ = _run(Layer, seg3, direct3, conf3, filter_estimates=True)
    assert int(dbg["selected"][0, 0]) == 2 * 56 + 40
    seg4, direct4, conf4 = _scene(boxes=((0, 40, 0, 40),))  # object larger than the background -> label 0
    out, dbg, _, _ = _run(Layer, seg4, direct4, conf4, filter_estimates=True)
    assert int(dbg["selected"][0, 0]) == -2 and float(out.abs().max()) == 0.0
    seg5, direct5, conf5 = _scene(boxes=())  # empty class
    out, dbg, _, _ = _run(Layer, seg5, direct5, conf5, filter_estimates=True)
    assert int(dbg["selected"][0, 0]) == -1 and float(out.abs().max()) == 0.0


def test_components_of_a_serpentine_and_diagonal_pixels(Layer):
    """Union-find stress: a one-pixel-wide serpentine is ONE component (long merge chains); pixels that touch
    only diagonally are separate components; two classes side by side do not merge."""
    h, w = 64, 64
    lab = np.zeros((h, w), np.int32)
    for r, y in enumerate(range(2, 40, 2)):  # class 1: rows joined alternately at the right / left end
        lab[y, 2:60] = 1
        lab[y + 1, 59 if r % 2 == 0 else 2] = 1
    lab[41, 2:60] = 0
    for i in range(10):  # class 2: ten diagonal single pixels and a 60-pixel bar right below class-1-free rows
        lab[44 + i, 3 + i] = 2
    lab[58:60, 5:35] = 2
    lab[57, 5:35] = 1  # a second class-1 component (30 px) touching the class-2 bar
    seg = np.zeros((1, h, w, 3), np.float32)
    seg[..., 0] = 1.0
    for c in (1, 2):
        seg[0, :, :, c] = np.where(lab == c, 4.0, 0.0)
    rng = np.random.default_rng(2)
    direct = rng.normal(size=(1, h, w, 4)).astype(np.float32)
    conf = rng.normal(size=(1, h, w, 2)).astype(np.float32)
    _, dbg, _, _ = _run(Layer, seg, direct, conf, filter_estimates=True)
    assert int(dbg["selected"][0, 0]) == 2 * w + 2  # the serpentine, rooted at its first pixel
    assert int(dbg["selected"][0, 1]) == 58 * w + 5  # the bar (the diagonal pixels are 1-px components)
    _run(Layer, seg, direct, conf, filter_estimates=True, output_second_largest_component=True)


def test_non_finite_input_raises_like_the_reference_assert(Layer):
    from casapose_b200._lib import CasaError
    from tests.test_oracle_ls import _scene

    seg, direct, conf = _scene()
    direct[0, 10, 10, 0] = np.nan
    layer = Layer("ls", 2, num_points=2)
    with pytest.raises(CasaError):
        layer([torch.from_numpy(seg).cuda(), torch.from_numpy(direct).cuda(), torch.from_numpy(conf).cuda()])


def test_tied_logits_list_a_pixel_for_every_class(Layer):
    """All-equal segmentation logits (a zero-initialised seg head): softmax(1e6 * seg) is 1/nc for EVERY class, so each
    pixel is listed oc times and the per-image lists need oc*h*w slots — the layer must give the reference's weighted
    solution (weights 1/nc), not zeros (the first attempt at h*w slots overflows and is retried with the measured need);
    the backward pass must see the same lists and give the gradient oracle's result (every pixel's gradient sums the
    four classes' terms with atomicAdd)."""
    from oracle import ls_voting_grad as G
    from tests.test_ls_backward import _check, _mask_singular

    rng = np.random.default_rng(11)
    b, h, w, nc, vn = 2, 24, 32, 5, 3
    seg = np.zeros((b, h, w, nc), np.float32)
    ang = rng.uniform(0, 2 * np.pi, (b, h, w, vn))
    direct = np.stack([np.sin(ang), np.cos(ang)], -1).reshape(b, h, w, 2 * vn).astype(np.float32)
    conf = rng.normal(size=(b, h, w, vn)).astype(np.float32)
    out, dbg, ref, _ = _run(Layer, seg, direct, conf)
    assert (dbg["tn"].cpu().numpy() == h * w).all()
    assert np.abs(ref).max() > 1.0  # a real solution, not the zeros of a gated class
    layer = Layer("ls", nc, num_points=vn)
    g = _mask_singular(rng.normal(size=(b, nc - 1, vn, 2)).astype(np.float32), seg, direct, conf, num_points=vn)
    assert (g != 0).all()  # every job is regular
    gd, gw = layer.backward([torch.from_numpy(seg).cuda(), torch.from_numpy(direct).cuda(), torch.from_numpy(conf).cuda()],
                            torch.from_numpy(g).cuda())
    _, rd, rw = G.ls_vote_with_grads(seg, direct, conf, g, num_points=vn)
    _check(gd.cpu().numpy(), rd, "grad_direct")
    _check(gw.cpu().numpy(), rw, "grad_conf")
    assert float(gd.abs().max()) > 0 and float(gw.abs().max()) > 0


@pytest.mark.parametrize("second", [False, True])
def test_salt_and_pepper_segmentation_has_more_runs_than_shared_memory_holds(Layer, second):
    """A noisy segmentation (early in training): thousands of one- and two-pixel runs per class, far more than the
    2048 runs k_cc_runs keeps in shared memory -> its global-memory run tables; components, selection and keypoints
    must still be the oracle's (and the pixel-level union-find's)."""
    rng = np.random.default_rng(5)
    h, w, vn = 96, 128, 3
    lab = rng.integers(0, 3, size=(h, w))
    lab[20:50, 30:90] = 1  # one solid blob per class on top of the noise
    lab[60:80, 10:60] = 2
    seg = np.zeros((1, h, w, 3), np.float32)
    for c in range(3):
        seg[0, :, :, c] = np.where(lab == c, 3.0, 0.0)
    direct = rng.normal(size=(1, h, w, 2 * vn)).astype(np.float32)
    conf = rng.normal(size=(1, h, w, vn)).astype(np.float32)
    _run(Layer, seg, direct, conf, filter_estimates=True, output_second_largest_component=second)


def test_ls_layer_with_three_calls_in_flight_equals_the_eager_calls(Layer):
    """casa_set_async(h, 3): consecutive casa_ls_vote calls rotate over three lanes (own workspace, own stream); after
    casa_join the results are the eager calls', bit for bit."""
    from casapose_b200 import _lib

    d = synthetic.make_frames(2, 120, 160, (1, 5, 6), variant="easy", with_logits=True)
    seg = torch.from_numpy(d["seg_logits"]).cuda()
    conf = torch.from_numpy(d["conf_logits"]).cuda()
    directs = [torch.from_numpy(np.roll(d["vertex"].reshape(2, 120, 160, 18), k, axis=3).copy()).cuda() for k in range(5)]
    layer = Layer("ls", seg.shape[3], num_points=9, filter_estimates=True)
    expect = [layer([seg, x, conf]).clone() for x in directs]
    torch.cuda.synchronize()
    _lib.set_async(0, 3)
    try:
        outs = [layer([seg, x, conf], check_finite=False) for x in directs]
        _lib.join(0)
        got = [o.clone() for o in outs]
        _lib.sync(0)
    finally:
        _lib.set_async(0, 0)
    for e, g in zip(expect, got):
        assert torch.equal(e, g)
