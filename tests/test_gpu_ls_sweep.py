"""CoordLSVotingWeighted across the code paths its kernels pick from the shape and the input, forward and backward.

Every GPU case goes through the bar of tests/test_gpu_ls.py (`_run`: float64 sums within 1e-7 of scale, keypoints
within 1e-3 px, the graph-replayed run-based call bit-equal to the pixel-union-find debug call) and the gradient bar
of tests/test_ls_backward.py (`_check` against oracle/ls_voting_grad.py: 2e-4 of scale, same zero pattern).  On top,
every case checks the per-job pixel counts (`tn`) and the int(hot + 0.1) label map against the numpy oracle.

The scene builders are plain numpy; the tests without the gpu marker check on the CPU that each scene delivers what it
promises (pixel counts, run counts, component sizes, softmax bands), so the GPU cases test what they claim to test.
"""
import ctypes as C

import numpy as np
import pytest
from scipy import ndimage

torch = pytest.importorskip("torch")

from casapose_b200 import synthetic  # noqa: E402
from oracle import ls_voting_grad as G  # noqa: E402
from oracle import ls_voting_np as L  # noqa: E402

F = np.float32
THR = F(13.942385)  # softplus branch point of Eigen's functor (-(log(eps_f32) + 2)), ls_vote.cuh ls_weight
MODES = [(False, False, False), (False, True, False), (True, False, False), (True, True, False), (True, False, True),
         (True, True, True)]  # (filter_estimates, sigmoid_weights, output_second_largest_component)
MODE_IDS = ["plain", "sigm", "filt", "filt-sigm", "filt-second", "filt-sigm-second"]


# ----------------------------------------------------------------------------------------------- scene builders
def _fields(rng, b, h, w, vn):
    """Random (dy, dx) per keypoint and confidence logits: a pixel's direction is arbitrary, so any 20 or more pixels
    give a well-conditioned 2x2 system."""
    direct = rng.normal(size=(b, h, w, 2 * vn)).astype(F)
    conf = rng.normal(size=(b, h, w, vn)).astype(F)
    return direct, conf


def _one_hot_logits(rng, lab, nc):
    """Logits whose softmax(1e6 * seg) is exactly one-hot at class `lab` (winner 1..2, the others -1..0)."""
    seg = rng.uniform(-1, 0, lab.shape + (nc,)).astype(F)
    np.put_along_axis(seg, lab[..., None], rng.uniform(1, 2, lab.shape + (1,)).astype(F), -1)
    return seg


def blocks_scene(b, h, w, nc, vn, bh, bw, seed=0, per_image=None):
    """Label map tiled by bh x bw blocks of random classes (0 = background); the last class owns the first block of
    every image.  per_image: classes (background included) an image draws from, the others stay empty."""
    rng = np.random.default_rng(seed)
    gy, gx = -(-h // bh), -(-w // bw)
    lab = np.empty((b, h, w), np.int64)
    for i in range(b):
        pool = np.arange(nc) if per_image is None else np.concatenate([[0, nc - 1], rng.choice(np.arange(1, nc - 1), per_image - 2, replace=False)])
        blk = rng.choice(pool, size=(gy, gx))
        blk[0, 0] = nc - 1
        lab[i] = np.kron(blk, np.ones((bh, bw), np.int64))[:h, :w]
    return (_one_hot_logits(rng, lab, nc),) + _fields(rng, b, h, w, vn) + (lab,)


TILE_TN = (255, 256, 257, 511, 512, 513, 1023, 1024, 1025)


def tile_edge_scene(vn, seed=1):
    """One image, class c+1 owns exactly TILE_TN[c] pixels (a raster-order range): jobs end just before, on and just
    after the 256-entry step, the 512-entry fused tile and the 1024-entry backward tile."""
    rng = np.random.default_rng(seed)
    h, w = 48, 160
    lab = np.zeros(h * w, np.int64)
    p = 17
    for c, n in enumerate(TILE_TN):
        lab[p:p + n] = c + 1
        p += n + 40
    lab = lab.reshape(1, h, w)
    return (_one_hot_logits(rng, lab, len(TILE_TN) + 1),) + _fields(rng, 1, h, w, vn) + (lab,)


RUN_BLOBS = ((2, 22, 4, 64), (2, 12, 70, 121))  # class 1: 20 runs (1200 px) and 10 runs (510 px) on the same rows


def run_count_scene(vn=3, seed=2):
    """Two images whose class 1 has exactly 2048 (image 0) and 2049 (image 1) horizontal runs: the largest run table
    k_cc_runs keeps in shared memory, and the first that goes to global memory.  Two blobs plus single-pixel runs on
    every other row and column; class 2 is a band at the bottom."""
    rng = np.random.default_rng(seed)
    h, w = 96, 128
    lab = np.zeros((2, h, w), np.int64)
    dots = [(y, x) for y in range(26, 90, 2) for x in range(0, w, 2)]
    for i, runs in enumerate((2048, 2049)):
        for y0, y1, x0, x1 in RUN_BLOBS:
            lab[i, y0:y1, x0:x1] = 1
        for y, x in dots[:runs - 30]:
            lab[i, y, x] = 1
        lab[i, 90:96, :] = 2
    return (_one_hot_logits(rng, lab, 3),) + _fields(rng, 2, h, w, vn) + (lab,)


def count_runs(m):
    """Horizontal runs of a boolean [h, w] map."""
    m = m.astype(np.int8)
    return int((np.diff(np.pad(m, ((0, 0), (1, 0))), axis=1) == 1).sum())


# class -> [(y0, y1, x0, x1)] boxes, in raster order of their first pixels (= the reference's component labels)
SIZE_BOXES = {
    1: [(2, 9, 2, 9), (2, 7, 20, 30), (2, 5, 40, 57)],   # 49, 50, 51 px: the < 50 rule on both sides
    2: [(12, 17, 2, 12), (12, 19, 20, 27)],              # 50 and 49 px
    3: [(25, 33, 2, 10), (25, 33, 30, 38)],              # two components of 64 px: the lower label wins
    4: [(25, 32, 60, 67), (25, 32, 80, 87)],             # two components of 49 px, both count 0
}
SIZE_EXPECT = {1: (49, 50, 51), 2: (50, 49), 3: (64, 64), 4: (49, 49)}
# selected root pixel (w = 160) for (largest, second largest), and the serpentine class 5 (blob first, snake second)
SIZE_SELECT = {1: (2 * 160 + 40, 2 * 160 + 20), 2: (12 * 160 + 2, 12 * 160 + 20), 3: (25 * 160 + 2, 25 * 160 + 30),
               4: (25 * 160 + 60, 25 * 160 + 80), 5: (40 * 160 + 0, 40 * 160 + 90)}


def component_scene(vn=3, seed=3):
    """Component edges in one 128 x 160 image (nc = 6): sizes 49 / 50 / 51, equal sizes, and class 5 with a 4800-px
    blob beside a serpentine on the same rows (6659 list entries: both components cross the 2048-entry trips of
    k_cc_runs, and their runs interleave in the list)."""
    rng = np.random.default_rng(seed)
    h, w = 128, 160
    lab = np.zeros((1, h, w), np.int64)
    for c, boxes in SIZE_BOXES.items():
        for y0, y1, x0, x1 in boxes:
            lab[0, y0:y1, x0:x1] = c
    lab[0, 40:100, 0:80] = 5
    for k, y in enumerate(range(40, 100, 2)):
        lab[0, y, 90:151] = 5
        if y + 1 < 99:
            lab[0, y + 1, 150 if k % 2 == 0 else 90] = 5
    return (_one_hot_logits(rng, lab, 6),) + _fields(rng, 1, h, w, vn) + (lab,)


def _set_gaps(seg, region, winner, gaps):
    """Logits near 0 so float32 resolves the gaps: the winner at 0, class c at -gaps[c] * 1e-6 (gap in units of
    1e6 * logit), every other class at -1 (exactly zero after the softmax)."""
    seg[region] = F(-1.0)
    sub = seg[region]
    sub[..., winner] = F(0.0)
    for c, g in gaps.items():
        sub[..., c] = F(-g * 1e-6)
    seg[region] = sub


# name -> (region (image, y0, y1, x0, x1), winner, {class: gap}, {class: (hot_lo, hot_hi)})
TIE_REGIONS = {
    "88": ((0, 2, 10, 2, 12), 1, {2: 2.0}, {1: (0.875, 0.885), 2: (0.115, 0.125)}),      # int(0.98) = 0
    "92": ((0, 2, 10, 20, 30), 1, {0: 2.4}, {1: (0.912, 0.922)}),                       # int(1.02) = 1
    "92bg": ((1, 2, 10, 2, 12), 0, {2: 2.4}, {2: (0.078, 0.088)}),                      # background wins 0.92
    "88bg": ((1, 2, 10, 20, 30), 2, {0: 2.0}, {2: (0.875, 0.885)}),
    "three": ((0, 14, 20, 2, 14), 1, {2: 0.7, 3: 1.5}, {1: (0.57, 0.59), 2: (0.28, 0.30), 3: (0.12, 0.14)}),
    "mid": ((1, 14, 20, 2, 14), 3, {1: 40.0}, {1: (1e-18, 1e-17)}),
    "sub90": ((0, 24, 30, 2, 12), 2, {3: 90.0}, {3: (1e-45, 1.1754944e-38)}),            # subnormal, not flushed
    "sub95": ((1, 24, 30, 2, 12), 1, {3: 95.0}, {3: (1e-45, 1.1754944e-38)}),
    "sub100": ((1, 24, 30, 20, 30), 2, {1: 100.0}, {1: (1e-45, 1.1754944e-38)}),
}
THREE_WAY = ("three",)


def tie_scene(vn=3, seed=4, names=tuple(TIE_REGIONS)):
    """Two 40 x 56 images (nc = 4) of one-hot blocks, with regions of near-tied logits: fractional hot at 0.88 and
    0.92 (either side of the int(hot + 0.1) boundary at a gap of ln 9), a three-way tie, a tiny normal runner-up, and
    subnormal runner-ups at gaps 90 / 95 / 100 that must still list the pixel for both classes."""
    seg, direct, conf, lab = blocks_scene(2, 40, 56, 4, vn, 8, 14, seed=seed)
    for n in names:
        (i, y0, y1, x0, x1), win, gaps, _ = TIE_REGIONS[n]
        _set_gaps(seg, (i, slice(y0, y1), slice(x0, x1)), win, gaps)
    return seg, direct, conf, lab


def overflow_scene(vn=3, seed=5):
    """Near ties (class 1 vs class 2, gap 0.3) over 80 % of the image: those pixels are listed twice, the per-image
    lists need more than h*w slots and the first attempt overflows and is retried with the measured need."""
    seg, direct, conf, lab = blocks_scene(1, 40, 60, 3, vn, 10, 12, seed=seed)
    _set_gaps(seg, (0, slice(0, 32), slice(0, 60)), 1, {2: 0.3})
    return seg, direct, conf, lab


def background_pick_scene(vn=3, seed=6):
    """filter_estimates selects label 0: class 1 covers 1600 of 2240 px, so top_k's rank 1 is the background.  The
    reference then keeps the class's listed pixels outside its int mask — here a 10 x 14 patch tied with the
    background (hot 0.38) — so the output is not zero."""
    rng = np.random.default_rng(seed)
    h, w = 40, 56
    lab = np.zeros((1, h, w), np.int64)
    lab[0, 0:40, 0:40] = 1
    lab[0, 28:38, 42:54] = 2
    seg = _one_hot_logits(rng, lab, 3)
    _set_gaps(seg, (0, slice(5, 15), slice(41, 55)), 0, {1: 0.5})
    return (seg,) + _fields(rng, 1, h, w, vn) + (lab,)


CONF_EDGES = np.array([THR, np.nextafter(THR, F(np.inf)), np.nextafter(THR, F(0)), -THR, np.nextafter(-THR, F(-np.inf)),
                       np.nextafter(-THR, F(0)), 90, -90, 100, -100], F)


def conf_edge_scene(vn=4, seed=7):
    """Confidence logits at the softplus branch points and their float32 neighbours, at +-90 (expf overflows /
    underflows) and +-100 (the sigmoid saturates), on a third of the pixels."""
    seg, direct, conf, lab = blocks_scene(2, 40, 56, 4, vn, 8, 14, seed=seed)
    rng = np.random.default_rng(seed + 100)
    pick = rng.random(conf.shape) < 1 / 3
    conf[pick] = rng.choice(CONF_EDGES, size=int(pick.sum()))
    return seg, direct, conf, lab


def _listed(seg):
    return L.hard_softmax_f32(seg)[..., 1:] != 0


# --------------------------------------------------------------------------------------- CPU checks of the builders
def test_blocks_scene_jobs_are_empty_or_large():
    for args in [(2, 37, 29, 2, 1, 8, 8), (2, 45, 23, 11, 10, 8, 8), (2, 33, 35, 12, 8, 6, 7), (2, 41, 27, 13, 9, 7, 9),
                 (2, 24, 44, 14, 16, 6, 11), (2, 16, 24, 33, 2, 4, 6), (2, 1, 300, 4, 3, 1, 20), (2, 300, 1, 4, 3, 20, 1)]:
        seg, _, _, lab = blocks_scene(*args)
        hot = L.hard_softmax_f32(seg)
        assert np.array_equal(hot, np.eye(args[3], dtype=F)[lab])  # exactly one-hot
        tn = _listed(seg).sum(axis=(1, 2))
        assert ((tn == 0) | (tn >= 20)).all(), tn
        assert (tn[:, -1] > 0).all()  # the last class (bit 31 of the membership word at nc = 33) is present
    seg, _, _, lab = blocks_scene(5, 40, 48, 6, 5, 8, 8, per_image=3)
    tn = _listed(seg).sum(axis=(1, 2))
    assert (tn == 0).sum() >= 5  # empty classes in some images


def test_tile_edge_scene_has_the_exact_job_sizes():
    seg, _, _, _ = tile_edge_scene(9)
    assert tuple(_listed(seg).sum(axis=(1, 2))[0]) == TILE_TN


def test_run_count_scene_has_2048_and_2049_runs():
    seg, _, _, lab = run_count_scene()
    hot_int = (L.hard_softmax_f32(seg)[..., 1:] + F(0.1)).astype(np.int32)
    assert [count_runs(hot_int[i, :, :, 0]) for i in range(2)] == [2048, 2049]
    for i in range(2):
        comp, n = ndimage.label(hot_int[i, :, :, 0])
        sizes = np.bincount(comp.ravel())[1:]
        assert sorted(sizes)[-2:] == [510, 1200] and (np.sort(sizes)[:-2] == 1).all()


def test_component_scene_has_the_promised_components():
    seg, _, _, _ = component_scene()
    hot_int = (L.hard_softmax_f32(seg)[..., 1:] + F(0.1)).astype(np.int32)[0]
    for c, want in SIZE_EXPECT.items():
        comp, n = ndimage.label(hot_int[:, :, c - 1])
        assert tuple(np.bincount(comp.ravel())[1:]) == want, c
    comp, n = ndimage.label(hot_int[:, :, 4])
    assert n == 2 and tuple(np.bincount(comp.ravel())[1:]) == (4800, 1859)
    assert hot_int[:, :, 4].sum() > 3 * 2048  # class 5's list spans four 2048-entry trips of k_cc_runs
    w = hot_int.shape[1]
    for c, (first, second) in SIZE_SELECT.items():  # the reference's selection picks the roots the GPU test expects
        for which, root in ((1, first), (2, second)):
            keep = L.select_component(hot_int[:, :, c - 1], 2 if which == 1 else 3, which).reshape(hot_int.shape[:2])
            ys, xs = np.nonzero(keep)
            assert ys[0] * w + xs[0] == root, (c, which)


def test_tie_scene_hot_values_are_in_their_bands():
    seg, _, _, _ = tie_scene()
    hot = L.hard_softmax_f32(seg)
    for name, ((i, y0, y1, x0, x1), win, gaps, bands) in TIE_REGIONS.items():
        h = hot[i, y0:y1, x0:x1]
        for c, (lo, hi) in bands.items():
            assert (h[..., c] >= lo).all() and (h[..., c] <= hi).all(), (name, c, h[..., c].min(), h[..., c].max())
        listed = (h[..., 1:] != 0).sum(-1)
        assert (listed == len([c for c in [win, *gaps] if c > 0])).all(), name
    hi_int = (hot + F(0.1)).astype(np.int32)
    # 0.88 sits below the int(hot + 0.1) boundary, 0.92 above it
    assert not hi_int[0, 2:10, 2:12].any() and hi_int[0, 2:10, 20:30, 1].all() and hi_int[1, 2:10, 2:12, 0].all()


def test_overflow_and_background_pick_scenes():
    seg, _, _, _ = overflow_scene()
    assert _listed(seg).sum() > 1.5 * 40 * 60  # more list entries than h*w slots
    seg, _, _, _ = background_pick_scene()
    hot = L.hard_softmax_f32(seg)[..., 1:]
    hot_int = (hot + F(0.1)).astype(np.int32)[0, :, :, 0]
    assert hot_int.sum() == 1600 and 40 * 56 - 1600 < 1600  # the object outranks the background
    keep = L.select_component(hot_int, 2, 1).reshape(40, 56)
    assert (keep[5:15, 41:55] == 1).all() and not keep[hot_int == 1].any()  # label 0 selected
    frac = hot[0, :, :, 0] * keep
    assert frac.sum() > 0 and ((frac == 0) | ((frac > 0.37) & (frac < 0.38))).all()


def test_conf_edge_values_are_on_both_sides_of_the_branch_points():
    _, _, conf, _ = conf_edge_scene()
    for v in CONF_EDGES:
        assert (conf == v).sum() > 10
    assert np.float32(np.nextafter(THR, F(np.inf))) > THR > np.float32(np.nextafter(THR, F(0)))
    sp = L.softplus_f32(CONF_EDGES)
    assert sp[0] == np.log(np.exp(THR) + F(1)) and sp[1] == CONF_EDGES[1]  # log branch at T, identity just above
    assert sp[7] > 0 and sp[7] < 1.1754944e-38  # softplus(-90) = exp(-90): subnormal
    assert L.sigmoid_f32(CONF_EDGES)[9] == 0 and L.sigmoid_f32(CONF_EDGES)[8] == 1


# ----------------------------------------------------------------------------------------------------- GPU cases
@pytest.fixture(scope="module")
def Layer(cuda_lib):
    assert torch.cuda.is_available()
    from casapose_b200.pose_estimation import CoordLSVotingWeighted

    return CoordLSVotingWeighted


def _cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _case(Layer, seg, direct, conf, mode=(False, False, False), seed=0, backward=True):
    """Forward through the shared bar, tn and label map against the oracle, then the backward against the gradient
    oracle.  Returns the debug call's (out, dbg) and the reference's (ref, rdbg)."""
    from tests.test_gpu_ls import _run
    from tests.test_ls_backward import _check, _mask_singular

    filt, sigm, second = mode
    kw = dict(filter_estimates=filt, sigmoid_weights=sigm, output_second_largest_component=second)
    vn = conf.shape[3]
    out, dbg, ref, rdbg = _run(Layer, seg, direct, conf, **kw)
    hot = L.hard_softmax_f32(seg)[..., 1:]
    assert np.array_equal(dbg["tn"].cpu().numpy(), (hot != 0).sum(axis=(1, 2)))
    hot_int = (hot + F(0.1)).astype(np.int32)
    labels = np.where(hot_int.any(-1), hot_int.argmax(-1) + 1, 0)
    assert np.array_equal(dbg["labels"].cpu().numpy(), labels)
    if not backward:
        return out, dbg, ref, rdbg
    b, oc = seg.shape[0], seg.shape[3] - 1
    g = np.random.default_rng(seed).normal(size=(b, oc, vn, 2)).astype(F)
    g = _mask_singular(g, seg, direct, conf, num_points=vn, **kw)
    layer = Layer("ls", seg.shape[3], num_points=vn, **kw)
    inp = _cuda(seg, direct, conf)
    tg = torch.from_numpy(g).cuda()
    gd, gw = layer.backward(inp, tg)
    _, rd, rw = G.ls_vote_with_grads(seg, direct, conf, g, num_points=vn, **kw)
    _check(gd.cpu().numpy(), rd, "grad_direct")
    _check(gw.cpu().numpy(), rw, "grad_conf")
    # A pixel listed for several classes collects its gradient with atomicAdd.  Two terms commute (0 + a + b ==
    # 0 + b + a), three do not associate ((a + b) + c != (a + c) + b), so the bits are only fixed below three.
    if (hot != 0).sum(-1).max() < 3:
        gd2, gw2 = layer.backward(inp, tg)
        assert torch.equal(gd, gd2) and torch.equal(gw, gw2)
    return out, dbg, ref, rdbg


SHAPES = {  # (b, h, w, nc, vn, block h, block w): one case per kernel path
    "nc2-vn1": (2, 37, 29, 2, 1, 8, 8),        # h*w = 1073: partial classify tile, scalar staging
    "nc11-vn10": (2, 45, 23, 11, 10, 8, 8),    # odd nc, (h*w*nc) % 4 != 0
    "nc12-vn8": (2, 33, 35, 12, 8, 6, 7),      # exactly 48 KB of staged logits (+ the kernel's static counters)
    "nc13-vn9": (2, 41, 27, 13, 9, 7, 9),      # first nc that needs the shared-memory opt-in; vn 9 backward gather
    "nc14-vn16": (2, 24, 44, 14, 16, 6, 11),   # 512-thread k_ls_fused blocks
    "nc33-vn2": (2, 16, 24, 33, 2, 4, 6),      # full membership word: class 32 sets bit 31
    "row": (2, 1, 300, 4, 3, 1, 20),           # one-pixel runs joined only horizontally
    "column": (2, 300, 1, 4, 3, 20, 1),        # runs of one pixel joined only vertically
    "b5-empty": (5, 40, 48, 6, 5, 8, 8),       # empty classes in some images
    "J288": (9, 16, 24, 33, 2, 4, 6),          # J = b * oc > 256: the 1024-thread k_plan
    "J1056": (33, 16, 24, 33, 2, 4, 6),        # J > 1024: k_plan loops
}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("shape", list(SHAPES))
def test_shapes(Layer, shape, mode):
    b, h, w, nc, vn, bh, bw = SHAPES[shape]
    seg, direct, conf, _ = blocks_scene(b, h, w, nc, vn, bh, bw, seed=len(shape), per_image=3 if shape == "b5-empty" else None)
    _case(Layer, seg, direct, conf, mode)


NC12_SCRIPT = r"""
import sys
sys.path.insert(0, %(root)r)
import numpy as np, torch
from casapose_b200.pose_estimation import CoordLSVotingWeighted
from oracle import ls_voting_np as L
from tests.test_gpu_ls_sweep import blocks_scene
seg, direct, conf, _ = blocks_scene(2, 33, 35, 12, 8, 6, 7)
out = CoordLSVotingWeighted("ls", 12, num_points=8)([torch.from_numpy(a).cuda() for a in (seg, direct, conf)])
err = float(np.abs(out.cpu().numpy() - L.coord_ls_voting_weighted(seg, direct, conf, num_points=8)).max())
assert err <= 1e-3, err
print("nc12 ok")
"""


@pytest.mark.gpu
def test_nc12_as_the_first_call_of_a_process(cuda_lib):
    """nc = 12 stages exactly 48 KB of logits; with k_ls_classify's static counters that is over the default limit,
    so the shared-memory opt-in is needed.  An earlier call with nc >= 13 leaves the attribute raised, so only a fresh
    process shows whether nc = 12 sets it itself."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", NC12_SCRIPT % {"root": root}], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "nc12 ok" in res.stdout, res.stdout + res.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [(True, False, False), (False, True, False)], ids=["filt", "sigm"])
def test_full_resolution_forward_and_backward(Layer, mode):
    d = synthetic.make_frames(1, 480, 640, synthetic.CONFIG_8_IDS, variant="easy", with_logits=True)
    _case(Layer, d["seg_logits"], d["vertex"].reshape(1, 480, 640, 18), d["conf_logits"], mode)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("vn", [9, 16])
def test_jobs_at_tile_edges(Layer, vn, mode):
    seg, direct, conf, _ = tile_edge_scene(vn)
    _, dbg, _, _ = _case(Layer, seg, direct, conf, mode)
    assert tuple(dbg["tn"].cpu().numpy()[0]) == TILE_TN


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_run_tables_at_the_shared_memory_limit(Layer, mode):
    seg, direct, conf, _ = run_count_scene()
    _, dbg, _, _ = _case(Layer, seg, direct, conf, mode)
    if mode[0]:
        (y0, _, x0, _), (y1, _, x1, _) = RUN_BLOBS
        want = y1 * 128 + x1 if mode[2] else y0 * 128 + x0
        assert dbg["selected"].cpu().numpy()[:, 0].tolist() == [want, want]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_component_edges(Layer, mode):
    seg, direct, conf, _ = component_scene()
    _, dbg, _, _ = _case(Layer, seg, direct, conf, mode)
    if mode[0]:
        sel = dbg["selected"].cpu().numpy()[0]
        assert [int(sel[c - 1]) for c in SIZE_SELECT] == [SIZE_SELECT[c][1 if mode[2] else 0] for c in SIZE_SELECT]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("names", [tuple(n for n in TIE_REGIONS if n not in THREE_WAY), THREE_WAY], ids=["two-way", "three-way"])
def test_near_tied_logits(Layer, names, mode):
    seg, direct, conf, _ = tie_scene(names=names)
    _case(Layer, seg, direct, conf, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_near_ties_over_most_of_the_image_retry_the_lists(Layer, mode):
    seg, direct, conf, _ = overflow_scene()
    _, dbg, _, _ = _case(Layer, seg, direct, conf, mode)
    assert int(dbg["tn"].sum()) > 40 * 60  # more than the first attempt's h*w slots


@pytest.mark.gpu
@pytest.mark.parametrize("second", [False, True])
@pytest.mark.parametrize("sigm", [False, True])
def test_background_selection_keeps_fractional_pixels(Layer, sigm, second):
    seg, direct, conf, _ = background_pick_scene()
    out, dbg, ref, _ = _case(Layer, seg, direct, conf, (True, sigm, second))
    if second:  # no third entry: nothing is kept
        assert int(dbg["selected"][0, 0]) == -1 and float(out[0, 0].abs().max()) == 0.0
    else:
        assert int(dbg["selected"][0, 0]) == -2 and np.abs(ref[0, 0]).max() > 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_confidence_logit_edges(Layer, mode):
    seg, direct, conf, _ = conf_edge_scene()
    _case(Layer, seg, direct, conf, mode)


# ------------------------------------------------------------------------------------------------------- alignment
def _offset(t):
    """A contiguous copy of `t` whose data pointer sits 4 bytes past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 == 4
    return v


ALIGN_SCENES = {"one-hot-nc9-vn9": lambda: blocks_scene(2, 60, 80, 9, 9, 10, 16, seed=8)[:3],
                "two-way-ties": lambda: tie_scene(names=("88", "92", "92bg", "sub90"))[:3]}


@pytest.mark.gpu
@pytest.mark.parametrize("filt", [False, True])
@pytest.mark.parametrize("scene", list(ALIGN_SCENES))
def test_ls_inputs_four_bytes_past_alignment(Layer, scene, filt):
    """seg, direct, conf and grad_out as views 4 bytes into an allocation: the results are the aligned inputs' bits
    (which meet the oracle bar)."""
    seg, direct, conf = ALIGN_SCENES[scene]()
    _case(Layer, seg, direct, conf, (filt, False, False))
    vn = conf.shape[3]
    layer = Layer("ls", seg.shape[3], num_points=vn, filter_estimates=filt)
    a = _cuda(seg, direct, conf)
    m = [_offset(t) for t in a]
    g = torch.from_numpy(np.random.default_rng(0).normal(size=(seg.shape[0], seg.shape[3] - 1, vn, 2)).astype(F)).cuda()
    assert torch.equal(layer(a), layer(m))  # graph-replayed forward
    oa, da = layer(a, return_debug=True)
    om, dm = layer(m, return_debug=True)
    assert torch.equal(oa, om) and all(torch.equal(da[k], dm[k]) for k in da)
    ga = layer.backward(a, g)
    gm = layer.backward(m, _offset(g))
    assert torch.equal(ga[0], gm[0]) and torch.equal(ga[1], gm[1])


@pytest.mark.gpu
def test_ls_abi_outputs_four_bytes_past_alignment(Layer):
    """out_points, grad_direct and grad_conf given to the C ABI as buffers 4 bytes into an allocation."""
    from casapose_b200 import _lib
    from casapose_b200._carrier import current_stream_ptr

    seg, direct, conf, _ = blocks_scene(2, 40, 56, 5, 3, 8, 14, seed=9)
    b, h, w, nc = seg.shape
    vn = conf.shape[3]
    layer = Layer("ls", nc, num_points=vn, filter_estimates=True)
    inp = _cuda(seg, direct, conf)
    g = torch.from_numpy(np.random.default_rng(1).normal(size=(b, nc - 1, vn, 2)).astype(F)).cuda()
    want = layer(inp)
    gd, gw = layer.backward(inp, g)
    dev = inp[0].device
    hdl = _lib.handle(dev.index, current_stream_ptr(dev))
    p = layer._params(b, h, w, nc, vn, True)
    out = _offset(torch.zeros_like(want))
    _lib.check(_lib.lib().casa_ls_vote(hdl, C.byref(p), *[t.data_ptr() for t in inp], out.data_ptr(), None,
                                       current_stream_ptr(dev)))
    out2, gd2, gw2 = _offset(torch.zeros_like(want)), _offset(torch.zeros_like(gd)), _offset(torch.zeros_like(gw))
    _lib.check(_lib.lib().casa_ls_vote_backward(hdl, C.byref(p), *[t.data_ptr() for t in inp], g.data_ptr(),
                                                out2.data_ptr(), gd2.data_ptr(), gw2.data_ptr(), current_stream_ptr(dev)))
    torch.cuda.synchronize()
    assert torch.equal(out, want) and torch.equal(out2, want)
    assert torch.equal(gd2, gd) and torch.equal(gw2, gw)


@pytest.mark.gpu
def test_voting_inputs_four_bytes_past_alignment(cuda_lib):
    """The RANSAC voting path with `mask` and `vertex` 4 bytes past alignment: the scalar mask staging and direction
    gather give the aligned inputs' votes and keypoints bit for bit."""
    from casapose_b200.pose_estimation import ransac_voting_layer_all_masks

    d = synthetic.make_frames(2, 120, 160, (1, 5, 6), variant="easy")
    mask, vertex = _cuda(d["mask"], d["vertex"])
    pa, da = ransac_voting_layer_all_masks(mask, vertex, 64, seed=3, return_debug=True)
    pm, dm = ransac_voting_layer_all_masks(_offset(mask), _offset(vertex), 64, seed=3, return_debug=True)
    torch.cuda.synchronize()
    assert torch.equal(pa, pm)
    for k in ("tn", "rounds", "counts", "win_idx", "win_pts"):
        assert torch.equal(da[k], dm[k]), k


# ---------------------------------------------------------------------------------------------------- handle state
@pytest.mark.gpu
def test_one_handle_across_changing_shapes(Layer):
    """One fresh handle (its own stream): nc, vn and the image shape go up and down, every call meets the oracle
    (the persistent grid size of k_ls_fused is fixed by the first call's 32 * vn); then more shapes than the
    16 cached graphs, and the first shape again gives its first result bit for bit."""
    seq = [(2, 24, 32, 4, 1), (1, 40, 56, 13, 16), (2, 16, 24, 33, 2), (3, 30, 20, 6, 9), (1, 24, 32, 4, 1),
           (2, 48, 40, 12, 8)]
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        first = None
        for i, (b, h, w, nc, vn) in enumerate(seq):
            seg, direct, conf, _ = blocks_scene(b, h, w, nc, vn, 8, 8, seed=20 + i)
            out, _, _, _ = _case(Layer, seg, direct, conf, (True, False, False), backward=False)
            first = out.clone() if first is None else first
        seg0, direct0, conf0, _ = blocks_scene(*seq[0][:4], seq[0][4], 8, 8, seed=20)
        for k in range(18):
            seg, direct, conf, _ = blocks_scene(1, 20 + k, 24, 3, 2, 8, 8, seed=40 + k)
            Layer("ls", 3, num_points=2, filter_estimates=True)(_cuda(seg, direct, conf))
        again = Layer("ls", 4, num_points=1, filter_estimates=True)(_cuda(seg0, direct0, conf0))
        s.synchronize()
    assert torch.equal(again, first)
