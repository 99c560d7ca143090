"""The RANSAC vote across the code paths its kernels pick from the shape, the input form and the pointer alignment.

Every GPU case goes through the bar of tests/test_gpu_ransac.py against oracle/ransac_voting_np.py: tn0, tn, rounds,
vote counts, winning indices, winning hypotheses and the refined flag bit-exact, keypoints within 1e-3 px.  On top,
every case checks that the graph-replayed call without debug outputs gives the same bits as the debug call, and the
device status word (`dbg["status"]`) holds exactly the CASA_STATUS_* bits the case expects.

Test ids name the path a case reaches:
  narrow / wide      k_score with 4 / 8 hypotheses per lane (hn mod 256 in 1..128 / otherwise)
  place9 / place0    k_place<9> / <0> gathering the directions while it scatters the pixels (fused)
  gather18 / gather0 k_gather_dirs<18> / <0>: capped jobs, a vector field 4 bytes past alignment, the host entry
  vec4 / scalar      the 128-bit and the per-element loops of k_mask_bits;  seg: k_seg_bits;  host: k_bits_in

The scene builders are plain numpy; the tests without the gpu marker check on the CPU that each scene delivers what it
claims (pixel counts per job, tile positions, the k_score class of hn, the job count), so the GPU cases test what they
claim to test.  The last two tests cover the 64-bit row offset of k_gather_dirs.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ransac_voting_np as O  # noqa: E402

F = np.float32
TOL_PX = 1e-3
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
NOT_BINARY, PIX_OVERFLOW, IDX_RANGE, EMPTY_AFTER_CAP = 1, 2, 4, 8  # include/casapose_b200.h
VARIANTS = {"easy": (3.0, 0.2), "hard": (35.0, 0.85)}  # (angular noise in degrees, outlier fraction): synthetic.py
gpu = pytest.mark.gpu


# ----------------------------------------------------------------------------------------------- scene builders
def aimed_field(lab, vn, rng, variant="easy", per_class=None, span=None):
    """(dy, dx) unit vectors from every labelled pixel's centre towards keypoints of its class (random points of the
    image, one set per image and class), with the angular noise and outliers of `variant`; zero on background.
    per_class = oc: a [b,h,w,oc,vn,2] field whose slot c holds those vectors for class c's pixels and random unit
    vectors everywhere else, so a gather from the wrong slot cannot agree with the oracle.
    span = (x0, x1, y0, y1): draw the keypoints there instead of inside the image."""
    b, h, w = lab.shape
    oc = int(lab.max()) if per_class is None else per_class
    noise, outlier = VARIANTS[variant]
    x0, x1, y0, y1 = span if span is not None else (0, w, 0, h)
    targets = rng.uniform([x0, y0], [x1, y1], size=(b, max(oc, 1), vn, 2))
    bi, ys, xs = np.nonzero(lab)
    t = targets[bi, lab[bi, ys, xs] - 1]
    ang = np.arctan2(t[..., 1] - (ys[:, None] + 0.5), t[..., 0] - (xs[:, None] + 0.5))
    ang = ang + np.deg2rad(noise) * rng.normal(size=ang.shape)
    out = rng.uniform(size=ang.shape[0]) < outlier
    ang[out] = rng.uniform(-np.pi, np.pi, size=(int(out.sum()), vn))
    if per_class is None:
        vertex = np.zeros((b, h, w, vn, 2), F)
        vertex[bi, ys, xs, :, 0], vertex[bi, ys, xs, :, 1] = np.sin(ang), np.cos(ang)
        return vertex
    junk = rng.uniform(-np.pi, np.pi, size=(b, h, w, oc, vn))
    vertex = np.stack([np.sin(junk), np.cos(junk)], -1).astype(F)
    vertex[bi, ys, xs, lab[bi, ys, xs] - 1, :, 0] = np.sin(ang)
    vertex[bi, ys, xs, lab[bi, ys, xs] - 1, :, 1] = np.cos(ang)
    return vertex


def one_hot(lab, oc):
    return np.stack([lab == c + 1 for c in range(oc)], -1).astype(F)


def box_labels(b, h, w, boxes):
    """boxes: {class: (y0, y1, x0, x1)} painted in order into every image."""
    lab = np.zeros((b, h, w), np.int64)
    for c, (y0, y1, x0, x1) in boxes.items():
        lab[:, y0:y1, x0:x1] = c + 1
    return lab


def grid_labels(b, h, w, oc, ch, cw):
    """ch x cw cells; cell k of image i belongs to label (7 k + 3 i) mod (oc + 1) (0 = background): every label shows
    up once there are oc + 1 cells, since 7 is prime to oc + 1 for the oc used here."""
    gy, gx = h // ch, w // cw
    lab = np.zeros((b, h, w), np.int64)
    for i in range(b):
        cells = ((7 * np.arange(gy * gx) + 3 * i) % (oc + 1)).reshape(gy, gx)
        lab[i, :gy * ch, :gx * cw] = np.kron(cells, np.ones((ch, cw), np.int64))
    return lab


def hn_class(hn):
    """k_score's instantiation for hn (ransac.cuh score_hpl): 4 hypotheses per lane if hn mod 256 is in 1..128."""
    return "narrow" if (hn - 1) % 256 < 128 else "wide"


HN_SWEEP = (1, 2, 127, 128, 129, 255, 256, 257, 384, 385)
HN_BOXES = {0: (8, 40, 10, 50), 1: (30, 60, 55, 90)}  # 1280 and 1050 px in a 64 x 96 image


def hn_scene(variant, seed=0):
    lab = box_labels(1, 64, 96, HN_BOXES)
    return one_hot(lab, 2), aimed_field(lab, 9, np.random.default_rng(seed), variant), lab


EDGE_TN = (127, 128, 129, 2047, 2048, 2049)  # kChunk = 128 scoring chunks, kVoteTile = 2048 refinement tiles
EDGE_HW = (160, 240)


def edge_ranges(kind):
    """Raster ranges (start, length) of the six jobs: after one another ("raster"), or each centred on its own
    1024-pixel (compaction tile) or 4096-pixel (k_place block) boundary."""
    if kind == "raster":
        out, p = [], 17
        for n in EDGE_TN:
            out.append((p, n))
            p += n + 40
        return out
    tile, first, step = (1024, 2, 3) if kind == "cross1024" else (4096, 1, 1)
    return [(tile * (first + step * k) - n // 2, n) for k, n in enumerate(EDGE_TN)]


def edge_scene(kind, seed=1):
    h, w = EDGE_HW
    lab = np.zeros(h * w, np.int64)
    for c, (s, n) in enumerate(edge_ranges(kind)):
        lab[s:s + n] = c + 1
    lab = lab.reshape(1, h, w)
    return one_hot(lab, len(EDGE_TN)), aimed_field(lab, 9, np.random.default_rng(seed)), lab


VN_SWEEP = (1, 2, 8, 9, 10, 16)
VN_BOXES = {0: (4, 24, 4, 30), 1: (26, 44, 30, 60)}  # 520 and 540 px in a 48 x 64 image
VN_CAP = 530.0  # max_num between the two: class 1 is capped (k_gather_dirs after k_cap_filter), class 0 is not


def vn_scene(vn, seed=2, per_class=None):
    lab = box_labels(1, 48, 64, VN_BOXES)
    return one_hot(lab, 2), aimed_field(lab, vn, np.random.default_rng(seed), per_class=per_class), lab


OC_CASES = {"oc1-vec4": (1, 48, 64, False), "oc31-vec4": (31, 48, 64, False), "oc31-scalar": (31, 47, 65, False),
            "oc32-vec4": (32, 48, 64, False), "oc32-scalar": (32, 48, 64, True)}  # (oc, h, w, mask 4 bytes past 16 B)


def oc_scene(oc, h, w, seed=3):
    lab = grid_labels(2, h, w, oc, 6, 8)
    return one_hot(lab, oc), aimed_field(lab, 9, np.random.default_rng(seed), per_class=None), lab


JOB_CASES = {256: (8, 32), 257: (257, 1), 1024: (32, 32), 1025: (205, 5), 2049: (683, 3)}  # J: (b, oc)


def jobs_scene(b, oc, seed=4):
    """12 x 16 images of 4 x 4 cells: 16 pixels per listed job, so the oracle stays cheap at 2049 jobs."""
    lab = grid_labels(b, 12, 16, oc, 4, 4)
    vertex = aimed_field(lab, 9, np.random.default_rng(seed)) if lab.max() == oc else None
    return one_hot(lab, oc), vertex, lab


def seg_argmax(seg):
    """k_seg_bits' arg-max, restated: scan the channels in order from channel 0, a score replaces the best only if it
    is strictly greater.  So the first maximum wins a tie, and a NaN score never wins (every comparison with NaN is
    false), unlike np.argmax, which returns the first NaN."""
    best, arg = seg[..., 0].copy(), np.zeros(seg.shape[:-1], np.int64)
    for c in range(1, seg.shape[-1]):
        up = seg[..., c] > best
        best = np.where(up, seg[..., c], best)
        arg = np.where(up, c, arg)
    return arg


SEG_OC = 5


def seg_scene(seed=5):
    """Scores [1, 48, 64, 6] with one clear winner per pixel, then regions of ties and NaN scores.  Returns the scores
    and the label map k_seg_bits must derive from them."""
    rng = np.random.default_rng(seed)
    lab = grid_labels(1, 48, 64, SEG_OC, 6, 8)
    seg = rng.uniform(-1, 0, lab.shape + (SEG_OC + 1,)).astype(F)
    np.put_along_axis(seg, lab[..., None], rng.uniform(1, 2, lab.shape + (1,)).astype(F), -1)
    r = seg[0]
    r[0:6, 0:16] = F(-1)
    r[0:6, 0:16, 2] = r[0:6, 0:16, 4] = F(1.5)           # tie of classes 2 and 4: class 2 (channel 2) wins
    r[6:12, 0:16] = F(-1)
    r[6:12, 0:16, 0] = r[6:12, 0:16, 1] = F(1.5)         # tie of the background and class 1: background
    r[12:18, 0:16] = F(-1)
    r[12:18, 0:16, 3], r[12:18, 0:16, 5] = np.nan, F(0.5)  # NaN in channel 3: channel 5 wins
    r[18:24, 0:16] = F(-1)
    r[18:24, 0:16, 1], r[18:24, 0:16, 2] = F(0.25), np.nan  # NaN after the best: channel 1 keeps it
    r[24:30, 0:16] = np.nan
    r[24:30, 0:16, 0], r[24:30, 0:16, 4] = F(-3), F(-2)  # NaN everywhere but two channels: channel 4
    return seg, seg_argmax(seg)


MASK_VALUES = {"negzero": (-0.0, 0), "nan": (np.nan, NOT_BINARY), "half": (0.5, NOT_BINARY), "two": (2.0, NOT_BINARY)}


def mask_value_scene(kind, seed=6):
    """Class 0: a 20 x 20 block of `value` (negzero: of ones, and -0.0 everywhere else in the channel); class 1: a
    10 x 10 block of ones."""
    lab = box_labels(1, 48, 64, {0: (4, 24, 4, 24), 1: (30, 40, 40, 50)})
    mask = one_hot(lab, 2)
    value = MASK_VALUES[kind][0]
    if kind == "negzero":
        mask[..., 0] = np.where(lab == 1, F(1), F(-0.0))
    else:
        mask[0, 4:24, 4:24, 0] = F(value)
    return mask, aimed_field(lab, 9, np.random.default_rng(seed)), lab


def gate_scene(sizes, h=32, w=64, seed=7):
    """One image, class c owns a raster range of sizes[c] pixels, 40 pixels behind the previous one."""
    lab = np.zeros((1, h * w), np.int64)
    p = 40
    for c, n in enumerate(sizes):
        lab[0, p:p + n] = c + 1
        p += n + 40
    lab = lab.reshape(1, h, w)
    return one_hot(lab, len(sizes)), aimed_field(lab, 9, np.random.default_rng(seed)), lab


SHAPE_CASES = {  # (h, w, object box (y0, y1, x0, x1), keypoints drawn in (x0, x1, y0, y1) or None: inside the image)
    "1xw": (1, 4099, (0, 1, 3000, 3300), (3000, 3300, -60, 60)),
    "hx1": (4099, 1, (700, 1000, 0, 1), (-60, 60, 700, 1000)),
    "odd-37x111": (37, 111, (3, 30, 85, 105), None),  # h*w = 4107: odd, not a multiple of 4 / 1024 / 4096
    "x65534-2x65535": (2, 65535, (0, 2, 65385, 65535), (65385, 65535, -60, 60)),
    "y65534-65535x2": (65535, 2, (65385, 65535, 0, 2), (-60, 60, 65385, 65535)),
}


def shape_scene(name, seed=8):
    """Thin images: the keypoints lie beside the object's line, so the pixels' directions are far from parallel."""
    h, w, box, span = SHAPE_CASES[name]
    lab = box_labels(1, h, w, {0: box})
    return one_hot(lab, 1), aimed_field(lab, 9, np.random.default_rng(seed), span=span), lab


# ---------------------------------------------------------------------------------------------------- the bar
def oracle(mask, vertex, hn, *, seed, inlier_thresh=0.99, confidence=0.99, max_iter=20, min_num=5, max_num=30000,
           image_offset=0, idxs=None, selection=None):
    """oracle/ransac_voting_np.py; a per-class field [b,h,w,oc,vn,2] is voted class by class on its own slot."""
    if vertex.ndim == 5:
        return O.ransac_voting_layer_all_masks(mask, vertex, hn, inlier_thresh, confidence, max_iter, min_num, max_num,
                                               seed=seed, image_offset=image_offset, idxs=idxs, selection=selection,
                                               return_debug=True)
    b, oc, vn = mask.shape[0], mask.shape[3], vertex.shape[4]
    ref = np.zeros((b, oc, vn, 2), F)
    rdbg = [[None] * oc for _ in range(b)]
    for i in range(b):
        for c in range(oc):
            r = O.ransac_voting_batch(mask[i, :, :, c], vertex[i, :, :, c], inlier_thresh, confidence, max_iter, min_num,
                                      max_num, hn, vn, seed=seed, image=image_offset + i, cls=c,
                                      idxs=None if idxs is None else idxs[i, c],
                                      selection=None if selection is None else selection[i, c])
            ref[i, c], rdbg[i][c] = r["points"], r
    return ref, rdbg


def check_bar(pts, dbg, ref, rdbg):
    b, oc = len(rdbg), len(rdbg[0])
    tn0, tn, rounds = (dbg[k].cpu().numpy() for k in ("tn0", "tn", "rounds"))
    counts, win_idx, win_pts, refined = (dbg[k].cpu().numpy() for k in ("counts", "win_idx", "win_pts", "refined"))
    for i in range(b):
        for c in range(oc):
            r = rdbg[i][c]
            assert (tn0[i, c], tn[i, c], rounds[i, c]) == (r["tn0"], r["tn"], r["rounds"]), (i, c)
            for k in range(r["rounds"]):
                assert np.array_equal(counts[i, c, k], r["counts"][k]), ("counts", i, c, k)
                assert np.array_equal(win_idx[i, c, k], r["win_idx"][k]), ("win_idx", i, c, k)
            assert np.array_equal(win_pts[i, c], r["win_pts"]), ("win_pts", i, c)
            assert int(refined[i, c]) == int(r["refined"]), ("refined", i, c)
    err = float(np.abs(pts.cpu().numpy() - ref).max())
    assert err <= TOL_PX, "refined keypoints differ by %g px" % err


def device_copy(a, misalign=0):
    """a on the GPU; misalign = k: the tensor starts k floats past an allocation (256-byte aligned) boundary."""
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    if not misalign:
        return t
    buf = torch.empty(t.numel() + misalign, device="cuda")
    v = buf[misalign:].view(t.shape)
    v.copy_(t)
    return v


def run(vote, mask, vertex, hn, *, seed=7, status=0, misalign_vertex=0, misalign_mask=0, seg=None, oracle_mask=None,
        idxs=None, selection=None, **kw):
    """Debug call against the oracle (the bar), status bits, and the graph-replayed call without debug outputs."""
    m = device_copy(seg if seg is not None else mask, misalign_mask)
    v = device_copy(vertex, misalign_vertex)
    if misalign_vertex:
        assert v.data_ptr() % 8 == 4
    extra = dict(kw, seed=seed, seg_scores=seg is not None)
    if idxs is not None:
        extra["idxs"] = torch.from_numpy(idxs).cuda()
    if selection is not None:
        extra["selection"] = torch.from_numpy(selection).cuda()
    pts, dbg = vote(m, v, hn, return_debug=True, **extra)
    torch.cuda.synchronize()
    okw = {k: kw[k] for k in ("inlier_thresh", "confidence", "max_iter", "min_num", "max_num", "image_offset") if k in kw}
    ref, rdbg = oracle(mask if oracle_mask is None else oracle_mask, vertex, hn, seed=seed, idxs=idxs,
                       selection=selection, **okw)
    check_bar(pts, dbg, ref, rdbg)
    assert dbg["status"] == status, "status 0x%x, expected 0x%x" % (dbg["status"], status)
    for _ in range(2):  # the first call without debug outputs builds the graph, the second patches and replays it
        assert torch.equal(vote(m, v, hn, **extra), pts)
    return pts, dbg, ref, rdbg


def last_status():
    from casapose_b200 import _lib

    st = C.c_uint32()
    _lib.check(_lib.lib().casa_last_status(_lib.handle(0), C.byref(st)))
    return st.value


@pytest.fixture(scope="module")
def vote(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from casapose_b200.pose_estimation import ransac_voting_layer_all_masks

    return ransac_voting_layer_all_masks


@pytest.fixture(scope="module")
def vote_host(cuda_lib):
    from casapose_b200.pose_estimation.ransac_voting import ransac_voting_layer_all_masks_host

    return ransac_voting_layer_all_masks_host


# ------------------------------------------------------------------------------------- CPU checks of the scenes
def test_scenes_hn_sweep_reaches_both_score_kernels_and_odd_pairs():
    assert {hn_class(hn) for hn in HN_SWEEP} == {"narrow", "wide"}
    assert [hn_class(hn) for hn in (1, 128, 129, 256, 257, 384, 385, 4096)] == \
        ["narrow", "narrow", "wide", "wide", "narrow", "narrow", "wide", "wide"]
    assert any(hn % 2 and hn_class(hn) == "wide" for hn in HN_SWEEP)  # a hypothesis without a pair partner
    _, _, lab = hn_scene("easy")
    assert [(lab == c + 1).sum() for c in range(2)] == [1280, 1050]


@pytest.mark.parametrize("kind", ["raster", "cross1024", "cross4096"])
def test_scenes_tile_edges(kind):
    _, _, lab = edge_scene(kind)
    flat = lab.reshape(-1)
    for c, ((s, n), want) in enumerate(zip(edge_ranges(kind), EDGE_TN)):
        idx = np.flatnonzero(flat == c + 1)
        assert idx.size == want and idx[0] == s and idx[-1] == s + n - 1
        if kind != "raster":
            tile = 1024 if kind == "cross1024" else 4096
            assert idx[0] // tile != idx[-1] // tile, (c, "does not cross a %d-pixel boundary" % tile)


def test_scenes_vn_and_caps():
    for vn in VN_SWEEP:
        mask, vertex, lab = vn_scene(vn)
        assert vertex.shape == (1, 48, 64, vn, 2)
    tn0 = mask.sum((0, 1, 2))
    assert tn0[0] < VN_CAP < tn0[1]  # one job gathered by k_place, one capped
    _, vpc, lab = vn_scene(9, per_class=2)
    assert vpc.shape == (1, 48, 64, 2, 9, 2)
    ys, xs = np.nonzero(lab[0] == 2)
    assert np.allclose(np.hypot(vpc[0, ys, xs, 1, :, 0], vpc[0, ys, xs, 1, :, 1]), 1, atol=1e-6)


@pytest.mark.parametrize("name", sorted(OC_CASES))
def test_scenes_classes(name):
    oc, h, w, misalign = OC_CASES[name]
    mask, _, lab = oc_scene(oc, h, w)
    counts = mask.sum((1, 2))
    assert (counts[:, oc - 1] > 0).all() and (counts[counts > 0] >= 5).all()
    vec4 = (h * w * oc) % 4 == 0 and not misalign
    assert vec4 == name.endswith("vec4")


@pytest.mark.parametrize("J", sorted(JOB_CASES))
def test_scenes_job_counts(J):
    b, oc = JOB_CASES[J]
    assert b * oc == J
    mask, vertex, lab = jobs_scene(b, oc)
    assert vertex is not None and mask.shape == (b, 12, 16, oc)
    tn0 = mask.sum((1, 2))
    assert (tn0 % 16 == 0).all() and tn0.max() <= 96 and tn0[:, oc - 1].max() > 0


def test_scenes_seg_argmax_rule():
    seg, lab = seg_scene()
    r = seg[0]
    assert (lab[0, 0:6, 0:16] == 2).all() and (lab[0, 6:12, 0:16] == 0).all()
    assert (lab[0, 12:18, 0:16] == 5).all() and (lab[0, 18:24, 0:16] == 1).all() and (lab[0, 24:30, 0:16] == 4).all()
    assert (np.argmax(r[12:18, 0:16], -1) == 3).all()  # np.argmax picks the NaN, the kernel's rule does not
    assert all((lab == c + 1).sum() >= 5 for c in range(SEG_OC))


def test_scenes_gates_and_shapes():
    mask, _, _ = gate_scene((4, 5, 19, 20, 300, 301))
    assert list(mask.sum((0, 1, 2))) == [4, 5, 19, 20, 300, 301]
    for name in SHAPE_CASES:
        mask, vertex, lab = shape_scene(name)
        n = int(mask.sum())
        assert 5 <= n <= 600, name
        ys, xs = np.nonzero(lab[0])
        if name.startswith("x65534"):
            assert xs.max() == 65534
        if name.startswith("y65534"):
            assert ys.max() == 65534
    assert (37 * 111) % 2 == 1 and all((37 * 111) % m for m in (4, 1024, 4096))


# ------------------------------------------------------------------------------------------- k_score, hn
@gpu
@pytest.mark.parametrize("variant", ["easy", "hard"])
@pytest.mark.parametrize("hn", HN_SWEEP, ids=["%s-hn%d" % (hn_class(hn), hn) for hn in HN_SWEEP])
def test_k_score_hypotheses_per_lane(vote, hn, variant):
    mask, vertex, _ = hn_scene(variant)
    _, _, _, rdbg = run(vote, mask, vertex, hn, max_iter=20 if variant == "easy" else 3)
    if variant == "hard":
        assert max(r["rounds"] for r in rdbg[0]) > 1, "the hard frame must take several rounds"


@gpu
def test_k_score_wide_hn4096_limit(vote):
    lab = box_labels(1, 24, 32, {0: (8, 20, 6, 26)})
    run(vote, one_hot(lab, 1), aimed_field(lab, 9, np.random.default_rng(9)), 4096, max_iter=2)


# ------------------------------------------------------------------------------- chunks and refinement tiles
@gpu
@pytest.mark.parametrize("kind", ["raster", "cross1024", "cross4096"])
def test_chunk_and_refine_tile_edges(vote, kind):
    mask, vertex, _ = edge_scene(kind)
    run(vote, mask, vertex, 64)


# ------------------------------------------------------------------------------------------ vn and gathers
ROUTES = {"fused": dict(), "capped": dict(max_num=VN_CAP), "misaligned": dict(misalign_vertex=1)}


def _route_id(route, vn):
    if route == "fused":
        return "place%d-vn%d" % (9 if vn == 9 else 0, vn)
    return "gather%d-%s-vn%d" % (18 if vn == 9 else 0, route, vn)


@gpu
@pytest.mark.parametrize("route,vn", [(r, vn) for r in ROUTES for vn in VN_SWEEP],
                         ids=[_route_id(r, vn) for r in ROUTES for vn in VN_SWEEP])
def test_keypoint_counts_on_each_gather(vote, route, vn):
    mask, vertex, _ = vn_scene(vn)
    _, dbg, _, _ = run(vote, mask, vertex, 48, max_iter=3, **ROUTES[route])
    if route == "capped":
        assert int(dbg["tn"][0, 1]) < int(dbg["tn0"][0, 1]) and int(dbg["tn"][0, 0]) == int(dbg["tn0"][0, 0])


# ----------------------------------------------------------------------------------------------- oc and J
@gpu
@pytest.mark.parametrize("name", sorted(OC_CASES))
def test_class_counts_and_the_top_membership_bit(vote, name):
    oc, h, w, misalign = OC_CASES[name]
    mask, vertex, _ = oc_scene(oc, h, w)
    _, dbg, _, _ = run(vote, mask, vertex, 32, max_iter=3, misalign_mask=misalign)
    assert (dbg["tn"][:, oc - 1] > 0).all()


@gpu
@pytest.mark.parametrize("J", sorted(JOB_CASES), ids=["k_plan-J%d" % j for j in sorted(JOB_CASES)])
def test_k_plan_job_counts(vote, J):
    b, oc = JOB_CASES[J]
    mask, vertex, _ = jobs_scene(b, oc)
    run(vote, mask, vertex, 16, max_iter=2)


# ------------------------------------------------------------------------------------------- mask forms
@gpu
def test_seg_scores_ties_first_maximum_and_nan_never_wins(vote):
    seg, lab = seg_scene()
    run(vote, one_hot(lab, SEG_OC), aimed_field(lab, 9, np.random.default_rng(10)), 32, max_iter=3, seg=seg)


@gpu
@pytest.mark.parametrize("oc", [8, 32], ids=["host-oc8", "host-oc32"])
def test_host_entry_packed_bits_and_mapped_field(vote, vote_host, oc):
    """casa_ransac_vote_host: the mask packed into membership words on host threads (k_bits_in), the pinned field read
    in place by k_gather_dirs; bit-equal to the device entry, which meets the oracle."""
    mask, vertex, _ = oc_scene(oc, 48, 64)
    pts, _, _, _ = run(vote, mask, vertex, 32, seed=11, max_iter=3)
    host = vote_host(torch.from_numpy(mask), torch.from_numpy(vertex).pin_memory(), 32, seed=11, max_iter=3)
    assert torch.equal(host, pts.cpu())
    assert last_status() == 0


# ------------------------------------------------------------------------------------------- mask values
@gpu
@pytest.mark.parametrize("path", ["vec4", "scalar"])
@pytest.mark.parametrize("kind", sorted(MASK_VALUES))
def test_mask_values(vote, path, kind):
    """-0.0 is not masked; NaN is masked (`!= 0`, like tf.not_equal) and, with 0.5 and 2.0, raises MASK_NOT_BINARY.
    The kernel counts masked pixels where the oracle sums the mask (foreground_num, ransac_voting.py:287); for these
    blocks both give the same gates, so the kernel meets the oracle on the raw mask and on the binarised one."""
    mask, vertex, _ = mask_value_scene(kind)
    status = MASK_VALUES[kind][1]
    run(vote, mask, vertex, 32, max_iter=3, status=status, misalign_mask=1 if path == "scalar" else 0)
    with np.errstate(invalid="ignore"):
        binary = (mask != 0).astype(F)
    run(vote, mask, vertex, 32, max_iter=3, status=status, oracle_mask=binary, misalign_mask=1 if path == "scalar" else 0)


@gpu
@pytest.mark.parametrize("value", [0.5, 2.0], ids=["half", "two"])
def test_non_binary_mask_gates_on_the_pixel_count(vote, value):
    """Where the sum and the count of a non-binary mask fall on different sides of a gate, the kernel gates on the
    count (documented in DESIGN.md): 4 pixels of 2.0 (sum 8) are gated at min_num = 5, 8 pixels of 0.5 (sum 4) are
    voted.  It then equals the oracle run on the binarised mask, and reports MASK_NOT_BINARY."""
    n = 4 if value == 2.0 else 8
    mask, vertex, _ = gate_scene((n, 40))
    mask[..., 0] *= F(value)
    binary = (mask != 0).astype(F)
    _, dbg, _, rdbg = run(vote, mask, vertex, 32, max_iter=3, status=NOT_BINARY, oracle_mask=binary)
    _, raw = oracle(mask, vertex, 32, seed=7, max_iter=3)
    assert (raw[0][0]["rounds"] > 0) == (value == 2.0) and (rdbg[0][0]["rounds"] > 0) == (value == 0.5)


# ------------------------------------------------------------------------------------------ per-class fields
@gpu
@pytest.mark.parametrize("route", ["place9-fused", "gather18-capped", "gather18-misaligned", "gather18-host"])
def test_vertex_per_class(vote, vote_host, route):
    mask, vertex, _ = vn_scene(9, per_class=2)
    kw = {"gather18-capped": dict(max_num=VN_CAP), "gather18-misaligned": dict(misalign_vertex=1)}.get(route, {})
    pts, _, _, _ = run(vote, mask, vertex, 48, max_iter=3, **kw)
    if route == "gather18-host":
        host = vote_host(torch.from_numpy(mask), torch.from_numpy(vertex).pin_memory(), 48, seed=7, max_iter=3)
        assert torch.equal(host, pts.cpu())


# ------------------------------------------------------------------------------------------------- gates
@gpu
@pytest.mark.parametrize("min_num", [5, 20])
def test_min_num_gate_edges(vote, min_num):
    mask, vertex, _ = gate_scene((4, 5, 19, 20))
    _, dbg, _, rdbg = run(vote, mask, vertex, 32, max_iter=3, min_num=min_num)
    assert [r["rounds"] > 0 for r in rdbg[0]] == [n >= min_num for n in (4, 5, 19, 20)]


@gpu
@pytest.mark.parametrize("sel", ["philox", "external"])
def test_max_num_cap_edges(vote, sel):
    mask, vertex, _ = gate_scene((300, 301))
    selection = np.random.default_rng(12).random((1, 2, 32, 64), dtype=F) if sel == "external" else None
    _, dbg, _, _ = run(vote, mask, vertex, 32, max_iter=3, max_num=300, selection=selection)
    assert int(dbg["tn"][0, 0]) == 300  # tn0 = max_num is not capped


@gpu
@pytest.mark.parametrize("sel", ["philox", "external"])
def test_cap_that_keeps_no_pixel(vote, sel):
    mask, vertex, _ = gate_scene((40, 60))
    kw = dict(max_num=0.0) if sel == "philox" else dict(max_num=30.0, selection=np.ones((1, 2, 32, 64), F))
    pts, dbg, _, _ = run(vote, mask, vertex, 32, max_iter=3, status=EMPTY_AFTER_CAP, **kw)
    assert dbg["tn"].cpu().numpy().tolist() == [[0, 0]] and not pts.any()


@gpu
def test_pix_capacity_exact_and_one_short(vote):
    """Overlapping channels list a pixel once per channel: the listed total is the capacity the call needs."""
    from casapose_b200 import _lib
    from casapose_b200._lib import CasaError

    mask, vertex, lab = vn_scene(9)
    mask[..., 1] = np.maximum(mask[..., 1], mask[..., 0])  # channel 1 = union of both boxes
    need = int(mask.sum())
    run(vote, mask, vertex, 32, max_iter=3, pix_capacity=need)
    m, v = torch.from_numpy(mask).cuda(), torch.from_numpy(vertex).cuda()
    with pytest.raises(CasaError):
        vote(m, v, 32, max_iter=3, pix_capacity=need - 1)
    assert last_status() == PIX_OVERFLOW
    stream = torch.cuda.current_stream().cuda_stream
    _lib.set_async(0, 2, stream)
    try:
        vote(m, v, 32, max_iter=3, pix_capacity=need - 1)
        _lib.join(0, stream)
        # CASA_ERR_WORKSPACE (-3) is the error of the PIX_OVERFLOW bit, whichever of the lane collection or casa_sync
        # reports it first
        with pytest.raises(CasaError, match=r"error -3: .*pix_capacity"):
            _lib.sync(0, stream)
    finally:
        _lib.set_async(0, 0, stream)


# ------------------------------------------------------------------------------------- shapes and coordinates
@gpu
@pytest.mark.parametrize("name", sorted(SHAPE_CASES))
def test_image_shapes_and_16_bit_coordinates(vote, name):
    mask, vertex, _ = shape_scene(name)
    run(vote, mask, vertex, 32, max_iter=3)


@gpu
def test_image_offset_near_2_31_and_a_64_bit_seed(vote):
    lab = box_labels(2, 48, 64, VN_BOXES)
    mask, vertex = one_hot(lab, 2), aimed_field(lab, 9, np.random.default_rng(13))
    run(vote, mask, vertex, 32, seed=(0xDEADBEEF << 32) | 0x12345678, image_offset=2 ** 31 - 2, max_iter=3, max_num=530)


# -------------------------------------------------------------------------------------------------- rounds
@gpu
def test_max_iter_1_and_64(vote):
    mask, vertex, _ = hn_scene("hard")
    run(vote, mask, vertex, 64, max_iter=1)
    vertex = vertex.copy()
    vertex[..., 4, :] = 0.0  # keypoint 4 gets no votes: no round meets the stop test
    _, dbg, _, _ = run(vote, mask, vertex, 8, max_iter=64)
    assert (dbg["rounds"] == 64).all()


@gpu
def test_confidence_stop_in_round_one(vote):
    lab = box_labels(1, 48, 64, VN_BOXES)
    mask, vertex = one_hot(lab, 2), aimed_field(lab, 9, np.random.default_rng(14))
    _, dbg, _, _ = run(vote, mask, vertex, 128)
    assert (dbg["rounds"] == 1).all()


@gpu
def test_external_idxs_out_of_range_are_clamped(vote):
    """An index outside [0, tn) raises IDX_RANGE (CasaError on a synchronous call); the kernel clamps it to
    [0, tn - 1], so its keypoints are the oracle's on the clamped indices."""
    from casapose_b200._lib import CasaError

    mask, vertex, _ = vn_scene(9)
    tn = mask.sum((1, 2)).astype(np.int64)[0]
    hn, mi = 32, 2
    rng = np.random.default_rng(15)
    idxs = np.stack([rng.integers(0, tn[c], size=(mi, hn, 9, 2)) for c in range(2)])[None].astype(np.int32)
    idxs[0, 0, 0, 3, 2, 1] = tn[0] + 7
    idxs[0, 1, 1, 5, 0, 0] = -3
    clamped = np.minimum(np.maximum(idxs, 0), (tn - 1)[None, :, None, None, None, None]).astype(np.int32)
    out = torch.empty((1, 2, 9, 2), device="cuda")
    with pytest.raises(CasaError):
        vote(torch.from_numpy(mask).cuda(), torch.from_numpy(vertex).cuda(), hn, seed=7, max_iter=mi,
             idxs=torch.from_numpy(idxs).cuda(), out=out)
    assert last_status() == IDX_RANGE
    ref, _ = oracle(mask, vertex, hn, seed=7, max_iter=mi, idxs=clamped)
    assert float(np.abs(out.cpu().numpy() - ref).max()) <= TOL_PX
    run(vote, mask, vertex, hn, max_iter=mi, idxs=clamped)  # the clamped indices themselves pass the full bar


# ------------------------------------------------------------------------- the 64-bit row offset of k_gather_dirs
def _layout_limits():
    """make_layout's limits on the vote's shape, read from the source."""
    src = open(os.path.join(ROOT, "casapose_b200", "csrc", "casa_api.cu")).read()
    body = src[src.index("int make_layout("):]
    vn = int(re.search(r"p->vn > (\d+)", body).group(1))
    oc = int(re.search(r"p->oc > (\d+)", body).group(1))
    hw = 1 << int(re.search(r"p->h \* p->w > \(1ll << (\d+)\)", body).group(1))
    return hw, vn, oc


BIG_SHARED = (8190, 8200, 16)      # h, w, vn: h*w just above 2^26, shared field
BIG_PER_CLASS = (1450, 1450, 16, 32)  # h, w, vn, oc: h*w just above 2^21, one field per class


def test_largest_row_offset_exceeds_int32():
    """k_gather_dirs reads a listed pixel's row at float offset pixel * vn * vpc * 2 of the image's field (vpc = oc
    for per-class fields).  Within make_layout's limits that offset passes INT32_MAX, so it must be formed in 64 bits;
    the GPU regression cases below sit just past 2^31."""
    hw, vn, oc = _layout_limits()
    assert (hw, vn, oc) == (1 << 30, 16, 32)
    int32_max = 2 ** 31 - 1
    assert (hw - 1) * vn * oc * 2 > int32_max
    h, w, vn = BIG_SHARED
    assert h * w <= hw and (h * w - 1) * vn * 2 > int32_max
    assert 2 ** 26 * vn * 2 == 2 ** 31  # shared field: from pixel 2^26 on
    h, w, vn, oc = BIG_PER_CLASS
    assert (h * w - 1) * vn * oc * 2 > int32_max and 2 ** 21 * vn * oc * 2 == 2 ** 31


def _free_bytes():
    return torch.cuda.mem_get_info()[0]


def _big_vote(vote, h, w, vn, oc, cls, rows, x0, x1, target):
    """One image on the device, zero except class `cls`: rows `rows`, columns x0..x1, all directions aimed at
    `target` (x, y).  Voted from the aligned field (k_place) and from a copy 4 bytes past alignment
    (k_gather_dirs); returns both results."""
    per_class = oc > 1
    shape = (1, h, w, oc, vn, 2) if per_class else (1, h, w, vn, 2)
    mask = torch.zeros((1, h, w, oc), device="cuda")
    mask[0, rows[0]:rows[1], x0:x1, cls] = 1.0
    ys, xs = torch.meshgrid(torch.arange(rows[0], rows[1], device="cuda", dtype=torch.float64),
                            torch.arange(x0, x1, device="cuda", dtype=torch.float64), indexing="ij")
    dx, dy = target[0] - (xs + 0.5), target[1] - (ys + 0.5)
    n = torch.sqrt(dx * dx + dy * dy)
    dirs = torch.stack([dy / n, dx / n], -1).float()[:, :, None, :].expand(-1, -1, vn, -1)
    field = torch.zeros(shape, device="cuda")
    if per_class:
        field[0, rows[0]:rows[1], x0:x1, cls] = dirs
    else:
        field[0, rows[0]:rows[1], x0:x1] = dirs
    cap = 4096
    pts_a, dbg_a = vote(mask, field, 64, seed=3, return_debug=True, pix_capacity=cap)
    torch.cuda.synchronize()
    buf = torch.empty(field.numel() + 1, device="cuda")
    off = buf[1:].view(shape)
    off.copy_(field)
    del field
    assert off.data_ptr() % 8 == 4
    pts_b, dbg_b = vote(mask, off, 64, seed=3, return_debug=True, pix_capacity=cap)
    torch.cuda.synchronize()
    del off, buf
    return (pts_a, dbg_a), (pts_b, dbg_b)


@gpu
@pytest.mark.parametrize("case", ["shared-vn16-8190x8200", "per-class-oc32-vn16-1450x1450"])
def test_gather_row_offset_past_2_31(vote, case):
    """A small object in the last rows, where pixel * vn * vpc * 2 > 2^31: k_gather_dirs (field 4 bytes past
    alignment) gives the bits of the fused gather of k_place, and the keypoints are the point the field aims at."""
    need = 18.5e9
    if _free_bytes() < need:
        pytest.skip("needs %.1f GB of free device memory" % (need / 1e9))
    if case.startswith("shared"):
        h, w, vn = BIG_SHARED
        oc, cls, rows, x0, x1 = 1, 0, (h - 4, h), 4000, 4100
        assert rows[0] * w * vn * 2 > 2 ** 31
    else:
        h, w, vn, oc = BIG_PER_CLASS
        cls, rows, x0, x1 = oc - 1, (h - 3, h), 600, 700
        assert rows[0] * w * vn * oc * 2 > 2 ** 31
    target = (float(x0 + 50.25), float(rows[0] - 36.5))
    (pa, da), (pb, db) = _big_vote(vote, h, w, vn, oc, cls, rows, x0, x1, target)
    try:
        assert torch.equal(pa, pb)
        for k in ("tn0", "tn", "rounds", "counts", "win_idx", "win_pts", "refined"):
            assert torch.equal(da[k], db[k]), k
        assert da["status"] == 0 and db["status"] == 0
        assert int(da["tn"][0, cls]) == (rows[1] - rows[0]) * (x1 - x0) and int(da["refined"][0, cls]) == 1
        err = (pa[0, cls].double().cpu() - torch.tensor(target, dtype=torch.float64)).abs().max().item()
        assert err <= TOL_PX, "keypoints %g px from the target" % err
    finally:
        del pa, pb, da, db
        torch.cuda.empty_cache()
