"""float16 and bfloat16 network outputs read natively by the RANSAC vote and the LS layer, forward and backward.

The contract: each 16-bit element is widened exactly to float32 at load and everything after that is the float32 path,
so every output of a 16-bit call is bit-identical to the float32 call on the upcast tensor (`x.float()`): keypoints,
every debug intermediate, status bits, rounds, gradients.  Every GPU case here compares bit patterns (`torch.equal` on
integer views, so NaN positions count too) against that float32 call.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from casapose_b200 import synthetic  # noqa: E402

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
HALF = [torch.float16, torch.bfloat16]
HALF_IDS = ["f16", "bf16"]
F32 = torch.float32


# ----------------------------------------------------------------------------------------------------------- helpers
def _bits(t):
    """Integer view of a tensor, so that equality compares bit patterns (NaN == NaN, -0 != +0)."""
    view = {torch.float32: torch.int32, torch.float64: torch.int64, torch.float16: torch.int16, torch.bfloat16: torch.int16}
    return t.contiguous().view(view[t.dtype]) if t.dtype in view else t


def _assert_bits_equal(a, b, what=""):
    if isinstance(a, dict):
        assert set(a) == set(b)
        for k in a:
            _assert_bits_equal(a[k], b[k], "%s[%s]" % (what, k))
        return
    if isinstance(a, (tuple, list)):
        assert len(a) == len(b), what
        for k, (x, y) in enumerate(zip(a, b)):
            _assert_bits_equal(x, y, "%s[%d]" % (what, k))
        return
    if isinstance(a, torch.Tensor):
        assert a.dtype == b.dtype and a.shape == b.shape, what
        assert torch.equal(_bits(a), _bits(b)), what
    else:
        assert a == b, what


def _offset_view(t):
    """Copy of t that starts one element into its allocation (2-byte aligned for 16-bit types)."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


def _frames(b=2, h=120, w=160, ids=(1, 5, 6), variant="easy", **kw):
    return synthetic.make_frames(b, h, w, ids, variant=variant, **kw)


def _vote(mask, vertex, hn=64, **kw):
    from casapose_b200.pose_estimation import ransac_voting_layer_all_masks

    out, dbg = ransac_voting_layer_all_masks(mask, vertex, hn, seed=7, return_debug=True, debug_hyps=True, **kw)
    torch.cuda.synchronize()
    return out, dbg


def _check_vote(mask, vertex, mdt, vdt, offset=False, **kw):
    """The vote on mask.to(mdt) / vertex.to(vdt) equals the float32 vote on their upcast copies, bit for bit."""
    m = mask.to(mdt)
    v = vertex.to(vdt)
    if offset:
        m, v = _offset_view(m), _offset_view(v)
    want = _vote(m.float(), v.float(), **kw)
    got = _vote(m, v, **kw)
    _assert_bits_equal(want[0], got[0], "out")
    _assert_bits_equal(want[1], got[1], "dbg")
    return got


@pytest.fixture(scope="module")
def gpu(cuda_lib):
    assert torch.cuda.is_available()
    return cuda_lib


# --------------------------------------------------------------------------------------------------- RANSAC vote
@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("pair", ["both", "f32mask", "f32field"])
def test_vote_dtype_pairs(gpu, dt, pair):
    d = _frames()
    mask, vertex = torch.from_numpy(d["mask"]).cuda(), torch.from_numpy(d["vertex"]).cuda()
    mdt = F32 if pair == "f32mask" else dt
    vdt = F32 if pair == "f32field" else dt
    _, dbg = _check_vote(mask, vertex, mdt, vdt)
    assert int(dbg["tn"].sum()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("case", ["oc8_vector", "oc3_scalar", "offset_by_one"])
def test_vote_mask_bits_paths(gpu, dt, case):
    """k_mask_bits' 128-bit path ((h*w*oc) % 8 == 0, 16-byte aligned base) and its scalar path (odd h*w*oc; a tensor
    one element into its allocation, which also moves the field off its pair alignment: k_gather_dirs gathers)."""
    if case == "oc8_vector":
        d = _frames(1, 120, 160, synthetic.CONFIG_8_IDS)
    elif case == "oc3_scalar":
        d = _frames(2, 121, 161)
    else:
        d = _frames(2, 120, 160)
    mask, vertex = torch.from_numpy(d["mask"]).cuda(), torch.from_numpy(d["vertex"]).cuda()
    _check_vote(mask, vertex, dt, dt, offset=case == "offset_by_one")


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("vn", [7, 16])
def test_vote_other_keypoint_counts(gpu, dt, vn):
    d = _frames()
    v = torch.from_numpy(d["vertex"]).cuda()
    vertex = v[..., :vn, :].contiguous() if vn < 9 else torch.cat([v, v.flip(3)[..., : vn - 9, :]], dim=3).contiguous()
    _check_vote(torch.from_numpy(d["mask"]).cuda(), vertex, dt, dt)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_vote_per_class_fields(gpu, dt):
    d = _frames()
    v = torch.from_numpy(d["vertex"]).cuda()
    per_class = torch.stack([v, -v, v.flip(3)], dim=3).contiguous()  # [b,h,w,oc,vn,2]
    _check_vote(torch.from_numpy(d["mask"]).cuda(), per_class, dt, dt)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_vote_cap_multi_round_and_gated_classes(gpu, dt):
    """max_num below the class sizes (k_gather_dirs gathers only the capped jobs), the hard scene (several rounds),
    and min_num above the smallest class (gated jobs)."""
    d = _frames(2, 120, 160, variant="hard")
    mask, vertex = torch.from_numpy(d["mask"]).cuda(), torch.from_numpy(d["vertex"]).cuda()
    _, dbg = _check_vote(mask, vertex, dt, dt, max_num=300, max_iter=6)
    assert int(dbg["rounds"].max()) > 1
    assert bool((dbg["tn"] < dbg["tn0"]).any())
    tn0 = d["mask"].sum(axis=(1, 2))
    gate = float(np.sort(tn0[tn0 > 0].ravel())[0]) + 1
    _check_vote(mask, vertex, dt, dt, min_num=gate)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_vote_odd_mask_values(gpu, dt):
    """A non-binary mask (status bit), -0 (not set) and NaN (set, like tf.not_equal) mask elements."""
    d = _frames()
    mask = torch.from_numpy(d["mask"]).cuda()
    m = mask.clone()
    m[0, 10:20, 10:20, 0] = 0.5
    _, dbg = _check_vote(m, torch.from_numpy(d["vertex"]).cuda(), dt, dt)
    assert dbg["status"] & 1
    m = mask.clone()
    m[m == 0] = -0.0
    m[1, 50:52, 60:70, 1] = float("nan")
    _check_vote(m, torch.from_numpy(d["vertex"]).cuda(), dt, dt)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_vote_non_finite_and_subnormal_directions(gpu, dt):
    d = _frames()
    v = torch.from_numpy(d["vertex"]).cuda()
    v[0, 40:44, :, 0, 0] = float("nan")
    v[0, 44:48, :, 1, 1] = float("inf")
    v[1, 40:44, :, 2, 0] = float("-inf")
    tiny = torch.finfo(dt).tiny / 4  # subnormal in the 16-bit type
    v[1, 44:60, :, 3, :] = tiny
    v[1, 60:64, :, 4, 0] = -0.0
    _check_vote(torch.from_numpy(d["mask"]).cuda(), v, dt, dt)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_seg_scores_with_heavy_ties(gpu, dt):
    """Scores on three levels, the labelled class on the top one plus less than a 16-bit step: the maximum ties on most
    pixels once the scores are rounded to 16 bits, and the first maximum still wins."""
    d = _frames()
    rng = np.random.default_rng(3)
    b, h, w, oc = d["mask"].shape
    seg = rng.integers(0, 3, (b, h, w, oc + 1)).astype(np.float32)
    top = np.eye(oc + 1, dtype=bool)[d["labels"]]
    seg[top] = 2 + rng.uniform(0, 1e-3, int(top.sum())).astype(np.float32)
    seg = torch.from_numpy(seg).cuda().to(dt)
    ties = (seg == seg.max(dim=-1, keepdim=True).values).sum(-1) > 1
    assert float(ties.float().mean()) > 0.2
    _check_vote(seg, torch.from_numpy(d["vertex"]).cuda(), dt, dt, seg_scores=True)


# ------------------------------------------------------------------------------------------------------- LS layer
def _ls_inputs(ids=(1, 5, 6), b=2, h=120, w=160):
    d = _frames(b, h, w, ids, with_logits=True)
    return (torch.from_numpy(d["seg_logits"]).cuda(), torch.from_numpy(d["vertex"].reshape(b, h, w, 18)).cuda(),
            torch.from_numpy(d["conf_logits"]).cuda())


def _check_ls(inp, dt, offset=False, debug=True, **kw):
    from casapose_b200.pose_estimation import CoordLSVotingWeighted

    layer = CoordLSVotingWeighted("ls", inp[0].shape[3], num_points=9, **kw)
    x = [t.to(dt) for t in inp]
    if offset:
        x = [_offset_view(t) for t in x]
    want = layer([t.float() for t in x], return_debug=debug)
    got = layer(x, return_debug=debug)
    torch.cuda.synchronize()
    _assert_bits_equal(want, got)
    return got


LS_MODES = [dict(), dict(sigmoid_weights=True), dict(filter_estimates=True),
            dict(filter_estimates=True, output_second_largest_component=True, sigmoid_weights=True)]
LS_MODE_IDS = ["plain", "sigm", "filt", "filt-second-sigm"]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("mode", LS_MODES, ids=LS_MODE_IDS)
@pytest.mark.parametrize("ids", [(1, 5, 6), synthetic.CONFIG_8_IDS], ids=["nc4", "nc9"])
def test_ls_forward(gpu, dt, mode, ids):
    inp = _ls_inputs(ids)
    _check_ls(inp, dt, debug=True, **mode)  # debug outputs (pixel-level components)
    _check_ls(inp, dt, debug=False, **mode)  # the graph-replayed forward (fused pass, run-based components)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("ids", [(1, 5, 6), synthetic.CONFIG_8_IDS], ids=["nc4", "nc9"])
def test_ls_forward_every_tensor_one_element_into_its_allocation(gpu, dt, ids):
    inp = _ls_inputs(ids)
    _check_ls(inp, dt, offset=True, debug=False, filter_estimates=True)
    _check_ls(inp, dt, offset=True, debug=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_ls_near_tied_logits_take_the_capacity_retry(gpu, dt):
    """Logits within a few units of 1e-6 of each other list pixels for several classes: the first attempt overflows
    h*w slots and the call is retried with the measured need."""
    seg, direct, conf = _ls_inputs()
    flat = torch.zeros_like(seg)
    flat[..., 1] = 1e-7
    _check_ls([flat, direct, conf], dt, debug=False)
    _check_ls([flat, direct, conf], dt, debug=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("filt", [False, True])
def test_ls_backward(gpu, dt, filt):
    from casapose_b200.pose_estimation import CoordLSVotingWeighted

    seg, direct, conf = _ls_inputs()
    layer = CoordLSVotingWeighted("ls", seg.shape[3], num_points=9, filter_estimates=filt)
    g = torch.randn(seg.shape[0], seg.shape[3] - 1, 9, 2, device="cuda")
    x = [t.to(dt) for t in (seg, direct, conf)]
    want = layer.backward([t.float() for t in x], g)
    got = layer.backward(x, g)
    torch.cuda.synchronize()
    assert got[0].dtype == got[1].dtype == F32
    _assert_bits_equal(want[0], got[0])
    _assert_bits_equal(want[1], got[1])
    # autograd: 16-bit leaves receive the float32 gradient rounded to their dtype
    d16 = x[1].clone().requires_grad_(True)
    c16 = x[2].clone().requires_grad_(True)
    (layer([x[0], d16, c16]) * g).sum().backward()
    assert d16.grad.dtype == dt and c16.grad.dtype == dt
    _assert_bits_equal(d16.grad, want[0].to(dt))
    _assert_bits_equal(c16.grad, want[1].to(dt))


@pytest.mark.gpu
def test_ls_mixed_dtypes_are_rejected(gpu):
    from casapose_b200.pose_estimation import CoordLSVotingWeighted

    seg, direct, conf = _ls_inputs()
    layer = CoordLSVotingWeighted("ls", seg.shape[3], num_points=9)
    with pytest.raises(TypeError):
        layer([seg, direct.bfloat16(), conf])
    with pytest.raises(TypeError):
        layer([seg.half(), direct.half(), conf.bfloat16()])
    with pytest.raises(TypeError):
        layer([seg.double(), direct.double(), conf.double()])


# ------------------------------------------------------------------------------------- one handle, several dtypes
@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [0, 4])
def test_alternating_dtypes_on_one_handle(gpu, lanes):
    """Calls of the same shape and different dtypes on one handle (and on four lanes): each dtype gets its own cached
    graph, so every call equals its own float32 reference."""
    from casapose_b200 import _lib
    from casapose_b200.pose_estimation import CoordLSVotingWeighted, ransac_voting_layer_all_masks

    d = _frames()
    mask, vertex = torch.from_numpy(d["mask"]).cuda(), torch.from_numpy(d["vertex"]).cuda()
    seg, direct, conf = _ls_inputs()
    layer = CoordLSVotingWeighted("ls", seg.shape[3], num_points=9, filter_estimates=True)
    order = [F32, torch.float16, torch.bfloat16] * 3
    want_v = {dt: ransac_voting_layer_all_masks(mask.to(dt).float(), vertex.to(dt).float(), 64, seed=3).clone() for dt in order[:3]}
    want_l = {dt: layer([t.to(dt).float() for t in (seg, direct, conf)]).clone() for dt in order[:3]}
    torch.cuda.synchronize()
    inputs = {dt: (mask.to(dt), vertex.to(dt), [t.to(dt) for t in (seg, direct, conf)]) for dt in order[:3]}
    if lanes:
        _lib.set_async(0, lanes)
    try:
        got = []
        for dt in order:
            m, v, ls_in = inputs[dt]
            got.append((dt, ransac_voting_layer_all_masks(m, v, 64, seed=3), layer(ls_in, check_finite=False)))
        if lanes:
            _lib.join(0)
        got = [(dt, a.clone(), b.clone()) for dt, a, b in got]
        if lanes:
            _lib.sync(0)
    finally:
        if lanes:
            _lib.set_async(0, 0)
    torch.cuda.synchronize()
    for dt, a, b in got:
        _assert_bits_equal(want_v[dt], a, str(dt))
        _assert_bits_equal(want_l[dt], b, str(dt))


# ------------------------------------------------------------------------------------------------- DLPack and eval
@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF, ids=HALF_IDS)
def test_dlpack_16_bit_capsules_from_a_non_torch_exporter(gpu, dt):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from dlpack_exporter import DLManagedTensor, CudaBuffer, cudart

    from casapose_b200 import _lib, dlpack_api

    class TypedBuffer(CudaBuffer):
        """CudaBuffer holding raw 16- or 64-bit elements, exported with the given DLPack (code, bits)."""

        def __init__(self, raw, code, bits):
            super().__init__(shape=(raw.size * raw.itemsize // 4 + 1,))
            self.shape, self.code, self.bits = tuple(raw.shape), code, bits
            assert cudart().cudaMemcpy(self.ptr, raw.ctypes.data_as(C.c_void_p), raw.nbytes, 1) == 0

        def __dlpack__(self, stream=None):
            cap = super().__dlpack__(stream)
            C.pythonapi.PyCapsule_GetPointer.restype = C.c_void_p
            C.pythonapi.PyCapsule_GetPointer.argtypes = [C.py_object, C.c_char_p]
            m = DLManagedTensor.from_address(C.pythonapi.PyCapsule_GetPointer(cap, b"dltensor"))
            m.dl_tensor.dtype.code, m.dl_tensor.dtype.bits = self.code, self.bits
            return cap

    code = 2 if dt == torch.float16 else 4
    d = _frames()
    m16, v16 = torch.from_numpy(d["mask"]).to(dt), torch.from_numpy(d["vertex"]).to(dt)
    raw = lambda t: t.view(torch.int16).numpy()  # noqa: E731
    b, oc, vn = m16.shape[0], m16.shape[3], v16.shape[3]
    want = CudaBuffer(shape=(b, oc, vn, 2))
    dlpack_api.ransac_voting_layer_all_masks_dlpack(CudaBuffer(m16.float().numpy()), CudaBuffer(v16.float().numpy()), want, 64, seed=5)
    for mm, vv in ((TypedBuffer(raw(m16), code, 16), TypedBuffer(raw(v16), code, 16)),
                   (CudaBuffer(m16.float().numpy()), TypedBuffer(raw(v16), code, 16))):
        out = CudaBuffer(shape=(b, oc, vn, 2))
        dlpack_api.ransac_voting_layer_all_masks_dlpack(mm, vv, out, 64, seed=5)
        _lib.sync(0)
        assert np.array_equal(want.numpy().view(np.int32), out.numpy().view(np.int32))
        assert (mm.deleter_calls, vv.deleter_calls, out.deleter_calls) == (1, 1, 1)
    # float64 capsules are still rejected in C, and every capsule is released once
    mm = TypedBuffer(d["mask"].astype(np.float64), 2, 64)
    vv, oo = TypedBuffer(raw(v16), code, 16), CudaBuffer(shape=(b, oc, vn, 2))
    with pytest.raises(_lib.CasaError, match="error -1"):
        dlpack_api.ransac_voting_layer_all_masks_dlpack(mm, vv, oo, 64, seed=5)
    assert (mm.deleter_calls, vv.deleter_calls, oo.deleter_calls) == (1, 1, 1)
    # a 16-bit `out` is rejected too: outputs stay float32
    bad_out = TypedBuffer(np.zeros((b, oc, vn, 2), np.int16), code, 16)
    with pytest.raises(_lib.CasaError, match="error -1"):
        dlpack_api.ransac_voting_layer_all_masks_dlpack(CudaBuffer(d["mask"]), CudaBuffer(d["vertex"]), bad_out, 64)
    assert bad_out.deleter_calls == 1


@pytest.mark.gpu
def test_device_evaluator_takes_bfloat16_outputs(gpu):
    from casapose_b200.pose_estimation import DeviceEvaluator
    from tests.test_gpu_pipeline import _inputs

    d, cams, offsets, kp3, target_seg, poses_gt, diam = _inputs()
    b, oc = diam.shape
    seg = torch.from_numpy(d["seg_logits"]).cuda().bfloat16()
    tgt = torch.from_numpy(target_seg).cuda()
    vert = torch.from_numpy(d["vertex"].reshape(b, 240, 320, 18)).cuda().bfloat16()
    ev = DeviceEvaluator(kp3[0, :, 0], cams[0], diam[0])
    s0, p0, k0 = ev(seg.float(), tgt, vert.float(), poses_gt[:, :, 0], offsets, seed=11)
    s1, p1, k1 = ev(seg, tgt, vert, poses_gt[:, :, 0], offsets, seed=11)
    _assert_bits_equal(k0, k1)
    _assert_bits_equal(p0, p1)
    for n in s0:
        assert np.array_equal(s0[n].view(np.int32), s1[n].view(np.int32)), n


# ----------------------------------------------------------------------------------------------------- no device
def test_host_entry_stays_float32_only():
    from casapose_b200.pose_estimation.ransac_voting import ransac_voting_layer_all_masks_host

    for dt in HALF:
        with pytest.raises(TypeError):
            ransac_voting_layer_all_masks_host(torch.zeros(1, 8, 8, 2, dtype=dt), torch.zeros(1, 8, 8, 9, 2, dtype=dt), 16)


def test_carrier_dtype_codes_match_the_header():
    import re

    from casapose_b200 import _carrier

    text = open(os.path.join(ROOT, "include", "casapose_b200.h")).read()
    codes = {n: int(v) for n, v in re.findall(r"CASA_(FLOAT32|FLOAT16|BFLOAT16) = (\d)", text)}
    assert codes == {"FLOAT32": 0, "FLOAT16": 1, "BFLOAT16": 2}
    assert _carrier.DTYPE_CODES == {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}
