"""Host-buffer entry (casa_ransac_vote_host): the status word and the launch count it reports cover exactly the image
ranges of the call, and its staged path (pageable vector field) returns what the device call returns."""
import ctypes as C

import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

NOT_BINARY = 1  # CASA_STATUS_MASK_NOT_BINARY
HN, SEED = 128, 77


@pytest.fixture
def fresh_handle(cuda_lib):
    """A handle of this test alone: the shared one carries lanes and state from other tests."""
    from casapose_b200 import _lib

    hp = C.c_void_p()
    _lib.check(cuda_lib.casa_create(0, C.byref(hp)))
    yield hp
    _lib.check(cuda_lib.casa_destroy(hp))


def _frames(b, seed, half_in=None):
    """[b,96,128,8] one-hot mask and [b,96,128,9,2] field; half_in: image whose first foreground value becomes 0.5."""
    from casapose_b200 import synthetic

    d = synthetic.make_frames(b, 96, 128, synthetic.CONFIG_8_IDS, seed=seed)
    mask, vertex = torch.from_numpy(d["mask"]), torch.from_numpy(d["vertex"])
    if half_in is not None:
        y, x, c = torch.nonzero(mask[half_in] == 1)[0].tolist()
        mask[half_in, y, x, c] = 0.5
    return mask, vertex


def _vote_params(mask, vertex, image_offset=0):
    from casapose_b200.pose_estimation.ransac_voting import _params

    b, h, w, oc = mask.shape
    return _params(b, h, w, oc, vertex.shape[3], HN, 0.99, 0.99, 20, 5, 30000, SEED, image_offset, 0, False)


def _host_vote(lib, hdl, mask, vertex):
    from casapose_b200 import _lib

    p = _vote_params(mask, vertex)
    out = torch.empty((mask.shape[0], mask.shape[3], vertex.shape[3], 2), dtype=torch.float32)
    _lib.check(lib.casa_ransac_vote_host(hdl, C.byref(p), mask.data_ptr(), vertex.data_ptr(), out.data_ptr()))
    return out


def _device_vote(lib, hdl, mask, vertex, image_offset=0):
    from casapose_b200 import _lib

    mask_d, vertex_d = mask.cuda(), vertex.cuda()
    p = _vote_params(mask, vertex, image_offset)
    out = torch.empty((mask.shape[0], mask.shape[3], vertex.shape[3], 2), dtype=torch.float32, device="cuda")
    _lib.check(lib.casa_ransac_vote(hdl, C.byref(p), mask_d.data_ptr(), vertex_d.data_ptr(), None, None, out.data_ptr(),
                                    None, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return out.cpu()


def _status(lib, hdl):
    from casapose_b200 import _lib

    s = C.c_uint32()
    _lib.check(lib.casa_last_status(hdl, C.byref(s)))
    return s.value


def _launches(lib, hdl):
    from casapose_b200 import _lib

    n = C.c_int64()
    _lib.check(lib.casa_last_launches(hdl, C.byref(n)))
    return n.value


@pytest.mark.parametrize("packed", [False, True], ids=["dma", "packed"])
def test_status_of_a_host_call_equals_the_device_call(cuda_lib, fresh_handle, monkeypatch, packed):
    # image 0 is the first of four ranges, each voted on a lane of its own: the status is the OR over the ranges
    if packed:
        monkeypatch.delenv("CASA_NO_HOST_PACK", raising=False)
    else:
        monkeypatch.setenv("CASA_NO_HOST_PACK", "1")  # every range is DMA-copied
    mask, vertex = _frames(8, 3, half_in=0)
    mask, vertex = mask.pin_memory(), vertex.pin_memory()
    got = _host_vote(cuda_lib, fresh_handle, mask, vertex)
    host_status = _status(cuda_lib, fresh_handle)
    want = _device_vote(cuda_lib, fresh_handle, mask, vertex)
    assert _status(cuda_lib, fresh_handle) & NOT_BINARY
    assert host_status & NOT_BINARY
    assert torch.equal(got, want)


def test_no_status_left_from_an_earlier_call(cuda_lib, fresh_handle, monkeypatch):
    from casapose_b200 import _lib

    monkeypatch.delenv("CASA_HOST_DEPTH", raising=False)  # two drivers: tickets 0 and 2 share one
    lib, hdl = cuda_lib, fresh_handle
    calls = [_frames(8, 4, half_in=7), _frames(8, 5), _frames(4, 6)]
    calls = [(m.pin_memory(), v.pin_memory()) for m, v in calls]
    outs = [torch.empty((m.shape[0], 8, 9, 2), dtype=torch.float32) for m, _ in calls]
    tickets = []

    def submit(i):
        m, v = calls[i]
        t = C.c_int64(-1)
        p = _vote_params(m, v)
        _lib.check(lib.casa_ransac_vote_host_async(hdl, C.byref(p), m.data_ptr(), v.data_ptr(), outs[i].data_ptr(),
                                                   C.byref(t)))
        tickets.append(t.value)

    submit(0)
    submit(1)
    _lib.check(lib.casa_host_wait(hdl, tickets[0]))
    assert _status(lib, hdl) & NOT_BINARY
    submit(2)  # b = 4 on the driver of the first call: two of its four lanes, the one that voted on the 0.5 idle
    _lib.check(lib.casa_host_wait(hdl, tickets[1]))
    assert _status(lib, hdl) == 0
    _lib.check(lib.casa_host_wait(hdl, tickets[2]))
    assert _status(lib, hdl) == 0


def test_launch_count_of_a_host_call(cuda_lib, fresh_handle):
    # 96 x 128 < max_num: no cap launches; the mapped field is gathered by k_gather_dirs, one launch per range more than
    # the device call, whose k_place gathers the directions itself
    mask, vertex = _frames(8, 7)
    mask, vertex = mask.pin_memory(), vertex.pin_memory()
    _host_vote(cuda_lib, fresh_handle, mask, vertex)
    host = _launches(cuda_lib, fresh_handle)
    dev = 0
    for k in range(4):
        _device_vote(cuda_lib, fresh_handle, mask[2 * k:2 * k + 2], vertex[2 * k:2 * k + 2], image_offset=2 * k)
        dev += _launches(cuda_lib, fresh_handle)
    assert host == dev + 4


@pytest.mark.parametrize("b", [1, 8])
def test_pageable_vector_field_is_staged(cuda_lib, fresh_handle, b):
    mask, vertex = _frames(b, 8)
    got = _host_vote(cuda_lib, fresh_handle, mask.pin_memory(), vertex)  # pageable field: copied in one piece
    host = _launches(cuda_lib, fresh_handle)
    want = _device_vote(cuda_lib, fresh_handle, mask, vertex)
    assert torch.equal(got, want)
    assert host == _launches(cuda_lib, fresh_handle)
