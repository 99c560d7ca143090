"""The C-ABI library loads without a GPU and exports every symbol include/casapose_b200.h declares."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _declared():
    text = open(os.path.join(ROOT, "include", "casapose_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(casa_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_expected_entry_points():
    names = _declared()
    for must in ("casa_create", "casa_destroy", "casa_last_error", "casa_ransac_vote", "casa_ransac_vote_host",
                 "casa_ransac_workspace_bytes", "casa_selftest_filter", "casa_measure_fp32_peak"):
        assert must in names


def test_library_exports_every_declared_symbol(cuda_lib):
    from casapose_b200 import _lib

    raw = C.CDLL(_lib.LIB_PATH)
    for name in _declared():
        assert hasattr(raw, name), "library does not export %s" % name
    # and the Python binding table covers the header
    assert sorted(_lib.EXPORTS) == _declared()


def test_version_and_error_without_gpu(cuda_lib):
    from casapose_b200 import _lib

    assert cuda_lib.casa_version() == 100
    p = _lib.RansacParams(b=1, h=480, w=640, oc=8, vn=9, round_hyp_num=512, max_iter=20, inlier_thresh=0.99,
                          confidence=0.99, min_num=5, max_num=30000)
    assert cuda_lib.casa_ransac_workspace_bytes(C.byref(p)) > 480 * 640 * 4
    bad = _lib.RansacParams(b=1, h=480, w=640, oc=40, vn=9, round_hyp_num=512, max_iter=20)
    assert cuda_lib.casa_ransac_workspace_bytes(C.byref(bad)) == 0
    assert b"oc=40" in cuda_lib.casa_last_error()


NO_DEVICE_SCRIPT = r'''
import sys
sys.path.insert(0, %(root)r)
import torch
from casapose_b200 import _lib
from casapose_b200.pose_estimation import ransac_voting_layer_all_masks

assert not torch.cuda.is_available()
try:
    _lib.handle(0)
    raise SystemExit("a handle was created without a device")
except _lib.CasaError:
    pass
try:
    ransac_voting_layer_all_masks(torch.zeros(1, 8, 8, 2), torch.zeros(1, 8, 8, 9, 2), 16)
    raise SystemExit("host tensors were accepted by the device entry point")
except ValueError:
    pass
print("no fallback ok")
'''


def test_product_path_fails_loudly_without_cuda(cuda_lib):
    """No CPU fallback: without a device the handle cannot be created and the Python layer raises.  Runs in a
    subprocess that sees no device, so that it checks the same on a machine with GPUs."""
    import subprocess
    import sys

    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", NO_DEVICE_SCRIPT % {"root": ROOT}], capture_output=True, text=True,
                         timeout=300, env=env)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "no fallback ok" in res.stdout


def test_pipelined_host_entry_rejects_bad_arguments_without_gpu(cuda_lib):
    """casa_ransac_vote_host_async / casa_host_wait validate their arguments before touching a device."""
    from casapose_b200 import _lib

    ticket = C.c_int64(-1)
    p = _lib.RansacParams(b=1, h=8, w=8, oc=2, vn=9, round_hyp_num=16, max_iter=2, inlier_thresh=0.99, confidence=0.99,
                          min_num=5, max_num=30000)
    assert cuda_lib.casa_ransac_vote_host_async(None, C.byref(p), None, None, None, C.byref(ticket)) == -1
    assert b"NULL" in cuda_lib.casa_last_error()
    assert cuda_lib.casa_host_wait(None, 0) == -1
    assert ticket.value == -1


def test_header_is_plain_c(tmp_path):
    """The boundary is a C ABI: include/casapose_b200.h compiles as C99 with warnings on (plain pointers and sizes,
    no C++ or torch types in the signatures)."""
    import shutil
    import subprocess

    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    src = tmp_path / "hdr.c"
    src.write_text('#include "casapose_b200.h"\nint main(void) { return casa_version() == 0; }\n')
    res = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
