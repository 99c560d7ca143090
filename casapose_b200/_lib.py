"""ctypes binding of libcasapose_b200.so (include/casapose_b200.h).

There is NO fallback: if the shared library is missing or a call fails, the Python layer raises.
PyTorch is used only as the carrier of device memory / streams (any ``__dlpack__`` exporter is
accepted and viewed zero-copy); no torch type crosses the C ABI.
"""
import ctypes as C
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("CASA_LIB_PATH") or os.path.join(CSRC, "libcasapose_b200.so")  # override: A/B runs only
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC", "-ldl", "-lpthread",
]

STATUS_BITS = {
    1: "MASK_NOT_BINARY",
    2: "PIX_OVERFLOW",
    4: "IDX_RANGE",
    8: "EMPTY_AFTER_CAP",
    16: "LS_NONFINITE",
}


class CasaError(RuntimeError):
    pass


class RansacParams(C.Structure):
    _fields_ = [
        ("b", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("oc", C.c_int32), ("vn", C.c_int32),
        ("round_hyp_num", C.c_int32), ("max_iter", C.c_int32),
        ("inlier_thresh", C.c_float), ("confidence", C.c_float), ("min_num", C.c_float), ("max_num", C.c_float),
        ("seed", C.c_uint64), ("image_offset", C.c_int32), ("pix_capacity", C.c_int32),
        ("force_exact", C.c_int32), ("vertex_per_class", C.c_int32),
    ]


class RansacDebug(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "tn0", "tn", "rounds", "counts", "win_idx", "hyps", "win_pts", "win_ratio",
        "ata", "atb", "refined", "pix", "pix_off", "stats")]


class LsParams(C.Structure):
    _fields_ = [
        ("b", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("num_classes", C.c_int32), ("vn", C.c_int32),
        ("sigmoid_weights", C.c_int32), ("filter_estimates", C.c_int32), ("second_largest", C.c_int32),
        ("min_component", C.c_int32), ("check_finite", C.c_int32), ("pix_capacity", C.c_int32),
    ]


class LsDebug(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("sums", "labels", "selected", "parent", "tn")]


EXPORTS = {
    # name: (restype, argtypes)
    "casa_version": (C.c_int, []),
    "casa_last_error": (C.c_char_p, []),
    "casa_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "casa_destroy": (C.c_int, [C.c_void_p]),
    "casa_ransac_workspace_bytes": (C.c_size_t, [C.POINTER(RansacParams)]),
    "casa_ransac_vote": (C.c_int, [C.c_void_p, C.POINTER(RansacParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.POINTER(RansacDebug), C.c_void_p]),
    "casa_ransac_vote_seg": (C.c_int, [C.c_void_p, C.POINTER(RansacParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.POINTER(RansacDebug), C.c_void_p]),
    "casa_ransac_vote_dlpack": (C.c_int, [C.c_void_p, C.POINTER(RansacParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                          C.c_void_p]),
    "casa_ransac_vote_host": (C.c_int, [C.c_void_p, C.POINTER(RansacParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    "casa_ransac_vote_host_async": (C.c_int, [C.c_void_p, C.POINTER(RansacParams), C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.POINTER(C.c_int64)]),
    "casa_host_wait": (C.c_int, [C.c_void_p, C.c_int64]),
    "casa_ls_vote": (C.c_int, [C.c_void_p, C.POINTER(LsParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.POINTER(LsDebug), C.c_void_p]),
    "casa_ls_vote_backward": (C.c_int, [C.c_void_p, C.POINTER(LsParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "casa_pnp": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                           C.c_void_p]),
    "casa_pnp_backward": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "casa_pose_errors": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "casa_set_async": (C.c_int, [C.c_void_p, C.c_int]),
    "casa_join": (C.c_int, [C.c_void_p, C.c_void_p]),
    "casa_sync": (C.c_int, [C.c_void_p]),
    "casa_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "casa_comm_init": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "casa_comm_attach": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "casa_comm_destroy": (C.c_int, [C.c_void_p]),
    "casa_allgather_points": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "casa_allgather_points_overlapped": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int]),
    "casa_gather_wait": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "casa_last_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "casa_last_launches": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "casa_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "casa_get_timing": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_uint64)]),
    "casa_selftest_pack": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int]),
    "casa_selftest_filter": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_float, C.c_float,
                                       C.POINTER(C.c_uint64)]),
    "casa_measure_fp32_peak": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

_lib = None
_lock = threading.Lock()
_handles = {}


def build(verbose=False):
    """Compile csrc/casa_api.cu for sm_100a into csrc/libcasapose_b200.so (nvcc cross-compiles without a GPU)."""
    src = os.path.join(CSRC, "casa_api.cu")
    cmd = ["nvcc"] + NVCC_FLAGS + ["-o", LIB_PATH, src]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise CasaError("nvcc failed:\n" + res.stdout + res.stderr)
    return res.stderr if verbose else LIB_PATH


def _sources_newer_than_lib():
    if os.environ.get("CASA_LIB_PATH"):
        return False
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    inc = os.path.join(_HERE, "..", "include", "casapose_b200.h")
    files = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))] + [inc]
    return any(os.path.exists(f) and os.path.getmtime(f) > t for f in files)


def lib():
    """Load the shared library, declaring every export of include/casapose_b200.h."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise CasaError(
                    "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(there is no CPU or PyTorch fallback for this path)" % LIB_PATH)
            L = C.CDLL(LIB_PATH)
            for name, (res, args) in EXPORTS.items():
                fn = getattr(L, name)  # AttributeError here = header and library disagree
                fn.restype = res
                fn.argtypes = args
            _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise CasaError("casapose_b200 error %d: %s" % (rc, lib().casa_last_error().decode()))


def handle(device, stream=0):
    """One library handle per (device, thread, CUDA stream).

    A handle owns one workspace and leaves refinement / solve running when a call returns, so two streams must
    never share one (include/casapose_b200.h: one handle per stream)."""
    key = (int(device), threading.get_ident(), int(stream or 0))
    h = _handles.get(key)
    if h is None:
        hp = C.c_void_p()
        check(lib().casa_create(int(device), C.byref(hp)))
        h = hp
        _handles[key] = h
    return h


def set_async(device, enable, stream=0):
    """Asynchronous calls on this (device, thread, stream) handle: consecutive votes queue back to back on the GPU;
    `sync(device)` waits for them and raises the first error any of them hit (casa_set_async / casa_sync)."""
    check(lib().casa_set_async(handle(device, stream), int(enable)))


def join(device, stream=0):
    """Two-lane mode (set_async(device, 2)): orders every vote issued so far on `stream` (casa_join)."""
    check(lib().casa_join(handle(device, stream), C.c_void_p(stream)))


def sync(device, stream=0):
    check(lib().casa_sync(handle(device, stream)))


def status_names(word):
    return [n for bit, n in STATUS_BITS.items() if word & bit]
