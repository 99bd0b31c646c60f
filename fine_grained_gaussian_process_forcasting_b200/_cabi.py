"""ctypes binding of libgpblur.so (include/gpblur.h).  No torch types cross this boundary: only raw
device pointers, sizes and the CUDA stream handle.

The product path has NO CPU / eager fallback: if the library is missing this module raises, and every
op in ``ops.py`` refuses non-CUDA tensors.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libgpblur.so"

GPBLUR_MAX_D = 128
GPBLUR_MAX_M = 1024

# covariance functions (GPBLUR_KERNEL_*): name used by ops.py -> kind
KERNEL_KINDS = {"rbf": 0, "matern12": 1, "matern32": 2, "matern52": 3, "rq": 4}

ERRORS = {
    -1: "GPBLUR_EINVAL (bad shape / null pointer / misaligned workspace)",
    -2: "GPBLUR_EWORKSPACE (workspace too small)",
    -3: "GPBLUR_ELAUNCH (CUDA launch failure)",
    -4: "GPBLUR_EUNSUPPORTED (D > 128 or M > 1024)",
}


class SvgpParams(C.Structure):
    """struct gpblur_svgp_params"""
    _fields_ = [
        ("inducing_points", C.c_void_p),
        ("raw_lengthscale", C.c_void_p),
        ("raw_outputscale", C.c_void_p),
        ("variational_mean", C.c_void_p),
        ("variational_stddev", C.c_void_p),
        ("mean_weights", C.c_void_p),
        ("mean_bias", C.c_void_p),
        ("raw_alpha", C.c_void_p),
    ]


# name -> (restype, argtypes); must list every symbol declared in include/gpblur.h
SIGNATURES = {
    "gpblur_svgp_grad_bucket_floats": (C.c_size_t, [C.c_int, C.c_int]),
    "gpblur_svgp_grad_bucket_floats_kind": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "gpblur_svgp_workspace_bytes": (C.c_size_t, [C.c_longlong, C.c_int, C.c_int, C.c_int]),
    "gpblur_svgp_forward": (C.c_int, [
        C.POINTER(SvgpParams), C.c_void_p, C.c_longlong, C.c_int, C.c_int,
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
        C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gpblur_svgp_param_stage_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "gpblur_svgp_backward": (C.c_int, [
        C.POINTER(SvgpParams), C.c_void_p, C.c_longlong, C.c_int, C.c_int,
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
        C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gpblur_svgp_stage_grad_doubles": (C.c_size_t, [C.c_int, C.c_int]),
    "gpblur_svgp_stage_grad_doubles_kind": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "gpblur_svgp_param_stage": (C.c_int, [
        C.POINTER(SvgpParams), C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
        C.c_size_t, C.c_void_p]),
    "gpblur_svgp_point_forward": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
        C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gpblur_svgp_point_backward": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
        C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
        C.c_size_t, C.c_void_p]),
    "gpblur_svgp_param_stage_backward": (C.c_int, [
        C.POINTER(SvgpParams), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
        C.c_void_p, C.c_size_t, C.c_void_p]),
    "gpblur_covariance": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
        C.c_void_p, C.c_void_p]),
    "gpblur_covariance_alpha": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
        C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpblur_covariance_backward_scratch_bytes": (C.c_size_t, [C.c_longlong, C.c_longlong, C.c_int, C.c_int]),
    "gpblur_covariance_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_int,
                                             C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "gpblur_covariance_backward_alpha": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int,
                                                   C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_size_t, C.c_void_p]),
    "gpblur_step_scratch_floats": (C.c_size_t, [C.c_int]),
    "gpblur_blur_apply_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int,
                                            C.c_void_p, C.c_void_p]),
    "gpblur_blur_apply_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpblur_loss_forward": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_longlong, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "gpblur_loss_backward": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "gpblur_window_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_longlong, C.c_int,
                                       C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpblur_ata_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong,
                                     C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpblur_ata_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                      C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    "gpblur_ata_forward_fused_stacks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong,
                                                  C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                  C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpblur_ata_backward_fused_stacks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong,
                                                   C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                   C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpblur_peer_comm_bytes": (C.c_size_t, [C.c_longlong]),
    "gpblur_peer_alloc": (C.c_int, [C.c_size_t, C.c_void_p, C.c_void_p]),
    "gpblur_peer_open": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gpblur_peer_close": (C.c_int, [C.c_void_p]),
    "gpblur_peer_free": (C.c_int, [C.c_void_p]),
    "gpblur_peer_allreduce": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_float, C.c_void_p]),
    "gpblur_elbo_forward": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
        C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]),
    "gpblur_elbo_backward": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
        C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpblur_elbo_backward_fused": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
        C.c_longlong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpblur_philox_bits": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_longlong, C.c_void_p, C.c_void_p]),
    "gpblur_philox_normal": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_longlong, C.c_void_p, C.c_void_p]),
    "gpblur_rsample_forward": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_longlong, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]),
    "gpblur_rsample_backward": (C.c_int, [
        C.c_void_p, C.c_void_p, C.c_longlong, C.c_uint64, C.c_uint64, C.c_uint32,
        C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpblur_debug_fetch": (C.c_int, [
        C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
        C.POINTER(C.c_int), C.c_void_p]),
    "gpblur_profile_enable": (C.c_int, [C.c_int]),
    "gpblur_debug_set_trace": (C.c_int, [C.c_void_p]),
    "gpblur_profile_collect": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_ulonglong), C.c_int]),
    "gpblur_launch_count": (C.c_ulonglong, []),
    "gpblur_last_cuda_error": (C.c_char_p, []),
    "gpblur_version": (C.c_char_p, []),
}

_lib = None


class GpblurLibraryMissing(ImportError):
    pass


def lib() -> C.CDLL:
    """Load libgpblur.so (once).  Fails loudly: there is no fallback implementation."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("GPBLUR_LIB", LIB_PATH))
    if not path.exists():
        raise GpblurLibraryMissing(
            f"{path} not found: the CUDA extension is not built.  Run "
            f"`python -m fine_grained_gaussian_process_forcasting_b200.build` (needs nvcc); "
            f"this package has no CPU or eager-PyTorch fallback.")
    handle = C.CDLL(str(path))
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(handle, name)   # AttributeError if the symbol is missing
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    detail = ""
    if rc == -3:
        detail = " : " + (lib().gpblur_last_cuda_error() or b"").decode()
    raise RuntimeError(f"{what} failed with {ERRORS.get(rc, rc)}{detail}")


STAGES = ("mm_fwd", "point_fwd", "point_bwd", "gram", "wx", "mm_bwd", "elbo_fwd", "elbo_bwd", "dx", "sg_reduce")


def profile_enable(on: bool) -> None:
    lib().gpblur_profile_enable(int(on))


def profile_collect() -> dict:
    """{stage: (total_ms, launches)} since the last collect (synchronises on the recorded events)."""
    n = len(STAGES)
    ms = (C.c_double * n)()
    cnt = (C.c_ulonglong * n)()
    check(lib().gpblur_profile_collect(ms, cnt, n), "gpblur_profile_collect")
    return {s: (float(ms[i]), int(cnt[i])) for i, s in enumerate(STAGES)}


def launch_count() -> int:
    return int(lib().gpblur_launch_count())
