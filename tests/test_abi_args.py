"""Argument checks of the split-form SVGP entry points and the dense covariance (CPU).

Every call below has exactly one bad argument and must return GPBLUR_EINVAL before it touches the device: the
pointers are fake 256-byte aligned device addresses that are never dereferenced, so no GPU is needed.
"""
import ctypes as C
import math

import pytest

from fine_grained_gaussian_process_forcasting_b200 import _cabi

EINVAL = -1
D, M, N = 16, 32, 100
BASE = 0x7F0000000000


def dev(i):
    """Fake 256-byte aligned device address number i."""
    return BASE + i * (1 << 24)


def params():
    return _cabi.SvgpParams(*[dev(i) for i in range(1, 8)])


def stage_bytes():
    return int(_cabi.lib().gpblur_svgp_param_stage_bytes(D, M))


def param_stage(**kw):
    a = dict(kind=0, extra_jitter=0.0, max_ctas=0, stage=dev(10), nbytes=stage_bytes())
    a.update(kw)
    p = params()
    return _cabi.lib().gpblur_svgp_param_stage(C.byref(p), D, M, a["kind"], a["extra_jitter"], a["max_ctas"], dev(11),
                                               dev(12), a["stage"], a["nbytes"], None)


def param_stage_backward(**kw):
    a = dict(kind=0, stage_grad=dev(13), grad_bucket=dev(14), max_ctas=0, stage=dev(10), nbytes=stage_bytes())
    a.update(kw)
    p = params()
    return _cabi.lib().gpblur_svgp_param_stage_backward(C.byref(p), D, M, a["kind"], a["stage_grad"], dev(15),
                                                        a["grad_bucket"], 0, a["max_ctas"], a["stage"], a["nbytes"],
                                                        None)


def point_forward(**kw):
    a = dict(stage=dev(10), kind=0, ws=dev(20))
    a.update(kw)
    ws_bytes = int(_cabi.lib().gpblur_svgp_workspace_bytes(N, D, M, 1))
    return _cabi.lib().gpblur_svgp_point_forward(a["stage"], dev(21), N, D, M, a["kind"], dev(22), dev(23), dev(24),
                                                 1, 0, 0, None, 1, a["ws"], ws_bytes, None)


def point_backward(**kw):
    a = dict(stage=dev(10), kind=0, starts=[0], stage_grad=dev(25))
    a.update(kw)
    nseg = a["nseg"] if "nseg" in a else len(a["starts"])
    starts = None if a["starts"] is None else (C.c_longlong * max(len(a["starts"]), 1))(*a["starts"])
    grads = [(C.c_void_p * 4)(*[dev(30 + 4 * k + s) for s in range(4)]) for k in range(3)]
    ws_bytes = int(_cabi.lib().gpblur_svgp_workspace_bytes(N, D, M, 1))
    return _cabi.lib().gpblur_svgp_point_backward(a["stage"], dev(21), N, D, M, a["kind"], nseg, starts, *grads,
                                                  dev(23), 1, 0, 0, None, dev(26), a["stage_grad"], dev(20), ws_bytes,
                                                  None)


@pytest.mark.parametrize("bad", [
    dict(kind=7), dict(kind=-1), dict(extra_jitter=-1.0), dict(extra_jitter=math.nan), dict(max_ctas=-1),
    dict(stage=dev(10) + 4), dict(stage=None),
])
def test_param_stage_rejects(bad):
    assert param_stage(**bad) == EINVAL


@pytest.mark.parametrize("bad", [
    dict(kind=4), dict(max_ctas=-1), dict(stage=dev(10) + 128), dict(stage=None), dict(stage_grad=None),
    dict(grad_bucket=None),
])
def test_param_stage_backward_rejects(bad):
    assert param_stage_backward(**bad) == EINVAL


@pytest.mark.parametrize("bad", [
    dict(kind=7), dict(stage=None), dict(stage=dev(10) + 16), dict(ws=dev(20) + 64),
])
def test_point_forward_rejects(bad):
    assert point_forward(**bad) == EINVAL


@pytest.mark.parametrize("bad", [
    dict(kind=9), dict(starts=[], nseg=0), dict(starts=[0, 10, 20, 30, 40]), dict(starts=[1]),
    dict(starts=[0, 50, 40]), dict(starts=[0, N + 1]), dict(starts=None, nseg=1), dict(stage=dev(10) + 8),
    dict(stage_grad=None),
])
def test_point_backward_rejects(bad):
    assert point_backward(**bad) == EINVAL


def test_covariance_rejects_unknown_kind():
    lib = _cabi.lib()
    assert lib.gpblur_covariance(dev(1), dev(2), 10, 12, D, 9, dev(3), 1, dev(4), dev(5), None) == EINVAL
    assert lib.gpblur_covariance_backward_scratch_bytes(10, 12, D, 9) == 0
    nbytes = int(lib.gpblur_covariance_backward_scratch_bytes(10, 12, D, 0))
    assert lib.gpblur_covariance_backward(dev(1), dev(2), 10, 12, D, 9, dev(3), 1, dev(4), dev(5), dev(6), dev(7),
                                          dev(8), dev(9), dev(10), nbytes, None) == EINVAL
