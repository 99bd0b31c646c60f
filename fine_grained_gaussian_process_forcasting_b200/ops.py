"""torch-facing ops over the gpblur C ABI: thin wrappers (device pointers + current CUDA stream in,
fresh tensors out), registered as ``torch.ops.gpblur.*`` custom ops, plus the autograd glue.

There is no CPU path: every op raises on non-CUDA tensors and the loader raises if libgpblur.so is
missing (``_cabi.lib``).
"""
from __future__ import annotations

import math

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _cabi

Tensor = torch.Tensor

# NVTX ranges around every op (forward ranges here, backward ranges inside the autograd Functions): visible in
# nsys / ncu --nvtx timelines; GPBLUR_NVTX=0 switches them off
import contextlib
import os

_NVTX = os.environ.get("GPBLUR_NVTX", "1") != "0"
_null_ctx = contextlib.nullcontext


def _ptr(t: Optional[Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    # raw handle of the current stream of the current device.  NOT torch.cuda.current_stream(): with device=None
    # that goes through torch.cuda.is_available() -> cudaGetDeviceCount on every call (~0.1 ms each here).
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "gpblur ops run only on CUDA tensors (B200 / sm_100a); there is no CPU fallback")


def _f32c(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _params_struct(Z, raw_ell, raw_os, m, s, w, b, raw_alpha=None) -> _cabi.SvgpParams:
    return _cabi.SvgpParams(Z.data_ptr(), raw_ell.data_ptr(), raw_os.data_ptr(), m.data_ptr(), s.data_ptr(),
                            None if w is None else w.data_ptr(), b.data_ptr(),
                            None if raw_alpha is None else raw_alpha.data_ptr())


def grad_bucket_floats(D: int, M: int, kind: int = 0) -> int:
    """Floats of the flat parameter-gradient bucket; the rational quadratic kind appends d raw_alpha."""
    return M * D + 2 * M + 2 * D + 2 + (1 if kind == _cabi.KERNEL_KINDS["rq"] else 0)


_WS_BYTES_CACHE = {}


def workspace_bytes(N: int, D: int, M: int, training: bool) -> int:
    key = (N, D, M, bool(training))
    n = _WS_BYTES_CACHE.get(key)
    if n is None:
        n = int(_cabi.lib().gpblur_svgp_workspace_bytes(N, D, M, int(training)))
        if len(_WS_BYTES_CACHE) < 4096:
            _WS_BYTES_CACHE[key] = n
    return n


# ------------------------------------------------------------------------------------------------
# raw calls
# ------------------------------------------------------------------------------------------------
_STAGE_BYTES_CACHE = {}


def param_stage_bytes(D: int, M: int) -> int:
    n = _STAGE_BYTES_CACHE.get((D, M))
    if n is None:
        n = int(_cabi.lib().gpblur_svgp_param_stage_bytes(D, M))
        if n == 0:
            raise RuntimeError(f"unsupported SVGP shape D={D} M={M} (D <= {_cabi.GPBLUR_MAX_D}, "
                               f"M <= {_cabi.GPBLUR_MAX_M})")
        _STAGE_BYTES_CACHE[(D, M)] = n
    return n


def svgp_forward_raw(x: Tensor, Z: Tensor, raw_ell: Tensor, raw_os: Tensor, m: Tensor, s: Tensor,
                     w: Optional[Tensor], b: Tensor, seed: int, offset: int, stream_id: int,
                     want_sample: bool, training: bool):
    """x [N, D] -> (mean [N], var [N], sample [N] | None, kl [1], info [1] int32, workspace uint8)."""
    _need_cuda(x, Z, raw_ell, raw_os, m, s, w, b)
    N, D = x.shape
    M = Z.shape[0]
    dev = x.device
    out = torch.empty((3 if want_sample else 2) * N + 1, device=dev, dtype=torch.float32)   # one allocation
    mean, var = out[:N], out[N:2 * N]
    sample = out[2 * N:3 * N] if want_sample else None
    kl = out[-1:]
    info = torch.empty(1, device=dev, dtype=torch.int32)
    ws = torch.empty(workspace_bytes(N, D, M, training), device=dev, dtype=torch.uint8)
    p = _params_struct(Z, raw_ell, raw_os, m, s, w, b)
    with torch.cuda.device(dev):
        rc = _cabi.lib().gpblur_svgp_forward(
            C.byref(p), _ptr(x), N, D, M, _ptr(mean), _ptr(var), _ptr(sample),
            seed & 0xFFFFFFFFFFFFFFFF, offset & 0xFFFFFFFFFFFFFFFF, stream_id & 0xFFFFFFFF,
            _ptr(kl), _ptr(info), int(training), _ptr(ws), ws.numel(), _stream())
    _cabi.check(rc, "gpblur_svgp_forward")
    return mean, var, sample, kl, info, ws


def svgp_backward_raw(x, Z, raw_ell, raw_os, m, s, w, b, g_mean, g_var, g_sample, g_kl, var, seed, offset,
                      stream_id, ws, need_dx: bool = True):
    """-> (dx [N, D] | None, bucket [M*D + 2M + 2D + 2])."""
    _need_cuda(x, Z, ws, g_mean, g_var, g_sample, g_kl, var)
    N, D = x.shape
    M = Z.shape[0]
    dev = x.device
    dx = torch.empty(N, D, device=dev, dtype=torch.float32) if need_dx else None
    bucket = torch.empty(grad_bucket_floats(D, M), device=dev, dtype=torch.float32)
    p = _params_struct(Z, raw_ell, raw_os, m, s, w, b)
    with torch.cuda.device(dev):
        rc = _cabi.lib().gpblur_svgp_backward(
            C.byref(p), _ptr(x), N, D, M, _ptr(g_mean), _ptr(g_var), _ptr(g_sample), _ptr(g_kl), _ptr(var),
            seed & 0xFFFFFFFFFFFFFFFF, offset & 0xFFFFFFFFFFFFFFFF, stream_id & 0xFFFFFFFF,
            _ptr(dx), _ptr(bucket), _ptr(ws), ws.numel(), _stream())
    _cabi.check(rc, "gpblur_svgp_backward")
    return dx, bucket


def split_bucket(bucket: Tensor, D: int, M: int, has_weights: bool, kernel: str = "rbf"):
    """Views of the flat gradient bucket in parameter order (see include/gpblur.h); `kernel` "rq" appends the view of
    d raw_alpha."""
    o = 0
    dZ = bucket[o:o + M * D].view(M, D); o += M * D
    dell = bucket[o:o + D]; o += D
    dos = bucket[o:o + 1]; o += 1
    dm = bucket[o:o + M]; o += M
    ds = bucket[o:o + M]; o += M
    dw = bucket[o:o + D] if has_weights else None; o += D
    db = bucket[o:o + 1]; o += 1
    if kernel == "rq":
        return dZ, dell, dos, dm, ds, dw, db, bucket[o:o + 1]
    return dZ, dell, dos, dm, ds, dw, db


def elbo_forward_raw(mean, var, y, raw_noise, kl, num_data: float):
    _need_cuda(mean, var, y, raw_noise, kl)
    B, L = mean.shape
    elbo = torch.empty(B, device=mean.device, dtype=torch.float32)
    with torch.cuda.device(mean.device):
        rc = _cabi.lib().gpblur_elbo_forward(_ptr(mean), _ptr(var), _ptr(y), _ptr(raw_noise), _ptr(kl),
                                             float(num_data), B, L, _ptr(elbo), _stream())
    _cabi.check(rc, "gpblur_elbo_forward")
    return elbo


_TICKETS = {}


def _next_ticket(dev) -> int:
    """Device address of a zeroed 4-byte ticket word for a last-block-done kernel (a pool of 256 per device, handed out
    round-robin; the kernels leave their word at 0)."""
    key = (dev.type, dev.index)
    ent = _TICKETS.get(key)
    if ent is None:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("gpblur: run one eager step before capturing a CUDA graph (ticket pool not allocated)")
        ent = [torch.zeros(256, device=dev, dtype=torch.int32), 0]
        _TICKETS[key] = ent
    ent[1] = (ent[1] + 1) % 256
    return ent[0].data_ptr() + 4 * ent[1]


def elbo_backward_raw(mean, var, y, raw_noise, g_elbo, num_data: float):
    _need_cuda(mean, var, y, raw_noise, g_elbo)
    B, L = mean.shape
    dev = mean.device
    g_mean = torch.empty(B, L, device=dev, dtype=torch.float32)
    g_var = torch.empty(B, L, device=dev, dtype=torch.float32)
    g_noise = torch.empty(1, device=dev, dtype=torch.float32)
    g_kl = torch.empty(1, device=dev, dtype=torch.float32)
    scratch = torch.empty(max(B, 1), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        if B >= 1:
            # one launch: the block with the last ticket reduces; tickets rotate so that concurrent calls never share one
            rc = _cabi.lib().gpblur_elbo_backward_fused(_ptr(mean), _ptr(var), _ptr(y), _ptr(raw_noise), _ptr(g_elbo),
                                                        float(num_data), B, L, _ptr(g_mean), _ptr(g_var), _ptr(g_noise),
                                                        _ptr(g_kl), _ptr(scratch), _next_ticket(dev), _stream())
        else:
            rc = _cabi.lib().gpblur_elbo_backward(_ptr(mean), _ptr(var), _ptr(y), _ptr(raw_noise), _ptr(g_elbo),
                                                  float(num_data), B, L, _ptr(g_mean), _ptr(g_var), _ptr(g_noise),
                                                  _ptr(g_kl), _ptr(scratch), _stream())
    _cabi.check(rc, "gpblur_elbo_backward")
    return g_mean, g_var, g_noise, g_kl


def philox_bits(seed: int, offset: int, n: int, stream_id: int = 0, device="cuda") -> Tensor:
    out = torch.empty(n, 4, device=device, dtype=torch.int32)
    _need_cuda(out)
    with torch.cuda.device(out.device):
        rc = _cabi.lib().gpblur_philox_bits(seed, offset, stream_id, n, _ptr(out), _stream())
    _cabi.check(rc, "gpblur_philox_bits")
    return out


def philox_normal(seed: int, offset: int, n: int, stream_id: int = 0, device="cuda") -> Tensor:
    out = torch.empty(n, device=device, dtype=torch.float32)
    _need_cuda(out)
    with torch.cuda.device(out.device):
        rc = _cabi.lib().gpblur_philox_normal(seed, offset, stream_id, n, _ptr(out), _stream())
    _cabi.check(rc, "gpblur_philox_normal")
    return out


def kernel_kind(kernel: str) -> int:
    """Covariance function name ("rbf", "matern12", "matern32", "matern52", "rq") -> GPBLUR_KERNEL_* kind."""
    kind = _cabi.KERNEL_KINDS.get(kernel)
    if kind is None:
        raise ValueError(f"unknown covariance function {kernel!r}: expected one of {sorted(_cabi.KERNEL_KINDS)}")
    return kind


def _rbf_covariance_raw(x1, x2, raw_lengthscale, raw_outputscale, ard: bool, kind: int = 0,
                        raw_alpha: Optional[Tensor] = None) -> Tensor:
    n1, D = x1.shape
    n2 = x2.shape[0]
    out = torch.empty(n1, n2, device=x1.device, dtype=torch.float32)
    with torch.cuda.device(x1.device):
        rc = _cabi.lib().gpblur_covariance_alpha(_ptr(x1), _ptr(x2), n1, n2, D, kind, _ptr(raw_lengthscale),
                                                 int(ard), _ptr(raw_outputscale), _ptr(raw_alpha), _ptr(out), _stream())
    _cabi.check(rc, "gpblur_covariance_alpha")
    return out


class _RbfCovFunction(torch.autograd.Function):
    """Dense ScaleKernel(RBF | Matern | RQ) covariance with its hand-written backward
    (gpblur_covariance_backward_alpha): gradients of the inputs, the raw lengthscale(s), the raw outputscale and (RQ)
    raw_alpha."""

    @staticmethod
    def forward(ctx, x1, x2, raw_lengthscale, raw_outputscale, ard, kind=0, raw_alpha=None):
        same = x2 is x1
        x1c, ellc, osc = _f32c(x1), _f32c(raw_lengthscale).reshape(-1), _f32c(raw_outputscale).reshape(-1)
        x2c = x1c if same else _f32c(x2)
        ac = None if raw_alpha is None else _f32c(raw_alpha).reshape(-1)
        ctx.save_for_backward(x1c, x2c, ellc, osc, ac)
        ctx.meta = (bool(ard), same, raw_lengthscale.shape, raw_outputscale.shape, int(kind),
                    None if raw_alpha is None else raw_alpha.shape)
        return _rbf_covariance_raw(x1c, x2c, ellc, osc, ard, kind, ac)

    @staticmethod
    def backward(ctx, g_out):
        x1, x2, ell, os_, ac = ctx.saved_tensors
        ard, same, ell_shape, os_shape, kind, a_shape = ctx.meta
        n1, D = x1.shape
        n2 = x2.shape[0]
        dev = x1.device
        need = ctx.needs_input_grad
        want_x1, want_x2 = need[0] or (same and need[1]), need[1] or (same and need[0])
        g_x1 = torch.empty(n1, D, device=dev, dtype=torch.float32) if want_x1 else None
        g_x2 = torch.empty(n2, D, device=dev, dtype=torch.float32) if want_x2 else None
        g_ell = torch.empty(D if ard else 1, device=dev, dtype=torch.float32)
        g_os = torch.empty(1, device=dev, dtype=torch.float32)
        g_a = None if ac is None else torch.empty(1, device=dev, dtype=torch.float32)
        nbytes = int(_cabi.lib().gpblur_covariance_backward_scratch_bytes(n1, n2, D, kind))
        scratch = torch.empty(nbytes, device=dev, dtype=torch.uint8)
        with torch.cuda.device(dev):
            rc = _cabi.lib().gpblur_covariance_backward_alpha(
                _ptr(x1), _ptr(x2), n1, n2, D, kind, _ptr(ell), int(ard), _ptr(os_), _ptr(ac), _ptr(_f32c(g_out)),
                _ptr(g_x1), _ptr(g_x2), _ptr(g_ell), _ptr(g_os), _ptr(g_a), _ptr(scratch), nbytes, _stream())
        _cabi.check(rc, "gpblur_covariance_backward_alpha")
        ga = None if g_a is None else g_a.reshape(a_shape)
        if same:                       # K(x, x): the one tensor is both arguments
            gx = g_x1 + g_x2 if (need[0] or need[1]) else None
            return gx if need[0] else None, None, g_ell.reshape(ell_shape), g_os.reshape(os_shape), None, None, ga
        return (g_x1 if need[0] else None, g_x2 if need[1] else None, g_ell.reshape(ell_shape), g_os.reshape(os_shape),
                None, None, ga)


def rbf_covariance(x1: Tensor, x2: Tensor, raw_lengthscale: Tensor, raw_outputscale: Tensor, ard: bool,
                   kernel: str = "rbf", raw_alpha: Optional[Tensor] = None) -> Tensor:
    """os * f(|(x1 - x2) / l|) [n1, n2] (f: exp(-d^2 / 2) for "rbf", the Matern functions of include/gpblur.h for
    "matern12" / "matern32" / "matern52", (1 + d^2 / (2 alpha))^-alpha for "rq", which needs `raw_alpha` [1]);
    differentiable w.r.t. x1, x2 and the raw hyper-parameters."""
    _need_cuda(x1, x2, raw_lengthscale, raw_outputscale, raw_alpha)
    if raw_lengthscale.numel() != (x1.shape[-1] if ard else 1):
        raise ValueError("rbf_covariance: raw_lengthscale must hold D values (ard) or one")
    kind = kernel_kind(kernel)
    if (kernel == "rq") != (raw_alpha is not None) or (raw_alpha is not None and raw_alpha.numel() != 1):
        raise ValueError("rbf_covariance: raw_alpha (one value) is given for kernel 'rq' and only for it")
    return _RbfCovFunction.apply(x1, x2, raw_lengthscale, raw_outputscale, bool(ard), kind, raw_alpha)


def debug_fetch(which: int, N: int, D: int, M: int, ws: Tensor) -> Tensor:
    """Test probe: 0 = L, 1 = Linv, 2 = Kzz + jitter (float64 [Mp, Mp]); 3 = A, 5 = W (float32 [N, Mp]); 6 = the
    folded upstream gradients g_mu, g_var of the last backward (float32 [2, N])."""
    mp = C.c_int(0)
    Mp = 32 if M <= 32 else 128 if M <= 128 else (M + 255) // 256 * 256
    if which == 4:
        out = torch.empty(32, device=ws.device, dtype=torch.int64)
    elif which in (3, 5):
        Nt = (N + 127) // 128 * 128 if Mp >= 128 else N     # tensor-core path: whole 128-point tiles, tile-major
        out = torch.empty(Nt, Mp, device=ws.device, dtype=torch.float32)
    elif which == 6:
        out = torch.empty(2, max(N, 1), device=ws.device, dtype=torch.float32)
    else:
        out = torch.empty(Mp, Mp, device=ws.device, dtype=torch.float64)
    with torch.cuda.device(ws.device):
        rc = _cabi.lib().gpblur_debug_fetch(which, N, D, M, _ptr(ws), _ptr(out), out.numel() * out.element_size(),
                                            C.byref(mp), _stream())
    _cabi.check(rc, "gpblur_debug_fetch")
    assert mp.value == Mp
    if which in (3, 5) and Mp >= 128:
        # [tile][Mp / 4 pieces][128 rows][4] -> [N, Mp]   (csrc/gpblur_common.cuh: tc_tiled_index)
        out = out.reshape(-1, Mp // 4, 128, 4).permute(0, 2, 1, 3).reshape(-1, Mp)[:N].contiguous()
    return out


# ------------------------------------------------------------------------------------------------
# autograd
# ------------------------------------------------------------------------------------------------
def stage_grad_doubles(D: int, M: int, kind: int = 0) -> int:
    return int(_cabi.lib().gpblur_svgp_stage_grad_doubles_kind(D, M, kind))


def param_stage_raw(Z, raw_ell, raw_os, m, s, w, b, out=None, extra_jitter: float = 0.0, max_ctas: int = 0,
                    kind: int = 0, raw_alpha: Optional[Tensor] = None):
    """Once-per-parameter-update M x M stage: -> (stage uint8 [param_stage_bytes], kl [1], info [1] int32).
    `out` = preallocated (stage, kl, info) (the call then only launches on the current stream).
    `extra_jitter` is added to the diagonal of Kzz on top of the variational jitter (psd_safe_cholesky retries).
    `max_ctas` > 0 bounds the cooperative grid (stages of a multi-output layer running side by side, see _Fork).
    `kind`: covariance function (kernel_kind); the point and backward calls on this stage must pass the same.
    `raw_alpha` [1]: the rational quadratic kind's shape parameter (read for that kind only)."""
    _need_cuda(Z, raw_ell, raw_os, m, s, w, b, raw_alpha)
    M, D = Z.shape
    dev = Z.device
    if out is None:
        stage = torch.empty(param_stage_bytes(D, M), device=dev, dtype=torch.uint8)
        kl = torch.empty(1, device=dev, dtype=torch.float32)
        info = torch.empty(1, device=dev, dtype=torch.int32)
    else:
        stage, kl, info = out
    p = _params_struct(Z, raw_ell, raw_os, m, s, w, b, raw_alpha)
    with torch.cuda.device(dev):
        rc = _cabi.lib().gpblur_svgp_param_stage(C.byref(p), D, M, int(kind), float(extra_jitter), int(max_ctas),
                                                 _ptr(kl), _ptr(info), _ptr(stage), stage.numel(), _stream())
    _cabi.check(rc, "gpblur_svgp_param_stage")
    return stage, kl, info


def point_forward_raw(stage: Tensor, x: Tensor, M: int, seed: int, offset: int, stream_id: int, want_sample: bool,
                      training: bool, out: Optional[Tensor] = None, offset_dev: Optional[Tensor] = None,
                      ws: Optional[Tensor] = None, kind: int = 0):
    """x [N, D] + parameter stage (read in place) -> (mean [N], var [N], sample [N] | None, workspace uint8).
    `out`: preallocated float32 [(3 | 2) * N] receiving mean | var | sample."""
    _need_cuda(x, stage)
    N, D = x.shape
    dev = x.device
    if out is None:
        out = torch.empty((3 if want_sample else 2) * N, device=dev, dtype=torch.float32)   # one allocation
    mean, var = out[:N], out[N:2 * N]
    sample = out[2 * N:3 * N] if want_sample else None
    if ws is None:
        ws = torch.empty(workspace_bytes(N, D, M, training), device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        rc = _cabi.lib().gpblur_svgp_point_forward(
            _ptr(stage), _ptr(x), N, D, M, int(kind), _ptr(mean), _ptr(var), _ptr(sample), seed & 0xFFFFFFFFFFFFFFFF,
            offset & 0xFFFFFFFFFFFFFFFF, stream_id & 0xFFFFFFFF, _ptr(offset_dev), int(training), _ptr(ws), ws.numel(),
            _stream())
    _cabi.check(rc, "gpblur_svgp_point_forward")
    return mean, var, sample, ws


def point_backward_raw(x: Tensor, M: int, g_mean, g_var, g_sample, var, seed, offset, stream_id, ws,
                       need_dx: bool = True, dx: Optional[Tensor] = None, sgrad: Optional[Tensor] = None,
                       offset_dev: Optional[Tensor] = None, stage: Optional[Tensor] = None, kind: int = 0,
                       seg_sizes=None):
    """-> (dx [N, D] | None, stage_grad float64 [stage_grad_doubles(D, M)]).
    Upstream gradients `g_mean` / `g_var` / `g_sample`: [N] tensors or None.  With `seg_sizes` (1 to 4 point counts
    summing to N) they come per segment of the point range instead: lists of one tensor or None per segment, indexed
    from the start of the segment.  `stage`: the parameter stage the matching point_forward_raw call read (None: the
    stage was built in `ws` itself by svgp_forward_raw).  `dx` / `sgrad`: preallocated outputs."""
    N, D = x.shape
    if seg_sizes is None:          # one segment: all N points
        seg_sizes, g_mean, g_var, g_sample = [N], [g_mean], [g_var], [g_sample]
    _need_cuda(x, ws, var, stage, *g_mean, *g_var, *g_sample)
    dev = x.device
    nseg = len(seg_sizes)
    starts, o = [], 0
    for n in seg_sizes:
        starts.append(o)
        o += int(n)
    assert o == N and 1 <= nseg <= 4

    def ptr_array(ts):
        return (C.c_void_p * nseg)(*[(_ptr(t) if t is not None else None) for t in ts])

    keep = [None if t is None else _f32c(t) for t in list(g_mean) + list(g_var) + list(g_sample)]   # alive until launch
    gm, gv, gs = keep[:nseg], keep[nseg:2 * nseg], keep[2 * nseg:]
    if not need_dx:
        dx = None
    elif dx is None:
        dx = torch.empty(N, D, device=dev, dtype=torch.float32)
    if sgrad is None:
        sgrad = torch.empty(stage_grad_doubles(D, M, kind), device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        rc = _cabi.lib().gpblur_svgp_point_backward(
            _ptr(stage), _ptr(x), N, D, M, int(kind), nseg, (C.c_longlong * nseg)(*starts), ptr_array(gm), ptr_array(gv),
            ptr_array(gs), _ptr(var), seed & 0xFFFFFFFFFFFFFFFF, offset & 0xFFFFFFFFFFFFFFFF, stream_id & 0xFFFFFFFF,
            _ptr(offset_dev), _ptr(dx), _ptr(sgrad), _ptr(ws), ws.numel(), _stream())
    _cabi.check(rc, "gpblur_svgp_point_backward")
    return dx, sgrad


def param_stage_backward_raw(Z, raw_ell, raw_os, m, s, w, b, sgrad: Tensor, g_kl: Optional[Tensor], stage: Tensor,
                             bucket: Optional[Tensor] = None, accumulate: bool = False, max_ctas: int = 0,
                             kind: int = 0, raw_alpha: Optional[Tensor] = None):
    """Summed stage gradient (+ g_kl) -> flat parameter-gradient bucket [grad_bucket_floats(D, M, kind)]
    (`accumulate`: added to `bucket` instead of overwriting it)."""
    _need_cuda(Z, sgrad, stage, g_kl, raw_alpha)
    M, D = Z.shape
    if bucket is None:
        bucket = torch.empty(grad_bucket_floats(D, M, kind), device=Z.device, dtype=torch.float32)
    p = _params_struct(Z, raw_ell, raw_os, m, s, w, b, raw_alpha)
    with torch.cuda.device(Z.device):
        rc = _cabi.lib().gpblur_svgp_param_stage_backward(
            C.byref(p), D, M, int(kind), _ptr(sgrad), _ptr(g_kl), _ptr(bucket), int(accumulate), int(max_ctas),
            _ptr(stage), stage.numel(), _stream())
    _cabi.check(rc, "gpblur_svgp_param_stage_backward")
    return bucket


# ---- side streams: the M x M stages of the H independent GPs of a multi-output layer run concurrently ----
_SIDE_STREAMS = {}
N_SIDE_STREAMS = 16
_SM_COUNT = {}


def _stage_cta_cap(dev, H: int) -> int:
    """Grid bound of each of the H concurrent M x M stages of a multi-output layer: the SMs are shared out among the
    stages that can be in flight at once (one per side stream), so that their cooperative grids are co-resident."""
    if H <= 1:
        return 0
    key = (dev.type, dev.index)
    sms = _SM_COUNT.get(key)
    if sms is None:
        sms = _SM_COUNT[key] = torch.cuda.get_device_properties(dev).multi_processor_count
    return max(8, sms // min(H, N_SIDE_STREAMS))


def _side_streams(dev):
    key = (dev.type, dev.index)
    st = _SIDE_STREAMS.get(key)
    if st is None:
        st = _SIDE_STREAMS[key] = [torch.cuda.Stream(device=dev) for _ in range(N_SIDE_STREAMS)]
    return st


class _Fork:
    """Round-robin fork of H independent launches onto side streams, joined back into the current stream.
    All buffers are allocated by the caller on the CURRENT stream before the fork; only launches happen inside.
    (Uses the raw set-stream call: torch.cuda.stream() / current_stream(None) cost ~0.1 ms each here because they
    go through torch.cuda.is_available().)"""

    def __init__(self, dev, H):
        self.H = H
        if H <= 1:
            return
        self.dev = dev
        self.cur = torch.cuda.current_stream(dev)
        self.side = _side_streams(dev)
        self.ev = torch.cuda.Event()
        self.ev.record(self.cur)
        for st in self.side[:H]:
            st.wait_event(self.ev)

    def enter(self, h):
        if self.H > 1:
            torch.cuda.set_stream(self.side[h % len(self.side)])

    def join(self):
        if self.H <= 1:
            return
        torch.cuda.set_stream(self.cur)
        for st in self.side[:self.H]:
            self.cur.wait_stream(st)


_ZERO64 = {}


def _zero64(dev):
    """One float64 zero per device, created once (a fresh torch.zeros per step is a fill kernel - and a graph node)."""
    key = (dev.type, dev.index)
    z = _ZERO64.get(key)
    if z is None:
        z = torch.zeros((), device=dev, dtype=torch.float64)
        if not (dev.type == "cuda" and torch.cuda.is_current_stream_capturing()):
            _ZERO64[key] = z                  # (memory of a capture's private pool is not kept across captures)
    return z


class _ParamStageFunction(torch.autograd.Function):
    """Parameters -> (token, kl, info).  `token` is a float64 carrier whose GRADIENT is the stage gradient
    (include/gpblur.h): every per-point call that uses this stage returns its contribution as d/d token, autograd
    adds them up, and the M x M backward (Cholesky backward, Kzz-path gradients) runs ONCE per parameter update no
    matter how many times the GP was evaluated (the reference evaluates it twice per step,
    denoise_model_2.py:50-51).  The stage buffer itself travels in `holder` (not differentiable).

    Multi-output layers (DeepGP.py:21-26: inducing points [H, M, D], H independent GPs) are handled in ONE node:
    parameters carry a leading H, token is [H, G], and the H M x M stages (forward and backward) are launched on
    side streams so that they overlap on the GPU."""

    @staticmethod
    def forward(ctx, Z, raw_ell, raw_os, m, s, w, b, holder, raw_alpha=None):
        batched = Z.dim() == 3
        H = Z.shape[0] if batched else 1
        M, D = Z.shape[-2], Z.shape[-1]
        Zc = _f32c(Z).reshape(H, M, D)
        ellc = _f32c(raw_ell).reshape(H, D)
        osc = _f32c(raw_os).reshape(H, 1)
        mc = _f32c(m).reshape(H, M)
        sc = _f32c(s).reshape(H, M)
        wc = None if w is None else _f32c(w).reshape(-1, D)           # [1, D] shared or [H, D]
        bc = _f32c(b).reshape(-1, 1)                                  # [1, 1] shared or [H, 1]
        ac = None if raw_alpha is None else _f32c(raw_alpha).reshape(H, 1)   # rational quadratic: [H, 1]
        dev = Zc.device
        _need_cuda(Zc)
        stage = torch.empty(H, param_stage_bytes(D, M), device=dev, dtype=torch.uint8)
        kl = torch.empty(H, device=dev, dtype=torch.float32)
        info = torch.empty(H, device=dev, dtype=torch.int32)
        fork = _Fork(dev, H)
        cap = _stage_cta_cap(dev, H)
        try:
            for h in range(H):
                fork.enter(h)
                param_stage_raw(Zc[h], ellc[h], osc[h], mc[h], sc[h], None if wc is None else wc[h % wc.shape[0]],
                                bc[h % bc.shape[0]], out=(stage[h], kl[h:h + 1], info[h:h + 1]),
                                extra_jitter=float(holder.get("extra_jitter", 0.0)), max_ctas=cap,
                                kind=holder["kind"], raw_alpha=None if ac is None else ac[h])
        finally:
            fork.join()
        holder["stage"] = stage
        holder["consumed"] = False
        ctx.holder = holder
        ctx.batched = batched
        ctx.save_for_backward(Zc, ellc, osc, mc, sc, wc, bc, ac)
        ctx.shapes = (Z.shape, raw_ell.shape, raw_os.shape, m.shape, s.shape, None if w is None else w.shape, b.shape,
                      None if raw_alpha is None else raw_alpha.shape)
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(info)
        G = stage_grad_doubles(D, M, holder["kind"])
        token = _zero64(dev).expand((H, G) if batched else (G,))   # carrier of the stage gradient: never written
        return token, (kl if batched else kl.reshape(())), info

    @staticmethod
    def backward(ctx, g_token, g_kl, _g_info):
        with torch.cuda.nvtx.range("gpblur.param_stage_backward") if _NVTX else _null_ctx():
            return _ParamStageFunction._backward(ctx, g_token, g_kl, _g_info)

    @staticmethod
    def _backward(ctx, g_token, g_kl, _g_info):
        Zc, ellc, osc, mc, sc, wc, bc, ac = ctx.saved_tensors
        holder = ctx.holder
        H, M, D = Zc.shape
        dev = Zc.device
        G = stage_grad_doubles(D, M, holder["kind"])
        if g_token is None:
            sgrad = torch.zeros(H, G, device=dev, dtype=torch.float64)
        else:
            sgrad = g_token.to(torch.float64).reshape(H, G).contiguous()
        gk = None if g_kl is None else _f32c(g_kl).reshape(-1).expand(H).contiguous()
        nb = grad_bucket_floats(D, M, holder["kind"])
        stage = holder["stage"]
        sink = holder.get("grad_sink")
        if sink is not None and H == 1 and wc is not None:
            # the caller's flat gradient buffer holds this layer's parameters contiguously in bucket order
            # (distributed.FlatGradBucket): the kernel accumulates straight into it, autograd gets no gradient to add
            param_stage_backward_raw(Zc[0], ellc[0], osc[0], mc[0], sc[0], wc[0], bc[0], sgrad[0],
                                     None if gk is None else gk[0:1], stage[0], bucket=sink, accumulate=True,
                                     kind=holder["kind"], raw_alpha=None if ac is None else ac[0])
            holder["consumed"] = True
            return (None,) * 9
        bucket = torch.empty(H, nb, device=dev, dtype=torch.float32)
        fork = _Fork(dev, H)
        cap = _stage_cta_cap(dev, H)
        try:
            for h in range(H):
                fork.enter(h)
                param_stage_backward_raw(Zc[h], ellc[h], osc[h], mc[h], sc[h],
                                         None if wc is None else wc[h % wc.shape[0]], bc[h % bc.shape[0]], sgrad[h],
                                         None if gk is None else gk[h:h + 1], stage[h], bucket=bucket[h], max_ctas=cap,
                                         kind=holder["kind"], raw_alpha=None if ac is None else ac[h])
        finally:
            fork.join()
        holder["consumed"] = True        # the graph behind this token is gone: the next forward rebuilds the stage
        o = 0
        dZ = bucket[:, o:o + M * D]; o += M * D
        dell = bucket[:, o:o + D]; o += D
        dos = bucket[:, o:o + 1]; o += 1
        dm = bucket[:, o:o + M]; o += M
        ds = bucket[:, o:o + M]; o += M
        dw = bucket[:, o:o + D]; o += D
        db = bucket[:, o:o + 1]; o += 1
        da = bucket[:, o:o + 1]                                       # rational quadratic: d raw_alpha
        shp = ctx.shapes
        need = ctx.needs_input_grad

        def shared(t, shape, n_rows):
            # a parameter shared by the H GPs (LinearMean of a multi-output layer) receives the sum over h
            return (t.sum(0) if (H > 1 and n_rows == 1) else t).reshape(shape)

        return (dZ.reshape(shp[0]) if need[0] else None,
                dell.reshape(shp[1]) if need[1] else None,
                dos.reshape(shp[2]) if need[2] else None,
                dm.reshape(shp[3]) if need[3] else None,
                ds.reshape(shp[4]) if need[4] else None,
                shared(dw, shp[5], wc.shape[0]) if (wc is not None and need[5]) else None,
                shared(db, shp[6], bc.shape[0]) if need[6] else None,
                None,
                da.reshape(shp[7]) if (ac is not None and need[8]) else None)


class _PointFunction(torch.autograd.Function):
    """Per-point part of the whitened SVGP predictive on a given parameter stage, hand-written backward.
    With an [H, G] token (multi-output layer) every output gains a trailing H: mean [..., H]."""

    @staticmethod
    def forward(ctx, x, token, holder, M, seed, offset, stream_id, want_sample, offset_dev, h_stride=None):
        shape = x.shape
        D = shape[-1]
        x2 = _f32c(x).reshape(-1, D)
        N = x2.shape[0]
        batched = token.dim() == 2
        H = token.shape[0] if batched else 1
        training = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        hs = N if h_stride is None else int(h_stride)       # Philox counter stride between the H GPs of a layer
        nout = 3 if want_sample else 2
        out = torch.empty(H, nout * N, device=x2.device, dtype=torch.float32)
        stage = holder["stage"]
        # the H GPs of a multi-output layer are independent: their (persistent, one CTA per SM) kernels alternate
        # between side streams so that each one starts in the tail of the previous one
        wss = [torch.empty(workspace_bytes(N, D, M, training), device=x2.device, dtype=torch.uint8) for _ in range(H)]
        fork = _Fork(x2.device, H)
        try:
            for h in range(H):
                fork.enter(h)
                point_forward_raw(stage[h], x2, M, seed, offset + h * hs, stream_id, want_sample, training,
                                  out=out[h], offset_dev=offset_dev, ws=wss[h], kind=holder["kind"])
        finally:
            fork.join()
        if training:
            ctx.save_for_backward(x2, out, *wss)
            ctx.stage = stage                                  # read in place by the backward kernels
            ctx.kind = holder["kind"]
        ctx.meta = (seed, offset, stream_id, M, shape, H, batched, nout, hs)
        ctx.offset_dev = offset_dev
        ctx.set_materialize_grads(False)
        out_shape = tuple(shape[:-1]) + ((H,) if batched else ())

        def view(i):
            t = out[:, i * N:(i + 1) * N]                      # [H, N]
            return (t.t() if batched else t[0]).reshape(out_shape)

        return view(0), view(1), (view(2) if want_sample else None)

    @staticmethod
    def backward(ctx, g_mean, g_var, g_sample):
        with torch.cuda.nvtx.range("gpblur.point_backward") if _NVTX else _null_ctx():
            return _PointFunction._backward(ctx, g_mean, g_var, g_sample)

    @staticmethod
    def _backward(ctx, g_mean, g_var, g_sample):
        x2, out, *wss = ctx.saved_tensors
        seed, offset, stream_id, M, shape, H, batched, nout, hs = ctx.meta
        N, D = x2.shape
        dev = x2.device

        def prep(g):
            if g is None:
                return None
            g = _f32c(g)
            return g.reshape(N, H).t().contiguous() if batched else g.reshape(1, N)

        gm, gv, gs = prep(g_mean), prep(g_var), prep(g_sample)
        need = ctx.needs_input_grad
        G = stage_grad_doubles(D, M, ctx.kind)
        sgrad = torch.empty(H, G, device=dev, dtype=torch.float64)
        dx = torch.empty(H, N, D, device=dev, dtype=torch.float32) if need[0] else None
        fork = _Fork(dev, H)
        try:
            for h in range(H):
                fork.enter(h)
                point_backward_raw(x2, M, None if gm is None else gm[h], None if gv is None else gv[h],
                                   None if gs is None else gs[h], out[h, N:2 * N], seed, offset + h * hs, stream_id,
                                   wss[h], need_dx=need[0], dx=None if dx is None else dx[h], sgrad=sgrad[h],
                                   offset_dev=ctx.offset_dev, stage=ctx.stage[h], kind=ctx.kind)
        finally:
            fork.join()
        if dx is not None:
            dx = (dx.sum(0) if H > 1 else dx[0]).reshape(shape)
        return (dx, (sgrad if batched else sgrad[0]) if need[1] else None, None, None, None, None, None, None, None,
                None)


def _stage_key(Z, raw_ell, raw_os, m, s, w, b, raw_alpha=None):
    key = tuple((t._version, t.data_ptr()) for t in (Z, raw_ell, raw_os, m, s, b))
    for t in (w, raw_alpha):
        if t is not None:
            key += ((t._version, t.data_ptr()),)
    return key + (tuple(Z.shape),)


class NotPSDError(RuntimeError):
    """Kzz + jitter is not positive definite even after the jitter retries (gpytorch.utils.errors.NotPSDError)."""


class NumericalWarning(RuntimeWarning):
    pass


# psd_safe_cholesky (gpytorch, fp32): on failure add 1e-6, 1e-5, 1e-4 to the diagonal, then give up
JITTER_RETRIES = (1e-6, 1e-5, 1e-4)


def svgp_param_stage(inducing_points: Tensor, raw_lengthscale: Tensor, raw_outputscale: Tensor,
                     variational_mean: Tensor, variational_stddev: Tensor, mean_weights: Optional[Tensor],
                     mean_bias: Tensor, stage_cache: Optional[dict] = None, check: bool = False,
                     grad_sink: Optional[Tensor] = None, kernel: str = "rbf", raw_alpha: Optional[Tensor] = None):
    """-> (token, kl, info, holder).  `kernel`: covariance function ("rbf", "matern12", "matern32", "matern52", "rq"); it
    is part of the stage-cache key and travels in `holder` to every call on the stage.  `raw_alpha` ([1], or [H, 1]
    for a multi-output layer): the shape parameter of "rq", differentiable like the other parameters; given for "rq"
    and only for it.  With `stage_cache` (a dict owned by the caller, one per GP layer) consecutive
    calls with unchanged parameter tensors (same `_version`) share one stage - and therefore one M x M backward -
    until a backward pass has consumed it.  Parameters with a leading H (inducing points [H, M, D]) describe the H
    independent GPs of a multi-output layer: kl is [H], token [H, G]."""
    params = (inducing_points, raw_lengthscale, raw_outputscale, variational_mean, variational_stddev, mean_weights,
              mean_bias)
    kind = kernel_kind(kernel)
    if (kernel == "rq") != (raw_alpha is not None):
        raise ValueError("raw_alpha is given for kernel 'rq' and only for it")
    want_grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in params + (raw_alpha,))
    key = None
    if stage_cache is not None:
        key = _stage_key(*params, raw_alpha) + (kind,)
        ent = stage_cache.get("entry")
        if ent is not None and stage_cache.get("key") == key and not ent[3]["consumed"] \
                and ent[0].requires_grad == want_grad:
            return ent
    holder = {"kind": kind}
    if grad_sink is not None:
        holder["grad_sink"] = grad_sink
    with torch.cuda.nvtx.range("gpblur.param_stage") if _NVTX else _null_ctx():
        token, kl, info = _ParamStageFunction.apply(*params, holder, raw_alpha)
    # Cholesky status (LAPACK-style info, 0 = ok).  Reading it synchronises with the device, as gpytorch's
    # psd_safe_cholesky does; it is skipped while a CUDA graph is being captured (check GraphedStep.check_info()).
    if check and not torch._C._cuda_isCurrentStreamCapturing():
        k = int(info.max().item())
        if k != 0:
            import warnings
            for jit in JITTER_RETRIES:
                holder = {"kind": kind, "extra_jitter": jit}
                if grad_sink is not None:
                    holder["grad_sink"] = grad_sink
                token, kl, info = _ParamStageFunction.apply(*params, holder, raw_alpha)
                if int(info.max().item()) == 0:
                    warnings.warn(f"Kzz + 1e-4 I is not positive definite (pivot {k}): added jitter of {jit:.1e} to the "
                                  f"diagonal", NumericalWarning)
                    break
            else:
                raise NotPSDError(f"Kzz is not positive definite after adding jitter up to {JITTER_RETRIES[-1]:.1e} "
                                  f"(first failing pivot {k})")
    ent = (token, kl, info, holder)
    if stage_cache is not None:
        stage_cache["key"] = key
        stage_cache["entry"] = ent
    return ent


def svgp_predict(x: Tensor, inducing_points: Tensor, raw_lengthscale: Tensor, raw_outputscale: Tensor,
                 variational_mean: Tensor, variational_stddev: Tensor, mean_weights: Optional[Tensor],
                 mean_bias: Tensor, seed: int = 0, offset: int = 0, stream_id: int = 0,
                 want_sample: bool = False, stage_cache: Optional[dict] = None,
                 offset_dev: Optional[Tensor] = None, h_stride: Optional[int] = None, check: bool = False,
                 grad_sink: Optional[Tensor] = None, kernel: str = "rbf", raw_alpha: Optional[Tensor] = None):
    """x [..., D] -> (mean [...], var [...], sample [...] | None, kl [], info [1]); with inducing points [H, M, D]
    (multi-output layer) the outputs are [..., H], kl [H], info [H], and GP h draws its sample with Philox counters
    offset + h * h_stride + n (h_stride defaults to the N points of this call; batch-sharded callers pass the GLOBAL
    point count so that the counters do not depend on the number of ranks).  `stage_cache`: see svgp_param_stage.  `offset_dev`: optional int64 device scalar added to
    `offset` when the kernels run (CUDA-graph replays draw fresh counters by bumping it between replays).  `kernel`,
    `raw_alpha`: covariance function, see svgp_param_stage."""
    token, kl, info, holder = svgp_param_stage(inducing_points, raw_lengthscale, raw_outputscale, variational_mean,
                                               variational_stddev, mean_weights, mean_bias, stage_cache, check=check,
                                               grad_sink=grad_sink, kernel=kernel, raw_alpha=raw_alpha)
    if x.numel() == 0:
        shp = tuple(x.shape[:-1]) + ((token.shape[0],) if token.dim() == 2 else ())
        e = x.new_empty(shp, dtype=torch.float32)
        return e, e.clone(), (e.clone() if want_sample else None), kl, info
    with torch.cuda.nvtx.range("gpblur.point_forward") if _NVTX else _null_ctx():
        mean, var, sample = _PointFunction.apply(x, token, holder, int(inducing_points.shape[-2]), int(seed), int(offset),
                                                 int(stream_id), bool(want_sample), offset_dev, h_stride)
    return mean, var, sample, kl, info


def as_one_buffer(xs) -> Tensor:
    """[..., D] activations -> their points back to back as ONE [N, D] tensor: a view when the tensors already sit
    back to back in one allocation (e.g. slices of a staging buffer), otherwise a concatenation (one copy kernel)."""
    D = xs[0].shape[-1]
    ok = all(t.is_contiguous() and t.dtype == torch.float32 and t.shape[-1] == D for t in xs)
    if ok:
        base = xs[0].untyped_storage().data_ptr()
        p = xs[0].data_ptr()
        for t in xs:
            ok = ok and t.untyped_storage().data_ptr() == base and t.data_ptr() == p
            p += t.numel() * 4
    if ok:
        n = sum(t.numel() for t in xs) // D
        return torch.as_strided(xs[0], (n, D), (D, 1))
    return torch.cat([_f32c(t).reshape(-1, D) for t in xs], dim=0)


class _PointSegFunction(torch.autograd.Function):
    """_PointFunction (single-output GP) on the CONCATENATED points of several activations: one launch per kernel for
    the whole step instead of one per activation.  Outputs come back per segment (views of one buffer) and the
    backward reads each segment's upstream gradients where autograd left them (no concatenation kernels)."""

    @staticmethod
    def forward(ctx, x, token, holder, M, seed, offset, stream_id, want_sample, offset_dev, seg_shapes):
        D = x.shape[-1]
        x2 = _f32c(x).reshape(-1, D)
        N = x2.shape[0]
        sizes = [int(math.prod(shp)) for shp in seg_shapes]
        if sum(sizes) != N:
            raise ValueError(f"segment shapes {seg_shapes} do not cover the {N} points of x")
        training = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        nout = 3 if want_sample else 2
        out = torch.empty(nout * N, device=x2.device, dtype=torch.float32)
        stage = holder["stage"]
        ws = torch.empty(workspace_bytes(N, D, M, training), device=x2.device, dtype=torch.uint8)
        point_forward_raw(stage[0], x2, M, seed, offset, stream_id, want_sample, training, out=out,
                          offset_dev=offset_dev, ws=ws, kind=holder["kind"])
        if training:
            ctx.save_for_backward(x2, out, ws)
            ctx.stage = stage
            ctx.kind = holder["kind"]
        ctx.meta = (seed, offset, stream_id, M, tuple(x.shape), sizes, nout)
        ctx.offset_dev = offset_dev
        ctx.set_materialize_grads(False)
        res, o = [], 0
        for shp, n in zip(seg_shapes, sizes):
            for k in range(3):
                res.append(out[k * N + o:k * N + o + n].view(tuple(shp)) if k < nout else None)
            o += n
        return tuple(res)

    @staticmethod
    def backward(ctx, *grads):
        x2, out, ws = ctx.saved_tensors
        seed, offset, stream_id, M, xshape, sizes, nout = ctx.meta
        N, D = x2.shape
        need = ctx.needs_input_grad
        gms, gvs, gss = list(grads[0::3]), list(grads[1::3]), list(grads[2::3])
        with torch.cuda.nvtx.range("gpblur.point_backward") if _NVTX else _null_ctx():
            dx, sgrad = point_backward_raw(x2, M, gms, gvs, gss, out[N:2 * N], seed, offset, stream_id, ws,
                                           need_dx=need[0], offset_dev=ctx.offset_dev, stage=ctx.stage[0], kind=ctx.kind,
                                           seg_sizes=sizes)
        return (dx.reshape(xshape) if dx is not None else None, sgrad if need[1] else None) + (None,) * 8


def svgp_predict_segments(x: Tensor, seg_shapes, inducing_points: Tensor, raw_lengthscale: Tensor,
                          raw_outputscale: Tensor, variational_mean: Tensor, variational_stddev: Tensor,
                          mean_weights: Optional[Tensor], mean_bias: Tensor, seed: int = 0, offset: int = 0,
                          stream_id: int = 0, want_sample: bool = False, stage_cache: Optional[dict] = None,
                          offset_dev: Optional[Tensor] = None, check: bool = False,
                          grad_sink: Optional[Tensor] = None, kernel: str = "rbf",
                          raw_alpha: Optional[Tensor] = None):
    """svgp_predict for a single-output GP on x [N, D] = the concatenated points of several activations;
    ``seg_shapes`` (e.g. [(B, 192), (B, 24)]) are the output shapes of the segments, in order.
    -> ([(mean, var, sample | None) per segment], kl, info)."""
    if inducing_points.dim() != 2:
        raise ValueError("svgp_predict_segments: single-output layers only")
    token, kl, info, holder = svgp_param_stage(inducing_points, raw_lengthscale, raw_outputscale, variational_mean,
                                               variational_stddev, mean_weights, mean_bias, stage_cache, check=check,
                                               grad_sink=grad_sink, kernel=kernel, raw_alpha=raw_alpha)
    with torch.cuda.nvtx.range("gpblur.point_forward") if _NVTX else _null_ctx():
        flat = _PointSegFunction.apply(x, token, holder, int(inducing_points.shape[-2]), int(seed), int(offset),
                                       int(stream_id), bool(want_sample), offset_dev,
                                       tuple(tuple(int(v) for v in shp) for shp in seg_shapes))
    return [tuple(flat[3 * i:3 * i + 3]) for i in range(len(seg_shapes))], kl, info


class _ElboFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mean, var, y, raw_noise, kl, num_data):
        L = mean.shape[-1]
        mean2 = _f32c(mean).reshape(-1, L)
        var2 = _f32c(var).reshape(-1, L)
        y2 = _f32c(y).expand(mean.shape).reshape(-1, L).contiguous()
        rn = _f32c(raw_noise).reshape(-1)
        klc = _f32c(kl).reshape(1)
        elbo = elbo_forward_raw(mean2, var2, y2, rn, klc, num_data)
        ctx.save_for_backward(mean2, var2, y2, rn)
        ctx.num_data = float(num_data)
        ctx.shapes = (mean.shape, var.shape, raw_noise.shape, kl.shape)
        return elbo.reshape(mean.shape[:-1])

    @staticmethod
    def backward(ctx, g_elbo):
        mean2, var2, y2, rn = ctx.saved_tensors
        g = _f32c(g_elbo).reshape(-1)
        g_mean, g_var, g_noise, g_kl = elbo_backward_raw(mean2, var2, y2, rn, g, ctx.num_data)
        shp = ctx.shapes
        need = ctx.needs_input_grad
        return (g_mean.reshape(shp[0]) if need[0] else None,
                g_var.reshape(shp[1]) if need[1] else None,
                None,
                g_noise.reshape(shp[2]) if need[3] else None,
                g_kl.reshape(shp[3]) if need[4] else None,
                None)


def variational_elbo(mean: Tensor, var: Tensor, y: Tensor, raw_noise: Tensor, kl: Tensor,
                     num_data: float) -> Tensor:
    """mean, var, y [..., L] -> elbo [...] (per window)."""
    return _ElboFunction.apply(mean, var, y, raw_noise, kl, float(num_data))


class _RsampleFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mean, var, seed, offset, stream_id):
        _need_cuda(mean, var)
        m = _f32c(mean).reshape(-1)
        v = _f32c(var).reshape(-1)
        out = torch.empty_like(m)
        with torch.cuda.device(m.device):
            rc = _cabi.lib().gpblur_rsample_forward(_ptr(m), _ptr(v), m.numel(), seed, offset, stream_id,
                                                    _ptr(out), _stream())
        _cabi.check(rc, "gpblur_rsample_forward")
        ctx.save_for_backward(v)
        ctx.rng = (seed, offset, stream_id)
        ctx.shape = mean.shape
        return out.reshape(mean.shape)

    @staticmethod
    def backward(ctx, g):
        (v,) = ctx.saved_tensors
        seed, offset, stream_id = ctx.rng
        gc = _f32c(g).reshape(-1)
        gm = torch.empty_like(gc)
        gv = torch.empty_like(gc)
        with torch.cuda.device(v.device):
            rc = _cabi.lib().gpblur_rsample_backward(_ptr(v), _ptr(gc), gc.numel(), seed, offset, stream_id,
                                                     _ptr(gm), _ptr(gv), _stream())
        _cabi.check(rc, "gpblur_rsample_backward")
        return gm.reshape(ctx.shape), gv.reshape(ctx.shape), None, None, None


def rsample(mean: Tensor, var: Tensor, seed: int, offset: int, stream_id: int = 0) -> Tensor:
    """Normal(mean, sqrt(var)).rsample() with explicit Philox counters (between DeepGP layers)."""
    return _RsampleFunction.apply(mean, var, int(seed), int(offset), int(stream_id))


# ------------------------------------------------------------------------------------------------
# torch.library registration (torch.ops.gpblur.*): the same raw calls behind dispatcher-visible ops
# ------------------------------------------------------------------------------------------------
def _register_custom_ops():
    try:
        from torch.library import custom_op
    except Exception:   # pragma: no cover
        return

    @custom_op("gpblur::svgp_fwd", mutates_args=(), device_types="cuda")
    def svgp_fwd(x: Tensor, Z: Tensor, raw_ell: Tensor, raw_os: Tensor, m: Tensor, s: Tensor, w: Optional[Tensor],
                 b: Tensor, seed: int, offset: int, stream_id: int, want_sample: bool,
                 training: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
        mean, var, sample, kl, info, ws = svgp_forward_raw(x, Z, raw_ell, raw_os, m, s, w, b, seed, offset,
                                                           stream_id, want_sample, training)
        if sample is None:
            sample = mean.new_empty(0)
        return mean, var, sample, kl, info, ws

    @custom_op("gpblur::svgp_bwd", mutates_args=(), device_types="cuda")
    def svgp_bwd(x: Tensor, Z: Tensor, raw_ell: Tensor, raw_os: Tensor, m: Tensor, s: Tensor, w: Optional[Tensor],
                 b: Tensor, g_mean: Optional[Tensor], g_var: Optional[Tensor], g_sample: Optional[Tensor],
                 g_kl: Optional[Tensor], var: Tensor, seed: int, offset: int, stream_id: int,
                 ws: Tensor) -> Tuple[Tensor, Tensor]:
        dx, bucket = svgp_backward_raw(x, Z, raw_ell, raw_os, m, s, w, b, g_mean, g_var, g_sample, g_kl, var,
                                       seed, offset, stream_id, ws, True)
        return dx, bucket

    @custom_op("gpblur::elbo_fwd", mutates_args=(), device_types="cuda")
    def elbo_fwd(mean: Tensor, var: Tensor, y: Tensor, raw_noise: Tensor, kl: Tensor, num_data: float) -> Tensor:
        return elbo_forward_raw(mean, var, y, raw_noise, kl, num_data)

    @custom_op("gpblur::elbo_bwd", mutates_args=(), device_types="cuda")
    def elbo_bwd(mean: Tensor, var: Tensor, y: Tensor, raw_noise: Tensor, g_elbo: Tensor,
                 num_data: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
        return elbo_backward_raw(mean, var, y, raw_noise, g_elbo, num_data)


_register_custom_ops()
