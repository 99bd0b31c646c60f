"""Batch-sharded data-parallel training of the GP blur model (SURVEY 8(e)).

The reference is single-process (no torch.distributed anywhere); this is new functionality:
forecast windows are sharded across ranks by batch, the GP parameters and the M x M Cholesky are
replicated, and the ONLY collective per step is one all-reduce of the flat GP-parameter-gradient
bucket (M*D + 2M + 2D + 3 floats, 68 KB at M=256, D=64) - NCCL over NVLink/NVSwitch on GPUs, gloo in
the CPU tests.  dX stays local.  Philox offsets are derived from the GLOBAL window index so that the
reparameterised samples are identical for any number of ranks.
"""
from __future__ import annotations

import os

from typing import Iterable, List, Optional, Tuple

import torch
import torch.distributed as dist
from torch import nn


def shard_range(n_global: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous shard [start, start + count) of n_global windows for `rank` (ragged tails go to the
    first ranks)."""
    base, rem = divmod(n_global, world)
    count = base + (1 if rank < rem else 0)
    start = rank * base + min(rank, rem)
    return start, count


def gp_parameters(module: nn.Module) -> List[nn.Parameter]:
    """Trainable parameters in a deterministic (name-sorted) order - identical on every rank."""
    return [p for _, p in sorted(module.named_parameters(), key=lambda kv: kv[0]) if p.requires_grad]


class FlatGradBucket:
    """One contiguous fp32 gradient buffer; every parameter's ``.grad`` is a view into it, so autograd
    accumulates straight into the bucket and the all-reduce needs no packing copy."""

    def __init__(self, params: Iterable[nn.Parameter], module: Optional[nn.Module] = None):
        """`module`: if given, every single-output GP layer with a linear mean whose parameters are all in `params`
        gets them laid out contiguously in the C-ABI bucket order (include/gpblur.h: Z, raw_lengthscale,
        raw_outputscale, variational_mean, variational_stddev, weights, bias, and raw_alpha for an RQKernel;
        layer._layer_params()) and becomes a GRADIENT SINK: its M x M
        backward kernel accumulates straight into this buffer (``layer._grad_sink``) and autograd launches no
        per-parameter accumulation kernels for it."""
        self.params = list(params)
        if not self.params:
            raise ValueError("no parameters")
        dev = self.params[0].device
        if any(p.dtype != torch.float32 or p.device != dev for p in self.params):
            raise ValueError("FlatGradBucket needs fp32 parameters on one device")
        sinks = []
        if module is not None:
            from .gpcompat import LinearMean
            have = {id(p) for p in self.params}
            taken = set()
            for layer in _gp_layers(module):
                mm = getattr(layer, "mean_module", None)
                if layer.output_dims is not None or not isinstance(mm, LinearMean) or mm.bias is None:
                    continue
                lp = list(layer._layer_params())
                if all(id(p) in have and id(p) not in taken for p in lp):
                    sinks.append((layer, lp))
                    taken.update(id(p) for p in lp)
            ordered = [p for _, lp in sinks for p in lp] + [p for p in self.params if id(p) not in taken]
            self.params = ordered
        n = sum(p.numel() for p in self.params)
        self.flat = torch.zeros(n, device=dev, dtype=torch.float32)
        o = 0
        starts = {}
        for p in self.params:
            starts[id(p)] = o
            p.grad = self.flat[o:o + p.numel()].view_as(p)
            o += p.numel()
        for layer, lp in sinks:
            a = starts[id(lp[0])]
            layer._grad_sink = self.flat[a:a + sum(p.numel() for p in lp)]

    def zero(self):
        self.flat.zero_()

    def enable_peer_allreduce(self, group=None) -> bool:
        """Switch all_reduce() to the library's one-shot exchange over NVLink peer memory (PeerAllReduce below; one
        node, one process per GPU).  Collective: every rank of `group` must call it.  Returns False (and keeps NCCL)
        when the peer mapping cannot be set up on some rank or GPBLUR_PEER_ALLREDUCE=0."""
        self._peer = None
        if os.environ.get("GPBLUR_PEER_ALLREDUCE", "1") == "0" or not self.flat.is_cuda:
            return False
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return False
        peer = PeerAllReduce(self.flat.numel(), self.flat.device, group)
        if peer.enabled:
            self._peer = peer
        return peer.enabled

    def all_reduce(self, group=None, average: bool = True, async_op: bool = False):
        """Sum (or mean) the bucket across ranks.  No-op when torch.distributed is not initialised."""
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return None
        if getattr(self, "_peer", None) is not None:
            self._peer(self.flat, average)          # stream-ordered kernel: nothing to wait for
            return None
        # NCCL averages inside the collective (no separate div_ kernel; capturable in a CUDA graph); gloo has no AVG
        use_avg = average and self.flat.is_cuda and dist.get_backend(group) == "nccl"
        op = dist.ReduceOp.AVG if use_avg else dist.ReduceOp.SUM
        work = dist.all_reduce(self.flat, op=op, group=group, async_op=async_op)
        if average and not use_avg:
            if async_op:
                work.wait()
                work = None
            self.flat.div_(dist.get_world_size(group))
        return work


class PeerAllReduce:
    """One-shot all-reduce of a small fp32 buffer over NVLink peer memory (csrc/gpblur_peer.cu): every rank maps the
    communication buffers of its peers through CUDA IPC once; per step ONE self-synchronising kernel stages the
    buffer, signals the peers, waits for theirs and sums all of them in rank order (bit-identical on every rank).
    ~8 us per step for the 17 k floats of the reference shape where the NCCL all-reduce takes ~30 us; capturable in
    a CUDA graph (device-resident step counter)."""

    def __init__(self, numel: int, device, group=None):
        import ctypes as C
        from . import _cabi
        lib = _cabi.lib()
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.numel, self.device = int(numel), torch.device(device)
        self.enabled = False
        self._own = None
        self._opened = []
        ok = self.world <= 16
        handle = (C.c_ubyte * 64)()
        own = C.c_void_p()
        if ok:
            with torch.cuda.device(self.device):
                ok = lib.gpblur_peer_alloc(lib.gpblur_peer_comm_bytes(self.numel), C.byref(own), handle) == 0
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle) if ok else None, group=group)
        ptrs = []
        if ok and all(h is not None for h in handles):
            self._own = own.value
            for r, h in enumerate(handles):
                if r == self.rank:
                    ptrs.append(own.value)
                    continue
                p = C.c_void_p()
                buf = (C.c_ubyte * 64).from_buffer_copy(h)
                with torch.cuda.device(self.device):
                    if lib.gpblur_peer_open(buf, C.byref(p)) != 0:
                        ok = False
                        break
                self._opened.append(p.value)
                ptrs.append(p.value)
        else:
            ok = False
        flag = torch.tensor([1 if ok else 0], device=self.device, dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)     # all ranks or none
        self.enabled = bool(flag.item())
        if self.enabled:
            self._arr = (C.c_void_p * self.world)(*ptrs)
        self._lib = lib

    def __call__(self, flat: torch.Tensor, average: bool = True):
        from . import _cabi
        if flat.numel() != self.numel or flat.dtype != torch.float32 or not flat.is_contiguous():
            raise ValueError("PeerAllReduce: buffer does not match the one it was set up for")
        with torch.cuda.device(self.device):
            rc = self._lib.gpblur_peer_allreduce(flat.data_ptr(), self.numel, self.world, self.rank, self._arr,
                                                 (1.0 / self.world) if average else 1.0,
                                                 torch.cuda.current_stream(self.device).cuda_stream)
        _cabi.check(rc, "gpblur_peer_allreduce")


def _gp_layers(module: nn.Module):
    from .gpcompat import DeepGPLayer
    return [m for m in module.modules() if isinstance(m, DeepGPLayer)]


def broadcast_parameters(module: nn.Module, src: int = 0, group=None) -> None:
    """Make every rank hold rank `src`'s parameters and buffers.

    The first-call variational initialisation (gpytorch: variational_mean <- 1e-3 randn from the rank's own RNG)
    is run BEFORE the broadcast, so that it cannot overwrite the broadcast values on the first forward and leave the
    replicas different for good.  The broadcast writes through ``p.detach()`` (shares the version counter, unlike
    ``p.data``), so parameter stages / KL values cached on the tensor versions are invalidated; they are also
    dropped explicitly."""
    layers = _gp_layers(module)
    for layer in layers:
        layer.variational_strategy._ensure_initialized()
    if not (dist.is_available() and dist.is_initialized()):
        return
    with torch.no_grad():
        for _, p in sorted(module.named_parameters(), key=lambda kv: kv[0]):
            dist.broadcast(p.detach(), src=src, group=group)
        for _, b in sorted(module.named_buffers(), key=lambda kv: kv[0]):
            dist.broadcast(b.detach(), src=src, group=group)
    for layer in layers:
        layer.invalidate_param_stage()


class ShardedGPBlur(nn.Module):
    """Data-parallel wrapper around a GP blur model (``DeepGPp`` / ``DeepGP2``).

    ``forward(x_local, y_local, first_global_window)`` runs the local shard with Philox counters offset
    to the shard's global position; ``sync_grads()`` all-reduces (averages) the flat gradient bucket.
    Rank-to-rank results are bit-identical to a single-rank run on the concatenated batch for the
    per-window outputs; parameter gradients agree up to fp32 summation order."""

    def __init__(self, model: nn.Module, group=None, broadcast: bool = True):
        super().__init__()
        self.model = model
        self.group = group
        if broadcast:
            broadcast_parameters(model, 0, group)
        self.bucket = FlatGradBucket(gp_parameters(model), module=model)
        if next(model.parameters()).is_cuda and os.environ.get("GPBLUR_PEER_ALLREDUCE", "0") == "1":
            self.bucket.enable_peer_allreduce(group)     # opt-in NVLink peer-memory exchange (default: NCCL, see DESIGN.md)
        self.step_index = 0

    def _layers(self):
        return _gp_layers(self.model)

    def forward(self, x_local, y_local=None, first_global_window: int = 0, global_windows: Optional[int] = None,
                num_data=None):
        L = x_local.shape[-2]
        total = (global_windows if global_windows is not None else x_local.shape[0]) * L
        for layer in self._layers():
            # counters of GP h, point n: step * total * H + h * total + (global n): identical for any rank count
            layer._rng_offset = self.step_index * total * max(1, layer.output_dims or 1) + first_global_window * L
            layer._rng_h_stride = total
        self.step_index += 1
        return self.model.blur(x_local, y_local, num_data=num_data)

    def zero_grad(self, set_to_none: bool = False):   # keep the views alive
        self.bucket.zero()

    def sync_grads(self, average: bool = True):
        return self.bucket.all_reduce(self.group, average=average)
