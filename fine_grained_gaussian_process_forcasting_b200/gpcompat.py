"""The slice of the gpytorch class protocol that the reference's GP blur path touches, re-implemented
on the gpblur CUDA ops (no gpytorch, no linear_operator, no autograd through library linear algebra).

Every class keeps gpytorch's constructor arguments, attribute names and state_dict key names so that

* ``fine_grained_gaussian_process_forcasting_b200.DeepGP`` / ``GPModel`` (this package's own modules), and
* the reference's UNCHANGED ``denoising_model/DeepGP.py`` (via the ``compat/gpytorch`` import shim)

both build the same module tree and checkpoints written by the reference load with ``strict=True``.

Reference call sites mirrored here (all in /root/reference):
  denoising_model/DeepGP.py:6-11      imports (MultivariateNormal, ScaleKernel, RBFKernel, GaussianLikelihood,
                                       ConstantMean, LinearMean, DeepGPLayer, DeepGP, VariationalStrategy,
                                       MeanFieldVariationalDistribution)
  denoising_model/DeepGP.py:28-49     module construction order
  denoising_model/DeepGP.py:62-73     __call__ protocol (are_samples, num_likelihood_samples)
  forecast_denoising.py:87-89         DeepApproximateMLL(VariationalELBO(likelihood, model, num_data))(dist, y)
  train.py:20, evaluate.py:134        gpytorch.settings.num_likelihood_samples(1)
"""
from __future__ import annotations

import math
import warnings
from typing import Optional

import torch
from torch import nn

from . import ops


# ------------------------------------------------------------------------------------------------
# settings
# ------------------------------------------------------------------------------------------------
class _ValueContext:
    """gpytorch.settings-style class-level value with context-manager override."""
    _global_value = None

    def __init__(self, value):
        self._new = value
        self._old = None

    @classmethod
    def value(cls):
        return cls._global_value

    @classmethod
    def _set_value(cls, v):
        cls._global_value = v

    def __enter__(self):
        self._old = self.__class__.value()
        self.__class__._set_value(self._new)
        return self

    def __exit__(self, *exc):
        self.__class__._set_value(self._old)
        return False


class num_likelihood_samples(_ValueContext):
    """Leading sample dimension of DeepGP outputs (gpytorch default 10; the reference runs under 1,
    train.py:20)."""
    _global_value = 10


class check_cholesky(_ValueContext):
    """If True (default, gpytorch's behaviour), building the M x M stage synchronises on the Cholesky ``info`` flag
    and follows psd_safe_cholesky: retry with 1e-6, 1e-5, 1e-4 extra diagonal jitter (NumericalWarning), then raise
    NotPSDError.  If False - and always while a CUDA graph is being captured - the flag is only kept on the layer
    (``last_info``; ``graphs.GraphedStep.check_info()`` reads it after a replay) and NaNs would propagate."""
    _global_value = True


class variational_cholesky_jitter:
    @staticmethod
    def value(dtype=torch.float32):
        return 1e-4


class min_variance:
    @staticmethod
    def value(dtype=torch.float32):
        return 1e-6


NotPSDError = ops.NotPSDError
NumericalWarning = ops.NumericalWarning


# ------------------------------------------------------------------------------------------------
# constraints
# ------------------------------------------------------------------------------------------------
class Interval(nn.Module):
    def __init__(self, lower_bound, upper_bound):
        super().__init__()
        self.register_buffer("lower_bound", torch.as_tensor(float(lower_bound)))
        self.register_buffer("upper_bound", torch.as_tensor(float(upper_bound)))

    def transform(self, raw):
        return torch.nn.functional.softplus(raw) + self.lower_bound

    def inverse_transform(self, value):
        v = torch.as_tensor(value) - self.lower_bound
        return v + torch.log(-torch.expm1(-v))


class GreaterThan(Interval):
    def __init__(self, lower_bound):
        super().__init__(lower_bound, math.inf)


class Positive(GreaterThan):
    def __init__(self):
        super().__init__(0.0)


# ------------------------------------------------------------------------------------------------
# means / kernels (parameter holders; evaluation happens inside the fused CUDA ops)
# ------------------------------------------------------------------------------------------------
class Mean(nn.Module):
    pass


class ConstantMean(Mean):
    def __init__(self, constant_prior=None, constant_constraint=None, batch_shape=torch.Size(), **kwargs):
        super().__init__()
        self.batch_shape = torch.Size(batch_shape)
        self.register_parameter("raw_constant", nn.Parameter(torch.zeros(self.batch_shape)))

    @property
    def constant(self):
        return self.raw_constant

    def forward(self, x):
        c = self.raw_constant
        return c.unsqueeze(-1).expand(*x.shape[:-1]) if c.dim() else c.expand(x.shape[:-1])


class LinearMean(Mean):
    def __init__(self, input_size, batch_shape=torch.Size(), bias=True):
        super().__init__()
        self.register_parameter("weights", nn.Parameter(torch.randn(*batch_shape, input_size, 1)))
        if bias:
            self.register_parameter("bias", nn.Parameter(torch.randn(*batch_shape, 1)))
        else:
            self.bias = None

    def forward(self, x):
        res = x.matmul(self.weights).squeeze(-1)
        if self.bias is not None:
            res = res + self.bias
        return res


class Kernel(nn.Module):
    has_lengthscale = False

    def __init__(self, ard_num_dims=None, batch_shape=torch.Size(), **kwargs):
        super().__init__()
        self.ard_num_dims = ard_num_dims
        self.batch_shape = torch.Size(batch_shape)
        if self.has_lengthscale:
            nd = 1 if ard_num_dims is None else ard_num_dims
            self.register_parameter("raw_lengthscale", nn.Parameter(torch.zeros(*self.batch_shape, 1, nd)))
            self.raw_lengthscale_constraint = Positive()

    @property
    def lengthscale(self):
        return self.raw_lengthscale_constraint.transform(self.raw_lengthscale)


class RBFKernel(Kernel):
    has_lengthscale = True


class MaternKernel(Kernel):
    """gpytorch's MaternKernel (imported by the reference at DeepGP.py:7): nu in {0.5, 1.5, 2.5}, evaluated by the same
    CUDA kernels as RBFKernel (include/gpblur.h: GPBLUR_KERNEL_MATERN*)."""
    has_lengthscale = True

    def __init__(self, nu=2.5, **kwargs):
        if nu not in {0.5, 1.5, 2.5}:
            raise RuntimeError("nu expected to be 0.5, 1.5, or 2.5")
        super().__init__(**kwargs)
        self.nu = nu

    @property
    def kernel_name(self):
        return {0.5: "matern12", 1.5: "matern32", 2.5: "matern52"}[self.nu]


class RQKernel(Kernel):
    """gpytorch's RQKernel: k = (1 + d^2 / (2 alpha))^-alpha with a learnable alpha = softplus(raw_alpha), raw_alpha
    of shape [*batch_shape, 1] (zeros: alpha = ln 2), evaluated by the same CUDA kernels as RBFKernel
    (include/gpblur.h: GPBLUR_KERNEL_RQ)."""
    has_lengthscale = True
    kernel_name = "rq"

    def __init__(self, alpha_constraint=None, **kwargs):
        super().__init__(**kwargs)
        self.register_parameter("raw_alpha", nn.Parameter(torch.zeros(*self.batch_shape, 1)))
        self.raw_alpha_constraint = Positive() if alpha_constraint is None else alpha_constraint

    @property
    def alpha(self):
        return self.raw_alpha_constraint.transform(self.raw_alpha)


class ScaleKernel(Kernel):
    def __init__(self, base_kernel, outputscale_prior=None, outputscale_constraint=None, **kwargs):
        kwargs.pop("ard_num_dims", None)
        super().__init__(**kwargs)
        self.base_kernel = base_kernel
        outputscale = torch.zeros(*self.batch_shape) if len(self.batch_shape) else torch.tensor(0.0)
        self.register_parameter("raw_outputscale", nn.Parameter(outputscale))
        self.raw_outputscale_constraint = Positive()

    @property
    def outputscale(self):
        return self.raw_outputscale_constraint.transform(self.raw_outputscale)

    def forward(self, x1, x2=None):
        """Dense ScaleKernel(RBF | Matern | RQ) covariance by the CUDA kernel, differentiable w.r.t. the inputs and the
        raw hyper-parameters (hand-written backward: gpblur_covariance_backward_alpha)."""
        x2 = x1 if x2 is None else x2
        bk = self.base_kernel
        if not isinstance(bk, _CUDA_KERNELS) or len(self.batch_shape):
            raise NotImplementedError("dense covariance: un-batched ScaleKernel(RBFKernel | MaternKernel | RQKernel) "
                                      "only")
        kernel = _base_kernel_name(bk)
        raw_alpha = bk.raw_alpha if isinstance(bk, RQKernel) else None
        lead = x1.shape[:-2]
        x1f = x1.reshape(-1, x1.shape[-2], x1.shape[-1])
        x2f = x2.reshape(-1, x2.shape[-2], x2.shape[-1])
        same = x2 is x1
        outs = [ops.rbf_covariance(a, a if same else b, bk.raw_lengthscale, self.raw_outputscale, bk.ard_num_dims is not None,
                                   kernel=kernel, raw_alpha=raw_alpha)
                for a, b in zip(x1f, x2f)]
        return torch.stack(outs).reshape(*lead, x1.shape[-2], x2.shape[-2])


def _base_kernel_name(base_kernel):
    return "rbf" if isinstance(base_kernel, RBFKernel) else base_kernel.kernel_name


_CUDA_KERNELS = (RBFKernel, MaternKernel, RQKernel)


def _kernel_raw_params(covar_module):
    """(raw_lengthscale, raw_outputscale, kernel name) of a ScaleKernel(RBFKernel | MaternKernel | RQKernel), and
    raw_alpha after them for an RQKernel - anything else is unsupported.  The name is what ops.svgp_predict takes as
    `kernel`."""
    if not isinstance(covar_module, ScaleKernel) or not isinstance(covar_module.base_kernel, _CUDA_KERNELS):
        raise NotImplementedError("the CUDA GP path implements ScaleKernel(RBFKernel | MaternKernel | "
                                  "RQKernel(ard_num_dims=D)) (DeepGP.py:46-49); got %r" % type(covar_module).__name__)
    bk = covar_module.base_kernel
    return (bk.raw_lengthscale, covar_module.raw_outputscale, _base_kernel_name(bk)) + \
        ((bk.raw_alpha,) if isinstance(bk, RQKernel) else ())


# ------------------------------------------------------------------------------------------------
# distributions
# ------------------------------------------------------------------------------------------------
class MultivariateNormal:
    """Diagonal view of the predictive (what the reference ever reads: .mean, .variance, event/batch
    shapes; DeepGP.py:97-99, forecast_denoising.py:89).  May also carry a dense covariance (prior)."""

    def __init__(self, mean, covariance_matrix=None, *, variance=None, sample=None, kl=None, layer=None):
        self._mean = mean
        self._covar = covariance_matrix
        self._variance = variance
        self._sample = sample
        self.kl = kl
        self._layer = layer

    @property
    def mean(self):
        return self._mean

    loc = mean

    @property
    def variance(self):
        if self._variance is not None:
            return self._variance
        cov = self.covariance_matrix
        v = cov.diagonal(dim1=-1, dim2=-2)
        mv = min_variance.value(v.dtype)
        if v.lt(mv).any():
            warnings.warn(f"Negative variance values detected. Rounding negative variances up to {mv}.",
                          NumericalWarning)
            v = v.clamp_min(mv)
        return v

    @property
    def stddev(self):
        return self.variance.sqrt()

    @property
    def covariance_matrix(self):
        if callable(self._covar):
            self._covar = self._covar()
        if self._covar is None:
            return torch.diag_embed(self._variance)
        return self._covar

    lazy_covariance_matrix = covariance_matrix

    @property
    def event_shape(self):
        return self._mean.shape[-1:]

    @property
    def batch_shape(self):
        return self._mean.shape[:-1]

    @property
    def sample_value(self):
        """Reparameterised blurred sample fused into the forward kernel (None if not requested)."""
        return self._sample

    def rsample(self, sample_shape=torch.Size()):
        """mean + sqrt(variance) * eps with Philox eps.  The first call returns the sample fused into the
        forward kernel; later calls draw fresh counters from the owning layer."""
        if len(sample_shape):
            raise NotImplementedError("sample_shape is not supported; use num_likelihood_samples")
        if self._sample is not None:
            s, self._sample = self._sample, None
            return s
        if self._layer is None:
            raise RuntimeError("distribution has no RNG owner")
        seed, offset, stream = self._layer._next_counters(self._mean.numel())
        return ops.rsample(self._mean, self.variance, seed, offset, stream)

    def sample(self, sample_shape=torch.Size()):
        with torch.no_grad():
            return self.rsample(sample_shape)

    def confidence_region(self):
        std2 = self.stddev * 2
        return self.mean - std2, self.mean + std2

    def expand(self, *shape):
        """Leading sample dimension S of DeepGP outputs.  S == 1 (the reference, train.py:20) is a pure view
        (``unsqueeze``: no reduction kernel in its backward); for S > 1 the single fused sample is dropped, so that
        ``rsample()`` draws S * n independent Philox counters like gpytorch's Normal(...).rsample() on the expanded
        distribution."""
        if len(shape) == self._mean.dim() + 1 and shape[0] == 1:
            def ex(t):
                return None if t is None else t.unsqueeze(0)
            keep_sample = True
        else:
            def ex(t):
                return None if t is None else t.expand(*shape)
            keep_sample = False
        return self.__class__(ex(self._mean), None, variance=ex(self._variance),
                              sample=ex(self._sample) if keep_sample else None, kl=self.kl, layer=self._layer)

    def __add__(self, other):
        return MultivariateNormal(self._mean + other, self._covar, variance=self._variance, sample=self._sample,
                                  kl=self.kl, layer=self._layer)


class MultitaskMultivariateNormal(MultivariateNormal):
    """Output of a hidden layer with output_dims = H: mean / variance [..., n, H] (independent tasks)."""

    @property
    def event_shape(self):
        return self._mean.shape[-2:]

    @property
    def batch_shape(self):
        return self._mean.shape[:-2]


# ------------------------------------------------------------------------------------------------
# variational pieces
# ------------------------------------------------------------------------------------------------
class MeanFieldVariationalDistribution(nn.Module):
    def __init__(self, num_inducing_points, batch_shape=torch.Size(), mean_init_std=1e-3, **kwargs):
        super().__init__()
        self.num_inducing_points = num_inducing_points
        self.batch_shape = torch.Size(batch_shape)
        self.mean_init_std = mean_init_std
        mean_init = torch.zeros(num_inducing_points).repeat(*self.batch_shape, 1)
        covar_init = torch.ones(num_inducing_points).repeat(*self.batch_shape, 1)
        self.register_parameter("variational_mean", nn.Parameter(mean_init))
        self.register_parameter("_variational_stddev", nn.Parameter(covar_init))

    @property
    def variational_stddev(self):
        # gpytorch masks with clamp_min(1e-8); covariance uses stddev^2 so the sign is irrelevant
        return self._variational_stddev

    def initialize_variational_distribution(self):
        """First-call init against the whitened prior N(0, I): m <- 0 + 1e-3 randn, s <- 1.
        Consumes the global torch RNG of the parameter's device, as gpytorch does."""
        with torch.no_grad():
            self.variational_mean.zero_()
            self.variational_mean.add_(torch.randn_like(self.variational_mean), alpha=self.mean_init_std)
            self._variational_stddev.fill_(1.0)


class VariationalStrategy(nn.Module):
    """Whitened variational strategy (parameters only; the math is the fused CUDA forward)."""

    def __init__(self, model, inducing_points, variational_distribution, learn_inducing_locations=True,
                 jitter_val=None):
        super().__init__()
        object.__setattr__(self, "model", model)
        inducing_points = inducing_points.clone()
        if inducing_points.dim() == 1:
            inducing_points = inducing_points.unsqueeze(-1)
        if learn_inducing_locations:
            self.register_parameter("inducing_points", nn.Parameter(inducing_points))
        else:
            self.register_buffer("inducing_points", inducing_points)
        self._variational_distribution = variational_distribution
        self.register_buffer("variational_params_initialized", torch.tensor(0))
        self.register_buffer("updated_strategy", torch.tensor(True))
        self._initialized_py = False
        self._last_kl = None
        self._last_kl_versions = None

    def _ensure_initialized(self):
        if self._initialized_py:
            return
        if not bool(self.variational_params_initialized.item()):
            self._variational_distribution.initialize_variational_distribution()
            self.variational_params_initialized.fill_(1)
        self._initialized_py = True

    def _load_from_state_dict(self, *args, **kwargs):
        super()._load_from_state_dict(*args, **kwargs)
        self._initialized_py = False
        self._last_kl = None

    def _versions(self):
        vd = self._variational_distribution
        return (vd.variational_mean._version, vd._variational_stddev._version,
                vd.variational_mean.data_ptr(), vd._variational_stddev.data_ptr())

    def _cache_kl(self, kl):
        self._last_kl = kl
        self._last_kl_versions = self._versions()

    def kl_divergence(self):
        """KL(q(u) || N(0, I)), summed over output dims.  Returns the value computed by the last fused
        forward (autograd-connected) when the variational parameters are unchanged since then; otherwise
        runs the M x M stage of the CUDA forward on zero points."""
        vd = self._variational_distribution
        want_grad = torch.is_grad_enabled() and (vd.variational_mean.requires_grad or
                                                 vd._variational_stddev.requires_grad)
        if self._last_kl is not None and self._last_kl_versions == self._versions() and \
                (self._last_kl.requires_grad or not want_grad):
            return self._last_kl
        layer = self.model
        kl = layer._kl_only()
        self._cache_kl(kl)
        return kl


class _DeepGPVariationalStrategy:
    def __init__(self, model):
        self.model = model

    @property
    def sub_variational_strategies(self):
        return [m.variational_strategy for m in self.model.modules() if isinstance(m, ApproximateGP)]

    def kl_divergence(self):
        terms = [s.kl_divergence() for s in self.sub_variational_strategies]
        if len(terms) == 1 and terms[0].numel() == 1:
            return terms[0].reshape(())              # one GP: a view, no reduction / accumulation kernels
        total = terms[0].sum()
        for t in terms[1:]:
            total = total + t.sum()
        return total


# ------------------------------------------------------------------------------------------------
# models
# ------------------------------------------------------------------------------------------------
class GP(nn.Module):
    def added_loss_terms(self):
        return iter(())

    def named_priors(self):
        return iter(())

    def named_added_loss_terms(self):
        return iter(())


class ApproximateGP(GP):
    def __init__(self, variational_strategy):
        super().__init__()
        self.variational_strategy = variational_strategy


class DeepGPLayer(ApproximateGP):
    """One (possibly multi-output) whitened SVGP layer evaluated by the fused CUDA ops.

    gpytorch's DeepGPLayer.__call__ -> ApproximateGP.__call__ -> VariationalStrategy.__call__/forward
    chain (batch-expanded inducing points, three kernel builds, fp64 Cholesky + solve per batch
    element) collapses into ONE ``ops.svgp_predict`` call per output dim."""

    def __init__(self, variational_strategy, input_dims, output_dims):
        super().__init__(variational_strategy)
        self.input_dims = input_dims
        self.output_dims = output_dims
        self._rng_seed = 0
        self._rng_offset = 0
        self._rng_stream = 0
        self._rng_h_stride = None          # Philox counter stride between the H GPs (None: the points of the call)
        self._grad_sink = None             # flat fp32 view the M x M backward accumulates into (FlatGradBucket)
        self.fused_sample = True
        self.last_info = None
        self.rng_offset_dev = None         # optional int64 device scalar added to the Philox offset (graphs.py)
        self.share_param_stage = True      # reuse Kzz / Cholesky / Linv between calls with unchanged parameters
        self._stage_caches = {}

    # ---- RNG counters of the fused sampler (Philox key = seed, counter = (offset + point, stream)) ----
    def set_rng(self, seed: int, offset: int = 0, stream: int = 0):
        self._rng_seed, self._rng_offset, self._rng_stream = int(seed), int(offset), int(stream)

    def invalidate_param_stage(self):
        """Drop the cached M x M stage (parameters are also tracked by tensor version, so an optimizer step
        invalidates it automatically; benchmarks that never step call this to stay honest)."""
        self._stage_caches = {}
        vs = self.variational_strategy
        vs._last_kl = None          # it references the autograd graph of the dropped stage
        vs._last_kl_versions = None

    def _next_counters(self, n: int):
        seed, off, stream = self._rng_seed, self._rng_offset, self._rng_stream
        self._rng_offset += int(n)
        return seed, off, stream

    def forward(self, x):   # pragma: no cover - subclasses define the prior
        raise NotImplementedError

    def _layer_params(self):
        """Parameter tensors of the layer in the C-ABI gradient-bucket order (include/gpblur.h): Z, raw_lengthscale,
        raw_outputscale, variational_mean, variational_stddev, weights, bias, and raw_alpha after them for an RQKernel.
        A multi-output layer (output_dims = H) passes its batched parameters ([H, M, D] inducing points ...) and is
        evaluated by ONE batched op."""
        vs = self.variational_strategy
        vd = vs._variational_distribution
        raw_ell, raw_os, _, *alpha = _kernel_raw_params(self.covar_module)
        Z, m, s = vs.inducing_points, vd.variational_mean, vd._variational_stddev
        mm = self.mean_module
        if isinstance(mm, LinearMean):
            w, b = mm.weights, (mm.bias if mm.bias is not None else torch.zeros(1, device=Z.device))
        elif isinstance(mm, ConstantMean):
            w, b = None, mm.raw_constant
        else:
            raise NotImplementedError("mean module %r" % type(mm).__name__)
        return (Z, raw_ell, raw_os, m, s, w, b, *alpha)

    def _op_args(self):
        """(the seven positional parameters of ops.svgp_*, keyword arguments kernel / raw_alpha)"""
        p = self._layer_params()
        return p[:7], {"kernel": _kernel_raw_params(self.covar_module)[2], "raw_alpha": p[7] if len(p) > 7 else None}

    def _stage_cache(self):
        return self._stage_caches.setdefault(None, {}) if self.share_param_stage else None

    def _kl_only(self):
        params, kw = self._op_args()
        _, kl, _, _ = ops.svgp_param_stage(*params, stage_cache=self._stage_cache(),
                                           check=bool(check_cholesky.value()), grad_sink=self._grad_sink, **kw)
        return kl.sum() if kl.dim() else kl

    def __call__(self, inputs, are_samples=False, **kwargs):
        vs = self.variational_strategy
        vs._ensure_initialized()
        if isinstance(inputs, MultitaskMultivariateNormal):
            inputs = inputs.rsample()
            are_samples = True
        elif isinstance(inputs, MultivariateNormal):
            inputs = inputs.rsample().unsqueeze(-1)
            are_samples = True
        if inputs.dim() == 1:
            inputs = inputs.unsqueeze(-1)
        if inputs.shape[-1] != self.input_dims:
            raise RuntimeError(f"Input shape did not match self.input_dims. Got total feature dims "
                               f"[{inputs.shape[-1]}], expected [{self.input_dims}]")
        H = self.output_dims
        n_pts = inputs.numel() // inputs.shape[-1]
        # GP h of a multi-output layer draws its sample with counters offset + h * n_pts + n
        seed, off, stream = self._next_counters(n_pts * (H or 1)) if self.fused_sample else (0, 0, 0)
        params, kw = self._op_args()
        mean, var, sample, kl, info = ops.svgp_predict(inputs, *params, seed, off, stream,
                                                       want_sample=self.fused_sample,
                                                       stage_cache=self._stage_cache(),
                                                       offset_dev=self.rng_offset_dev, h_stride=self._rng_h_stride,
                                                       check=bool(check_cholesky.value()),
                                                       grad_sink=self._grad_sink, **kw)
        self.last_info = info
        if H is None:
            cls = MultivariateNormal
        else:
            kl = kl.sum()
            cls = MultitaskMultivariateNormal
        vs._cache_kl(kl)
        dist = cls(mean, None, variance=var, sample=sample, kl=kl, layer=self)
        if not are_samples:
            S = num_likelihood_samples.value()
            dist = dist.expand(S, *mean.shape)
        return dist


    def call_segments(self, x_flat, seg_shapes):
        """ONE fused evaluation on x_flat [N, D] = the concatenated points of several activations (the reference
        blurs the encoder and the decoder activations of a step with the same GP, denoise_model_2.py:50-51).
        ``seg_shapes``: output shape of every segment, e.g. [(B, 192), (B, 24)].  Returns one distribution per
        segment, exactly what separate calls return (same Philox counters: segment s starts where s - 1 ended)."""
        vs = self.variational_strategy
        vs._ensure_initialized()
        if self.output_dims is not None:
            raise NotImplementedError("call_segments: single-output layers only")
        if x_flat.dim() != 2 or x_flat.shape[-1] != self.input_dims:
            raise RuntimeError(f"call_segments expects [N, {self.input_dims}] points, got {tuple(x_flat.shape)}")
        n_pts = x_flat.shape[0]
        seed, off, stream = self._next_counters(n_pts) if self.fused_sample else (0, 0, 0)
        params, kw = self._op_args()
        segs, kl, info = ops.svgp_predict_segments(x_flat, seg_shapes, *params, seed, off, stream,
                                                   want_sample=self.fused_sample, stage_cache=self._stage_cache(),
                                                   offset_dev=self.rng_offset_dev,
                                                   check=bool(check_cholesky.value()), grad_sink=self._grad_sink, **kw)
        self.last_info = info
        vs._cache_kl(kl)
        S = num_likelihood_samples.value()
        return [MultivariateNormal(m, None, variance=v, sample=sm, kl=kl, layer=self).expand(S, *m.shape)
                for (m, v, sm) in segs]


class DeepGP(GP):
    def __init__(self):
        super().__init__()
        self.variational_strategy = _DeepGPVariationalStrategy(self)

    def forward(self, x):   # pragma: no cover
        raise NotImplementedError

    def __call__(self, *args, **kwargs):
        return self.forward(*args, **kwargs)


# ------------------------------------------------------------------------------------------------
# likelihood and marginal log likelihoods
# ------------------------------------------------------------------------------------------------
class HomoskedasticNoise(nn.Module):
    def __init__(self, noise_prior=None, noise_constraint=None, batch_shape=torch.Size()):
        super().__init__()
        if noise_constraint is None:
            noise_constraint = GreaterThan(1e-4)
        self.register_parameter("raw_noise", nn.Parameter(torch.zeros(*batch_shape, 1)))
        self.raw_noise_constraint = noise_constraint

    @property
    def noise(self):
        return self.raw_noise_constraint.transform(self.raw_noise)


class GaussianLikelihood(nn.Module):
    def __init__(self, noise_prior=None, noise_constraint=None, batch_shape=torch.Size(), **kwargs):
        super().__init__()
        self.noise_covar = HomoskedasticNoise(noise_prior, noise_constraint, batch_shape)

    @property
    def noise(self):
        return self.noise_covar.noise

    @property
    def raw_noise(self):
        return self.noise_covar.raw_noise

    def forward(self, function_samples):
        raise NotImplementedError

    def __call__(self, dist, *args, **kwargs):
        """Marginal p(y | x): same mean, variance + noise (GaussianLikelihood.marginal)."""
        if not isinstance(dist, MultivariateNormal):
            raise NotImplementedError("likelihood(function_samples) is not on the reference's path")
        out = dist.__class__(dist.mean, None, variance=dist.variance + self.noise, sample=None, kl=dist.kl,
                             layer=dist._layer)
        return out

    def expected_log_prob(self, target, dist):
        noise = self.noise
        mean, var = dist.mean, dist.variance
        return -0.5 * (((target - mean) ** 2 + var) / noise + noise.log() + math.log(2 * math.pi))


class VariationalELBO(nn.Module):
    """ELBO with the fused CUDA likelihood + KL term (forecast_denoising.py:87-88)."""

    def __init__(self, likelihood, model, num_data, beta=1.0, combine_terms=True):
        super().__init__()
        object.__setattr__(self, "likelihood", likelihood)
        object.__setattr__(self, "model", model)
        self.num_data = num_data
        self.beta = beta
        self.combine_terms = combine_terms

    def forward(self, approximate_dist_f, target, **kwargs):
        mean, var = approximate_dist_f.mean, approximate_dist_f.variance
        kl = self.model.variational_strategy.kl_divergence()
        target = target.expand(mean.shape) if target.shape != mean.shape else target
        return ops.variational_elbo(mean, var, target, self.likelihood.raw_noise, kl,
                                    float(self.num_data) / float(self.beta))


class DeepApproximateMLL(nn.Module):
    def __init__(self, base_mll):
        super().__init__()
        self.base_mll = base_mll

    def forward(self, approximate_dist_f, target, **params):
        return self.base_mll(approximate_dist_f, target, **params).mean(0)


class ExactMarginalLogLikelihood(nn.Module):
    """gpytorch.mlls.ExactMarginalLogLikelihood for a Gaussian likelihood: ``mll(model(train_x), train_y)`` =
    log N(y | mean, K + noise I) / n - the objective an ``ExactGPModel`` (GPModel.py:4-13) is trained with.  The
    covariance comes from the CUDA kernel with its hand-written backward; the n x n factorisation is a library call
    (cuSOLVER through torch.linalg), as gpytorch's is."""

    def __init__(self, likelihood, model):
        super().__init__()
        object.__setattr__(self, "likelihood", likelihood)
        object.__setattr__(self, "model", model)

    def forward(self, function_dist, target, **params):
        K = function_dist.covariance_matrix
        n = K.shape[-1]
        Kn = K + self.likelihood.noise * torch.eye(n, device=K.device, dtype=K.dtype)
        Lc = torch.linalg.cholesky(Kn)
        r = (target - function_dist.mean).unsqueeze(-1)
        alpha = torch.cholesky_solve(r, Lc)
        quad = (r * alpha).sum((-2, -1))
        logdet = 2.0 * torch.diagonal(Lc, dim1=-2, dim2=-1).log().sum(-1)
        return -0.5 * (quad + logdet + n * math.log(2 * math.pi)) / n


# ------------------------------------------------------------------------------------------------
# exact GP (GPModel.py)
# ------------------------------------------------------------------------------------------------
class ExactGP(GP):
    """gpytorch.models.ExactGP protocol: train mode returns the prior at the train inputs, eval mode the
    posterior conditioned on (train_inputs, train_targets)."""

    def __init__(self, train_inputs, train_targets, likelihood):
        super().__init__()
        if train_inputs is not None and torch.is_tensor(train_inputs):
            train_inputs = (train_inputs,)
        self.train_inputs = None if train_inputs is None else tuple(
            t.unsqueeze(-1) if t.dim() == 1 else t for t in train_inputs)
        self.train_targets = train_targets
        self.likelihood = likelihood

    def __call__(self, *args, **kwargs):
        x = args[0]
        if x.dim() == 1:
            x = x.unsqueeze(-1)
        if self.training or self.train_inputs is None:
            return self.forward(x)
        xt = self.train_inputs[0]
        full = self.forward(torch.cat([xt, x], dim=-2))
        n = xt.shape[-2]
        cov = full.covariance_matrix
        mean = full.mean
        noise = self.likelihood.noise
        Ktt = cov[..., :n, :n] + noise * torch.eye(n, device=cov.device, dtype=cov.dtype)
        Kst = cov[..., n:, :n]
        Kss = cov[..., n:, n:]
        Lc = torch.linalg.cholesky(Ktt)
        alpha = torch.cholesky_solve((self.train_targets - mean[..., :n]).unsqueeze(-1), Lc).squeeze(-1)
        V = torch.linalg.solve_triangular(Lc, Kst.transpose(-1, -2), upper=False)
        post_mean = mean[..., n:] + (Kst @ alpha.unsqueeze(-1)).squeeze(-1)
        post_cov = Kss - V.transpose(-1, -2) @ V
        return MultivariateNormal(post_mean, post_cov)
