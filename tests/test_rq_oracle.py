"""CPU checks of the rational quadratic kernel (gpytorch RQKernel) of the oracle, the gpytorch shim and the C ABI.

* External anchor: scikit-learn's RationalQuadratic(length_scale=1, alpha) on inputs divided by the lengthscales, for
  the SVGP predictive (m = L^-1 y_z, s = 0 is the exact-GP posterior, as in test_pin_sklearn.py) and the exact GP.
* alpha -> infinity is the RBF kernel.
* Closed form == reference order (gpytorch op order); fp64 gradcheck including raw_alpha; the kernel-order backward
  (the algorithm of the CUDA kernels, with the alpha gradient) against autograd.
* The shim: an RQKernel layer has gpytorch's state_dict keys and alpha = ln 2; the reference DeepGP.py imports
  RQKernel from the shim; the ABI rejects RQ without raw_alpha and still rejects unknown kinds.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import gp_oracle as O
from oracle import rq_oracle as RO

NAMES = ["inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean", "variational_stddev", "weights",
         "bias"]
ALPHAS = [0.3, math.log(2.0), 20.0]


def _raw(alpha):
    return torch.tensor([math.log(math.expm1(alpha))], dtype=torch.float64)   # softplus^-1


def _sk():
    sk = pytest.importorskip("sklearn.gaussian_process")
    from sklearn.gaussian_process.kernels import RationalQuadratic, ConstantKernel
    return sk, RationalQuadratic, ConstantKernel


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("D,M,B,L", [(5, 7, 3, 4), (16, 32, 4, 6)])
def test_svgp_oracle_against_sklearn_rq(alpha, D, M, B, L):
    sk, RQ, ConstantKernel = _sk()
    p = O.clone_params(O.init_params_exercise(D, M, seed=D + M), torch.float64)
    p["raw_alpha"] = _raw(alpha)
    g = torch.Generator().manual_seed(D)
    p["raw_outputscale"] = torch.tensor(0.37, dtype=torch.float64)
    ell = O.softplus(p["raw_lengthscale"]).reshape(-1)
    os_ = O.softplus(p["raw_outputscale"]).reshape(())
    Z = p["inducing_points"]
    yz = torch.randn(M, generator=g, dtype=torch.float64)
    Kzz = RO.scale_direct(Z, Z, ell, os_, "rq", alpha) + 1e-4 * torch.eye(M, dtype=torch.float64)
    Lc = torch.linalg.cholesky(Kzz)
    p["variational_mean"] = torch.linalg.solve_triangular(Lc, yz.unsqueeze(-1), upper=False).squeeze(-1)
    p["variational_stddev"] = torch.zeros(M, dtype=torch.float64)
    p["weights"] = torch.zeros_like(p["weights"])
    p["bias"] = torch.zeros_like(p["bias"])
    x = 0.7 * torch.randn(B, L, D, generator=g, dtype=torch.float64)

    kern = ConstantKernel(float(os_), "fixed") * RQ(1.0, alpha, "fixed", "fixed")
    gpr = sk.GaussianProcessRegressor(kern, alpha=1e-4, optimizer=None).fit((Z / ell).numpy(), yz.numpy())
    mean_s, std_s = gpr.predict((x.reshape(-1, D) / ell).numpy(), return_std=True)
    want_mean = torch.from_numpy(mean_s).reshape(B, L)
    want_var = torch.from_numpy(std_s ** 2).reshape(B, L) + 1e-4
    scale = max(1.0, float(want_mean.abs().max()))
    for fn in (RO.svgp_predict_closed_form, RO.svgp_predict_reference_order):
        mean, var = fn(p, x, kernel="rq")
        assert (mean - want_mean).abs().max() < 1e-7 * scale, fn.__name__
        assert (var - want_var.clamp_min(1e-6)).abs().max() < 1e-7 * float(os_), fn.__name__


@pytest.mark.parametrize("alpha", ALPHAS)
def test_exact_gp_oracle_against_sklearn_rq(alpha):
    sk, RQ, ConstantKernel = _sk()
    g = torch.Generator().manual_seed(3)
    n, ns, D = 40, 9, 4
    tx, ty = torch.randn(n, D, generator=g, dtype=torch.float64), torch.randn(n, generator=g, dtype=torch.float64)
    sx = torch.randn(ns, D, generator=g, dtype=torch.float64)
    c, rl, ro, rn = (torch.tensor(v, dtype=torch.float64) for v in (0.3, 0.8, -0.4, -1.5))
    ra = _raw(alpha)
    ell, os_, noise = float(O.softplus(rl)), float(O.softplus(ro)), float(O.softplus(rn)) + 1e-4
    kern = ConstantKernel(os_, "fixed") * RQ(1.0, alpha, "fixed", "fixed")
    _, cov = RO.exact_gp_prior(tx, c, rl, ro, "rq", ra)
    assert np.abs(cov.numpy() - kern((tx / ell).numpy())).max() < 1e-12
    gpr = sk.GaussianProcessRegressor(kern, alpha=noise, optimizer=None).fit((tx / ell).numpy(), (ty - c).numpy())
    mean_s, cov_s = gpr.predict((sx / ell).numpy(), return_cov=True)
    pm, pc = RO.exact_gp_posterior(tx, ty, sx, c, rl, ro, rn, "rq", ra)
    assert np.abs(pm.numpy() - (mean_s + float(c))).max() < 1e-9 and np.abs(pc.numpy() - cov_s).max() < 1e-9


def test_large_alpha_is_rbf():
    p = O.clone_params(O.init_params_exercise(8, 12, seed=4), torch.float64)
    x, _, _, _ = O.make_inputs(3, 5, 8, 2, dtype=torch.float64)
    q = dict(p, raw_alpha=torch.tensor([1e6], dtype=torch.float64))
    for a, b in zip(RO.svgp_predict_closed_form(q, x, kernel="rq"), O.svgp_predict_closed_form(p, x)):
        assert (a - b).abs().max() < 1e-6 * max(1.0, float(b.abs().max()))


@pytest.mark.parametrize("alpha", ALPHAS)
def test_closed_form_equals_reference_order(alpha):
    p = O.clone_params(O.init_params_exercise(16, 24, seed=4), torch.float64)
    p["raw_alpha"] = _raw(alpha)
    x, _, _, _ = O.make_inputs(3, 5, 16, 2, dtype=torch.float64)
    m1, v1 = RO.svgp_predict_closed_form(p, x, kernel="rq")
    m2, v2 = RO.svgp_predict_reference_order(p, x, kernel="rq")
    assert (m1 - m2).abs().max() < 1e-9 * max(1.0, float(m1.abs().max()))
    assert (v1 - v2).abs().max() < 1e-9


def test_closed_form_gradcheck_with_raw_alpha():
    D, M = 3, 5
    p = O.clone_params(O.init_params_exercise(D, M, seed=11), torch.float64)
    p["raw_alpha"] = torch.tensor([0.2], dtype=torch.float64)
    x, _, _, _ = O.make_inputs(2, 3, D, 5, dtype=torch.float64)
    names = ["inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean", "variational_stddev",
             "raw_alpha"]

    def f(xx, *vals):
        q = dict(p)
        q.update(zip(names, vals))
        mean, var = RO.svgp_predict_closed_form(q, xx, kernel="rq")
        return mean.sum() + (var * torch.linspace(0.5, 1.5, var.numel(), dtype=torch.float64).reshape(var.shape)).sum()

    args = [x.clone().requires_grad_(True)] + [p[k].clone().requires_grad_(True) for k in names]
    assert torch.autograd.gradcheck(f, args, eps=1e-6, atol=1e-6, rtol=1e-5)


@pytest.mark.parametrize("raw_alpha", [-1.0, 0.0, 2.0])
def test_kernel_order_backward_matches_autograd(raw_alpha):
    D, M, B, L = 6, 10, 3, 4
    p = O.clone_params(O.init_params_exercise(D, M, seed=7), torch.float64)
    p["raw_alpha"] = torch.tensor([raw_alpha], dtype=torch.float64)
    p = O.clone_params(p, torch.float64, requires_grad=True)
    x, _, _, _ = O.make_inputs(B, L, D, 3, dtype=torch.float64)
    x = x.requires_grad_(True)
    g = torch.Generator().manual_seed(1)
    gm = torch.randn(B, L, generator=g, dtype=torch.float64)
    gv = torch.randn(B, L, generator=g, dtype=torch.float64)
    mean, var = RO.svgp_predict_closed_form(p, x, kernel="rq")
    ((gm * mean).sum() + (gv * var).sum() + 0.3 * O.kl_meanfield(p)).backward()
    got, da = RO.svgp_backward_kernel_order({k: v.detach() for k, v in p.items()}, x.detach(), gm, gv, 0.3,
                                            kernel="rq")

    def close(a, b):
        return (a - b).abs().max() <= 1e-9 * max(1.0, float(b.abs().max()))

    assert close(got.dx, x.grad)
    for name in NAMES:
        assert close(getattr(got, name).reshape(p[name].grad.shape), p[name].grad), name
    assert close(da, p["raw_alpha"].grad)


def test_rq_oracle_other_kernels_are_matern_oracle():
    from oracle import matern_oracle as MO
    p = O.clone_params(O.init_params_exercise(6, 10, seed=7), torch.float64)
    x, _, _, _ = O.make_inputs(3, 4, 6, 3, dtype=torch.float64)
    for kernel in ("rbf", "matern32"):
        for a, b in zip(RO.svgp_predict_closed_form(p, x, kernel=kernel), MO.svgp_predict_closed_form(p, x, kernel=kernel)):
            assert torch.equal(a, b)
    with pytest.raises(ValueError):
        RO.scale_direct(x[0], x[0], 1.0, 1.0, "rq")            # "rq" needs alpha


def test_shim_rq_layer_state_dict_and_default_alpha():
    import fine_grained_gaussian_process_forcasting_b200 as pkg
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    gpytorch = pkg.install_gpytorch_shim()
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import ToyDeepGPHiddenLayer

    D, M = 8, 16
    rbf_layer = ToyDeepGPHiddenLayer(D, None, 0, num_inducing=M, mean_type="linear")
    rq_layer = ToyDeepGPHiddenLayer(D, None, 0, num_inducing=M, mean_type="linear")
    rq_layer.covar_module = gpytorch.kernels.ScaleKernel(gpytorch.kernels.RQKernel(ard_num_dims=D))
    keys, rbf_keys = set(rq_layer.state_dict().keys()), set(rbf_layer.state_dict().keys())
    assert rbf_keys < keys
    extra = keys - rbf_keys
    assert "covar_module.base_kernel.raw_alpha" in extra
    assert all(k.startswith("covar_module.base_kernel.raw_alpha") for k in extra), extra
    assert any(k.startswith("covar_module.base_kernel.raw_alpha_constraint.") for k in extra), extra
    bk = rq_layer.covar_module.base_kernel
    assert tuple(bk.raw_alpha.shape) == (1,) and abs(bk.alpha.item() - math.log(2.0)) < 1e-7
    raw = gpcompat._kernel_raw_params(rq_layer.covar_module)
    assert raw[2] == "rq" and raw[3] is bk.raw_alpha
    lp = rq_layer._layer_params()
    assert len(lp) == 8 and lp[7] is bk.raw_alpha            # bucket order: raw_alpha after the bias
    assert len(rbf_layer._layer_params()) == 7
    batched = gpytorch.kernels.ScaleKernel(gpytorch.kernels.RQKernel(ard_num_dims=D, batch_shape=torch.Size([3])),
                                           batch_shape=torch.Size([3]))
    assert tuple(batched.base_kernel.raw_alpha.shape) == (3, 1)


def test_reference_kernel_imports_include_rq():
    """The reference DeepGP.py's kernel import, with RQKernel added the gpytorch way, resolves against the shim."""
    import fine_grained_gaussian_process_forcasting_b200 as pkg
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    pkg.install_gpytorch_shim()
    from gpytorch.kernels import ScaleKernel, RBFKernel, MaternKernel, RQKernel        # DeepGP.py:7 + RQKernel
    assert RQKernel is gpcompat.RQKernel and ScaleKernel is gpcompat.ScaleKernel
    k = ScaleKernel(RQKernel(ard_num_dims=4))
    assert gpcompat._kernel_raw_params(k)[2] == "rq"


def _lib():
    from fine_grained_gaussian_process_forcasting_b200 import _cabi
    try:
        return _cabi, _cabi.lib()
    except OSError as e:                     # pragma: no cover - library not built
        pytest.skip(f"libgpblur.so not loadable: {e}")


def test_abi_rq_needs_raw_alpha_and_unknown_kinds_fail():
    _cabi, lib = _lib()
    EINVAL = -1
    D, M = 8, 16
    fake = C.c_void_p(1 << 20)               # 256-byte aligned, never dereferenced: validation fails first
    p = _cabi.SvgpParams(fake, fake, fake, fake, fake, fake, fake, None)
    nbytes = int(lib.gpblur_svgp_param_stage_bytes(D, M))
    for kind in (_cabi.KERNEL_KINDS["rq"], 5, -1):
        rc = lib.gpblur_svgp_param_stage(C.byref(p), D, M, kind, 0.0, 0, fake, fake, fake, nbytes, None)
        assert rc == EINVAL, kind
        rc = lib.gpblur_svgp_param_stage_backward(C.byref(p), D, M, kind, fake, None, fake, 0, 0, fake, nbytes, None)
        assert rc == EINVAL, kind
    for kind in (5, -1):
        assert lib.gpblur_svgp_point_forward(fake, fake, 10, D, M, kind, fake, fake, None, 0, 0, 0, None, 0, fake,
                                             1 << 30, None) == EINVAL
    rq = _cabi.KERNEL_KINDS["rq"]
    assert lib.gpblur_covariance_alpha(fake, fake, 4, 4, D, rq, fake, 1, fake, None, fake, None) == EINVAL
    assert lib.gpblur_covariance(fake, fake, 4, 4, D, rq, fake, 1, fake, fake, None) == EINVAL
    nb = int(lib.gpblur_covariance_backward_scratch_bytes(4, 4, D, rq))
    assert nb > int(lib.gpblur_covariance_backward_scratch_bytes(4, 4, D, 0))
    assert lib.gpblur_covariance_backward_alpha(fake, fake, 4, 4, D, rq, fake, 1, fake, None, fake, None, None, fake,
                                                fake, fake, fake, nb, None) == EINVAL
    assert lib.gpblur_covariance_backward_alpha(fake, fake, 4, 4, D, 5, fake, 1, fake, fake, fake, None, None, fake,
                                                fake, fake, fake, nb, None) == EINVAL


def test_abi_sizes_of_rq():
    _cabi, lib = _lib()
    from fine_grained_gaussian_process_forcasting_b200 import ops
    rq = _cabi.KERNEL_KINDS["rq"]
    for D, M in [(5, 3), (64, 256), (128, 1024)]:
        base = int(lib.gpblur_svgp_grad_bucket_floats(D, M))
        assert base == ops.grad_bucket_floats(D, M)
        for kind in range(4):
            assert int(lib.gpblur_svgp_grad_bucket_floats_kind(D, M, kind)) == base
            assert int(lib.gpblur_svgp_stage_grad_doubles_kind(D, M, kind)) == int(
                lib.gpblur_svgp_stage_grad_doubles(D, M))
        assert int(lib.gpblur_svgp_grad_bucket_floats_kind(D, M, rq)) == base + 1 == ops.grad_bucket_floats(D, M, rq)
        assert int(lib.gpblur_svgp_stage_grad_doubles_kind(D, M, rq)) == int(
            lib.gpblur_svgp_stage_grad_doubles(D, M)) + 1
        assert int(lib.gpblur_svgp_grad_bucket_floats_kind(D, M, 5)) == 0
    bucket = torch.arange(float(ops.grad_bucket_floats(4, 3, rq)))
    views = ops.split_bucket(bucket, 4, 3, True, kernel="rq")
    assert len(views) == 8 and views[7].item() == bucket[-1].item()
    assert len(ops.split_bucket(bucket[:-1], 4, 3, True)) == 7
