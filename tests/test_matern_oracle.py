"""CPU checks of the Matern kernels (nu = 1/2, 3/2, 5/2) of the oracle and the gpytorch shim.

* External anchor: scikit-learn's GaussianProcessRegressor(ConstantKernel(os) * Matern(ell, nu), alpha=1e-4), as in
  test_pin_sklearn.py: with m = L^-1 y_z and s = 0 the whitened SVGP predictive is that exact GP posterior.
* Closed form == reference order (gpytorch op order: centre, divide, sq_dist, clamp, sqrt).
* fp64 gradcheck of the closed form away from coincident points, and the analytic kernel-order backward (the
  algorithm of the CUDA kernels: W = kbar o g, outputscale through kbar o k) against autograd.
* The shim: a layer with gpytorch.kernels.MaternKernel builds with the RBF layer's state_dict keys; nu = 2.0 raises.
"""
import numpy as np
import pytest
import torch

from oracle import gp_oracle as O
from oracle import matern_oracle as MO

KERNELS = ["matern12", "matern32", "matern52"]
NU = {"matern12": 0.5, "matern32": 1.5, "matern52": 2.5}


def _sk():
    sk = pytest.importorskip("sklearn.gaussian_process")
    from sklearn.gaussian_process.kernels import Matern, ConstantKernel
    return sk, Matern, ConstantKernel


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("D,M,B,L", [(5, 7, 3, 4), (16, 32, 4, 6)])
def test_svgp_oracle_against_sklearn_matern(kernel, D, M, B, L):
    sk, Matern, ConstantKernel = _sk()
    p = O.clone_params(O.init_params_exercise(D, M, seed=D + M), torch.float64)
    g = torch.Generator().manual_seed(D)
    p["raw_outputscale"] = torch.tensor(0.37, dtype=torch.float64)
    ell = O.softplus(p["raw_lengthscale"]).reshape(-1)
    os_ = O.softplus(p["raw_outputscale"]).reshape(())
    Z = p["inducing_points"]
    yz = torch.randn(M, generator=g, dtype=torch.float64)
    Kzz = MO.matern_scale_direct(Z, Z, ell, os_, kernel) + 1e-4 * torch.eye(M, dtype=torch.float64)
    Lc = torch.linalg.cholesky(Kzz)
    p["variational_mean"] = torch.linalg.solve_triangular(Lc, yz.unsqueeze(-1), upper=False).squeeze(-1)
    p["variational_stddev"] = torch.zeros(M, dtype=torch.float64)
    p["weights"] = torch.zeros_like(p["weights"])
    p["bias"] = torch.zeros_like(p["bias"])
    x = 0.7 * torch.randn(B, L, D, generator=g, dtype=torch.float64)

    kern = ConstantKernel(float(os_), "fixed") * Matern(ell.numpy(), "fixed", nu=NU[kernel])
    gpr = sk.GaussianProcessRegressor(kern, alpha=1e-4, optimizer=None).fit(Z.numpy(), yz.numpy())
    mean_s, std_s = gpr.predict(x.reshape(-1, D).numpy(), return_std=True)
    want_mean = torch.from_numpy(mean_s).reshape(B, L)
    want_var = torch.from_numpy(std_s ** 2).reshape(B, L) + 1e-4
    scale = max(1.0, float(want_mean.abs().max()))
    for fn in (MO.svgp_predict_closed_form, MO.svgp_predict_reference_order):
        mean, var = fn(p, x, kernel=kernel)
        assert (mean - want_mean).abs().max() < 1e-7 * scale, fn.__name__
        assert (var - want_var.clamp_min(1e-6)).abs().max() < 1e-7 * float(os_), fn.__name__


@pytest.mark.parametrize("kernel", KERNELS)
def test_exact_gp_oracle_against_sklearn_matern(kernel):
    sk, Matern, ConstantKernel = _sk()
    g = torch.Generator().manual_seed(3)
    n, ns, D = 40, 9, 4
    tx, ty = torch.randn(n, D, generator=g, dtype=torch.float64), torch.randn(n, generator=g, dtype=torch.float64)
    sx = torch.randn(ns, D, generator=g, dtype=torch.float64)
    c, rl, ro, rn = (torch.tensor(v, dtype=torch.float64) for v in (0.3, 0.8, -0.4, -1.5))
    ell, os_, noise = float(O.softplus(rl)), float(O.softplus(ro)), float(O.softplus(rn)) + 1e-4
    kern = ConstantKernel(os_, "fixed") * Matern(ell, "fixed", nu=NU[kernel])
    _, cov = MO.exact_gp_prior(tx, c, rl, ro, kernel=kernel)
    assert np.abs(cov.numpy() - kern(tx.numpy())).max() < 1e-12
    gpr = sk.GaussianProcessRegressor(kern, alpha=noise, optimizer=None).fit(tx.numpy(), (ty - c).numpy())
    mean_s, cov_s = gpr.predict(sx.numpy(), return_cov=True)
    pm, pc = MO.exact_gp_posterior(tx, ty, sx, c, rl, ro, rn, kernel=kernel)
    assert np.abs(pm.numpy() - (mean_s + float(c))).max() < 1e-9 and np.abs(pc.numpy() - cov_s).max() < 1e-9


@pytest.mark.parametrize("kernel", KERNELS)
def test_closed_form_equals_reference_order(kernel):
    p = O.clone_params(O.init_params_exercise(16, 24, seed=4), torch.float64)
    x, _, _, _ = O.make_inputs(3, 5, 16, 2, dtype=torch.float64)
    m1, v1 = MO.svgp_predict_closed_form(p, x, kernel=kernel)
    m2, v2 = MO.svgp_predict_reference_order(p, x, kernel=kernel)
    assert (m1 - m2).abs().max() < 1e-9 * max(1.0, float(m1.abs().max()))
    assert (v1 - v2).abs().max() < 1e-9


@pytest.mark.parametrize("kernel", KERNELS)
def test_closed_form_gradcheck(kernel):
    D, M = 3, 5
    p = O.clone_params(O.init_params_exercise(D, M, seed=11), torch.float64)
    x, _, _, _ = O.make_inputs(2, 3, D, 5, dtype=torch.float64)
    names = ["inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean", "variational_stddev"]

    def f(xx, *vals):
        q = dict(p)
        q.update(zip(names, vals))
        mean, var = MO.svgp_predict_closed_form(q, xx, kernel=kernel)
        return mean.sum() + (var * torch.linspace(0.5, 1.5, var.numel(), dtype=torch.float64).reshape(var.shape)).sum()

    args = [x.clone().requires_grad_(True)] + [p[k].clone().requires_grad_(True) for k in names]
    assert torch.autograd.gradcheck(f, args, eps=1e-6, atol=1e-6, rtol=1e-5)


@pytest.mark.parametrize("kernel", ["rbf"] + KERNELS)
def test_kernel_order_backward_matches_autograd(kernel):
    D, M, B, L = 6, 10, 3, 4
    p = O.clone_params(O.init_params_exercise(D, M, seed=7), torch.float64, requires_grad=True)
    x, _, _, _ = O.make_inputs(B, L, D, 3, dtype=torch.float64)
    x = x.requires_grad_(True)
    g = torch.Generator().manual_seed(1)
    gm = torch.randn(B, L, generator=g, dtype=torch.float64)
    gv = torch.randn(B, L, generator=g, dtype=torch.float64)
    g_kl = 0.3
    mean, var = MO.svgp_predict_closed_form(p, x, kernel=kernel)
    obj = (gm * mean).sum() + (gv * var).sum() + g_kl * O.kl_meanfield(p)
    obj.backward()
    got = MO.svgp_backward_kernel_order({k: v.detach() for k, v in p.items()}, x.detach(), gm, gv, g_kl, kernel=kernel)

    def close(a, b):
        return (a - b).abs().max() <= 1e-9 * max(1.0, float(b.abs().max()))

    assert close(got.dx, x.grad)
    for name in ("inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean", "variational_stddev",
                 "weights", "bias"):
        assert close(getattr(got, name).reshape(p[name].grad.shape), p[name].grad), name


def test_shim_matern_layer_state_dict_and_nu_check():
    import fine_grained_gaussian_process_forcasting_b200 as pkg
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    gpytorch = pkg.install_gpytorch_shim()
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import ToyDeepGPHiddenLayer

    D, M = 8, 16
    rbf_layer = ToyDeepGPHiddenLayer(D, None, 0, num_inducing=M, mean_type="linear")
    mat_layer = ToyDeepGPHiddenLayer(D, None, 0, num_inducing=M, mean_type="linear")
    mat_layer.covar_module = gpytorch.kernels.ScaleKernel(gpytorch.kernels.MaternKernel(nu=1.5, ard_num_dims=D))
    assert sorted(mat_layer.state_dict().keys()) == sorted(rbf_layer.state_dict().keys())
    assert gpcompat._kernel_raw_params(mat_layer.covar_module)[2] == "matern32"
    batched = gpytorch.kernels.ScaleKernel(gpytorch.kernels.MaternKernel(nu=0.5, ard_num_dims=D,
                                                                         batch_shape=torch.Size([3])),
                                           batch_shape=torch.Size([3]))
    ell, os_, kind = gpcompat._kernel_raw_params(batched)
    assert tuple(ell.shape) == (3, 1, D) and tuple(os_.shape) == (3,) and kind == "matern12"
    with pytest.raises(RuntimeError):
        gpytorch.kernels.MaternKernel(nu=2.0, ard_num_dims=D)


def test_matern_oracle_rbf_is_gp_oracle():
    """With kernel="rbf" the restated functions compute what gp_oracle computes."""
    D, M = 6, 10
    p = O.clone_params(O.init_params_exercise(D, M, seed=7), torch.float64)
    x, _, _, _ = O.make_inputs(3, 4, D, 3, dtype=torch.float64)
    for a, b in zip(MO.svgp_predict_closed_form(p, x), O.svgp_predict_closed_form(p, x)):
        assert torch.equal(a, b)
    for a, b in zip(MO.svgp_predict_reference_order(p, x), O.svgp_predict_reference_order(p, x)):
        assert torch.equal(a, b)
    gm, gv = torch.ones(3, 4, dtype=torch.float64), 0.5 * torch.ones(3, 4, dtype=torch.float64)
    ga, gb = MO.svgp_backward_kernel_order(p, x, gm, gv, 0.3), O.svgp_backward_kernel_order(p, x, gm, gv, 0.3)
    for name in ("dx", "inducing_points", "raw_lengthscale", "variational_mean", "variational_stddev"):
        assert torch.equal(getattr(ga, name), getattr(gb, name)), name
    # the outputscale term is summed as sum(Kbar o K) here and as sum(W) there: the same value up to rounding
    assert torch.allclose(ga.raw_outputscale, gb.raw_outputscale, rtol=1e-12, atol=0)
