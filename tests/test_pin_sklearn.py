"""An EXTERNAL anchor for the GP oracle (the suite does not run gpytorch itself):
scikit-learn's exact GP regression, an independent implementation of the same kernel algebra.

* Whitened SVGP predictive.  With the inducing points as "training inputs", whitened variational mean m = L^-1 y_z and
  s = 0, the predictive of /root/reference/denoising_model/DeepGP.py:56-73 (gpytorch VariationalStrategy) is the exact
  GP posterior given noise-free observations y_z at Z with the variational jitter as nugget:
      mean = k_x^T (Kzz + 1e-4 I)^-1 y_z ,   var = os + 1e-4 - k_x^T (Kzz + 1e-4 I)^-1 k_x
  which is GaussianProcessRegressor(ConstantKernel(os) * RBF(ell), alpha=1e-4).  This pins the ARD kernel, the
  outputscale, where the jitter goes, the whitening and the variance formula of BOTH oracle restatements
  (reference order and closed form).  gpytorch-only conventions (1e-6 variance clamp, ELBO scaling) are not touched.
* Exact GP (GPModel.py:4-13): prior covariance and eval-mode posterior against the same class.
"""
import numpy as np
import pytest
import torch

from oracle import gp_oracle as O

sk = pytest.importorskip("sklearn.gaussian_process")
from sklearn.gaussian_process.kernels import RBF, ConstantKernel  # noqa: E402


@pytest.mark.parametrize("D,M,B,L", [(5, 7, 3, 4), (16, 32, 4, 6), (64, 96, 2, 8)])
def test_svgp_oracle_against_sklearn_exact_gp(D, M, B, L):
    p = O.clone_params(O.init_params_exercise(D, M, seed=D + M), torch.float64)
    g = torch.Generator().manual_seed(D)
    p["raw_outputscale"] = torch.tensor(0.37, dtype=torch.float64)
    ell = O.softplus(p["raw_lengthscale"]).reshape(-1)
    os_ = O.softplus(p["raw_outputscale"]).reshape(())
    Z = p["inducing_points"]
    yz = torch.randn(M, generator=g, dtype=torch.float64)
    Kzz = O.rbf_scale_direct(Z, Z, ell, os_) + 1e-4 * torch.eye(M, dtype=torch.float64)
    Lc = torch.linalg.cholesky(Kzz)
    p["variational_mean"] = torch.linalg.solve_triangular(Lc, yz.unsqueeze(-1), upper=False).squeeze(-1)
    p["variational_stddev"] = torch.zeros(M, dtype=torch.float64)
    p["weights"] = torch.zeros_like(p["weights"])
    p["bias"] = torch.zeros_like(p["bias"])
    x = 0.7 * torch.randn(B, L, D, generator=g, dtype=torch.float64)

    kern = ConstantKernel(float(os_), "fixed") * RBF(ell.numpy(), "fixed")
    gpr = sk.GaussianProcessRegressor(kern, alpha=1e-4, optimizer=None).fit(Z.numpy(), yz.numpy())
    mean_s, std_s = gpr.predict(x.reshape(-1, D).numpy(), return_std=True)
    want_mean = torch.from_numpy(mean_s).reshape(B, L)
    want_var = torch.from_numpy(std_s ** 2).reshape(B, L) + 1e-4          # the jitter gpytorch adds to diag(Kxx)
    scale = max(1.0, float(want_mean.abs().max()))
    for fn in (O.svgp_predict_closed_form, O.svgp_predict_reference_order):
        mean, var = fn(p, x)
        # (the reference-order restatement forms squared distances by norm expansion: a few ulps at these scales)
        assert (mean - want_mean).abs().max() < 1e-7 * scale, fn.__name__
        assert (var - want_var.clamp_min(1e-6)).abs().max() < 1e-7 * float(os_), fn.__name__


def test_exact_gp_oracle_against_sklearn():
    g = torch.Generator().manual_seed(3)
    n, ns, D = 40, 9, 4
    tx, ty = torch.randn(n, D, generator=g, dtype=torch.float64), torch.randn(n, generator=g, dtype=torch.float64)
    sx = torch.randn(ns, D, generator=g, dtype=torch.float64)
    c, rl, ro, rn = (torch.tensor(v, dtype=torch.float64) for v in (0.3, 0.8, -0.4, -1.5))
    ell, os_, noise = float(O.softplus(rl)), float(O.softplus(ro)), float(O.softplus(rn)) + 1e-4
    kern = ConstantKernel(os_, "fixed") * RBF(ell, "fixed")
    _, cov = O.exact_gp_prior(tx, c, rl, ro)
    assert np.abs(cov.numpy() - kern(tx.numpy())).max() < 1e-12
    gpr = sk.GaussianProcessRegressor(kern, alpha=noise, optimizer=None).fit(tx.numpy(), (ty - c).numpy())
    mean_s, cov_s = gpr.predict(sx.numpy(), return_cov=True)
    pm, pc = O.exact_gp_posterior(tx, ty, sx, c, rl, ro, rn)
    assert np.abs(pm.numpy() - (mean_s + float(c))).max() < 1e-9 and np.abs(pc.numpy() - cov_s).max() < 1e-9


def test_elbo_terms_against_independent_implementations():
    """KL(q(u) || p(u)) against torch.distributions' own closed form, and the expected log likelihood of
    GaussianLikelihood.expected_log_prob against Gauss-Hermite quadrature of log N(y | f, noise) under f ~ N(mu, var)
    (numpy's nodes): the two terms of forecast_denoising.py:87-89's ELBO, each pinned outside the restatement."""
    g = torch.Generator().manual_seed(9)
    M, B, L, num_data = 24, 3, 5, 32.0
    p = O.clone_params(O.init_params_exercise(8, M, seed=5), torch.float64)
    p["raw_noise"] = torch.tensor([0.3], dtype=torch.float64)
    m, s = p["variational_mean"], p["variational_stddev"]
    q = torch.distributions.MultivariateNormal(m, covariance_matrix=torch.diag(s * s))
    prior = torch.distributions.MultivariateNormal(torch.zeros(M, dtype=torch.float64), torch.eye(M, dtype=torch.float64))
    kl = O.kl_meanfield(p)
    assert abs(float(kl) - float(torch.distributions.kl_divergence(q, prior))) < 1e-10
    mu = torch.randn(B, L, generator=g, dtype=torch.float64)
    var = torch.rand(B, L, generator=g, dtype=torch.float64) + 0.1
    y = torch.randn(B, L, generator=g, dtype=torch.float64)
    noise = O.noise_variance(p)
    nodes, weights = np.polynomial.hermite.hermgauss(40)
    f = mu.unsqueeze(-1) + torch.sqrt(2.0 * var).unsqueeze(-1) * torch.from_numpy(nodes)
    logp = torch.distributions.Normal(f, float(noise.sqrt())).log_prob(y.unsqueeze(-1))
    ell = (logp * torch.from_numpy(weights)).sum(-1) / np.sqrt(np.pi)             # E_q[log p(y | f)] per point
    want = ell.mean(-1) - kl / num_data                                           # VariationalELBO: / L and KL / num_data
    got = O.elbo_per_window(mu, var, y, noise, kl, num_data)
    assert (got - want).abs().max() < 1e-10
