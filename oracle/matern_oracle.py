"""Matern kernels (gpytorch MaternKernel, nu = 1/2, 3/2, 5/2) for the float64 oracle.

The functions of gp_oracle.py that evaluate the layer's kernel, restated with a ``kernel`` argument ("rbf",
"matern12", "matern32", "matern52").  With ``kernel="rbf"`` each one computes what its gp_oracle namesake computes;
everything that does not depend on the kernel (parameters, ELBO, Philox, KL) is gp_oracle's own.

  x~ = (x - c) / ell,  d2 = |x~ - z~|^2,  r = sqrt(max(d2, 1e-30))   (gpytorch covar_dist)
  k  = os f(r):  f = exp(-r) | (1 + sqrt3 r) exp(-sqrt3 r) | (1 + sqrt5 r + 5/3 r^2) exp(-sqrt5 r)
  g  = -2 os df/d(d2): the weight of every distance gradient (W = kbar o g; g = k for RBF), 0 where the clamp is active
"""
from __future__ import annotations

import math
from typing import Dict, Tuple

import torch

from . import gp_oracle as GO


# Matern kernels (gpytorch MaternKernel, nu = 1/2, 3/2, 5/2): k = os f(r), r = sqrt(max(d2, 1e-30)) (covar_dist)
KERNELS = ("rbf", "matern12", "matern32", "matern52")


def _check_kernel(kernel):
    if kernel not in KERNELS:
        raise ValueError(f"unknown kernel {kernel!r}")


def matern_from_d2(d2, os, kernel):
    """os f(r) and g = -2 os df/d(d2) (the weight of every distance gradient; 0 where the clamp is active)."""
    r = d2.clamp_min(1e-30).sqrt()
    live = d2 > 1e-30
    if kernel == "matern12":
        e = os * torch.exp(-r)
        k, g = e, e / r
    elif kernel == "matern32":
        sr = math.sqrt(3.0) * r
        e = os * torch.exp(-sr)
        k, g = (1.0 + sr) * e, 3.0 * e
    else:
        sr = math.sqrt(5.0) * r
        e = os * torch.exp(-sr)
        k, g = (1.0 + sr + sr * sr / 3.0) * e, (5.0 / 3.0) * (1.0 + sr) * e
    return k, torch.where(live, g, torch.zeros_like(g))


def matern_scale_direct(x1, x2, ell, os, kernel="matern52"):
    """ScaleKernel(MaternKernel(nu)) by direct differences; kernel in matern12 / matern32 / matern52."""
    diff = (x1.unsqueeze(-2) - x2.unsqueeze(-3)) / ell
    return matern_from_d2(diff.pow(2).sum(-1), os, kernel)[0]


def matern_scale_reference_order(x1, x2, ell, os, kernel="matern52"):
    """gpytorch MaternKernel.forward order: centre on the mean of x1, divide by the lengthscale, sq_dist, clamp,
    sqrt."""
    mean = x1.reshape(-1, x1.shape[-1]).mean(0)
    d2 = GO.sq_dist_reference_order((x1 - mean) / ell, (x2 - mean) / ell)
    return matern_from_d2(d2, os, kernel)[0]


def scale_direct(x1, x2, ell, os, kernel="rbf"):
    _check_kernel(kernel)
    return GO.rbf_scale_direct(x1, x2, ell, os) if kernel == "rbf" else matern_scale_direct(x1, x2, ell, os, kernel)


def scale_reference_order(x1, x2, ell, os, kernel="rbf"):
    _check_kernel(kernel)
    if kernel == "rbf":
        return GO.rbf_scale_reference_order(x1, x2, ell, os)
    return matern_scale_reference_order(x1, x2, ell, os, kernel)


def scale_direct_kg(x1, x2, ell, os, kernel="rbf"):
    """(K, G) by direct differences: G = -2 os df/d(d2) (G = K for RBF)."""
    if kernel == "rbf":
        k = GO.rbf_scale_direct(x1, x2, ell, os)
        return k, k
    diff = (x1.unsqueeze(-2) - x2.unsqueeze(-3)) / ell
    return matern_from_d2(diff.pow(2).sum(-1), os, kernel)


def svgp_predict_reference_order(p: Dict[str, torch.Tensor], x: torch.Tensor,
                                 linalg_dtype=torch.float64, kernel="rbf") -> Tuple[torch.Tensor, torch.Tensor]:
    """``ToyDeepGPHiddenLayer.__call__`` -> whitened ``VariationalStrategy.forward`` for
    output_dims=None, linear mean (DeepGP.py:56-73; SURVEY 3.3).  x [B, L, D] -> mean, var [B, L].

    Op order follows gpytorch: inducing points expanded over the batch, ONE kernel evaluation on
    cat([Z, x]) per batch element, jitter on Kzz, Cholesky + solve in ``linalg_dtype``, cast back.
    Differentiable w.r.t. x and every entry of ``p`` by torch autograd.
    """
    Z = p["inducing_points"]
    B, L, D = x.shape
    M = Z.shape[0]
    ell = GO.softplus(p["raw_lengthscale"])               # [1, D]
    os = GO.softplus(p["raw_outputscale"])
    Zb = Z.unsqueeze(0).expand(B, M, D)
    full = torch.cat([Zb, x], dim=-2)                  # [B, M+L, D]
    full_mean = (full @ p["weights"]).squeeze(-1) + p["bias"]      # LinearMean
    full_covar = scale_reference_order(full, full, ell, os, kernel)    # [B, M+L, M+L]
    test_mean = full_mean[..., M:]
    eye = torch.eye(M, dtype=x.dtype)
    Kzz = full_covar[..., :M, :M] + GO.JITTER * eye
    Kzx = full_covar[..., :M, M:]
    Lc = torch.linalg.cholesky(Kzz.to(linalg_dtype))
    A = torch.linalg.solve_triangular(Lc, Kzx.to(linalg_dtype), upper=False).to(x.dtype)   # [B, M, L]
    m = p["variational_mean"]
    s = p["variational_stddev"]
    mean = (A.transpose(-1, -2) @ m.unsqueeze(-1)).squeeze(-1) + test_mean
    # diag(Kxx): gpytorch evaluates the diagonal with diag=True on identical inputs -> d2 = 0 exactly
    kxx_diag = os * torch.ones(B, L, dtype=x.dtype)
    var = kxx_diag + GO.JITTER + ((s.pow(2) - 1.0).unsqueeze(-1) * A.pow(2)).sum(-2)
    var = var.clamp_min(GO.MIN_VARIANCE)
    return mean, var


def svgp_predict_closed_form(p: Dict[str, torch.Tensor], x: torch.Tensor,
                             kernel="rbf") -> Tuple[torch.Tensor, torch.Tensor]:
    """Same predictive in the shared-Z closed form of SURVEY Appendix A (ONE MxM Cholesky, direct
    squared distances).  Intended for float64 "truth" runs."""
    Z = p["inducing_points"]
    B, L, D = x.shape
    M = Z.shape[0]
    ell = GO.softplus(p["raw_lengthscale"]).reshape(D)
    os = GO.softplus(p["raw_outputscale"])
    Kzz = scale_direct(Z, Z, ell, os, kernel) + GO.JITTER * torch.eye(M, dtype=x.dtype)
    Lc = torch.linalg.cholesky(Kzz)
    X = x.reshape(B * L, D)
    Kzx = scale_direct(Z, X, ell, os, kernel)          # [M, N]
    A = torch.linalg.solve_triangular(Lc, Kzx, upper=False)
    m = p["variational_mean"]
    s = p["variational_stddev"]
    mean = A.t() @ m + (X @ p["weights"]).squeeze(-1) + p["bias"]
    var = os + GO.JITTER + ((s.pow(2) - 1.0).unsqueeze(-1) * A.pow(2)).sum(0)
    var = var.clamp_min(GO.MIN_VARIANCE)
    return mean.reshape(B, L), var.reshape(B, L)


def mll_error(p, x, y, num_data, reference_order=True, kernel="rbf") -> torch.Tensor:
    """``-mll(dist, y_true.permute(2,0,1)).mean()`` of forecast_denoising.py:89."""
    fn = svgp_predict_reference_order if reference_order else svgp_predict_closed_form
    mean, var = fn(p, x, kernel=kernel)
    e = GO.elbo_per_window(mean, var, y, GO.noise_variance(p), GO.kl_meanfield(p), num_data)
    return -e.mean()


def svgp_backward_kernel_order(p, x, g_mean, g_var, g_kl=0.0, kernel="rbf") -> GO.SvgpGrads:
    """Analytic gradient of  sum(g_mean*mean) + sum(g_var*var) + g_kl*KL  in the op order of the
    CUDA backward: whitening through the explicit inverse Linv, Gram S = sum_n g_var a a^T,
    E = m u^T + 2 diag(c) S, Gbar = Linv^T E, Lbar = -tril(Gbar), Cholesky backward via
    Kbar = sym(Linv^T Phi(L^T Lbar) Linv).  All tensors float64.  Matern kernels: the distance gradients take
    W = Kbar o G (G = -2 os df/d(d2), scale_direct_kg) in place of Kbar o K; the outputscale takes Kbar o K."""
    Z = p["inducing_points"]
    B, L_, D = x.shape
    M = Z.shape[0]
    N = B * L_
    X = x.reshape(N, D)
    gm = g_mean.reshape(N)
    gv = g_var.reshape(N)
    ell = GO.softplus(p["raw_lengthscale"]).reshape(D)
    os = GO.softplus(p["raw_outputscale"])
    m = p["variational_mean"]
    s = p["variational_stddev"]
    w = p["weights"].reshape(D)
    cvec = s.pow(2) - 1.0

    Kzz0, Gzz = scale_direct_kg(Z, Z, ell, os, kernel)
    Lc = torch.linalg.cholesky(Kzz0 + GO.JITTER * torch.eye(M, dtype=X.dtype))
    Linv = torch.linalg.solve_triangular(Lc, torch.eye(M, dtype=X.dtype), upper=False)
    K, G = scale_direct_kg(X, Z, ell, os, kernel)      # [N, M]
    A = K @ Linv.t()                                   # [N, M]
    var_raw = os + GO.JITTER + (A.pow(2) * cvec).sum(-1)
    gv = torch.where(var_raw < GO.MIN_VARIANCE, torch.zeros_like(gv), gv)   # clamp kills the gradient

    Abar = gm[:, None] * m[None, :] + 2.0 * gv[:, None] * cvec[None, :] * A
    Kbar = Abar @ Linv                                 # k_bar_n = Linv^T a_bar_n
    W = Kbar * G
    r = W.sum(1)
    csum = W.sum(0)
    Xt = X / ell
    Zt = Z / ell
    dx = (W @ Zt - r[:, None] * Xt) / ell + gm[:, None] * w[None, :]
    WX = W.t() @ Xt                                    # [M, D]
    dZ = (WX - csum[:, None] * Zt) / ell
    q = (r[:, None] * Xt.pow(2)).sum(0)
    dell = (q - 2.0 * (Zt * WX).sum(0) + (csum[:, None] * Zt.pow(2)).sum(0)) / ell
    dos = (Kbar * K).sum() / os + gv.sum()
    u = (gm[:, None] * A).sum(0)                       # sum_n g_mu a
    S = A.t() @ (gv[:, None] * A)                      # Gram
    dm = u + g_kl * m
    ds = 2.0 * s * torch.diagonal(S) + g_kl * (s - 1.0 / s)
    dw = (gm[:, None] * X).sum(0)
    db = gm.sum()

    # Cholesky backward
    E = m[:, None] * u[None, :] + 2.0 * cvec[:, None] * S
    Gbar = Linv.t() @ E
    Lbar = -torch.tril(Gbar)
    P = Lc.t() @ Lbar
    Phi = torch.tril(P)
    Phi = Phi - 0.5 * torch.diag(torch.diagonal(P))
    Kb = Linv.t() @ Phi @ Linv
    Kb = 0.5 * (Kb + Kb.t())
    Wzz = Kb * Gzz
    rz = Wzz.sum(1)
    dZ = dZ + 2.0 * (Wzz @ Zt - rz[:, None] * Zt) / ell
    diff2 = (Zt.unsqueeze(1) - Zt.unsqueeze(0)).pow(2)   # [M, M, D]
    dell = dell + (Wzz.unsqueeze(-1) * diff2).sum((0, 1)) / ell
    dos = dos + (Kb * Kzz0).sum() / os

    sig = torch.sigmoid
    return GO.SvgpGrads(
        dx=dx.reshape(B, L_, D),
        inducing_points=dZ,
        raw_lengthscale=(dell * sig(p["raw_lengthscale"]).reshape(D)).reshape(1, D),
        raw_outputscale=dos * sig(p["raw_outputscale"]),
        variational_mean=dm,
        variational_stddev=ds,
        weights=dw.reshape(D, 1),
        bias=db.reshape(1),
    )


def hidden_layer_predict(p1, x, closed_form=True, kernel="rbf"):
    """Layer with output_dims=H: DeepGPLayer expands the input over H and runs H independent
    whitened SVGPs.  Returns mean, var [B, L, H]."""
    H = p1["inducing_points"].shape[0]
    means, vars_ = [], []
    fn = svgp_predict_closed_form if closed_form else svgp_predict_reference_order
    for h in range(H):
        ph = {
            "inducing_points": p1["inducing_points"][h],
            "raw_lengthscale": p1["raw_lengthscale"][h],
            "raw_outputscale": p1["raw_outputscale"][h],
            "variational_mean": p1["variational_mean"][h],
            "variational_stddev": p1["variational_stddev"][h],
            "weights": p1["weights"],
            "bias": p1["bias"],
        }
        mu, v = fn(ph, x, kernel=kernel)
        means.append(mu)
        vars_.append(v)
    return torch.stack(means, -1), torch.stack(vars_, -1)


def deepgp2_predict(p1, p2, x, eps, closed_form=True, kernel="rbf"):
    """Two-layer stack: layer 1 (D -> H), elementwise Normal(mean, sqrt(var)).rsample() with the
    given eps [B, L, H], layer 2 (H -> scalar).  Returns (mean, var, hidden_sample)."""
    mu1, v1 = hidden_layer_predict(p1, x, closed_form, kernel=kernel)
    h = GO.rsample(mu1, v1, eps)
    fn = svgp_predict_closed_form if closed_form else svgp_predict_reference_order
    mu2, v2 = fn(p2, h, kernel=kernel)
    return mu2, v2, h


def exact_gp_prior(x, constant, raw_lengthscale, raw_outputscale, kernel="rbf"):
    """``ExactGPModel.forward`` (GPModel.py:10-13): ConstantMean + ScaleKernel(RBF, no ARD).
    x [n, D] -> (mean [n], covar [n, n])."""
    ell = GO.softplus(raw_lengthscale).reshape(())
    os = GO.softplus(raw_outputscale).reshape(())
    mean = constant.reshape(()).expand(x.shape[-2])
    covar = scale_direct(x, x, ell, os, kernel)
    return mean, covar


def exact_gp_posterior(train_x, train_y, test_x, constant, raw_lengthscale, raw_outputscale, raw_noise, kernel="rbf"):
    """gpytorch ``ExactGP.__call__`` in eval mode: condition on (train_x, train_y) through the
    Cholesky of K + noise I.  Returns (mean [n*], covar [n*, n*])."""
    ell = GO.softplus(raw_lengthscale).reshape(())
    os = GO.softplus(raw_outputscale).reshape(())
    noise = GO.softplus(raw_noise).reshape(()) + GO.NOISE_LOWER
    c = constant.reshape(())
    Ktt = scale_direct(train_x, train_x, ell, os, kernel) + noise * torch.eye(train_x.shape[0], dtype=train_x.dtype)
    Kst = scale_direct(test_x, train_x, ell, os, kernel)
    Kss = scale_direct(test_x, test_x, ell, os, kernel)
    Lc = torch.linalg.cholesky(Ktt)
    alpha = torch.cholesky_solve((train_y - c).unsqueeze(-1), Lc).squeeze(-1)
    V = torch.linalg.solve_triangular(Lc, Kst.t(), upper=False)
    return c + Kst @ alpha, Kss - V.t() @ V
