"""Rational quadratic kernel (gpytorch RQKernel, learnable alpha) for the float64 oracle.

matern_oracle.py's kernel-dependent functions, restated with a further kernel "rq".  Every function takes the same
``kernel`` argument as its matern_oracle namesake and computes what that one computes for "rbf" and the Matern
kernels; for "rq" the shape parameter comes as ``alpha`` (kernel evaluations) or as the parameter ``raw_alpha``
(``p["raw_alpha"]`` of a layer, an argument of the exact-GP functions), alpha = softplus(raw_alpha).

  x~ = x / ell,  d2 = clamp_min(sq_dist(x~, z~), 0)   (gpytorch square_dist=True: no 1e-30 clamp)
  u  = d2 / (2 alpha),  k = os (1 + u)^-alpha
  g  = -2 os df/d(d2) = k / (1 + u)                    (the weight of every distance gradient: W = kbar o g)
  ka = dk/dalpha = k (u / (1 + u) - log1p(u))
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch

from . import gp_oracle as GO
from . import matern_oracle as MO

KERNELS = MO.KERNELS + ("rq",)


def _check_kernel(kernel, alpha):
    if kernel not in KERNELS:
        raise ValueError(f"unknown kernel {kernel!r}")
    if (kernel == "rq") != (alpha is not None):
        raise ValueError("alpha is given for kernel 'rq' and only for it")


def rq_from_d2(d2, os, alpha):
    """(k, g, ka) of the rational quadratic kernel from the squared distances."""
    u = d2 / (2.0 * alpha)
    lp = torch.log1p(u)
    k = os * torch.exp(-alpha * lp)
    q = 1.0 / (1.0 + u)
    return k, k * q, k * (u * q - lp)


def _d2_direct(x1, x2, ell):
    diff = (x1.unsqueeze(-2) - x2.unsqueeze(-3)) / ell
    return diff.pow(2).sum(-1)


def scale_direct(x1, x2, ell, os, kernel="rbf", alpha=None):
    _check_kernel(kernel, alpha)
    if kernel != "rq":
        return MO.scale_direct(x1, x2, ell, os, kernel)
    return rq_from_d2(_d2_direct(x1, x2, ell), os, alpha)[0]


def scale_reference_order(x1, x2, ell, os, kernel="rbf", alpha=None):
    """gpytorch order; RQKernel.forward: divide by the lengthscale, sq_dist (clamp_min 0), div(2 alpha), add(1),
    pow(-alpha)."""
    _check_kernel(kernel, alpha)
    if kernel != "rq":
        return MO.scale_reference_order(x1, x2, ell, os, kernel)
    d2 = GO.sq_dist_reference_order(x1 / ell, x2 / ell)
    return os * d2.div(alpha * 2).add(1).pow(-alpha)


def scale_direct_kga(x1, x2, ell, os, kernel="rbf", alpha=None):
    """(K, G, KA) by direct differences: G = -2 os df/d(d2), KA = dK/dalpha (None but for "rq")."""
    _check_kernel(kernel, alpha)
    if kernel != "rq":
        return MO.scale_direct_kg(x1, x2, ell, os, kernel) + (None,)
    return rq_from_d2(_d2_direct(x1, x2, ell), os, alpha)


def scale_direct_kg(x1, x2, ell, os, kernel="rbf", alpha=None):
    return scale_direct_kga(x1, x2, ell, os, kernel, alpha)[:2]


def _alpha(p, kernel):
    return GO.softplus(p["raw_alpha"]).reshape(()) if kernel == "rq" else None


def svgp_predict_reference_order(p: Dict[str, torch.Tensor], x: torch.Tensor, linalg_dtype=torch.float64,
                                 kernel="rbf") -> Tuple[torch.Tensor, torch.Tensor]:
    """matern_oracle.svgp_predict_reference_order (gpytorch op order), p["raw_alpha"] [1] for "rq"."""
    Z = p["inducing_points"]
    B, L, D = x.shape
    M = Z.shape[0]
    ell = GO.softplus(p["raw_lengthscale"])
    os = GO.softplus(p["raw_outputscale"])
    full = torch.cat([Z.unsqueeze(0).expand(B, M, D), x], dim=-2)
    full_mean = (full @ p["weights"]).squeeze(-1) + p["bias"]
    full_covar = scale_reference_order(full, full, ell, os, kernel, _alpha(p, kernel))
    Kzz = full_covar[..., :M, :M] + GO.JITTER * torch.eye(M, dtype=x.dtype)
    Kzx = full_covar[..., :M, M:]
    Lc = torch.linalg.cholesky(Kzz.to(linalg_dtype))
    A = torch.linalg.solve_triangular(Lc, Kzx.to(linalg_dtype), upper=False).to(x.dtype)
    m, s = p["variational_mean"], p["variational_stddev"]
    mean = (A.transpose(-1, -2) @ m.unsqueeze(-1)).squeeze(-1) + full_mean[..., M:]
    var = os * torch.ones(B, L, dtype=x.dtype) + GO.JITTER + ((s.pow(2) - 1.0).unsqueeze(-1) * A.pow(2)).sum(-2)
    return mean, var.clamp_min(GO.MIN_VARIANCE)


def svgp_predict_closed_form(p: Dict[str, torch.Tensor], x: torch.Tensor,
                             kernel="rbf") -> Tuple[torch.Tensor, torch.Tensor]:
    """matern_oracle.svgp_predict_closed_form (one M x M Cholesky, direct distances), p["raw_alpha"] for "rq"."""
    Z = p["inducing_points"]
    B, L, D = x.shape
    M = Z.shape[0]
    ell = GO.softplus(p["raw_lengthscale"]).reshape(D)
    os = GO.softplus(p["raw_outputscale"])
    a = _alpha(p, kernel)
    Kzz = scale_direct(Z, Z, ell, os, kernel, a) + GO.JITTER * torch.eye(M, dtype=x.dtype)
    Lc = torch.linalg.cholesky(Kzz)
    X = x.reshape(B * L, D)
    A = torch.linalg.solve_triangular(Lc, scale_direct(Z, X, ell, os, kernel, a), upper=False)
    m, s = p["variational_mean"], p["variational_stddev"]
    mean = A.t() @ m + (X @ p["weights"]).squeeze(-1) + p["bias"]
    var = (os + GO.JITTER + ((s.pow(2) - 1.0).unsqueeze(-1) * A.pow(2)).sum(0)).clamp_min(GO.MIN_VARIANCE)
    return mean.reshape(B, L), var.reshape(B, L)


def mll_error(p, x, y, num_data, reference_order=True, kernel="rbf") -> torch.Tensor:
    fn = svgp_predict_reference_order if reference_order else svgp_predict_closed_form
    mean, var = fn(p, x, kernel=kernel)
    e = GO.elbo_per_window(mean, var, y, GO.noise_variance(p), GO.kl_meanfield(p), num_data)
    return -e.mean()


def svgp_backward_kernel_order(p, x, g_mean, g_var, g_kl=0.0, kernel="rbf"):
    """matern_oracle.svgp_backward_kernel_order (the CUDA backward's op order) -> (SvgpGrads, d raw_alpha | None).
    RQ: d alpha = sum Kbar o KA (points) + sum sym(Kbar_zz) o KA_zz (inducing pairs)."""
    if kernel != "rq":
        return MO.svgp_backward_kernel_order(p, x, g_mean, g_var, g_kl, kernel), None
    Z = p["inducing_points"]
    B, L_, D = x.shape
    M = Z.shape[0]
    N = B * L_
    X = x.reshape(N, D)
    gm, gv = g_mean.reshape(N), g_var.reshape(N)
    ell = GO.softplus(p["raw_lengthscale"]).reshape(D)
    os = GO.softplus(p["raw_outputscale"])
    a = _alpha(p, kernel)
    m, s = p["variational_mean"], p["variational_stddev"]
    w = p["weights"].reshape(D)
    cvec = s.pow(2) - 1.0

    Kzz0, Gzz, KAzz = scale_direct_kga(Z, Z, ell, os, kernel, a)
    Lc = torch.linalg.cholesky(Kzz0 + GO.JITTER * torch.eye(M, dtype=X.dtype))
    Linv = torch.linalg.solve_triangular(Lc, torch.eye(M, dtype=X.dtype), upper=False)
    K, G, KA = scale_direct_kga(X, Z, ell, os, kernel, a)
    A = K @ Linv.t()
    var_raw = os + GO.JITTER + (A.pow(2) * cvec).sum(-1)
    gv = torch.where(var_raw < GO.MIN_VARIANCE, torch.zeros_like(gv), gv)

    Kbar = (gm[:, None] * m[None, :] + 2.0 * gv[:, None] * cvec[None, :] * A) @ Linv
    W = Kbar * G
    r, csum = W.sum(1), W.sum(0)
    Xt, Zt = X / ell, Z / ell
    dx = (W @ Zt - r[:, None] * Xt) / ell + gm[:, None] * w[None, :]
    WX = W.t() @ Xt
    dZ = (WX - csum[:, None] * Zt) / ell
    dell = ((r[:, None] * Xt.pow(2)).sum(0) - 2.0 * (Zt * WX).sum(0) + (csum[:, None] * Zt.pow(2)).sum(0)) / ell
    dos = (Kbar * K).sum() / os + gv.sum()
    da = (Kbar * KA).sum()
    u = (gm[:, None] * A).sum(0)
    S = A.t() @ (gv[:, None] * A)

    E = m[:, None] * u[None, :] + 2.0 * cvec[:, None] * S
    Lbar = -torch.tril(Linv.t() @ E)
    P = Lc.t() @ Lbar
    Phi = torch.tril(P) - 0.5 * torch.diag(torch.diagonal(P))
    Kb = Linv.t() @ Phi @ Linv
    Kb = 0.5 * (Kb + Kb.t())
    Wzz = Kb * Gzz
    dZ = dZ + 2.0 * (Wzz @ Zt - Wzz.sum(1)[:, None] * Zt) / ell
    diff2 = (Zt.unsqueeze(1) - Zt.unsqueeze(0)).pow(2)
    dell = dell + (Wzz.unsqueeze(-1) * diff2).sum((0, 1)) / ell
    dos = dos + (Kb * Kzz0).sum() / os
    da = da + (Kb * KAzz).sum()

    sig = torch.sigmoid
    grads = GO.SvgpGrads(
        dx=dx.reshape(B, L_, D),
        inducing_points=dZ,
        raw_lengthscale=(dell * sig(p["raw_lengthscale"]).reshape(D)).reshape(1, D),
        raw_outputscale=dos * sig(p["raw_outputscale"]),
        variational_mean=u + g_kl * m,
        variational_stddev=2.0 * s * torch.diagonal(S) + g_kl * (s - 1.0 / s),
        weights=(gm[:, None] * X).sum(0).reshape(D, 1),
        bias=gm.sum().reshape(1),
    )
    return grads, (da * sig(p["raw_alpha"])).reshape(p["raw_alpha"].shape)


def hidden_layer_predict(p1, x, closed_form=True, kernel="rbf"):
    """Layer with output_dims=H (H independent whitened SVGPs; "rq": p1["raw_alpha"] [H, 1]).  -> mean, var
    [B, L, H]."""
    H = p1["inducing_points"].shape[0]
    fn = svgp_predict_closed_form if closed_form else svgp_predict_reference_order
    means, vars_ = [], []
    for h in range(H):
        ph = {k: p1[k][h] for k in ("inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean",
                                    "variational_stddev")}
        ph["weights"], ph["bias"] = p1["weights"], p1["bias"]
        if kernel == "rq":
            ph["raw_alpha"] = p1["raw_alpha"][h]
        mu, v = fn(ph, x, kernel=kernel)
        means.append(mu)
        vars_.append(v)
    return torch.stack(means, -1), torch.stack(vars_, -1)


def deepgp2_predict(p1, p2, x, eps, closed_form=True, kernel="rbf"):
    """matern_oracle.deepgp2_predict.  -> (mean, var, hidden_sample)."""
    mu1, v1 = hidden_layer_predict(p1, x, closed_form, kernel=kernel)
    h = GO.rsample(mu1, v1, eps)
    fn = svgp_predict_closed_form if closed_form else svgp_predict_reference_order
    mu2, v2 = fn(p2, h, kernel=kernel)
    return mu2, v2, h


def exact_gp_prior(x, constant, raw_lengthscale, raw_outputscale, kernel="rbf", raw_alpha=None):
    """ConstantMean + ScaleKernel(kernel, no ARD).  x [n, D] -> (mean [n], covar [n, n])."""
    ell = GO.softplus(raw_lengthscale).reshape(())
    os = GO.softplus(raw_outputscale).reshape(())
    a = None if raw_alpha is None else GO.softplus(raw_alpha).reshape(())
    return constant.reshape(()).expand(x.shape[-2]), scale_direct(x, x, ell, os, kernel, a)


def exact_gp_posterior(train_x, train_y, test_x, constant, raw_lengthscale, raw_outputscale, raw_noise, kernel="rbf",
                       raw_alpha=None):
    """gpytorch ExactGP.__call__ in eval mode.  -> (mean [n*], covar [n*, n*])."""
    ell = GO.softplus(raw_lengthscale).reshape(())
    os = GO.softplus(raw_outputscale).reshape(())
    a = None if raw_alpha is None else GO.softplus(raw_alpha).reshape(())
    noise = GO.softplus(raw_noise).reshape(()) + GO.NOISE_LOWER
    c = constant.reshape(())
    Ktt = scale_direct(train_x, train_x, ell, os, kernel, a) + noise * torch.eye(train_x.shape[0], dtype=train_x.dtype)
    Kst = scale_direct(test_x, train_x, ell, os, kernel, a)
    Kss = scale_direct(test_x, test_x, ell, os, kernel, a)
    Lc = torch.linalg.cholesky(Ktt)
    alpha = torch.cholesky_solve((train_y - c).unsqueeze(-1), Lc).squeeze(-1)
    V = torch.linalg.solve_triangular(Lc, Kst.t(), upper=False)
    return c + Kst @ alpha, Kss - V.t() @ V
