"""The closed form of the Cholesky backward that the M x M stage backward relies on, checked in float64 on the CPU.

mm_backward_kernel does not run the chain  Lbar = -tril(Linv^T X), Phi(L^T Lbar), Kbar = Linv^T Phi Linv, sym(Kbar)
(X = m u^T + 2 diag(c) S).  It computes

    sym(Kbar) = Linv^T P Linv,   P_ik = -1/2 (m_hi u_lo + 2 c_hi S_hi,lo),   hi = max(i, k), lo = min(i, k),

with P built from the row-major S that stage_grad_reduce_kernel makes exactly symmetric by writing each lower
element to both (i, j) and (j, i).  These tests pin that algebra against the chain of the fp64 oracle and against
torch autograd through cholesky + inv, including identity padding, an ill-conditioned Kzz and an S whose two
triangles differ by rounding.
"""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import gp_oracle as O  # noqa: E402

DT = torch.float64


def lower_mirrored(S):
    """What stage_grad_reduce_kernel leaves: the lower element of every pair on both sides."""
    return torch.tril(S) + torch.tril(S, -1).t()


def closed_form(Linv, m, u, c, S):
    """sym(Kbar) as the kernel forms it: P from the row-major read of the (lower-mirrored) S, then two products."""
    Ssym = lower_mirrored(S)
    n = S.shape[0]
    idx = torch.arange(n)
    upper = idx[None, :] >= idx[:, None]          # k >= i: hi = k, lo = i
    P = torch.where(upper, -(c[None, :] * Ssym + 0.5 * m[None, :] * u[:, None]),
                    -(c[:, None] * Ssym + 0.5 * m[:, None] * u[None, :]))
    return Linv.t() @ (P @ Linv), P


def oracle_chain(Lc, Linv, m, u, c, S):
    """The Kbar chain of oracle.gp_oracle.svgp_backward_kernel_order, operation for operation."""
    E = m[:, None] * u[None, :] + 2.0 * c[:, None] * S
    Gbar = Linv.t() @ E
    Lbar = -torch.tril(Gbar)
    P = Lc.t() @ Lbar
    Phi = torch.tril(P)
    Phi = Phi - 0.5 * torch.diag(torch.diagonal(P))
    Kb = Linv.t() @ Phi @ Linv
    return 0.5 * (Kb + Kb.t())


def autograd_kbar(Kzz, Knz, gm, gv, m, c):
    """d/dKzz of  sum_n gm_n m.a_n + sum_n gv_n c.(a_n o a_n),  a_n = inv(cholesky(Kzz)) k_n  (symmetrised)."""
    K = Kzz.clone().requires_grad_(True)
    Linv = torch.linalg.inv(torch.linalg.cholesky(K))
    A = Knz @ Linv.t()
    loss = (gm[:, None] * A * m[None, :]).sum() + (gv[:, None] * c[None, :] * A.pow(2)).sum()
    (g,) = torch.autograd.grad(loss, K)
    return 0.5 * (g + g.t())


def problem(M, D, N, seed, near_duplicates=False):
    gen = torch.Generator().manual_seed(seed)
    p = O.init_params_exercise(D, M, seed)
    Z = p["inducing_points"].to(DT)
    if near_duplicates:
        Z[1] = Z[0] + 1e-3 * torch.randn(D, generator=gen, dtype=DT)
        Z[3] = Z[2] + 1e-3 * torch.randn(D, generator=gen, dtype=DT)
    ell = O.softplus(p["raw_lengthscale"].to(DT)).reshape(D)
    os_ = O.softplus(p["raw_outputscale"].to(DT))
    Kzz = O.rbf_scale_direct(Z, Z, ell, os_) + O.JITTER * torch.eye(M, dtype=DT)
    X = torch.randn(N, D, generator=gen, dtype=DT)
    Knz = O.rbf_scale_direct(X, Z, ell, os_)
    gm = torch.randn(N, generator=gen, dtype=DT)
    gv = torch.randn(N, generator=gen, dtype=DT)
    m = torch.randn(M, generator=gen, dtype=DT)
    c = p["variational_stddev"].to(DT).pow(2) - 1.0 + 0.3 * torch.randn(M, generator=gen, dtype=DT)
    Lc = torch.linalg.cholesky(Kzz)
    Linv = torch.linalg.solve_triangular(Lc, torch.eye(M, dtype=DT), upper=False)
    A = Knz @ Linv.t()
    u = (gm[:, None] * A).sum(0)
    S = A.t() @ (gv[:, None] * A)
    return dict(Kzz=Kzz, Knz=Knz, gm=gm, gv=gv, m=m, c=c, Lc=Lc, Linv=Linv, u=u, S=S)


def rel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


@pytest.mark.parametrize("M", [32, 64, 200])
def test_closed_form_matches_oracle_chain_and_autograd(M):
    pb = problem(M, 16, 3 * M, seed=M)
    got, _ = closed_form(pb["Linv"], pb["m"], pb["u"], pb["c"], pb["S"])
    assert rel(got, oracle_chain(pb["Lc"], pb["Linv"], pb["m"], pb["u"], pb["c"], pb["S"])) < 1e-12
    assert rel(got, autograd_kbar(pb["Kzz"], pb["Knz"], pb["gm"], pb["gv"], pb["m"], pb["c"])) < 1e-10


def test_closed_form_ill_conditioned_kzz():
    M = 64
    pb = problem(M, 8, 4 * M, seed=7, near_duplicates=True)
    assert torch.linalg.cond(pb["Kzz"]).item() >= 1e5
    got, _ = closed_form(pb["Linv"], pb["m"], pb["u"], pb["c"], pb["S"])
    assert rel(got, oracle_chain(pb["Lc"], pb["Linv"], pb["m"], pb["u"], pb["c"], pb["S"])) < 1e-9
    assert rel(got, autograd_kbar(pb["Kzz"], pb["Knz"], pb["gm"], pb["gv"], pb["m"], pb["c"])) < 1e-7


def test_closed_form_identity_padding():
    """MP > M: Kzz, L and Linv padded with the identity, m, u, c, S with zeros - P is 0 in the padding and the
    M x M block of sym(Kbar) is that of the unpadded problem."""
    M, MP = 40, 64
    pb = problem(M, 16, 3 * M, seed=3)
    pad = lambda v: torch.cat([v, torch.zeros(MP - M, dtype=DT)])
    Sp = torch.zeros(MP, MP, dtype=DT)
    Sp[:M, :M] = pb["S"]
    Linvp = torch.eye(MP, dtype=DT)
    Linvp[:M, :M] = pb["Linv"]
    gotp, P = closed_form(Linvp, pad(pb["m"]), pad(pb["u"]), pad(pb["c"]), Sp)
    assert torch.all(P[M:, :] == 0) and torch.all(P[:, M:] == 0)
    assert torch.all(gotp[M:, :] == 0) and torch.all(gotp[:, M:] == 0)
    got, _ = closed_form(pb["Linv"], pb["m"], pb["u"], pb["c"], pb["S"])
    assert rel(gotp[:M, :M], got) < 1e-14
    assert rel(gotp[:M, :M], oracle_chain(pb["Lc"], pb["Linv"], pb["m"], pb["u"], pb["c"], pb["S"])) < 1e-12


def test_closed_form_asymmetric_rounding_S():
    """The Gram computes S_ij and S_ji separately, so its two triangles differ in the last bits.  The chain reads
    only the lower triangle of X = m u^T + 2 diag(c) S, so mirroring the lower elements (as the stage gradient
    reduction does) gives the chain's result for the unmirrored S, and the row-major read of the mirrored S is
    exactly S(hi, lo)."""
    M = 96
    pb = problem(M, 16, 3 * M, seed=11)
    A = (pb["Knz"] @ pb["Linv"].t()).float()
    gv = pb["gv"].float()
    S32 = torch.zeros(M, M, dtype=torch.float32)
    for i in range(M):   # each element summed on its own, in a different order for (i, j) and (j, i)
        S32[i] = (A[:, i:i + 1] * (gv[:, None] * A)).sum(0)
    S = S32.to(DT)
    assert not torch.equal(S, S.t())
    Ssym = lower_mirrored(S)
    assert torch.equal(Ssym, Ssym.t())
    got, P = closed_form(pb["Linv"], pb["m"], pb["u"], pb["c"], S)
    assert torch.equal(P, P.t())
    assert rel(got, oracle_chain(pb["Lc"], pb["Linv"], pb["m"], pb["u"], pb["c"], S)) < 1e-12
    # the upper triangle of S does not enter: the chain fed the mirrored S gives the same result
    assert rel(got, oracle_chain(pb["Lc"], pb["Linv"], pb["m"], pb["u"], pb["c"], Ssym)) < 1e-12
