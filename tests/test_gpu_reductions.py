"""The backward N-reductions of the tensor-core path (Mp >= 128) against fp64 torch on the operands they reduce.

One backward call leaves the saved A = k Linv^T, W and the folded upstream gradients g_mu, g_var in its workspace;
its stage gradient must hold u = A^T g_mu, the column sums of W, S = A^T diag(g_var) A (full and symmetric) and
W^T X, whatever the Gram / W^T X tiling and split layout.  Two identical calls must give bit-identical results.
"""
import pytest
import torch

from oracle import gp_oracle as O

pytestmark = pytest.mark.gpu

# (N, D, M): Mp = 128 / 256 / 512 / 1024, Dp = 16 / 64 / 128; N ragged (not a multiple of 32 or 128), below the split
# count of the one-wave launch (N < 148), and large enough for many splits
CASES = [
    (37, 16, 100), (4133, 64, 100), (20011, 128, 128),
    (50, 64, 256), (9001, 16, 256), (55296, 64, 256), (12345, 128, 256),
    (131, 128, 400), (6007, 64, 512),
    (97, 16, 1000), (5003, 64, 1024), (3001, 128, 1024),
]


def _padded_m(M):
    return 128 if M <= 128 else (M + 255) // 256 * 256


def _padded_d(D):
    return 16 if D <= 16 else 32 if D <= 32 else 64 if D <= 64 else 128


def _backward(ops, cuda, N, D, M, seed):
    p = {k: v.to(cuda) for k, v in O.init_params_exercise(D, M, seed=seed).items()}
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(N, D, generator=g).to(cuda)
    gm, gv, gs = (torch.randn(N, generator=g).to(cuda) for _ in range(3))
    mean, var, sample, kl, info, ws = ops.svgp_forward_raw(
        x, p["inducing_points"], p["raw_lengthscale"].reshape(-1), p["raw_outputscale"].reshape(1),
        p["variational_mean"], p["variational_stddev"], p["weights"].reshape(-1), p["bias"], 7, 3, 0, True, True)
    _, sgrad = ops.point_backward_raw(x, M, gm, gv, gs, var, 7, 3, 0, ws, need_dx=False)
    torch.cuda.synchronize()
    return x, ws, sgrad


@pytest.mark.parametrize("N,D,M", CASES)
def test_stage_gradient_reductions(cuda, N, D, M):
    from fine_grained_gaussian_process_forcasting_b200 import ops
    x, ws, sgrad = _backward(ops, cuda, N, D, M, seed=31)
    Mp, Dp = _padded_m(M), _padded_d(D)
    A = ops.debug_fetch(3, N, D, M, ws).double()
    W = ops.debug_fetch(5, N, D, M, ws).double()
    g_mu, g_var = ops.debug_fetch(6, N, D, M, ws).double()[:, :N]
    xp = torch.zeros(N, Dp, dtype=torch.float64, device=cuda)
    xp[:, :D] = x.double()
    vec_len = Mp + 2 * Dp + 4
    sg = sgrad.double()
    u = sg[:Mp]
    colsum = sg[Mp:2 * Mp]
    S = sg[Mp + vec_len:Mp + vec_len + Mp * Mp].reshape(Mp, Mp)
    WX = sg[Mp + vec_len + Mp * Mp:].reshape(Mp, Dp)

    def check(name, got, want, scale):
        # error against the sum of absolute terms: 3xTF32 products and fp32 partial sums, independent of cancellation
        err = ((got - want).abs() / (scale + 1e-30)).max().item()
        assert err < 1e-5, f"{name}: {err:.2e}"

    check("u", u, A.T @ g_mu, A.abs().T @ g_mu.abs())
    check("colsum", colsum, W.sum(0), W.abs().sum(0))
    check("S", S, A.T @ (g_var[:, None] * A), A.abs().T @ (g_var.abs()[:, None] * A.abs()))
    assert torch.equal(S, S.T) or (S - S.T).abs().max() <= 1e-5 * S.abs().max()
    check("WX", WX, W.T @ xp, W.abs().T @ xp.abs())


@pytest.mark.parametrize("N,D,M", [(55296, 64, 256), (6007, 64, 512), (131, 16, 1000)])
def test_backward_bit_identical(cuda, N, D, M):
    from fine_grained_gaussian_process_forcasting_b200 import ops
    _, _, s1 = _backward(ops, cuda, N, D, M, seed=41)
    _, _, s2 = _backward(ops, cuda, N, D, M, seed=41)
    assert torch.equal(s1, s2)


def test_parameter_gradients_bit_identical(cuda):
    from fine_grained_gaussian_process_forcasting_b200 import ops
    B, L, D, M = 64, 24, 64, 256
    p32 = O.init_params_exercise(D, M, seed=51)
    x32, _, gm32, gv32 = O.make_inputs(B, L, D, seed=52)
    grads = []
    for _ in range(2):
        pd = {k: v.to(cuda).requires_grad_(True) for k, v in p32.items()}
        xd = x32.to(cuda).requires_grad_(True)
        mean, var, _, kl, _ = ops.svgp_predict(xd, pd["inducing_points"], pd["raw_lengthscale"], pd["raw_outputscale"],
                                               pd["variational_mean"], pd["variational_stddev"], pd["weights"],
                                               pd["bias"], seed=5, offset=0, stream_id=0, want_sample=True)
        ((gm32.to(cuda) * mean).sum() + (gv32.to(cuda) * var).sum() + 0.3 * kl).backward()
        torch.cuda.synchronize()
        grads.append({k: v.grad.clone() for k, v in pd.items() if v.grad is not None})
    assert "inducing_points" in grads[0] and "variational_mean" in grads[0]
    for k in grads[0]:
        assert torch.equal(grads[0][k], grads[1][k]), k
