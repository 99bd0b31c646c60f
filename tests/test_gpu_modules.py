"""GPU tests at the module boundary (the calls the reference's forecast_denoising.py / denoise_model_2.py make),
against the oracle and the committed golden fixtures, plus size-independent properties at BASELINE sizes."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import gp_oracle as O

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def rel(a, b):
    a = torch.as_tensor(a).detach().double().cpu()
    b = torch.as_tensor(b).detach().double().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-300)).item()


def load_params(model, p):
    hl = model.hidden_layer
    with torch.no_grad():
        hl.variational_strategy.inducing_points.copy_(p["inducing_points"])
        hl.covar_module.base_kernel.raw_lengthscale.copy_(p["raw_lengthscale"].reshape(1, -1))
        hl.covar_module.raw_outputscale.copy_(p["raw_outputscale"].reshape(()))
        hl.variational_strategy._variational_distribution.variational_mean.copy_(p["variational_mean"])
        hl.variational_strategy._variational_distribution._variational_stddev.copy_(p["variational_stddev"])
        hl.mean_module.weights.copy_(p["weights"].reshape(-1, 1))
        hl.mean_module.bias.copy_(p["bias"].reshape(1))
        if "raw_noise" in p:
            model.likelihood.noise_covar.raw_noise.copy_(p["raw_noise"].reshape(1))
        hl.variational_strategy.variational_params_initialized.fill_(1)


def test_predict_and_mll_protocol_like_the_reference(cuda):
    """denoise_model_2.add_gp_noise + forecast_denoising.py:87-89, verbatim call sequence."""
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat as gpytorch_like
    B, L, D, M = 16, 24, 32, 64
    p = O.init_params_exercise(D, M, 3)
    x, y, _, _ = O.make_inputs(B, L, D, 4)
    with gpytorch_like.num_likelihood_samples(1):
        deep_gp = DeepGPp(D, 1234, num_inducing=M).to(cuda)
        load_params(deep_gp, p)
        proj_up = torch.nn.Linear(1, D).to(cuda)
        xd = x.to(cuda).requires_grad_(True)
        eps_gp, dist = deep_gp.predict(xd)                       # denoise_model_2.py:36
        assert eps_gp.shape == (1, B, L) and dist.mean.shape == (1, B, L) and dist.event_shape == (L,)
        x_noisy = xd + proj_up(eps_gp.permute(1, 2, 0))          # :37-38
        y_true = y.to(cuda).unsqueeze(-1)                        # [B, L, 1]
        mll = gpytorch_like.DeepApproximateMLL(
            gpytorch_like.VariationalELBO(deep_gp.likelihood, deep_gp, D))
        mll_error = -mll(dist, y_true.permute(2, 0, 1)).mean()   # forecast_denoising.py:89
        loss = x_noisy.pow(2).mean() + 0.005 * mll_error
        loss.backward()
    p64 = O.clone_params(p, torch.float64, requires_grad=True)
    x64 = x.double().requires_grad_(True)
    mo, vo = O.svgp_predict_closed_form(p64, x64)
    w64, b64 = proj_up.weight.detach().double().cpu(), proj_up.bias.detach().double().cpu()
    xn = x64 + mo.unsqueeze(-1) * w64.reshape(1, 1, D) + b64
    eo = O.elbo_per_window(mo, vo, y.double(), O.noise_variance(p64), O.kl_meanfield(p64), float(D))
    lo = xn.pow(2).mean() + 0.005 * (-eo.mean())
    lo.backward()
    assert rel(eps_gp[0], mo) < 1e-5 and rel(dist.variance[0], vo) < 1e-5
    assert abs(mll_error.item() + eo.mean().item()) < 1e-5 * abs(eo.mean().item())
    assert rel(xd.grad, x64.grad) < 2e-4
    hl = deep_gp.hidden_layer
    assert rel(hl.variational_strategy.inducing_points.grad, p64["inducing_points"].grad) < 2e-4
    assert rel(hl.covar_module.base_kernel.raw_lengthscale.grad, p64["raw_lengthscale"].grad) < 2e-4
    assert rel(hl.variational_strategy._variational_distribution._variational_stddev.grad,
               p64["variational_stddev"].grad) < 2e-4
    assert rel(deep_gp.likelihood.noise_covar.raw_noise.grad, p64["raw_noise"].grad) < 2e-4
    # default sample count outside the context is 10 (gpytorch default)
    _, d10 = deep_gp.predict(x.to(cuda))
    assert d10.mean.shape == (10, B, L)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "svgp_*.npz"))))
def test_cuda_matches_golden_fixtures(cuda, path):
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    g = np.load(path)
    p = {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("p_")}
    x = torch.from_numpy(g["x"])
    B, L, D = x.shape
    M = p["inducing_points"].shape[0]
    seed, off, stream = (int(v) for v in g["philox_seed_offset_stream"])
    with gpcompat.num_likelihood_samples(1):
        model = DeepGPp(D, 0, num_inducing=M).to(cuda)
        load_params(model, p)
        model.hidden_layer.set_rng(seed, off, stream)
        xd = x.to(cuda).requires_grad_(True)
        out = model.blur(xd, torch.from_numpy(g["y"]).to(cuda), num_data=D)
        loss = -out.elbo.mean() + (torch.from_numpy(g["g_mean"]).to(cuda) * out.mean[0]).sum() + \
            (torch.from_numpy(g["g_sample"]).to(cuda) * out.sample[0]).sum()
        loss.backward()
    assert rel(out.mean[0], g["mean"]) < 1e-5 and rel(out.variance[0], g["var"]) < 1e-5
    assert rel(out.elbo[0], g["elbo"]) < 1e-5 and rel(out.kl, g["kl"]) < 1e-5
    assert rel(out.sample[0], g["sample"]) < 1e-5
    # the scalar is a sum of cancelling fp32 terms: compare against the magnitude of what was summed
    scale = float(np.abs(g["g_mean"] * g["mean"]).sum() + np.abs(g["g_sample"] * g["sample"]).sum() + abs(g["elbo"]).mean())
    assert abs(loss.item() - float(g["loss"])) < 1e-5 * scale
    assert rel(xd.grad, g["dx"]) < 2e-4
    hl = model.hidden_layer
    got = {"inducing_points": hl.variational_strategy.inducing_points.grad,
           "raw_lengthscale": hl.covar_module.base_kernel.raw_lengthscale.grad,
           "raw_outputscale": hl.covar_module.raw_outputscale.grad,
           "variational_mean": hl.variational_strategy._variational_distribution.variational_mean.grad,
           "variational_stddev": hl.variational_strategy._variational_distribution._variational_stddev.grad,
           "weights": hl.mean_module.weights.grad, "bias": hl.mean_module.bias.grad,
           "raw_noise": model.likelihood.noise_covar.raw_noise.grad}
    for k, v in got.items():
        assert rel(v.reshape(-1), g["d_" + k].reshape(-1)) < 2e-4, k


def test_eval_mode_and_no_grad(cuda):
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    D, M = 16, 32
    p = O.init_params_exercise(D, M, 3)
    x, _, _, _ = O.make_inputs(5, 24, D, 4)
    with gpcompat.num_likelihood_samples(1):
        m = DeepGPp(D, 1, num_inducing=M).to(cuda).eval()
        load_params(m, p)
        with torch.no_grad():
            mean, dist = m.predict(x.to(cuda))
    mo, vo = O.svgp_predict_closed_form(O.clone_params(p, torch.float64), x.double())
    assert rel(mean[0], mo) < 1e-5 and rel(dist.variance[0], vo) < 1e-5 and not mean.requires_grad


def test_two_layer_deepgp_matches_oracle(cuda):
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGP2
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    B, L, D, H, M = 6, 24, 16, 4, 32
    p1 = O.init_params_hidden_layer(D, H, M, 5)
    p2 = O.init_params_exercise(H, M, 6)
    x, y, _, _ = O.make_inputs(B, L, D, 7)
    with gpcompat.num_likelihood_samples(1):
        net = DeepGP2(D, 11, hidden_dims=H, num_inducing=M).to(cuda)
        l1, l2 = net.hidden_layer, net.last_layer
        with torch.no_grad():
            l1.variational_strategy.inducing_points.copy_(p1["inducing_points"])
            l1.covar_module.base_kernel.raw_lengthscale.copy_(p1["raw_lengthscale"])
            l1.covar_module.raw_outputscale.copy_(p1["raw_outputscale"])
            l1.variational_strategy._variational_distribution.variational_mean.copy_(p1["variational_mean"])
            l1.variational_strategy._variational_distribution._variational_stddev.copy_(p1["variational_stddev"])
            l1.mean_module.weights.copy_(p1["weights"]); l1.mean_module.bias.copy_(p1["bias"])
            l1.variational_strategy.variational_params_initialized.fill_(1)
            l2.variational_strategy.inducing_points.copy_(p2["inducing_points"])
            l2.covar_module.base_kernel.raw_lengthscale.copy_(p2["raw_lengthscale"])
            l2.variational_strategy._variational_distribution.variational_mean.copy_(p2["variational_mean"])
            l2.variational_strategy._variational_distribution._variational_stddev.copy_(p2["variational_stddev"])
            l2.mean_module.weights.copy_(p2["weights"]); l2.mean_module.bias.copy_(p2["bias"])
            l2.variational_strategy.variational_params_initialized.fill_(1)
        l1.set_rng(77, 0, stream=1)
        xd = x.to(cuda).requires_grad_(True)
        mean, dist = net.predict(xd)
        mll = gpcompat.DeepApproximateMLL(gpcompat.VariationalELBO(net.likelihood, net, D))
        loss = -mll(dist, y.to(cuda).unsqueeze(0)).mean()
        loss.backward()
    # oracle with the same Philox draws: layer 1 output h uses counters offset = h * N + n, stream 1
    N = B * L
    eps = torch.stack([torch.from_numpy(O.philox_normal(77, h * N, N, 1)).reshape(B, L) for h in range(H)], -1).double()
    p1_64 = O.clone_params(p1, torch.float64, requires_grad=True)
    p2_64 = O.clone_params(p2, torch.float64, requires_grad=True)
    x64 = x.double().requires_grad_(True)
    mo, vo, ho = O.deepgp2_predict(p1_64, p2_64, x64, eps)
    kl = O.kl_hidden_layer(p1_64) + O.kl_meanfield(p2_64)
    noise = O.softplus(torch.zeros((), dtype=torch.float64)) + O.NOISE_LOWER
    lo = -O.elbo_per_window(mo, vo, y.double(), noise, kl, float(D)).mean()
    lo.backward()
    assert rel(mean[0], mo) < 2e-5 and rel(dist.variance[0], vo) < 2e-5
    assert abs(loss.item() - lo.item()) < 2e-5 * abs(lo.item())
    assert rel(xd.grad, x64.grad) < 5e-4
    assert rel(l1.variational_strategy.inducing_points.grad, p1_64["inducing_points"].grad) < 5e-4
    assert rel(l2.variational_strategy.inducing_points.grad, p2_64["inducing_points"].grad) < 5e-4
    assert rel(l1.mean_module.weights.grad, p1_64["weights"].grad) < 5e-4


def test_exact_gp_model(cuda):
    from fine_grained_gaussian_process_forcasting_b200.GPModel import ExactGPModel
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    g = torch.Generator().manual_seed(0)
    tx, ty, sx = torch.randn(20, 3, generator=g), torch.randn(20, generator=g), torch.randn(7, 3, generator=g)
    lik = gpcompat.GaussianLikelihood().to(cuda)
    m = ExactGPModel(tx.to(cuda), ty.to(cuda), lik).to(cuda)
    prior = m(tx.to(cuda))                                       # train mode: prior at the inputs
    z = torch.zeros((), dtype=torch.float64)
    mean_o, cov_o = O.exact_gp_prior(tx.double(), z, z, z)
    assert rel(prior.covariance_matrix, cov_o) < 1e-5 and rel(prior.mean + 1.0, mean_o + 1.0) < 1e-6
    m.eval()
    post = m(sx.to(cuda))
    pm, pc = O.exact_gp_posterior(tx.double(), ty.double(), sx.double(), z, z, z, z)
    assert rel(post.mean, pm) < 1e-4 and rel(post.covariance_matrix, pc) < 1e-4


def test_exact_gp_model_trains(cuda):
    """GPModel.py:4-13 trained the gpytorch way: loss = -ExactMarginalLogLikelihood(likelihood, model)(model(train_x),
    train_y); gradients of the raw lengthscale / outputscale / noise / constant against fp64 autograd on the oracle."""
    from fine_grained_gaussian_process_forcasting_b200.GPModel import ExactGPModel
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    g = torch.Generator().manual_seed(4)
    tx, ty = torch.randn(48, 6, generator=g), torch.randn(48, generator=g)
    lik = gpcompat.GaussianLikelihood().to(cuda)
    m = ExactGPModel(tx.to(cuda), ty.to(cuda), lik).to(cuda)
    with torch.no_grad():
        m.covar_module.base_kernel.raw_lengthscale.fill_(1.2)
        m.covar_module.raw_outputscale.fill_(0.4)
        m.mean_module.raw_constant.fill_(0.1)
        lik.noise_covar.raw_noise.fill_(-1.0)
    mll = gpcompat.ExactMarginalLogLikelihood(lik, m)
    loss = -mll(m(tx.to(cuda)), ty.to(cuda))
    loss.backward()
    c, rl, ro, rn = (torch.tensor(v, dtype=torch.float64, requires_grad=True) for v in (0.1, 1.2, 0.4, -1.0))
    mean_o, cov_o = O.exact_gp_prior(tx.double(), c, rl, ro)
    Kn = cov_o + (O.softplus(rn) + 1e-4) * torch.eye(48, dtype=torch.float64)
    want = -torch.distributions.MultivariateNormal(mean_o, covariance_matrix=Kn).log_prob(ty.double()) / 48
    want.backward()
    assert rel(loss, want) < 1e-5
    assert rel(m.covar_module.base_kernel.raw_lengthscale.grad.reshape(()), rl.grad) < 1e-4
    assert rel(m.covar_module.raw_outputscale.grad, ro.grad) < 1e-4
    assert rel(lik.noise_covar.raw_noise.grad.reshape(()), rn.grad) < 1e-4
    assert rel(m.mean_module.raw_constant.grad, c.grad) < 1e-4


def test_shard_invariance_and_bit_exact_samples(cuda):
    """Size-independent property at a BASELINE size (C3: B=1024, L=24, D=64, M=128): running the batch in
    two shards with global Philox offsets reproduces the single-shot per-window outputs BIT-exactly."""
    from fine_grained_gaussian_process_forcasting_b200 import ops
    B, L, D, M = 1024, 24, 64, 128
    p = {k: v.to(cuda) for k, v in O.init_params_exercise(D, M, 9).items()}
    x = torch.randn(B, L, D, device=cuda, generator=torch.Generator(device=cuda).manual_seed(1))

    def run(xs, off):
        return ops.svgp_predict(xs, p["inducing_points"], p["raw_lengthscale"], p["raw_outputscale"],
                                p["variational_mean"], p["variational_stddev"], p["weights"], p["bias"],
                                seed=5, offset=off, stream_id=0, want_sample=True)
    m_all, v_all, s_all, _, _ = run(x, 0)
    h = 384
    m_a, v_a, s_a, _, _ = run(x[:h], 0)
    m_b, v_b, s_b, _, _ = run(x[h:], h * L)
    assert torch.equal(torch.cat([m_a, m_b]), m_all)
    assert torch.equal(torch.cat([v_a, v_b]), v_all)
    assert torch.equal(torch.cat([s_a, s_b]), s_all)


def test_backward_linearity_at_full_size(cuda):
    """Property at C5 size (B=8192, L=24, D=64, M=64): the backward is linear in the upstream gradients,
    grads(g1 + 2 g2) == grads(g1) + 2 grads(g2), and deterministic run to run."""
    from fine_grained_gaussian_process_forcasting_b200 import ops
    B, L, D, M = 8192, 24, 64, 64
    gen = torch.Generator(device=cuda).manual_seed(2)
    p = {k: v.to(cuda).requires_grad_(True) for k, v in O.init_params_exercise(D, M, 9).items()}
    x = torch.randn(B, L, D, device=cuda, generator=gen).requires_grad_(True)
    g1m, g2m = (torch.randn(B, L, device=cuda, generator=gen) for _ in range(2))
    g1v, g2v = (torch.randn(B, L, device=cuda, generator=gen) for _ in range(2))
    names = ["inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean", "variational_stddev",
             "weights", "bias"]

    def grads(gm, gv):
        mean, var, _, kl, _ = ops.svgp_predict(x, *(p[k] for k in names))
        return torch.autograd.grad([mean, var], [x] + [p[k] for k in names], [gm, gv])
    ga, gb = grads(g1m, g1v), grads(g2m, g2v)
    gc = grads(g1m + 2 * g2m, g1v + 2 * g2v)
    gc2 = grads(g1m + 2 * g2m, g1v + 2 * g2v)
    for a, b, c, c2 in zip(ga, gb, gc, gc2):
        assert torch.equal(c, c2)                                     # deterministic reductions
        assert rel(a + 2 * b, c) < 2e-4


@pytest.mark.parametrize("D,M", [(64, 256), (128, 256), (64, 512)])
def test_tile_position_invariance_of_the_tensor_core_kernels(cuda, D, M):
    """The tensor-core point kernels are persistent: a CTA that owns several 128-point tiles lets its producer groups
    run ahead of each other across slab / tile boundaries (two producer groups in the forward; row owners, loaders and
    per-chunk barriers in the backward; two gates when D = 128; two column blocks when M = 512).  One shot over 282
    tiles (two tiles on most CTAs) must reproduce three shards of 94 tiles (one tile per CTA): outputs bit-exactly,
    dx to rounding, parameter gradients up to the order of the fp32 / fp64 partial sums."""
    from fine_grained_gaussian_process_forcasting_b200 import ops
    B, L = 1500, 24
    gen = torch.Generator(device=cuda).manual_seed(11)
    names = ["inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean", "variational_stddev",
             "weights", "bias"]
    p = {k: v.to(cuda).requires_grad_(True) for k, v in O.init_params_exercise(D, M, 5).items()}
    x = torch.randn(B, L, D, device=cuda, generator=gen).requires_grad_(True)
    gm = torch.randn(B, L, device=cuda, generator=gen)
    gv = torch.randn(B, L, device=cuda, generator=gen)

    def run(lo, hi):
        xs = x[lo:hi].detach().requires_grad_(True)
        mean, var, _, _, _ = ops.svgp_predict(xs, *(p[k] for k in names))
        g = torch.autograd.grad([mean, var], [xs] + [p[k] for k in names], [gm[lo:hi], gv[lo:hi]])
        return mean.detach(), var.detach(), g
    m_all, v_all, g_all = run(0, B)
    parts = [run(lo, lo + 500) for lo in (0, 500, 1000)]
    assert torch.equal(torch.cat([q[0] for q in parts]), m_all)
    assert torch.equal(torch.cat([q[1] for q in parts]), v_all)
    assert rel(torch.cat([q[2][0] for q in parts]), g_all[0]) < 1e-6                     # dx: per-point work only
    for i in range(1, len(g_all)):
        assert rel(sum(q[2][i] for q in parts), g_all[i]) < 2e-4, names[i - 1]


def test_sharded_wrapper_single_process(cuda):
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200.distributed import ShardedGPBlur
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    D, M, B, L = 16, 32, 8, 24
    with gpcompat.num_likelihood_samples(1):
        model = DeepGPp(D, 3, num_inducing=M).to(cuda)
        load_params(model, O.init_params_exercise(D, M, 3))
        dp = ShardedGPBlur(model)
        x, y, _, _ = O.make_inputs(B, L, D, 4)
        out = dp(x.to(cuda).requires_grad_(True), y.to(cuda), first_global_window=0, global_windows=B)
        (-out.elbo.mean()).backward()
        dp.sync_grads()
    assert dp.bucket.flat.abs().sum().item() > 0
    assert model.hidden_layer.variational_strategy.inducing_points.grad.data_ptr() >= dp.bucket.flat.data_ptr()


def test_param_stage_is_shared_between_calls_and_invalidated_by_updates(cuda):
    """The enc / dec calls of one step share the M x M stage (gpblur_svgp_param_stage); an in-place parameter
    update (optimizer step) bumps the tensor version and forces a recompute."""
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat, _cabi
    D, M = 32, 256
    p = O.init_params_exercise(D, M, 3)
    x_enc, _, _, _ = O.make_inputs(4, 48, D, 4)
    x_dec, y, _, _ = O.make_inputs(4, 24, D, 5)
    with gpcompat.num_likelihood_samples(1):
        model = DeepGPp(D, 1, num_inducing=M).to(cuda)
        load_params(model, p)
        hl = model.hidden_layer
        _cabi.profile_enable(True)
        m1, _ = model.predict(x_enc.to(cuda).requires_grad_(True))
        m2, d2 = model.predict(x_dec.to(cuda).requires_grad_(True))
        torch.cuda.synchronize()
        prof = _cabi.profile_collect()
        assert prof["mm_fwd"][1] == 1 and prof["point_fwd"][1] == 2          # one factorisation, two point passes
        # gradients through the cached call
        mll = gpcompat.DeepApproximateMLL(gpcompat.VariationalELBO(model.likelihood, model, D))
        (-mll(d2, y.to(cuda).unsqueeze(0)).mean() + m1.sum()).backward()
        torch.cuda.synchronize()
        prof_b = _cabi.profile_collect()
        # two per-point backward passes, ONE M x M backward (the stage gradients of both calls are summed first)
        assert prof_b["point_bwd"][1] == 2 and prof_b["mm_bwd"][1] == 1 and prof_b["sg_reduce"][1] == 2
        hl.share_param_stage = False
        m2_ref, d2_ref = model.predict(x_dec.to(cuda))
        assert torch.equal(m2, m2_ref) and torch.equal(d2.variance, d2_ref.variance)
        hl.share_param_stage = True
        torch.cuda.synchronize()
        _cabi.profile_collect()
        with torch.no_grad():
            hl.variational_strategy.inducing_points.add_(0.01)                # "optimizer step"
        m3, _ = model.predict(x_dec.to(cuda))
        torch.cuda.synchronize()
        prof = _cabi.profile_collect()
        _cabi.profile_enable(False)
        assert prof["mm_fwd"][1] == 1                                          # recompute after the update
    p2 = dict(p, inducing_points=p["inducing_points"] + 0.01)
    mo, _ = O.svgp_predict_closed_form(O.clone_params(p2, torch.float64), x_dec.double())
    assert rel(m3[0], mo) < 1e-4


def test_two_calls_on_one_stage_match_the_oracle_gradients(cuda):
    """enc + dec call of one step (denoise_model_2.py:50-51) on ONE parameter stage: every parameter gradient is
    the sum over both calls, computed by a single M x M backward."""
    from fine_grained_gaussian_process_forcasting_b200 import ops
    for (D, M) in ((16, 32), (32, 256)):
        p = O.init_params_exercise(D, M, 11)
        x1, _, gm1, gv1 = O.make_inputs(3, 40, D, 12)
        x2, _, gm2, gv2 = O.make_inputs(5, 24, D, 13)
        names = ("inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean", "variational_stddev",
                 "weights", "bias")
        pd = {k: p[k].to(cuda).clone().requires_grad_(True) for k in names}
        cache = {}
        xs = [x1.to(cuda).requires_grad_(True), x2.to(cuda).requires_grad_(True)]
        outs, grads = [], []
        kl = None
        for x, gm, gv in zip(xs, (gm1, gm2), (gv1, gv2)):
            mean, var, _, kl, _ = ops.svgp_predict(x, *(pd[k] for k in names), stage_cache=cache)
            outs += [mean, var]
            grads += [gm.to(cuda), gv.to(cuda)]
        torch.autograd.backward(outs + [kl], grads + [torch.tensor(0.3, device=cuda)])
        p64 = O.clone_params(p, torch.float64, requires_grad=True)
        xo = [x1.double().requires_grad_(True), x2.double().requires_grad_(True)]
        loss = 0.3 * O.kl_meanfield(p64)
        for x, gm, gv in zip(xo, (gm1, gm2), (gv1, gv2)):
            mo, vo = O.svgp_predict_closed_form(p64, x)
            loss = loss + (gm.double() * mo).sum() + (gv.double() * vo).sum()
        loss.backward()
        tol = 2e-4
        for k in names:
            assert rel(pd[k].grad.reshape(-1), p64[k].grad.reshape(-1)) < tol, (D, M, k)
        for xg, xr in zip(xs, xo):
            assert rel(xg.grad, xr.grad) < tol


def test_graphed_step_matches_eager_and_draws_fresh_samples(cuda):
    """CUDA-graph capture of forward + backward (graphs.GraphedStep): replays reproduce the eager step bit for bit
    (same Philox counters), and consecutive replays draw different samples through the device-resident offset."""
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    from fine_grained_gaussian_process_forcasting_b200.graphs import GraphedStep
    from fine_grained_gaussian_process_forcasting_b200.distributed import FlatGradBucket, gp_parameters
    B, L, D, M = 8, 24, 32, 128
    p = O.init_params_exercise(D, M, 21)
    x, y, gm, _ = O.make_inputs(B, L, D, 22)
    with gpcompat.num_likelihood_samples(1):
        model = DeepGPp(D, 5, num_inducing=M).to(cuda)
        load_params(model, p)
        model.train()
        hl = model.hidden_layer
        hl.set_rng(99, 0, 0)
        bucket = FlatGradBucket(gp_parameters(model))
        gmd = gm.to(cuda).unsqueeze(0)
        dx_static = torch.zeros(B, L, D, device=cuda)

        def step(xin, yin):
            bucket.zero()
            xl = xin.detach().requires_grad_(True)
            out = model.blur(xl, yin, num_data=D)
            torch.autograd.backward([out.mean, out.sample, out.elbo],
                                    [gmd, gmd, torch.full((1, B), -1.0 / B, device=cuda)])
            dx_static.copy_(xl.grad)
            return out.mean, out.sample, out.elbo

        g = GraphedStep(model, step, [x.to(cuda), y.to(cuda).unsqueeze(0)])
        mean1, sample1, elbo1 = [t.clone() for t in g.replay()]
        grads1, dx1 = bucket.flat.clone(), dx_static.clone()
        mean2, sample2, elbo2 = [t.clone() for t in g.replay()]
        torch.cuda.synchronize()
        assert torch.equal(mean1, mean2) and torch.equal(elbo1, elbo2)
        assert not torch.equal(sample1, sample2)                      # fresh counters on every replay
        # eager reference with the counters of replay 1 (offset 0) and replay 2 (offset N)
        hl.rng_offset_dev = None
        for k, (mean_g, sample_g) in enumerate(((mean1, sample1), (mean2, sample2))):
            hl.invalidate_param_stage()
            hl._rng_offset = k * B * L
            m_e, s_e, e_e = step(x.to(cuda), y.to(cuda).unsqueeze(0))
            assert torch.equal(m_e, mean_g) and torch.equal(s_e, sample_g)
        # gradients of replay 1 against an eager step with offset 0
        hl.invalidate_param_stage()
        hl._rng_offset = 0
        step(x.to(cuda), y.to(cuda).unsqueeze(0))
        torch.cuda.synchronize()
        assert torch.equal(bucket.flat, grads1) and torch.equal(dx_static, dx1)


def test_anomaly_mode_and_concurrent_threads(cuda):
    """The reference enables torch.autograd.set_detect_anomaly(True) at import (forecast_denoising.py:11) and runs
    optuna with n_jobs=4 threads, each with its own model on the same device (train.py:86): the ops must produce no
    NaN / Inf in backward and be re-entrant."""
    import threading
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    B, L, D, M = 8, 24, 32, 128
    p = O.init_params_exercise(D, M, 31)
    x, y, _, _ = O.make_inputs(B, L, D, 32)
    results, errors = {}, []

    def worker(k):
        try:
            model = DeepGPp(D, 100 + k, num_inducing=M).to(cuda)
            load_params(model, p)
            for _ in range(3):
                xd = x.to(cuda).requires_grad_(True)
                m_enc, _ = model.predict(xd)                 # two calls on one stage, like the reference
                _, dist = model.predict(xd)
                mll = gpcompat.DeepApproximateMLL(gpcompat.VariationalELBO(model.likelihood, model, D))
                loss = -mll(dist, y.to(cuda).unsqueeze(0)).mean() + m_enc.mean()
                model.zero_grad()
                loss.backward()
            torch.cuda.synchronize()
            g = model.hidden_layer.variational_strategy.inducing_points.grad
            assert torch.isfinite(g).all() and torch.isfinite(xd.grad).all()
            results[k] = (loss.item(), g.double().cpu())
        except Exception as e:    # pragma: no cover
            errors.append(repr(e))

    # anomaly mode is a process-global switch (the reference flips it at import): set it around the threads, not
    # inside them, and restore it - a leaked anomaly mode would break CUDA-graph capture in later tests
    # The same holds for num_likelihood_samples: like gpytorch's settings it is a PROCESS-wide value, and the reference
    # enters it once around everything (train.py:20).  Entered per thread, the first thread to leave restored 10 while
    # the others were still in their last step (valid, but S = 10 accumulates the gradients in another order: this
    # test then failed about once in five runs).
    torch.autograd.set_detect_anomaly(True, check_nan=True)
    try:
        with gpcompat.num_likelihood_samples(1):
            threads = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
            for t in threads:
                t.start()
            for t in threads:
                t.join()
    finally:
        torch.autograd.set_detect_anomaly(False)
    assert not errors, errors
    # identical parameters and inputs in every thread -> identical results (deterministic kernels)
    for k in range(1, 4):
        assert results[k][0] == results[0][0] and torch.equal(results[k][1], results[0][1])


def test_call_streams_match_single_stream(cuda):
    """graphs.CallStreams: the encoder- and decoder-side call of one step on two streams (eagerly and inside a
    CUDA-graph capture) give bit-identical outputs and gradients to the single-stream step."""
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    from fine_grained_gaussian_process_forcasting_b200.graphs import GraphedStep, CallStreams
    from fine_grained_gaussian_process_forcasting_b200.distributed import FlatGradBucket, gp_parameters
    D, M = 32, 256
    p = O.init_params_exercise(D, M, 41)
    x_enc, _, g_enc, _ = O.make_inputs(16, 96, D, 42)
    x_dec, y, g_dec, _ = O.make_inputs(16, 24, D, 43)
    with gpcompat.num_likelihood_samples(1):
        model = DeepGPp(D, 7, num_inducing=M).to(cuda)
        load_params(model, p)
        model.train()
        hl = model.hidden_layer
        hl.set_rng(5, 0, 0)
        bucket = FlatGradBucket(gp_parameters(model))
        ge, gd = g_enc.to(cuda).unsqueeze(0), g_dec.to(cuda).unsqueeze(0)
        cs = CallStreams(cuda, 2)
        dxs = [torch.zeros(16, 96, D, device=cuda), torch.zeros(16, 24, D, device=cuda)]

        def step(xe, xd, yy, streams):
            bucket.zero()
            hl.invalidate_param_stage()
            hl._rng_offset = 0
            hl._kl_only()
            xe = xe.detach().requires_grad_(True)
            xd = xd.detach().requires_grad_(True)
            o1 = streams.run(0, lambda: model.blur(xe)) if streams else model.blur(xe)
            o2 = streams.run(1, lambda: model.blur(xd, yy, num_data=D)) if streams else model.blur(xd, yy, num_data=D)
            if streams:
                streams.join()
            torch.autograd.backward([o1.mean, o1.sample, o2.mean, o2.elbo],
                                    [ge, ge, gd, torch.full((1, 16), -1.0 / 16, device=cuda)])
            if streams:
                streams.join()
            dxs[0].copy_(xe.grad)
            dxs[1].copy_(xd.grad)
            return o1.mean, o1.sample, o2.mean, o2.elbo

        ins = [x_enc.to(cuda), x_dec.to(cuda), y.to(cuda).unsqueeze(0)]
        ref = [t.detach().clone() for t in step(*ins, None)]      # detached: keep no autograd graph alive
        torch.cuda.synchronize()
        ref_b, ref_dx = bucket.flat.clone(), [d.clone() for d in dxs]
        got = [t.detach().clone() for t in step(*ins, cs)]
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(ref, got))
        assert torch.equal(bucket.flat, ref_b) and all(torch.equal(a, b) for a, b in zip(dxs, ref_dx))
        g = GraphedStep(model, lambda a, b, c: step(a, b, c, cs), ins)
        got = [t.clone() for t in g.replay()]
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(ref, got))
        assert torch.equal(bucket.flat, ref_b) and all(torch.equal(a, b) for a, b in zip(dxs, ref_dx))
