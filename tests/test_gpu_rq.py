"""Rational quadratic kernel (gpytorch RQKernel, learnable alpha) on the CUDA path against the float64 oracle
(oracle/rq_oracle.py).

Same metric and tolerances as the RBF and Matern parity tests: max|cuda - oracle| / max|oracle|, 1e-5 on mean /
variance on the FP32-FFMA path (M <= 32), 1e-4 on the tcgen05 3xTF32 path, 2e-4 on every gradient, raw_alpha
included.
"""
import math

import pytest
import torch

from oracle import gp_oracle as O
from oracle import rq_oracle as RO

pytestmark = pytest.mark.gpu

TOL_GRAD = 2e-4
NAMES = ["inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean", "variational_stddev", "weights",
         "bias"]
RAW_ALPHAS = [0.0, 1.5]          # alpha = ln 2 (gpytorch's default) and 1.70


def rel(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-300)).item()


def fwd_tol(M):
    return 1e-4 if M > 32 else 1e-5


# (B, L, D, M): both paths, ragged padding of M and D, ragged N (test_gpu_matern.SHAPES)
SHAPES = [
    (3, 7, 5, 3),
    (64, 24, 16, 16),
    (256, 24, 64, 32),
    (5, 13, 48, 100),
    (40, 24, 64, 64),
    (8, 192, 16, 256),
    (3, 24, 128, 300),
    (2, 24, 64, 1024),
]


def _params(D, M, seed, raw_alpha):
    p = O.init_params_exercise(D, M, seed=seed)
    p["raw_alpha"] = torch.tensor([raw_alpha], dtype=torch.float32)
    return p


def _run(ops, p32, x32, seed=1234, offset=5):
    """CUDA forward (mean, var, fused sample, kl) + backward of sum(gm mean + gv var + gs sample) + 0.3 kl."""
    dev = torch.device("cuda")
    pd = {k: v.to(dev).requires_grad_(True) for k, v in p32.items()}
    xd = x32.to(dev).requires_grad_(True)
    mean, var, sample, kl, info = ops.svgp_predict(xd, *(pd[k] for k in NAMES), seed, offset, 0, want_sample=True,
                                                   kernel="rq", raw_alpha=pd["raw_alpha"])
    g = torch.Generator().manual_seed(99)
    gm, gv, gs = (torch.randn(mean.shape, generator=g).to(dev) for _ in range(3))
    loss = (gm * mean).sum() + (gv * var).sum() + (gs * sample).sum() + 0.3 * kl
    loss.backward()
    torch.cuda.synchronize()
    assert int(info.max().item()) == 0
    return mean, var, sample, kl, xd.grad, {k: pd[k].grad for k in NAMES + ["raw_alpha"]}, (gm.cpu(), gv.cpu(),
                                                                                              gs.cpu())


def _oracle(p32, x32, gms, seed=1234, offset=5):
    from fine_grained_gaussian_process_forcasting_b200 import ops
    p64 = O.clone_params(p32, torch.float64, requires_grad=True)
    x64 = x32.double().requires_grad_(True)
    mo, vo = RO.svgp_predict_closed_form(p64, x64, kernel="rq")
    eps = ops.philox_normal(seed, offset, mo.numel(), 0).cpu().double().reshape(mo.shape)
    so = mo + vo.sqrt() * eps
    kl = O.kl_meanfield(p64)
    gm, gv, gs = (t.double() for t in gms)
    ((gm * mo).sum() + (gv * vo).sum() + (gs * so).sum() + 0.3 * kl).backward()
    return mo, vo, so, kl, x64.grad, {k: p64[k].grad for k in NAMES + ["raw_alpha"]}


@pytest.mark.parametrize("raw_alpha", RAW_ALPHAS)
@pytest.mark.parametrize("B,L,D,M", SHAPES)
def test_rq_parity(cuda, raw_alpha, B, L, D, M):
    from fine_grained_gaussian_process_forcasting_b200 import ops
    p32 = _params(D, M, 11, raw_alpha)
    x32, _, _, _ = O.make_inputs(B, L, D, seed=12)
    mean, var, sample, kl, dx, grads, gms = _run(ops, p32, x32)
    mo, vo, so, klo, dxo, go = _oracle(p32, x32, gms)
    errs = {"mean": rel(mean, mo), "var": rel(var, vo), "sample": rel(sample, so), "dx": rel(dx, dxo)}
    errs.update({k: rel(grads[k].reshape(go[k].shape), go[k]) for k in NAMES + ["raw_alpha"]})
    # raw_outputscale and raw_alpha are ONE number each, a sum of terms of both signs over all points and inducing
    # pairs: measured against the size of the terms (the same gradient with |upstream gradients|), as test_gpu_matern
    scale = _oracle(p32, x32, tuple(t.abs() for t in gms))[5]
    for k in ("raw_outputscale", "raw_alpha"):
        errs[k] = ((grads[k].double().cpu().reshape(go[k].shape) - go[k]).abs()
                   / torch.maximum(go[k].abs(), scale[k].abs())).max().item()
    print(f"rq raw_alpha={raw_alpha} B={B} L={L} D={D} M={M}:", {k: f"{v:.1e}" for k, v in errs.items()})
    tol = fwd_tol(M)
    assert errs["mean"] < tol and errs["var"] < tol and errs["sample"] < tol, errs
    assert abs(kl.item() - klo.item()) <= 1e-5 * max(1.0, abs(klo.item()))
    for k in ["dx"] + NAMES + ["raw_alpha"]:
        assert errs[k] < TOL_GRAD, (k, errs)


@pytest.mark.parametrize("M", [32, 256])
def test_rq_repeated_backward_bit_identical(cuda, M):
    from fine_grained_gaussian_process_forcasting_b200 import ops
    p32 = _params(64, M, 3, 0.5)
    x32, _, _, _ = O.make_inputs(64, 24, 64, seed=4)
    r1 = _run(ops, p32, x32)
    r2 = _run(ops, p32, x32)
    assert torch.equal(r1[4], r2[4])
    for k in NAMES + ["raw_alpha"]:
        assert torch.equal(r1[5][k], r2[5][k]), k


@pytest.mark.parametrize("M", [32, 100, 256, 600, 1024])
def test_rq_stage_bit_identical_across_grids(cuda, M):
    """The M x M stage and its backward (RQ: the alpha term summed per product tile in fixed order) give the same
    bits whatever cooperative grid they run on (max_ctas, as the multi-output layers bound it)."""
    from fine_grained_gaussian_process_forcasting_b200 import ops
    D = 20
    kind = ops.kernel_kind("rq")
    p = {k: v.cuda() for k, v in _params(D, M, 17, 0.7).items()}
    args = [p[k].reshape(-1) if k in ("raw_lengthscale", "weights") else p[k] for k in NAMES]
    G = ops.stage_grad_doubles(D, M, kind)
    sgrad = torch.randn(G, generator=torch.Generator().manual_seed(5), dtype=torch.float64).cuda()
    gkl = torch.tensor([0.3], device="cuda")
    res = []
    for cap in (0, 8, 13, 37, 74):
        stage, kl, info = ops.param_stage_raw(*args, max_ctas=cap, kind=kind, raw_alpha=p["raw_alpha"])
        bucket = ops.param_stage_backward_raw(*args, sgrad, gkl, stage, max_ctas=cap, kind=kind,
                                              raw_alpha=p["raw_alpha"])
        torch.cuda.synchronize()
        assert int(info.item()) == 0
        # L and Linv: their lower triangles (the stage leaves the upper half of the diagonal blocks unwritten)
        res.append((torch.tril(ops.debug_fetch(0, 0, D, M, stage).cpu()),
                    torch.tril(ops.debug_fetch(1, 0, D, M, stage).cpu()), kl.cpu(), bucket.cpu()))
    assert res[0][3].numel() == ops.grad_bucket_floats(D, M, kind) == ops.grad_bucket_floats(D, M) + 1
    assert torch.isfinite(res[0][3]).all() and res[0][3][-1] != 0
    for r in res[1:]:
        for u, v in zip(res[0], r):
            assert torch.equal(u, v)


@pytest.mark.parametrize("M", [32, 256])
def test_rq_multi_output_layer(cuda, M):
    """Batched [H, M, D] parameters with a per-GP alpha (raw_alpha [H, 1]) against the per-GP oracle."""
    from fine_grained_gaussian_process_forcasting_b200 import ops
    D, H, B, L = 16, 3, 8, 24
    p1 = O.init_params_hidden_layer(D, H, M, seed=5)
    p1["raw_alpha"] = torch.tensor([[-0.5], [0.0], [1.2]])
    x32, _, _, _ = O.make_inputs(B, L, D, seed=6)
    dev = torch.device("cuda")
    pd = {k: v.to(dev).requires_grad_(True) for k, v in p1.items()}
    xd = x32.to(dev).requires_grad_(True)
    mean, var, _, kl, _ = ops.svgp_predict(xd, *(pd[k] for k in NAMES), kernel="rq", raw_alpha=pd["raw_alpha"])
    (mean.sum() + var.sum() + kl.sum()).backward()
    p64 = O.clone_params(p1, torch.float64, requires_grad=True)
    x64 = x32.double().requires_grad_(True)
    mo, vo = RO.hidden_layer_predict(p64, x64, kernel="rq")
    (mo.sum() + vo.sum() + O.kl_hidden_layer(p64)).backward()
    assert rel(mean, mo) < fwd_tol(M) and rel(var, vo) < fwd_tol(M)
    assert rel(xd.grad, x64.grad) < TOL_GRAD
    for k in NAMES + ["raw_alpha"]:
        assert rel(pd[k].grad, p64[k].grad) < TOL_GRAD, k


def test_rq_segments_equal_separate_calls(cuda):
    from fine_grained_gaussian_process_forcasting_b200 import ops
    D, M = 32, 256
    p32 = _params(D, M, 8, 0.3)
    dev = torch.device("cuda")
    xa, _, _, _ = O.make_inputs(8, 192, D, seed=1)
    xb, _, _, _ = O.make_inputs(8, 24, D, seed=2)
    res = []
    for joint in (False, True):
        pd = {k: v.to(dev).requires_grad_(True) for k, v in p32.items()}
        a, b = xa.to(dev).requires_grad_(True), xb.to(dev).requires_grad_(True)
        args = [pd[k] for k in NAMES]
        kw = dict(want_sample=True, kernel="rq", raw_alpha=pd["raw_alpha"])
        if joint:
            x = torch.cat([a.reshape(-1, D), b.reshape(-1, D)])
            segs, kl, _ = ops.svgp_predict_segments(x, [(8, 192), (8, 24)], *args, 7, 0, 0, **kw)
            (ma, va, sa), (mb, vb, sb) = segs
        else:
            ma, va, sa, kl, _ = ops.svgp_predict(a, *args, 7, 0, 0, **kw)
            mb, vb, sb, _, _ = ops.svgp_predict(b, *args, 7, a.numel() // D, 0, **kw)
        (ma.sum() + 2 * va.sum() + sa.sum() + mb.sum() + vb.sum() + 3 * sb.sum() + kl).backward()
        res.append(([ma, va, sa, mb, vb, sb], [a.grad, b.grad] + [pd[k].grad for k in NAMES + ["raw_alpha"]]))
    for u, v in zip(res[0][0], res[1][0]):
        assert torch.equal(u, v)
    for u, v in zip(res[0][1], res[1][1]):
        assert rel(u, v) < 1e-5


@pytest.mark.parametrize("ard", [True, False])
def test_rq_dense_covariance(cuda, ard):
    from fine_grained_gaussian_process_forcasting_b200 import ops
    g = torch.Generator().manual_seed(2)
    n1, n2, D = 37, 21, 5
    x1, x2 = torch.randn(n1, D, generator=g), torch.randn(n2, D, generator=g)
    rl = 0.3 * torch.randn(D if ard else 1, generator=g)
    ro, ra = torch.tensor([0.4]), torch.tensor([-0.3])
    dev = torch.device("cuda")
    a, b, l, o, al = (t.to(dev).requires_grad_(True) for t in (x1, x2, rl, ro, ra))
    K = ops.rbf_covariance(a, b, l, o, ard, kernel="rq", raw_alpha=al)
    G = torch.randn(n1, n2, generator=g)
    (K * G.to(dev)).sum().backward()
    a64, b64, l64, o64, al64 = (t.double().requires_grad_(True) for t in (x1, x2, rl, ro, ra))
    Ko = RO.scale_direct(a64, b64, O.softplus(l64), O.softplus(o64).reshape(()), "rq", O.softplus(al64).reshape(()))
    (Ko * G.double()).sum().backward()
    assert rel(K, Ko) < 1e-5
    for u, v in [(a.grad, a64.grad), (b.grad, b64.grad), (l.grad, l64.grad), (o.grad, o64.grad), (al.grad, al64.grad)]:
        assert rel(u, v) < TOL_GRAD


def test_rq_exact_gp_trains(cuda):
    """gpcompat.ScaleKernel(RQKernel) evaluates the dense covariance by the CUDA kernel, and an exact GP with it
    trains under ExactMarginalLogLikelihood: the loss falls and alpha moves."""
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    k = gpcompat.ScaleKernel(gpcompat.RQKernel()).cuda()
    x = torch.randn(30, 3, device="cuda")
    want = RO.scale_direct(x.double().cpu(), x.double().cpu(), O.softplus(torch.zeros(1, dtype=torch.float64)),
                           O.softplus(torch.zeros((), dtype=torch.float64)), "rq", math.log(2.0))
    assert rel(k(x), want) < 1e-5

    from fine_grained_gaussian_process_forcasting_b200.GPModel import ExactGPModel
    g = torch.Generator().manual_seed(4)
    tx, ty = torch.randn(48, 6, generator=g), torch.randn(48, generator=g)
    lik = gpcompat.GaussianLikelihood().cuda()
    m = ExactGPModel(tx.cuda(), ty.cuda(), lik).cuda()
    m.covar_module = gpcompat.ScaleKernel(gpcompat.RQKernel()).cuda()
    with torch.no_grad():
        m.covar_module.base_kernel.raw_lengthscale.fill_(1.2)
        m.covar_module.base_kernel.raw_alpha.fill_(-0.4)
        m.covar_module.raw_outputscale.fill_(0.4)
        m.mean_module.raw_constant.fill_(0.1)
        lik.noise_covar.raw_noise.fill_(-1.0)
    mll = gpcompat.ExactMarginalLogLikelihood(lik, m)
    loss = -mll(m(tx.cuda()), ty.cuda())
    loss.backward()
    c, rl, ro, rn, ra = (torch.tensor(v, dtype=torch.float64, requires_grad=True) for v in (0.1, 1.2, 0.4, -1.0, -0.4))
    mean_o, cov_o = RO.exact_gp_prior(tx.double(), c, rl, ro, "rq", ra)
    Kn = cov_o + (O.softplus(rn) + 1e-4) * torch.eye(48, dtype=torch.float64)
    want = -torch.distributions.MultivariateNormal(mean_o, covariance_matrix=Kn).log_prob(ty.double()) / 48
    want.backward()
    assert rel(loss, want) < 1e-5
    assert rel(m.covar_module.base_kernel.raw_alpha.grad.reshape(()), ra.grad) < 1e-4
    assert rel(m.covar_module.base_kernel.raw_lengthscale.grad.reshape(()), rl.grad) < 1e-4
    assert rel(m.covar_module.raw_outputscale.grad, ro.grad) < 1e-4
    opt = torch.optim.Adam(m.parameters(), lr=0.05)
    losses = []
    for _ in range(20):
        opt.zero_grad()
        loss = -mll(m(tx.cuda()), ty.cuda())
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(math.isfinite(v) for v in losses)
    assert losses[-1] < losses[0], losses
    assert m.covar_module.base_kernel.raw_alpha.item() != -0.4


def _rq_covar(layer, gpcompat):
    ard = layer.covar_module.base_kernel.ard_num_dims
    bs = layer.covar_module.batch_shape
    return gpcompat.ScaleKernel(gpcompat.RQKernel(ard_num_dims=ard, batch_shape=bs), batch_shape=bs)


def test_rq_deepgp2_both_layers(cuda):
    """DeepGP2 with RQ kernels in both layers (a multi-output first layer with per-GP alpha): forward and backward run
    and every gradient, raw_alpha included, is finite."""
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGP2
    import inspect
    D = 16
    sig = inspect.signature(DeepGP2.__init__)
    model = DeepGP2(D, 1234, **({"num_inducing": 32} if "num_inducing" in sig.parameters else {})).cuda()
    layers = [m for m in model.modules() if isinstance(m, gpcompat.DeepGPLayer)]
    assert len(layers) >= 2
    for layer in layers:
        layer.covar_module = _rq_covar(layer, gpcompat).cuda()
        assert gpcompat._kernel_raw_params(layer.covar_module)[2] == "rq"
    x = torch.randn(4, 24, D, device="cuda")
    with gpcompat.num_likelihood_samples(1):
        out = model(x)
        dist = out[1] if isinstance(out, tuple) else out
        (dist.mean.sum() + dist.variance.sum()).backward()
    for layer in layers:
        ga = layer.covar_module.base_kernel.raw_alpha.grad
        assert ga is not None and torch.isfinite(ga).all() and (ga != 0).any()
    for p in model.parameters():
        if p.grad is not None:
            assert torch.isfinite(p.grad).all()


@pytest.mark.parametrize("M", [32, 256])
def test_rq_graph_replayed_step_with_flat_bucket(cuda, M):
    """A GraphedStep with an RQ layer whose gradients go through a FlatGradBucket (the layer is a gradient sink: its
    M x M backward accumulates into the flat buffer, raw_alpha last) computes what the eager step computes."""
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200.distributed import FlatGradBucket
    from fine_grained_gaussian_process_forcasting_b200.graphs import GraphedStep
    D = 32
    p = O.init_params_exercise(D, M, 7)

    def build():
        model = DeepGPp(D, 1234, num_inducing=M)
        hl = model.hidden_layer
        hl.covar_module = _rq_covar(hl, gpcompat)
        with torch.no_grad():
            hl.variational_strategy.inducing_points.copy_(p["inducing_points"])
            hl.covar_module.base_kernel.raw_lengthscale.copy_(p["raw_lengthscale"])
            hl.covar_module.base_kernel.raw_alpha.fill_(0.4)
            hl.variational_strategy.variational_params_initialized.fill_(1)
        return model.cuda()

    x = torch.randn(16, 24, D, device="cuda")
    gm = torch.randn(1, 16, 24, device="cuda")

    def stepper(model):
        def step(xin):
            out = model.blur(xin.detach().requires_grad_(True))
            torch.autograd.backward([out.mean], [gm])
            return (out.mean,)
        return step

    with gpcompat.num_likelihood_samples(1):
        eager = build()
        want = stepper(eager)(x)[0].detach().clone()
        want_g = {n: q.grad.clone() for n, q in eager.named_parameters() if q.grad is not None}
        assert "hidden_layer.covar_module.base_kernel.raw_alpha" in want_g
        model = build()
        flat = FlatGradBucket(list(model.parameters()), module=model)
        assert model.hidden_layer._grad_sink is not None
        assert model.hidden_layer._grad_sink.numel() == sum(q.numel() for q in model.hidden_layer._layer_params())
        graphed = GraphedStep(model, stepper(model), [x], warmup=1)
        flat.zero()
        got = graphed.replay()[0]
        torch.cuda.synchronize()
    assert torch.equal(got, want)
    params = dict(model.named_parameters())
    for n, g in want_g.items():
        assert rel(params[n].grad, g) < 1e-6, n
