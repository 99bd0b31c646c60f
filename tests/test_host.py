"""CPU tests of the host logic: the C-ABI library loads and exports every symbol include/gpblur.h
declares (no compute calls without a GPU), the module boundary mirrors the reference (constructor,
state_dict keys, RNG order), the product path fails loudly off-GPU, the gpytorch import shim, the
data-parallel gradient bucket over gloo (world_size 2), the bench.py reference-arm contract and (on a GPU) the
bench.py result line and --dump-outputs."""
import ctypes
import json
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from fine_grained_gaussian_process_forcasting_b200 import _cabi
    header = open(os.path.join(ROOT, "include", "gpblur.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(gpblur_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 15
    assert declared == set(_cabi.SIGNATURES), declared ^ set(_cabi.SIGNATURES)
    lib = ctypes.CDLL(str(_cabi.LIB_PATH))
    for name in declared:
        assert hasattr(lib, name), name
    assert b"sm_100a" in _cabi.lib().gpblur_version()


def test_host_only_entry_points():
    from fine_grained_gaussian_process_forcasting_b200 import _cabi, ops
    lib = _cabi.lib()
    assert lib.gpblur_svgp_grad_bucket_floats(64, 32) == 32 * 64 + 2 * 32 + 2 * 64 + 2 == ops.grad_bucket_floats(64, 32)
    small = lib.gpblur_svgp_workspace_bytes(100, 64, 32, 0)
    train = lib.gpblur_svgp_workspace_bytes(100, 64, 32, 1)
    big = lib.gpblur_svgp_workspace_bytes(100000, 64, 32, 1)
    assert 0 < small < train < big and small % 256 == 0 and train % 256 == 0
    assert lib.gpblur_svgp_workspace_bytes(10, 129, 32, 1) == 0      # D > GPBLUR_MAX_D
    assert lib.gpblur_svgp_workspace_bytes(10, 64, 1025, 1) == 0     # M > GPBLUR_MAX_M
    assert lib.gpblur_svgp_workspace_bytes(0, 1, 1, 1) > 0           # empty batch is legal


def test_cuda_kernels_are_sm100a_sass():
    from fine_grained_gaussian_process_forcasting_b200 import _cabi
    try:
        out = subprocess.run(["cuobjdump", "-lelf", str(_cabi.LIB_PATH)], capture_output=True, text=True, timeout=60)
    except FileNotFoundError:
        pytest.skip("cuobjdump not available")
    assert "sm_100a" in out.stdout


def test_ops_fail_loudly_without_cuda():
    from fine_grained_gaussian_process_forcasting_b200 import ops
    x = torch.randn(4, 3, 8)
    Z = torch.randn(5, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.svgp_predict(x, Z, torch.zeros(1, 8), torch.zeros(()), torch.zeros(5), torch.ones(5), torch.zeros(8, 1),
                         torch.zeros(1))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.variational_elbo(torch.zeros(2, 3), torch.ones(2, 3), torch.zeros(2, 3), torch.zeros(1), torch.zeros(()), 8.0)


def test_missing_library_raises(monkeypatch, tmp_path):
    from fine_grained_gaussian_process_forcasting_b200 import _cabi
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setenv("GPBLUR_LIB", str(tmp_path / "nope.so"))
    with pytest.raises(_cabi.GpblurLibraryMissing):
        _cabi.lib()


EXPECTED_KEYS = {
    "hidden_layer.variational_strategy.inducing_points",
    "hidden_layer.variational_strategy.variational_params_initialized",
    "hidden_layer.variational_strategy.updated_strategy",
    "hidden_layer.variational_strategy._variational_distribution.variational_mean",
    "hidden_layer.variational_strategy._variational_distribution._variational_stddev",
    "hidden_layer.mean_module.weights",
    "hidden_layer.mean_module.bias",
    "hidden_layer.covar_module.raw_outputscale",
    "hidden_layer.covar_module.base_kernel.raw_lengthscale",
    "hidden_layer.covar_module.base_kernel.raw_lengthscale_constraint.lower_bound",
    "hidden_layer.covar_module.base_kernel.raw_lengthscale_constraint.upper_bound",
    "hidden_layer.covar_module.raw_outputscale_constraint.lower_bound",
    "hidden_layer.covar_module.raw_outputscale_constraint.upper_bound",
    "likelihood.noise_covar.raw_noise",
    "likelihood.noise_covar.raw_noise_constraint.lower_bound",
    "likelihood.noise_covar.raw_noise_constraint.upper_bound",
}


def test_deepgpp_constructor_and_state_dict():
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from oracle import gp_oracle as O
    m = DeepGPp(32, 1234)                                    # positional (num_hidden_dims, seed), DeepGP.py:77
    sd = m.state_dict()
    assert set(sd) == EXPECTED_KEYS
    ref = O.init_params_reference(32, 1234, M=256)           # reference RNG order: Z first, then w, b
    hl = m.hidden_layer
    assert torch.equal(hl.variational_strategy.inducing_points, ref["inducing_points"])
    assert torch.equal(hl.mean_module.weights, ref["weights"]) and torch.equal(hl.mean_module.bias, ref["bias"])
    assert sd["hidden_layer.covar_module.base_kernel.raw_lengthscale"].shape == (1, 32)
    assert sd["hidden_layer.covar_module.raw_outputscale"].shape == ()
    assert sd["likelihood.noise_covar.raw_noise"].shape == (1,)
    assert abs(m.likelihood.noise.item() - (0.6931471805599453 + 1e-4)) < 1e-6
    m2 = DeepGPp(32, 99)
    m2.load_state_dict(sd, strict=True)
    assert torch.equal(m2.hidden_layer.variational_strategy.inducing_points, ref["inducing_points"])
    assert len(list(m.parameters())) == 8 and m.training
    m.eval()
    assert not m.hidden_layer.training


def test_hidden_layer_multi_output_shapes():
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import ToyDeepGPHiddenLayer, DeepGP2
    hl = ToyDeepGPHiddenLayer(16, 5, seed=3, num_inducing=12)            # default mean_type='constant'
    assert hl.variational_strategy.inducing_points.shape == (5, 12, 16)
    assert hl.mean_module.raw_constant.shape == (5,)
    assert hl.covar_module.raw_outputscale.shape == (5,)
    assert hl.covar_module.base_kernel.raw_lengthscale.shape == (5, 1, 16)
    assert hl.variational_strategy._variational_distribution.variational_mean.shape == (5, 12)
    d2 = DeepGP2(16, 3, hidden_dims=4, num_inducing=8)
    assert d2.last_layer.input_dims == 4


def test_first_call_initialisation_semantics():
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    m = DeepGPp(8, 5, num_inducing=16)
    vs = m.hidden_layer.variational_strategy
    assert int(vs.variational_params_initialized) == 0
    torch.manual_seed(123)
    vs._ensure_initialized()
    torch.manual_seed(123)
    want = 1e-3 * torch.randn(16)
    assert torch.allclose(vs._variational_distribution.variational_mean.detach(), want)
    assert int(vs.variational_params_initialized) == 1
    before = vs._variational_distribution.variational_mean.detach().clone()
    vs._ensure_initialized()
    assert torch.equal(before, vs._variational_distribution.variational_mean.detach())


def test_settings_context():
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    assert gpcompat.num_likelihood_samples.value() == 10
    with gpcompat.num_likelihood_samples(1):
        assert gpcompat.num_likelihood_samples.value() == 1
    assert gpcompat.num_likelihood_samples.value() == 10


def test_gpytorch_shim_imports():
    import fine_grained_gaussian_process_forcasting_b200 as pkg
    g = pkg.install_gpytorch_shim()
    assert getattr(g, "IS_GPBLUR_SHIM", False)
    from gpytorch.mlls import DeepApproximateMLL, VariationalELBO            # forecast_denoising.py:5
    from gpytorch.models.deep_gps import DeepGPLayer, DeepGP                 # DeepGP.py:10
    from gpytorch.variational import VariationalStrategy, MeanFieldVariationalDistribution   # DeepGP.py:11
    from gpytorch.kernels import ScaleKernel, RBFKernel, MaternKernel        # DeepGP.py:7
    import gpytorch
    assert gpytorch.likelihoods.GaussianLikelihood is not None               # train.py:57
    with gpytorch.settings.num_likelihood_samples(1):                        # train.py:20
        pass
    assert callable(gpytorch.models.ExactGP)                                 # GPModel.py:4


def test_shard_range():
    from fine_grained_gaussian_process_forcasting_b200.distributed import shard_range
    for n, w in [(1024, 8), (10, 4), (3, 8), (0, 2)]:
        spans = [shard_range(n, r, w) for r in range(w)]
        assert sum(c for _, c in spans) == n
        pos = 0
        for s, c in spans:
            assert s == pos
            pos += c


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp
    from fine_grained_gaussian_process_forcasting_b200.distributed import (FlatGradBucket, gp_parameters,
                                                                            broadcast_parameters)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    model = DeepGPp(8, 100 + rank, num_inducing=16)          # different seeds: broadcast must equalise
    broadcast_parameters(model, 0)
    params = gp_parameters(model)
    bucket = FlatGradBucket(params)
    # a stand-in loss on the parameters (the GP ops need CUDA): rank-dependent so the average is checkable
    loss = sum(((rank + 1.0) * (i + 1) * p).sum() for i, p in enumerate(params))
    loss.backward()
    assert all(p.grad.data_ptr() >= bucket.flat.data_ptr() for p in params)   # grads live in the bucket
    bucket.all_reduce(average=True)
    want = (1 + world) / 2.0
    ok = all(torch.allclose(p.grad, torch.full_like(p, want * (i + 1))) for i, p in enumerate(params))
    z0 = model.hidden_layer.variational_strategy.inducing_points.detach().clone()
    gathered = [torch.zeros_like(z0) for _ in range(world)]
    dist.all_gather(gathered, z0)
    same = all(torch.equal(gathered[0], g) for g in gathered)
    # the first-call variational init (1e-3 randn from each rank's own RNG) ran BEFORE the broadcast and cannot run
    # again on the first forward: the replicas hold rank 0's variational mean and keep it
    vs = model.hidden_layer.variational_strategy
    torch.manual_seed(1000 + rank)
    vs._ensure_initialized()                                  # what the first forward does: must be a no-op now
    vm = vs._variational_distribution.variational_mean.detach().clone()
    gvm = [torch.zeros_like(vm) for _ in range(world)]
    dist.all_gather(gvm, vm)
    same = same and all(torch.equal(gvm[0], g) for g in gvm) and bool(vm.abs().max() > 0) \
        and int(vs.variational_params_initialized) == 1
    bucket.zero()
    zeroed = all(float(p.grad.abs().max()) == 0.0 for p in params)
    if rank == 0:
        with open(out, "w") as f:
            json.dump({"ok": ok, "same": same, "zeroed": zeroed, "n": bucket.flat.numel()}, f)
    dist.destroy_process_group()


def test_flat_grad_bucket_allreduce_gloo_world2(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "res.json")
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, out), nprocs=2, join=True)
    res = json.load(open(out))
    assert res["ok"] and res["same"] and res["zeroed"]
    assert res["n"] == 16 * 8 + 2 * 16 + 2 * 8 + 3           # M*D + 2M + 2D + 3 (SURVEY 8e)


def test_bench_reference_arm_contract():
    env = dict(os.environ, GPBLUR_CPU_SAMPLE_B="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--workload", "c1"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "windows/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["higher_is_better"] is True
    assert line["config"]["workload"] == "c1"


@pytest.mark.gpu
def test_bench_result_line_and_dump_outputs(cuda, tmp_path):
    """bench.py prints one short JSON result line on stdout, and --dump-outputs writes what the last timed step
    computed (float32, at most 64 MiB); two runs with the same arguments write the same arrays."""
    import numpy as np
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", "3",
                              "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = out.stdout.strip().splitlines()
        assert len(lines) == 1 and len(lines[0]) < 2000, lines
        line = json.loads(lines[0])
        assert line["steps"] == 3 and line["config"]["workload"] == "c1" and line["value"] > 0
        dumps.append({f.stem: np.load(f) for f in sorted(d.glob("*.npy"))})
    a, b = dumps
    assert {"mean_0", "sample_0", "dx_0", "elbo", "grad_hidden_layer.variational_strategy.inducing_points"} <= set(a)
    assert a["dx_0"].shape == (256, 24, 64) and a["mean_0"].shape == (1, 256, 24) and a["elbo"].shape == (1, 256)
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
