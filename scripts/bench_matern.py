"""Step time of the GP blur with each covariance function: RBF, Matern nu = 1/2, 3/2, 5/2 and rational quadratic.

For the workloads c1 (FP32-FFMA point kernels, M = 32), c2 (two calls per step, M = 256) and c5_m256 of bench.py, the
model of bench.make_model (exercise_init parameters) is built once per covariance function - the Matern and RQ layers
take the same raw parameter values (RQ: raw_alpha = 0, alpha = ln 2), only covar_module is swapped, the gpytorch
idiom - and its forward + backward step is
captured in a CUDA graph (GraphedStep).  The kernels are then timed in rounds that alternate between them, so that a
drift of the clocks or of the other work on the machine hits them alike.  Prints the card name and power limit, one
JSON line per workload with the median ms per step and the ratio to RBF, and (c2) the per-stage times of the library's
profile hooks from one extra eager step per kernel.

    python scripts/bench_matern.py [--steps 50] [--rounds 7]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

KERNELS = {"rbf": None, "matern12": 0.5, "matern32": 1.5, "matern52": 2.5, "rq": "rq"}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:     # the measurement does not depend on it
        return f"unavailable ({e!r})"


def swap_kernel(model, nu):
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    for layer in [m for m in model.modules() if isinstance(m, gpcompat.DeepGPLayer)]:
        old = layer.covar_module
        bs = old.batch_shape
        ard = old.base_kernel.ard_num_dims
        base = (gpcompat.RQKernel(ard_num_dims=ard, batch_shape=bs) if nu == "rq"
                else gpcompat.MaternKernel(nu=nu, ard_num_dims=ard, batch_shape=bs))
        new = gpcompat.ScaleKernel(base, batch_shape=bs)
        # same raw lengthscale / outputscale values (RQ keeps its own raw_alpha)
        missing, unexpected = new.load_state_dict(old.state_dict(), strict=False)
        assert not unexpected and all(k.startswith("base_kernel.raw_alpha") for k in missing), (missing, unexpected)
        layer.covar_module = new.to(old.raw_outputscale.device)


def build(wl, kernel, device):
    import bench
    from fine_grained_gaussian_process_forcasting_b200.graphs import GraphedStep
    model = bench.make_model(wl, device)
    if KERNELS[kernel] is not None:
        swap_kernel(model, KERNELS[kernel])
    model.train()
    B, D, calls = wl["B"], wl["D"], wl["calls"]
    g = torch.Generator(device=device).manual_seed(1234)
    xs = [torch.randn(B, L, D, device=device, generator=g) for L in calls]
    y = torch.randn(1, B, calls[-1], device=device, generator=g)
    gms = [torch.randn(1, B, L, device=device, generator=g) for L in calls]

    def step(*ins):
        xin, yin = ins[:-1], ins[-1]
        outs, grads = [], []
        for c, x in enumerate(xin):
            last = c == len(xin) - 1
            o = model.blur(x.detach().requires_grad_(True), yin if last else None, num_data=D)
            outs += [o.mean, o.sample]
            grads += [gms[c], gms[c]]
            if last:
                outs.append(o.elbo)
                grads.append(torch.full_like(o.elbo, -1.0 / B))
        torch.autograd.backward(outs, grads)
        return (outs[-1],)

    for p in model.parameters():
        p.grad = torch.zeros_like(p)
    return model, step, xs + [y], GraphedStep(model, step, xs + [y])


def time_graph(graphed, steps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        graphed.replay()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / steps


def stage_times(model, step, inputs):
    from fine_grained_gaussian_process_forcasting_b200 import _cabi
    step(*inputs)
    torch.cuda.synchronize()
    _cabi.profile_enable(True)
    step(*inputs)
    torch.cuda.synchronize()
    _cabi.profile_enable(False)
    return {name: round(ms * 1e3, 1) for name, (ms, _) in _cabi.profile_collect().items()}   # microseconds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--workloads", default="c1,c2,c5_m256")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_matern.py needs a CUDA device")
    import bench
    device = torch.device("cuda", 0)
    print(json.dumps({"card": card()}), flush=True)
    for name in args.workloads.split(","):
        wl = bench.WORKLOADS[name]
        built = {k: build(wl, k, device) for k in KERNELS}
        times = {k: [] for k in KERNELS}
        for k in KERNELS:
            time_graph(built[k][3], 5)
        for _ in range(args.rounds):
            for k in KERNELS:
                times[k].append(time_graph(built[k][3], args.steps))
        med = {k: statistics.median(v) for k, v in times.items()}
        line = {"workload": name, "ms_per_step": {k: round(v, 4) for k, v in med.items()},
                "spread_ms": {k: round(max(v) - min(v), 4) for k, v in times.items()},
                "ratio_to_rbf": {k: round(med[k] / med["rbf"], 3) for k in KERNELS}}
        if name == "c2":
            line["stage_us"] = {k: stage_times(*built[k][:3]) for k in KERNELS}
        print(json.dumps(line), flush=True)
        del built
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
