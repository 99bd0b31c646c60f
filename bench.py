#!/usr/bin/env python
"""GP-blur fwd+bwd throughput (windows/s) on B200 - the metric of BASELINE.json.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference]
                  [--sweep] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic forecast windows per GPU:
whitened-SVGP predictive (mean, variance, fused Philox sample) of every GP call of the workload, the
ELBO on the decoder-side call, and the full hand-written backward (dX + every GP parameter gradient);
for N > 1 the flat GP-gradient bucket is all-reduced over NCCL inside the step.  The inputs and
parameters are seeded, so runs with the same arguments see the same inputs.

Workloads (BASELINE.json `configs`; per-GPU batch is fixed => weak scaling):
  c2      configs[1]: the two GP-blur calls of the traffic-shape train step, enc [256,192,64] and
          dec [256,24,64], M=256 (reference default), ELBO on the decoder call.   <- default
          (the forecaster / denoiser around them are outside the hot path, SURVEY section 8)
  c1      configs[0]: B=256, L=24, D=64, M=32
  c3      configs[2]: B=1024, L=24, D=64, M=128
  c4      configs[3]: two-layer DeepGP, B=2048, L=24, D=64, M=256, hidden width H=10
  c5_mM   configs[4]: B=8192, L=24, D=64, M in {64,128,256,512,1024}

The run prints ONE JSON result line for --workload on stdout, and the breakdown (roofline,
roofline_per_point_kernel, stage_ms_per_step and what --sweep adds) as one JSON line on stderr.
  value     K = --steps timed steps on inputs resident in HBM: per-step CUDA events (max over ranks),
            a 256 MiB L2 flush (write) and 3 rotating input sets between timed steps.
  e2e       the same steps through the public module API from pinned host buffers: step i + 1's
            inputs travel on a copy stream while step i computes; the per-window ELBO goes back into
            pinned memory and the host reads EVERY step's result one step behind the launches, the
            last one before the clock stops.
  cpu_baseline  the oracle's reference-order restatement of the gpytorch path on the host cores
            (gpytorch itself when it can be imported).  `--impl reference` times that CPU path alone.
  roofline  the dominant kernel, and roofline_per_point_kernel the dominant per-point kernel
            (per-stage CUDA-event times from the library's profile hooks).  "achieved" counts
            ALGORITHMIC bytes or flops; the tensor peak is the TF32 dense rate, 1/2 of the bf16 peak
            (a 3xTF32 kernel issues 3 MMAs per product, so its ceiling is frac = 1/3; M <= 32 runs
            FP32 FFMA, ~74 TFLOP/s).  The once-per-update M x M stages (mm_fwd / mm_bwd / sg_reduce)
            are latency-bound fp64 work with no per-window traffic.  "traffic" is the measured DRAM
            bytes per launch recorded in profiles/ncu_traffic.json for that workload and kernel.
--sweep adds `workloads` (the other BASELINE.json configurations, measured the same way in the same
process) and `next_rows` (the kernels on either side of the GP blur, each beside the torch-eager
sequence it replaces).
--dump-outputs DIR writes, after the timed steps, what the last timed step computed (dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the benchmark writes nothing into the tree it runs from

import torch  # noqa: E402

WORKLOADS = {
    "c1": dict(B=256, calls=[24], D=64, M=32, desc="configs[0]: GPModel blur B=256 L=24 D=64 M=32"),
    "c2": dict(B=256, calls=[192, 24], D=64, M=256,
               desc="configs[1] GP-blur calls of the traffic-shape step: enc [256,192,64] + dec [256,24,64], M=256"),
    "c3": dict(B=1024, calls=[24], D=64, M=128, desc="configs[2]: electricity shape B=1024 L=24 D=64 M=128"),
}
for _m in (64, 128, 256, 512, 1024):
    WORKLOADS[f"c5_m{_m}"] = dict(B=8192, calls=[24], D=64, M=_m,
                                  desc=f"configs[4]: inducing sweep point B=8192 L=24 D=64 M={_m}")
WORKLOADS["c3"]["strong"] = True     # configs[2]: B = 1024 GLOBAL, batch-sharded (128 windows per GPU on 8)
EXTRA_WORKLOADS = ["c1", "c3", "c4", "c5_m64", "c5_m256", "c5_m1024"]
WORKLOADS["c4"] = dict(B=2048, calls=[24], D=64, M=256, H=10,
                       desc="configs[3]: two-layer DeepGP blur B=2048 L=24 D=64 M=256, hidden width H=10 "
                            "(H independent GPs D->H, reparameterised sample, one GP H->1)")
DEFAULT_WORKLOAD = "c2"
METRIC = "gp_blur_fwd_bwd_windows_per_sec"
UNIT = "windows/s"
L2_FLUSH_BYTES = 256 << 20
DUMP_LIMIT_BYTES = 64 << 20
# printed on stderr: the result line on stdout stays short enough to be read back from the end of the output
DETAIL_KEYS = ("roofline", "roofline_per_point_kernel", "stage_ms_per_step", "workloads", "next_rows")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]),
                    bf16_tflops_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


# --------------------------------------------------------------------------------------------------
# algorithmic work model (DESIGN.md section 4; SURVEY 8(d))
# --------------------------------------------------------------------------------------------------
def stage_work(stage: str, N: int, D: int, M: int):
    """(algorithmic bytes, algorithmic flops) of one launch of `stage` over N points."""
    if stage == "point_fwd":
        return N * (4 * D + 12), N * (2 * M * D + M * M)
    if stage == "point_bwd":          # dX is fused into the backward kernel: x and upstream grads in, dx out
        return N * (8 * D + 16), N * (4 * M * D + M * M)
    if stage == "dx":
        return N * 8 * D, 2 * N * M * D
    if stage == "gram":
        return 0, N * M * M
    if stage == "wx":
        return 0, 2 * N * M * D
    if stage == "mm_fwd":
        return 4 * M * D, 2 * M * M * D + M ** 3 // 3 + M ** 3 // 3
    if stage == "mm_bwd":
        return 4 * M * D, 4 * M ** 3
    return 0, 0


def bytes_per_window(L, D):
    return 12 * L * D + 32 * L + 4


# --------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock + throttle reasons DURING the timed region (NVML from a background thread, ~1 ms period;
    falls back to one `nvidia-smi` query)."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = False
        self._thread = None

    def _init(self):
        """NVML set-up (import, nvmlInit, handle: tens of ms) - done by start() BEFORE the timed region, so that only
        the cheap per-sample queries run beside it (initialising inside the sampling thread overlapped the first timed
        steps with driver work and, at 20 steps, left a single sample)."""
        import pynvml
        pynvml.nvmlInit()
        self._nv = pynvml
        self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        self._names = {"hw_slowdown": getattr(pynvml, "nvmlClocksEventReasonHwSlowdown", 0x8),
                       "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                       "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                       "sw_power_cap": getattr(pynvml, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        self._get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")

    def _run(self):
        try:
            while not self._stop:
                self.samples.append(float(self._nv.nvmlDeviceGetClockInfo(self._h, self._nv.NVML_CLOCK_SM)))
                mask = int(self._get_reasons(self._h))
                for nm, bit in self._names.items():
                    if mask & bit:
                        self.reasons.add(nm)
                time.sleep(0.001)
        except Exception:
            pass

    def start(self):
        import threading
        try:
            self._init()
        except Exception:
            return                                   # stop() falls back to one nvidia-smi query
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop = True
        if self._thread is not None:
            self._thread.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if self.samples:
            sm = sorted(self.samples)
            out["sm_mhz"] = sm[len(sm) // 2]
        else:
            try:
                r = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits",
                                    "-i", str(self.index)], capture_output=True, text=True, timeout=10).stdout.split(",")
                out["sm_mhz"], out["sm_max_mhz"] = float(r[0]), float(r[1])
            except Exception:
                pass
        return out


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference's own algorithm on the host cores (oracle restatement; gpytorch is absent)
# --------------------------------------------------------------------------------------------------
def cpu_reference_step_fn(wl, B_cpu, seed=1234):
    from oracle import gp_oracle as O
    D, M = wl["D"], wl["M"]
    if "H" in wl:
        return cpu_reference_step_fn_two_layer(wl, B_cpu, seed)
    p = O.clone_params(O.init_params_exercise(D, M, seed), requires_grad=True)
    calls = []
    for i, L in enumerate(wl["calls"]):
        x, y, gm, gv = O.make_inputs(B_cpu, L, D, seed + 1 + i)
        calls.append((x.requires_grad_(True), y, gm, gv))

    def step():
        for q in p.values():
            q.grad = None
        loss = 0.0
        for i, (x, y, gm, gv) in enumerate(calls):
            x.grad = None
            mean, var = O.svgp_predict_reference_order(p, x)
            loss = loss + (gm * mean).sum()
            if i == len(calls) - 1:
                e = O.elbo_per_window(mean, var, y, O.noise_variance(p), O.kl_meanfield(p), float(D))
                loss = loss - e.mean()
        loss.backward()
        return float(loss.detach())
    return step


def cpu_reference_step_fn_two_layer(wl, B_cpu, seed=1234):
    from oracle import gp_oracle as O
    D, M, H, L = wl["D"], wl["M"], wl["H"], wl["calls"][0]
    p1 = O.clone_params(O.init_params_hidden_layer(D, H, M, seed), requires_grad=True)
    p2 = O.clone_params(O.init_params_exercise(H, M, seed + 1), requires_grad=True)
    x, y, gm, gv = O.make_inputs(B_cpu, L, D, seed + 2)
    x.requires_grad_(True)
    eps = torch.randn(B_cpu, L, H, generator=torch.Generator().manual_seed(seed + 3))

    def step():
        for q in list(p1.values()) + list(p2.values()):
            q.grad = None
        x.grad = None
        mean, var, _ = O.deepgp2_predict(p1, p2, x, eps, closed_form=False)
        kl = O.kl_hidden_layer(p1) + O.kl_meanfield(p2)
        e = O.elbo_per_window(mean, var, y, O.noise_variance(p2), kl, float(D))
        loss = (gm * mean).sum() - e.mean()
        loss.backward()
        return float(loss.detach())
    return step


def gpytorch_step_fn(wl, B_cpu, seed=1234):
    """The reference's OWN classes on real gpytorch (BASELINE.md section 2) - only when gpytorch can be imported and
    the reference tree is installed under baseline/_ref."""
    for extra in (os.path.join(ROOT, "baseline", "_ref"),):
        if os.path.isdir(extra) and extra not in sys.path:
            sys.path.append(extra)
    import gpytorch                                    # noqa: F401  (ImportError -> caller falls back to the port)
    from denoising_model.DeepGP import DeepGPp         # the reference's unmodified module
    if "H" in wl:
        raise ImportError("the reference defines no two-layer model")
    D, M = wl["D"], wl["M"]
    from oracle import gp_oracle as O
    model = DeepGPp(D, seed)
    if M != 256:
        from denoising_model.DeepGP import ToyDeepGPHiddenLayer
        model.hidden_layer = ToyDeepGPHiddenLayer(input_dims=D, output_dims=None, seed=seed, num_inducing=M,
                                                  mean_type="linear")
    calls = [O.make_inputs(B_cpu, L, D, seed + 1 + i) for i, L in enumerate(wl["calls"])]

    def step():
        model.zero_grad(set_to_none=True)
        loss = 0.0
        with gpytorch.settings.num_likelihood_samples(1):
            for i, (x, y, gm, gv) in enumerate(calls):
                x = x.detach().requires_grad_(True)
                mean, dist = model.predict(x)
                loss = loss + (gm * mean[0]).sum()
                if i == len(calls) - 1:
                    mll = gpytorch.mlls.DeepApproximateMLL(gpytorch.mlls.VariationalELBO(model.likelihood, model, D))
                    loss = loss - mll(dist, y.unsqueeze(0)).mean()
        loss.backward()
        return float(loss.detach())
    return step, f"gpytorch {gpytorch.__version__}"


def time_cpu_reference(wl, steps, warmup, budget_s=100.0):
    """Times the reference's CPU implementation of the path on all host cores: `warmup` + `steps` steps on a bounded
    sample B_cpu <= B of the workload, sized from one calibration step so that the whole run fits `budget_s`."""
    torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    kind, impl = "port", (f"oracle reference-order restatement of the gpytorch path (fp32 kernels, fp64 batched "
                          f"Cholesky/solve, autograd backward), torch {torch.__version__} CPU")
    make = cpu_reference_step_fn
    try:
        gpytorch_step_fn(wl, 2)
        make = lambda w, b: gpytorch_step_fn(w, b)[0]      # noqa: E731
        kind, impl = "reference", gpytorch_step_fn(wl, 2)[1] + " (the reference's own DeepGPp) on CPU"
    except Exception as e:                                  # gpytorch / linear_operator are not installable here
        impl += f"; gpytorch unavailable ({type(e).__name__})"
    B = wl["B"]
    B_cpu = os.environ.get("GPBLUR_CPU_SAMPLE_B")
    if B_cpu is None:
        # calibration: one step on a small sample, then the largest B_cpu <= B whose (warmup + steps) steps fit
        b0 = max(2, min(B, 4))
        cal = make(wl, b0)
        cal()
        t0 = time.perf_counter()
        cal()
        per_window = (time.perf_counter() - t0) / b0
        B_cpu = int(max(2, min(B, budget_s / max(per_window * (steps + warmup), 1e-9))))
    B_cpu = int(B_cpu)
    step = make(wl, B_cpu)
    for _ in range(max(0, warmup)):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    full = B_cpu == B
    return dict(value=B_cpu / dt, unit=UNIT, cores=cores, kind=kind, nproc=os.cpu_count(),
                sample=f"{steps} steps (+{warmup} warm-up) of B={B_cpu} windows "
                       f"({'the full workload' if full else 'a bounded sample of the workload, B=' + str(B)}), "
                       f"calls L={wl['calls']}, {impl}"), dt, B_cpu


def run_reference(args, wl, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb, dt, B_cpu = time_cpu_reference(wl, max(1, args.steps), max(0, args.warmup))
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": max(1, args.steps), "warmup": max(0, args.warmup), "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": name, "desc": wl["desc"], "B_per_gpu": wl["B"], "B_cpu_sample": B_cpu, "L": wl["calls"],
                   "D": wl["D"], "M": wl["M"], "regime": "R-exercise (SURVEY 8d)"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def exercise_init(layer, seed):
    """"R-exercise" parameter regime of SURVEY 8(d) for one (possibly multi-output) whitened SVGP layer:
    lengthscales ~ sqrt(D) so that K(x, Z) is O(0.1..1) instead of underflowing, non-trivial q(u)."""
    import math
    vs = layer.variational_strategy
    vd = vs._variational_distribution
    Z = vs.inducing_points
    Dd = Z.shape[-1]
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        Z.copy_(torch.randn(Z.shape, generator=g))
        rl = layer.covar_module.base_kernel.raw_lengthscale
        ell = math.sqrt(Dd) * (0.75 + 0.5 * torch.rand(rl.shape, generator=g))
        rl.copy_(torch.log(torch.expm1(ell)))
        vd.variational_mean.copy_(0.5 * torch.randn(vd.variational_mean.shape, generator=g))
        vd._variational_stddev.copy_(0.5 + torch.rand(vd._variational_stddev.shape, generator=g))
        layer.mean_module.weights.copy_(torch.randn(layer.mean_module.weights.shape, generator=g) / math.sqrt(Dd))
        layer.mean_module.bias.copy_(torch.randn(layer.mean_module.bias.shape, generator=g))
        vs.variational_params_initialized.fill_(1)


def dump_outputs(dirname, outputs, model):
    """Writes what one step hands its caller as DIR/<name>.npy (float32): the per-call mean / sample and dX
    (mean_<c>, sample_<c>, dx_<c>, c = index of the GP call), the per-window ELBO and every parameter gradient
    (grad_<parameter name>).  When together they exceed DUMP_LIMIT_BYTES, every array larger than an equal share
    of the limit is replaced by the same seeded sample of its flattened elements (sorted indices) in every run."""
    import numpy as np
    arrays = dict(outputs)
    arrays.update({"grad_" + n: p.grad for n, p in model.named_parameters() if p.grad is not None})
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    share = DUMP_LIMIT_BYTES // len(arrays)
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES and a.nbytes > share:
            keep = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(keep)]
        np.save(os.path.join(dirname, name + ".npy"), a)


def make_model(wl, device, seed=1234):
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import DeepGPp, DeepGP2
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat
    gpcompat.num_likelihood_samples._set_value(1)       # train.py:20
    if "H" in wl:
        model = DeepGP2(wl["D"], seed, hidden_dims=wl["H"], num_inducing=wl["M"])
        exercise_init(model.hidden_layer, seed)
        exercise_init(model.last_layer, seed + 1)
    else:
        model = DeepGPp(wl["D"], seed, num_inducing=wl["M"])
        exercise_init(model.hidden_layer, seed)
    return model.to(device)


def run_ours(args, wl, name):
    """The result line: --workload in full, plus (with --sweep) a `workloads` dict with the other BASELINE.json
    configurations measured the same way in the same process (c3 strong-scaled: B = 1024 global) and `next_rows`."""
    from fine_grained_gaussian_process_forcasting_b200 import _cabi
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the GP blur path has no CPU fallback); "
                         "use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    _cabi.lib()
    ctx = dict(world=world, rank=rank, local_rank=local_rank, device=device, dist=dist)
    line = measure(args, wl, name, ctx, primary=True)
    if args.sweep:
        extra = {}
        for other in EXTRA_WORKLOADS:
            if other == name:
                continue
            wlo = dict(WORKLOADS[other])
            if wlo.get("strong"):                         # fixed GLOBAL batch: B / world windows per GPU
                wlo["B"] = max(1, wlo["B"] // world)
            sub = measure(args, wlo, other, ctx, primary=False)
            if rank == 0:
                extra[other] = sub
        if rank == 0:
            line["workloads"] = extra
            try:
                line["next_rows"] = measure_next_rows(device, load_peaks())
            except Exception as e:      # the headline line must survive a failure of the side measurements
                line["next_rows"] = {"error": repr(e)}
    if rank == 0:
        detail = {k: line.pop(k) for k in DETAIL_KEYS if k in line}
        print(json.dumps(detail), file=sys.stderr, flush=True)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def measure(args, wl, name, ctx, primary=True):
    from fine_grained_gaussian_process_forcasting_b200 import _cabi
    from fine_grained_gaussian_process_forcasting_b200.distributed import FlatGradBucket, gp_parameters
    world, rank, local_rank, device, dist = ctx["world"], ctx["rank"], ctx["local_rank"], ctx["device"], ctx["dist"]

    B, D, M, calls = wl["B"], wl["D"], wl["M"], wl["calls"]
    model = make_model(wl, device)
    model.train()
    bucket = FlatGradBucket(gp_parameters(model), module=model)
    peer_allreduce = bucket.enable_peer_allreduce() if (world > 1 and args.peer_allreduce) else False
    g = torch.Generator(device=device).manual_seed(1234 + rank)
    nbuf = 3   # rotate inputs; an L2 flush is also issued between timed steps
    # the activations of a step sit back to back in one buffer (what a caller that wants ONE fused GP evaluation per
    # step provides, see DeepGPp.blur_segments); xs[k][c] are the per-call [B, L, D] views
    def seg_views(flat):
        out, o = [], 0
        for L in calls:
            out.append(flat[o:o + B * L].view(B, L, D))
            o += B * L
        return out
    xflat = [torch.randn(B * sum(calls), D, device=device, generator=g) for _ in range(nbuf)]
    xs = [seg_views(f) for f in xflat]
    fused = bool(args.fuse_calls and len(calls) > 1 and hasattr(model, "blur_segments"))
    ys = [torch.randn(1, B, calls[-1], device=device, generator=g) for _ in range(nbuf)]
    gms = [torch.randn(1, B, L, device=device, generator=g) for L in calls]
    gss = [torch.randn(1, B, L, device=device, generator=g) for L in calls]
    g_elbo = torch.full((1, B), -1.0 / B, device=device)
    xh = [[x.cpu().pin_memory() for x in xs[0]]]
    yh = ys[0].cpu().pin_memory()
    elbo_h = torch.empty(1, B).pin_memory()
    flush = torch.empty(L2_FLUSH_BYTES // 4, device=device)
    from fine_grained_gaussian_process_forcasting_b200.gpcompat import DeepGPLayer
    from fine_grained_gaussian_process_forcasting_b200.graphs import GraphedStep
    layers = [m for m in model.modules() if isinstance(m, DeepGPLayer)]

    # The GP calls of one step are independent given the shared parameter stage; the small decoder-side call only
    # fills a third of the SMs, so it is issued on a second stream and runs in the tail of the encoder-side kernels
    # (autograd replays each call's backward on the stream of its forward).
    from fine_grained_gaussian_process_forcasting_b200.graphs import CallStreams
    call_streams = CallStreams(device, len(calls)) if (args.call_streams and len(calls) > 1 and not fused) else None

    def step_body(xin, yin):
        """forward (mean, variance, fused sample, ELBO) + backward (dX, every GP parameter gradient); returns what
        the caller receives besides the parameter gradients, by name (dump_outputs), the ELBO under "elbo"."""
        bucket.zero()
        outs, grads = [], []
        res = {}
        if fused:
            # ONE fused evaluation for all the activations of the step (one launch per kernel, one leaf for dX)
            from fine_grained_gaussian_process_forcasting_b200 import ops as _ops
            xf = _ops.as_one_buffer(list(xin)).detach().requires_grad_(True)
            segs = model.blur_segments(xf, [(B, L) for L in calls], yin, num_data=D)
            for c, o in enumerate(segs):
                outs += [o.mean, o.sample]
                grads += [gms[c], gss[c]]
                res[f"mean_{c}"], res[f"sample_{c}"] = o.mean, o.sample
            res["elbo"] = segs[-1].elbo
            outs.append(res["elbo"])
            grads.append(g_elbo)
            torch.autograd.backward(outs, grads)
            if world > 1 and allreduce_in_step[0]:
                bucket.all_reduce(average=True)
            res.update((f"dx_{c}", g_) for c, g_ in enumerate(seg_views(xf.grad)))
            return res
        if call_streams is not None:
            for ly in layers:                             # the shared stage is built once, on the main stream
                ly._kl_only()
        leaves = []
        for c, L in enumerate(calls):
            x = xin[c].detach().requires_grad_(True)      # fresh leaf: dX flows back to the forecaster
            leaves.append(x)
            last = c == len(calls) - 1
            fn = (lambda x=x, last=last: model.blur(x, yin if last else None, num_data=D))
            out = call_streams.run(c, fn) if call_streams is not None else fn()
            outs += [out.mean, out.sample]
            grads += [gms[c], gss[c]]
            res[f"mean_{c}"], res[f"sample_{c}"] = out.mean, out.sample
            if last:
                res["elbo"] = out.elbo
                outs.append(out.elbo)
                grads.append(g_elbo)
        if call_streams is not None:
            call_streams.join()
        torch.autograd.backward(outs, grads)
        if call_streams is not None:
            call_streams.join()
        if world > 1 and allreduce_in_step[0]:
            bucket.all_reduce(average=True)               # NCCL AVG on the flat bucket: part of the captured step
        res.update((f"dx_{c}", x.grad) for c, x in enumerate(leaves))
        return res

    allreduce_in_step = [not args.allreduce_after_replay]

    def eager_step(i, xin, yin):
        for ly in layers:               # a real training step changes the parameters: recompute Kzz / Cholesky once
            ly.invalidate_param_stage()
            # Philox counters by GLOBAL point index (and, for the H GPs of a multi-output layer, a stride of the global
            # point count between them): the samples do not depend on the number of ranks
            H_ = max(1, ly.output_dims or 1)
            total = world * B * sum(calls)
            ly._rng_offset = i * total * H_ + rank * B * sum(calls)
            ly._rng_h_stride = total if H_ > 1 else None
        return step_body(xin, yin)

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- warm-up (eager) ----
    launches0 = _cabi.launch_count()
    eager_step(0, xs[0], ys[0])
    launches_per_step = _cabi.launch_count() - launches0
    for i in range(1, max(3, args.warmup)):
        eager_step(i, xs[i % nbuf], ys[i % nbuf])
    sync_all()

    # ---- the step as ONE CUDA graph (graphs.GraphedStep): static inputs, device-resident Philox offsets ----
    graphed = None
    graph_note = "eager launches (--eager)"
    if not args.eager:
        for attempt in (0, 1):
            try:
                if fused:     # static inputs: the flat activation buffer + targets
                    graphed = GraphedStep(model, lambda xf, y: (step_body(seg_views(xf), y),), [xflat[0], ys[0]],
                                          warmup=2, world=world, rank=rank)
                else:
                    graphed = GraphedStep(model, lambda *ins: (step_body(ins[:-1], ins[-1]),), list(xs[0]) + [ys[0]],
                                          warmup=2, world=world, rank=rank)
                graph_note = "whole step (fwd + bwd" + (" + NCCL all-reduce of the gradient bucket" if world > 1 and
                             allreduce_in_step[0] else "") + ") replayed as one CUDA graph" + \
                             ("; NCCL all-reduce issued after the replay" if world > 1 and not allreduce_in_step[0] else "")
                break
            except Exception as e:    # pragma: no cover - report and fall back
                graphed = None
                for ly in layers:
                    ly.rng_offset_dev = None
                if world > 1 and allreduce_in_step[0] and attempt == 0:
                    allreduce_in_step[0] = False         # retry with the collective outside the graph
                    continue
                graph_note = f"CUDA graph capture failed ({type(e).__name__}: {e}); eager launches"
                break
    sync_all()
    g_inputs = None
    if graphed is not None:       # the graph's static inputs as [x per call ..., y]
        g_inputs = (seg_views(graphed.inputs[0]) + [graphed.inputs[1]]) if fused else list(graphed.inputs)

    def run_step(i, xin, yin):
        """one step on inputs already in HBM; returns the per-window ELBO"""
        if graphed is None:
            return eager_step(i, xin, yin)["elbo"]
        for dst, src in zip(g_inputs, list(xin) + [yin]):
            if dst.data_ptr() != src.data_ptr():
                dst.copy_(src, non_blocking=True)
        (res,) = graphed.replay()
        if world > 1 and not allreduce_in_step[0]:
            bucket.all_reduce(average=True)
        return res["elbo"]

    for i in range(3):
        run_step(i, xs[i % nbuf], ys[i % nbuf])
    sync_all()

    # ---- timed region 1: inputs resident in HBM ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sync_all()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        if graphed is not None:                         # stage this step's inputs in the graph's static buffers
            for dst, src in zip(g_inputs, list(xs[i % nbuf]) + [ys[i % nbuf]]):
                dst.copy_(src, non_blocking=True)
        flush.zero_()                                   # L2 flush between timed iterations (outside the events)
        evs[i][0].record()
        if graphed is not None:
            (last,) = graphed.replay()
            if world > 1 and not allreduce_in_step[0]:
                bucket.all_reduce(average=True)
        else:
            last = eager_step(i, xs[i % nbuf], ys[i % nbuf])
        evs[i][1].record()
    sync_all()
    t_wall = time.perf_counter() - t_wall0
    launches = launches_per_step * args.steps
    ms_dev = sum(a.elapsed_time(b) for a, b in evs)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms_dev], device=device, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and primary and rank == 0:     # before anything below runs the step again
        dump_outputs(args.dump_outputs, last, model)

    # ---- timed region 2: end to end through the module API with host buffers ----
    if graphed is not None:
        xdev, ydev = g_inputs[:-1], g_inputs[-1]
    else:
        xdev = seg_views(torch.empty_like(xflat[0]))
        ydev = torch.empty_like(ys[0])
    # Every step's inputs start in PINNED HOST memory and its result is read on the host; all copies are inside the
    # timed region.  Like any training input pipeline, the host->device copy of step i + 1 is issued on a copy stream
    # before the host waits for step i (double-buffered device staging), so it overlaps step i's kernels.
    cur = torch.cuda.current_stream(device)
    copy_stream = torch.cuda.Stream(device=device)
    stage_x = [[torch.empty_like(x) for x in xs[0]] for _ in range(2)]
    stage_y = [torch.empty_like(ys[0]) for _ in range(2)]
    h2d_done = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def issue_h2d(k):
        copy_stream.wait_event(consumed[k])              # the staging buffers were read by an earlier step
        with torch.cuda.stream(copy_stream):
            for c in range(len(calls)):
                stage_x[k][c].copy_(xh[0][c], non_blocking=True)
            stage_y[k].copy_(yh, non_blocking=True)
            h2d_done[k].record(copy_stream)

    def e2e_step(i):
        k = i & 1
        cur.wait_event(h2d_done[k])
        for c in range(len(calls)):                      # device-side hand-over into the step's input buffers
            xdev[c].copy_(stage_x[k][c], non_blocking=True)
        ydev.copy_(stage_y[k], non_blocking=True)
        consumed[k].record(cur)
        elbo = run_step(i, xdev, ydev)
        elbo_hh[k].copy_(elbo.detach(), non_blocking=True)
        result_ready[k].record(cur)

    # The host reads EVERY step's result (the per-window ELBO) inside the timed region, one step behind the launches:
    # while step i runs it waits for and reads step i - 1 (double-buffered pinned result), as an asynchronous training
    # loop does for its loss - the device never idles waiting for the host to come back from a synchronize.
    elbo_hh = [elbo_h, torch.empty_like(elbo_h).pin_memory()]
    result_ready = [torch.cuda.Event(), torch.cuda.Event()]
    host_acc = [0.0]
    for k in range(2):
        consumed[k].record(cur)
    issue_h2d(0)                                         # untimed warm-up of the pinned-copy path
    e2e_step(0)
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    issue_h2d(0)
    for i in range(args.steps):
        if i + 1 < args.steps:
            issue_h2d((i + 1) & 1)                       # next step's inputs travel while this step computes
        e2e_step(i)
        if i > 0:
            result_ready[(i - 1) & 1].synchronize()      # the caller reads step i - 1's result on the host
            host_acc[0] += float(elbo_hh[(i - 1) & 1][0, 0])
    result_ready[(args.steps - 1) & 1].synchronize()
    host_acc[0] += float(elbo_hh[(args.steps - 1) & 1][0, 0])
    e1.record()
    sync_all()
    t2 = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / (float(t2.item()) * 1e-3)
    h2d = sum(x.numel() for x in xh[0]) * 4 + yh.numel() * 4
    d2h = elbo_h.numel() * 4

    # ---- eager timing for comparison (host-issue bound on the small shapes) ----
    ev_e = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    for ly in layers:
        ly.rng_offset_dev = None
    sync_all()
    n_e = max(3, min(args.steps, 10))
    for i in range(3):                                   # the caching allocator re-grows outside the graph pool
        eager_step(i, xs[i % nbuf], ys[i % nbuf])
    sync_all()
    ev_e[0].record()
    for i in range(n_e):
        eager_step(i, xs[i % nbuf], ys[i % nbuf])
    ev_e[1].record()
    sync_all()
    eager_ms = ev_e[0].elapsed_time(ev_e[1]) / n_e

    # ---- per-stage device times (library profile hooks: CUDA events on the launching stream) ----
    stage_ms = {}
    if rank == 0 or True:
        _cabi.profile_enable(True)
        nprof = max(3, min(args.steps, 10))
        for i in range(nprof):
            flush.zero_()
            eager_step(i, xs[i % nbuf], ys[i % nbuf])
        torch.cuda.synchronize()
        prof = _cabi.profile_collect()
        _cabi.profile_enable(False)
        stage_ms = {k: (ms / nprof, cnt / nprof) for k, (ms, cnt) in prof.items() if cnt}
    sync_all()

    # ---- --check (N > 1): the all-reduced gradient bucket against ONE rank's run on the concatenated batch ----
    allreduce_check = None
    if args.check and world > 1:
        zs = [torch.zeros_like(g_) for g_ in gss]          # no sample gradient: the counters of a window depend on its rank
        saved = list(gss)
        gss[:] = zs
        eager_step(0, xs[0], ys[0])                         # sharded: bucket = mean over ranks (all-reduce in the step)
        if not allreduce_in_step[0]:
            bucket.all_reduce(average=True)
        sharded = bucket.flat.clone()
        gx = [[torch.empty_like(x) for _ in range(world)] for x in xs[0]]
        for c in range(len(calls)):
            dist.all_gather(gx[c], xs[0][c])
        gy = [torch.empty_like(ys[0]) for _ in range(world)]
        dist.all_gather(gy, ys[0])
        ggm = [[torch.empty_like(g_) for _ in range(world)] for g_ in gms]
        for c in range(len(calls)):
            dist.all_gather(ggm[c], gms[c])
        if rank == 0:
            keep = (list(gms), g_elbo)
            xin = [torch.cat(gx[c], 0) for c in range(len(calls))]
            yin = torch.cat(gy, 1)
            gms[:] = [torch.cat(ggm[c], 1) / world for c in range(len(calls))]
            gss[:] = [torch.zeros_like(g_) for g_ in gms]
            g_elbo_full = torch.full((1, B * world), -1.0 / (B * world), device=device)
            was = allreduce_in_step[0]
            allreduce_in_step[0] = False
            for ly in layers:
                ly.invalidate_param_stage()
                ly._rng_offset, ly._rng_h_stride = 0, None      # step 0 on the concatenated batch: the same counters
            bucket.zero()
            outs, grads = [], []
            for c, L_ in enumerate(calls):
                x = xin[c].detach().requires_grad_(True)
                last = c == len(calls) - 1
                out = model.blur(x, yin if last else None, num_data=D)
                outs += [out.mean, out.sample]
                grads += [gms[c], gss[c]]
                if last:
                    outs.append(out.elbo)
                    grads.append(g_elbo_full)
            bucket.zero()
            torch.autograd.backward(outs, grads)
            full = bucket.flat.clone()
            allreduce_in_step[0] = was
            gms[:] = keep[0]
            allreduce_check = float(((sharded - full).abs().max() / full.abs().max().clamp_min(1e-30)).item())
        gss[:] = saved
        sync_all()

    if rank == 0:
        peaks = load_peaks()
        N_total = B * sum(calls)
        # dominant kernel and its roofline; the once-per-update M x M kernels (mm_fwd / mm_bwd / sg_reduce) are
        # latency-bound fp64 work with no per-window traffic, so the dominant PER-POINT kernel is reported too
        dom = max(stage_ms.items(), key=lambda kv: kv[1][0])[0] if stage_ms else None
        point_stages = {k: v for k, v in stage_ms.items() if k in ("point_fwd", "point_bwd", "dx", "gram", "wx")}
        dom_point = max(point_stages.items(), key=lambda kv: kv[1][0])[0] if point_stages else None
        roofs = {}
        for which, dom in (("roofline", dom), ("roofline_per_point_kernel", dom_point)):
          roof = None
          if dom is not None:
              ms_dom, launches_dom = stage_ms[dom]
              per_launch_s = ms_dom * 1e-3 / max(launches_dom, 1)
              n_per_launch = N_total / max(launches_dom, 1)
              if "H" in wl:                       # two-layer stack: H + 1 launches per stage, each over all N points
                  n_per_launch = N_total          # (work model uses the layer-1 dims D, M: H of the H + 1 launches)
              by, fl = stage_work(dom, int(n_per_launch), D, M)
              tf32_peak = peaks["bf16_tflops"] / 2.0
              intensity = fl / max(by, 1)
              if by > 0 and intensity < tf32_peak * 1e12 / (peaks["hbm_gbs"] * 1e9):
                  roof = {"bound": "hbm", "achieved": by / per_launch_s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s"}
              else:
                  roof = {"bound": "tensor", "achieved": fl / per_launch_s / 1e12, "peak": tf32_peak, "unit": "TFLOP/s"}
              roof["frac"] = roof["achieved"] / roof["peak"]
              if roof["bound"] == "tensor" and M > 32 and dom in point_stages:
                  roof["frac_of_3xtf32_ceiling"] = 3.0 * roof["frac"]
              if M <= 32 and dom in point_stages:     # FP32-FFMA path: CUDA-core bound long before HBM
                  roof["ffma_tflops_achieved"] = fl / per_launch_s / 1e12
                  roof["ffma_frac_of_74_tflops"] = roof["ffma_tflops_achieved"] / 74.0
              # measured DRAM traffic of that kernel (ncu --set full capture of this same command, per launch)
              roof["traffic"] = None
              try:
                  tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
                  ent = tj.get(name, {}).get(dom)
                  if ent:
                      roof["traffic"] = ent["bytes_per_launch"]
              except Exception:
                  pass
              roof["algorithmic_bytes_per_launch"] = by
              roof["algorithmic_flops_per_launch"] = fl
              roof["kernel"] = dom
              roof["kernel_ms_per_launch"] = per_launch_s * 1e3
              roof["peak_source"] = peaks["source"]
              roof["hbm_frac_whole_step"] = (B * sum(bytes_per_window(L, D) for L in calls) / (ms_per_step * 1e-3) / 1e9
                                             / peaks["hbm_gbs"])
          roofs[which] = roof
        cb = None if (args.no_cpu_baseline or not primary) else time_cpu_reference(wl, 3, 1, budget_s=20.0)[0]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if wl.get("strong") else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": name, "B_per_gpu": B, "B_global": B * world, "L": calls, "D": D, "M": M,
                       "parallelism": f"dp{world}",
                       "launch": graph_note,
                       "call_streams": call_streams is not None,
                       "calls_fused": fused,
                       "allreduce": (None if world == 1 else "one-shot kernel over NVLink peer memory (CUDA IPC), rank-ordered sum"
                                     if peer_allreduce else "NCCL all-reduce (AVG)"),
                       "regime": "R-exercise (SURVEY 8d)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofs.get("roofline"),
            "roofline_per_point_kernel": roofs.get("roofline_per_point_kernel"),
            "cpu_baseline": cb,
            "stage_ms_per_step": {k: round(v[0], 5) for k, v in stage_ms.items()},
            "wall_ms_per_step": t_wall * 1e3 / args.steps,
            "eager_ms_per_step": eager_ms,
        }
        if allreduce_check is not None:
            line["allreduce_check"] = allreduce_check
            line["allreduce_check_note"] = ("max |mean over ranks of the per-rank gradient buckets - bucket of ONE rank on "
                                            "the concatenated batch| / max |.| (sample gradients off: the Philox "
                                            "counters of a window depend on its rank's offset)")
        return line
    return None


# --------------------------------------------------------------------------------------------------
# SURVEY 8(f) rows on either side of the GP blur: each kernel timed alone (CUDA events per launch on the launching
# stream, L2 flushed between launches, median), ALGORITHMIC bytes / time against the measured HBM peak, and the same
# operation done the reference's way beside it (torch eager ops on the same GPU = the library baseline; host pandas
# slicing for the sampler)
# --------------------------------------------------------------------------------------------------
def measure_next_rows(device, peaks, reps=12):
    import numpy as np
    from fine_grained_gaussian_process_forcasting_b200 import ATA as ata_mod
    from fine_grained_gaussian_process_forcasting_b200 import base_train as bt
    from fine_grained_gaussian_process_forcasting_b200 import step_ops
    flush = torch.empty(L2_FLUSH_BYTES // 4, device=device)

    def timed(fn):
        # launches replayed from a CUDA graph (as the GP step is): the interval holds the kernels, not Python
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            for _ in range(3):
                fn()
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            fn()
        ts = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graph.replay()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        del graph
        return float(np.median(ts))

    def row(t, by, **kw):
        d = {"ms": t * 1e3, "algorithmic_bytes": int(by), "achieved_gbs": by / t / 1e9,
             "hbm_frac": by / t / 1e9 / peaks["hbm_gbs"]}
        d.update(kw)
        return d

    out = {"timing": "each operation captured once and replayed as a CUDA graph; CUDA events per replay, median of %d, "
                     "%d MiB L2 flush before every replay" % (reps, L2_FLUSH_BYTES >> 20)}
    g = torch.Generator(device=device).manual_seed(99)
    # ---- rank 4: window gather, traffic shape (time_steps 240 = 192 + 24 + 24, F = 4), one epoch of 256-window batches
    rows, F, T, ne, pl = 1 << 20, 4, 240, 192, 24
    rs = np.random.RandomState(3)
    nwin = 65536
    ws = bt.WindowSet(rs.randn(rows, F).astype(np.float32), rs.randn(rows).astype(np.float32),
                      rs.randint(0, rows - T, size=nwin).astype(np.int64), T, ne, pl, device=device)
    per_win = ((T - pl) * F + pl) * 4 * 2                     # every gathered float is read once and written once
    t_epoch = timed(lambda: ws.gather(0, nwin))
    t_batch = timed(lambda: ws.gather(0, 256))
    t0 = time.perf_counter()                                  # the reference's way: one slice + copy per window on the host
    nh = 2048
    enc = np.zeros((nh, ne, F)); dec = np.zeros((nh, T - ne - pl, F)); yy = np.zeros((nh, pl, 1))
    for i, st in enumerate(ws.starts_host[:nh]):
        enc[i] = ws.table_host[st:st + ne]; dec[i] = ws.table_host[st + ne:st + T - pl]; yy[i, :, 0] = ws.target_host[st + T - pl:st + T]
    t_host = (time.perf_counter() - t0) / nh
    out["window_gather"] = row(t_epoch, per_win * nwin, windows=nwin, windows_per_s=nwin / t_epoch,
                               batch256_us=t_batch * 1e6,
                               host_numpy_windows_per_s=1.0 / t_host,
                               note="host figure: numpy slice + copy per window (the reference slices a pandas frame "
                                    "per window, slower still) and excludes its per-batch .to(device)")
    # ---- rank 1: blur application x + proj_up(mean), c2 shape
    N, D = 256 * (192 + 24), 64
    x = torch.randn(N, D, device=device, generator=g, requires_grad=True)
    mean = torch.randn(N, device=device, generator=g, requires_grad=True)
    up = torch.nn.Linear(1, D).to(device)
    go = torch.randn(N, D, device=device, generator=g)

    def fused_blur():
        o = step_ops.blur_apply(x, mean, up.weight, up.bias)
        torch.autograd.grad(o, (x, mean, up.weight, up.bias), go)

    def eager_blur():
        o = x + up(mean.unsqueeze(-1))
        torch.autograd.grad(o, (x, mean, up.weight, up.bias), go)

    by = N * D * 4 * 3 + N * 4 * 3                           # fwd: x in, out; bwd: g_out in (+ mean in / g_mean out)
    out["blur_apply_fwd_bwd"] = row(timed(fused_blur), by, torch_eager_ms=timed(eager_blur) * 1e3)
    # ---- rank 2: loss assembly (final projection + MSE + clipped-lambda ELBO term), decoder states of configs[1] and
    # the same at 32 x the batch (the c2 shape is one launch latency: 6 144 rows)
    for tag, Bl in (("loss_assembly_fwd_bwd", 256), ("loss_assembly_fwd_bwd_B8192", 8192)):
        P = 24
        hdec = torch.randn(Bl, 48, D, device=device, generator=g, requires_grad=True)
        yt = torch.randn(Bl, P, 1, device=device, generator=g)
        elbo = torch.randn(Bl, device=device, generator=g, requires_grad=True)
        lam = torch.full((1,), 0.003, device=device, requires_grad=True)
        fin = torch.nn.Linear(D, 1).to(device)

        def fused_loss():
            f, loss, mse = step_ops.forecast_loss(fin, hdec[:, -P:, :], yt, elbo, lam)
            torch.autograd.grad(loss, (hdec, fin.weight, fin.bias, elbo, lam))

        def eager_loss():                                      # forecast_denoising.py:84, 87-89, 102-104
            f = fin(hdec[:, -P:, :])
            mll_error = -elbo.mean()
            mse = torch.nn.functional.mse_loss(yt, f)
            loss = mse + torch.clip(lam, min=0, max=0.005) * mll_error
            torch.autograd.grad(loss, (hdec, fin.weight, fin.bias, elbo, lam))

        by = Bl * P * D * 4 * 3                                # h read forward and backward, g_h written
        out[tag] = row(timed(fused_loss), by, torch_eager_ms=timed(eager_loss) * 1e3, rows=Bl * P)
    # ---- rank 3: ATA core, encoder self-attention of configs[1] (b = 256, 8 heads, l = l_k = 192, d_k = d_v = 4)
    b, h, l, dk = 256, 8, 192, 4
    qp = torch.relu(torch.randn(b, h, l, 4 * dk, device=device, generator=g)).requires_grad_(True)
    kp = torch.relu(torch.randn(b, h, l, 4 * dk, device=device, generator=g)).requires_grad_(True)
    v = torch.randn(b, l, h, dk, device=device, generator=g).transpose(1, 2).requires_grad_(True)
    gc = torch.randn(b, h, l, dk, device=device, generator=g)

    def fused_ata():
        c = ata_mod.ata_core(qp, kp, v, dk)[0]
        torch.autograd.grad(c, (qp, kp, v), gc)

    def eager_ata():                                          # ATA.py:56-65 verbatim
        Q, _ = torch.topk(qp, dim=-1, k=1)
        K, _ = torch.topk(kp, dim=-1, k=1)
        scores = torch.einsum('bhqd,bhkd->bhqk', Q, K) / np.sqrt(dk)
        attn = torch.softmax(scores, -1)
        c = torch.einsum('bhqk,bhkd->bhqd', attn, v)
        torch.autograd.grad(c, (qp, kp, v), gc)

    by = (2 * b * h * l * 4 * dk * 2 + b * h * l * dk * 4) * 4    # q_proj, k_proj in + their gradients out; V, ctx, g_ctx, g_V
    out["ata_core_fwd_bwd"] = row(timed(fused_ata), by, torch_eager_ms=timed(eager_ata) * 1e3,
                                  attn_bytes_never_materialised=b * h * l * l * 4,
                                  note="exp / FMA bound on the CUDA cores (2 x b h l l_k exp per step), not HBM bound")
    # the whole head as its caller uses it (multi_head_attention.py:49-51: a NEW module per forward): wall clock per
    # call incl. the host side, fresh construction + the reference's op sequence vs ATA.cached + the fused core
    q_s = torch.randn(b, l, h, dk, device=device, generator=g).transpose(1, 2).requires_grad_(True)

    def head_reference_style():
        head = ata_mod.ATA(d_k=dk, device=device, h=h, seed=1234)
        Qr, Kr = q_s.reshape(b, -1, l), q_s.reshape(b, -1, l)
        Q_l = [head.conv_list_q[i](Qr) for i in range(4)]
        K_l = [head.conv_list_k[i](Kr) for i in range(4)]
        Q_p = torch.cat(Q_l, dim=0).reshape(b, h, l * 4, -1).reshape(b, h, l, -1)
        K_p = torch.cat(K_l, dim=0).reshape(b, h, l * 4, -1).reshape(b, h, l, -1)
        Q, _ = torch.topk(Q_p, dim=-1, k=1)
        K, _ = torch.topk(K_p, dim=-1, k=1)
        attn = torch.softmax(torch.einsum('bhqd,bhkd->bhqk', Q, K) / np.sqrt(dk), -1)
        c = torch.einsum('bhqk,bhkd->bhqd', attn, q_s)
        torch.autograd.grad(c, (q_s,), gc)

    def head_ours():
        c, _ = ata_mod.ATA.cached(d_k=dk, device=device, h=h, seed=1234)(Q=q_s, K=q_s, V=q_s)
        torch.autograd.grad(c, (q_s,), gc)

    def wall(fn, n=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize(device)
        return (time.perf_counter() - t0) / n

    out["ata_head_fwd_bwd_wall"] = {"ms": wall(head_ours) * 1e3, "reference_style_ms": wall(head_reference_style) * 1e3,
                                    "shape": "b=256 h=8 l=192 d_k=4 (d_model 32), self-attention",
                                    "note": "convolutions / batch norm are cuDNN calls in both columns"}
    return out



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default=os.environ.get("GPBLUR_WORKLOAD", DEFAULT_WORKLOAD), choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the host-CPU leg (profiling runs)")
    ap.add_argument("--no-call-streams", dest="call_streams", action="store_false",
                    help="issue the GP calls of a step on one stream (default: one extra stream per additional call)")
    ap.add_argument("--peer-allreduce", dest="peer_allreduce", action="store_true",
                    help="N > 1: the library's one-shot all-reduce over NVLink peer memory instead of NCCL (measured: "
                         "equal at 2 GPUs, slower than NCCL's in-switch reduction at 8)")
    ap.add_argument("--allreduce-after-replay", action="store_true",
                    help="N > 1: issue the NCCL all-reduce after the graph replay instead of capturing it in the step")
    ap.add_argument("--no-fuse-calls", dest="fuse_calls", action="store_false",
                    help="evaluate the GP once per activation (blur) instead of once per step (blur_segments)")
    ap.add_argument("--eager", action="store_true", help="launch every kernel from Python instead of replaying the "
                    "step as a CUDA graph")
    ap.add_argument("--sweep", action="store_true", help="also measure the other BASELINE.json workloads (`workloads`) "
                    "and the kernels on either side of the GP blur (`next_rows`)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step "
                    "computed as DIR/<name>.npy (float32, at most 64 MiB in all)")
    ap.add_argument("--check", action="store_true", help="N > 1: verify the all-reduced gradient bucket against a "
                    "single-rank run on the concatenated batch (adds `allreduce_check` to the line)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl, args.workload)
    else:
        run_ours(args, wl, args.workload)


if __name__ == "__main__":
    main()
