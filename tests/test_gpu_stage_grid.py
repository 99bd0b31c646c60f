"""The M x M stage (mm_forward_kernel / mm_backward_kernel, M > 32) at every grid size its launchers can pick.

These are the only multi-CTA kernels whose division of work depends on gridDim.x G: the Kzz tiles of phase 1 are
strided over G - 1 CTAs, the look-ahead Cholesky of phase 2 has G - 1 workers looping over each step's items, phase 4
splits the TF32 operand images into `parts` that follow G, and every product phase of the backward strides over G.
Every output element is written by exactly one CTA with arithmetic that does not depend on G, and the cross-tile sums
are added in a fixed order, so the stage and its gradient bucket are bit-identical for every G.  This file holds that:

* `stage_grid` restates launch_mm_forward / launch_mm_backward (csrc/gpblur_mm.cu) and the phase quantities that
  depend on G; `critical_grids` picks, per Mp class, the grids where the work division changes (CPU tests).
* The sweep builds the stage and runs the point calls and the stage backward at every critical grid, checks from the
  profiler trace that each launch got the grid the mirror predicts, and requires torch.equal with a run at the
  default grid; once per cell the run at G = 8 is compared with the float64 oracle.
* Multi-output layers as they run in production (H stages on side streams, grid bounded by ops._stage_cta_cap)
  against H single-output evaluations at the default grid, bit for bit.
* The Cholesky failure report: a NaN in inducing point k gives info = k + 1 at any grid and in the M <= 32 kernel.

Not covered here: GPBLUR_MM_COOP=0 (plain launch + counter barrier), whose grid barrier needs every CTA resident at
once, which a plain launch does not guarantee on a shared GPU; the peer all-reduce (several GPUs); the grids of the
point kernels (test_gpu_dispatch_matrix and the tile-position tests).
"""
import json
import time

import pytest
import torch

from oracle import gp_oracle as O
from test_gpu_dispatch_matrix import (KIND_ID, NAMES, _inputs, _stage_fp64, kernel_id, oracle, padded_d, padded_m,
                                      rel)

TB = 32                 # block size of the blocked factorisation
CTA_LIMIT = 148         # launchers: at most 148 CTAs
MIN_CTAS = 8            # launchers: at least 8 CTAs
K_THREADS = 256
B200_SMS = 148


# ---------------------------------------------------------------------------------------------------------------------
# Grid mirror
# ---------------------------------------------------------------------------------------------------------------------
def tc_bw(MP):
    return 256 if MP >= 256 else MP


def tc_bq(MP):
    return 128 if MP >= 128 else MP


def image_counts(MP):
    """(n_fwd, n_bwd): TF32 images of Linv (forward point kernel) and of (diag(c) Linv)^T (backward), phase 4."""
    if MP < 128:
        return 0, 0
    nsl = MP // 32
    BW, BT = tc_bw(MP), tc_bq(MP)
    NP, spb, NPT, spt = MP // BW, BW // 32, MP // BT, BT // 32
    return spb * NP * (NP + 1) // 2, NPT * nsl - spt * NPT * (NPT - 1) // 2


def half_tiles(MP):
    """mm_backward_kernel<16, .> (16-row items) while 2 nb^2 <= 296, else <32, .>."""
    nb = MP // TB
    return 2 * nb * nb <= 2 * CTA_LIMIT


def stage_grid(direction, M, D, max_ctas, sms=B200_SMS):
    """Grid of mm_forward_kernel ("fwd") / mm_backward_kernel ("bwd") for `max_ctas` (0: unbounded); 1 for the one-CTA
    kernels of M <= 32.  coop_grid caps the grid at occupancy x SMs: both kernels fit at least one CTA per SM, so the
    cap is taken as `sms`, which is exact whenever the GPU has >= 148 SMs."""
    MP, DP = padded_m(M), padded_d(D)
    nb = MP // TB
    if nb == 1:
        return 1
    if direction == "fwd":
        n_fwd, n_bwd = image_counts(MP)
        want = nb * nb + nb + 3 * (n_fwd + n_bwd)
        if max_ctas > 0 and want > max_ctas:
            want = max_ctas
        want = max(want, MIN_CTAS)
    elif direction == "bwd":
        want = (2 if half_tiles(MP) else 1) * nb * nb
        want = max(want, -(-MP * DP // K_THREADS))
        if max_ctas > 0 and want > max_ctas:
            want = max(max_ctas, MIN_CTAS)
    else:
        raise ValueError(direction)
    return min(want, CTA_LIMIT, sms)


def n_items(MP, kb):
    """Worker items of step kb of the forward's phase 2 (trailing tiles but CTA 0's + inverse partial sums)."""
    nb = MP // TB
    nrb = nb - kb - 1
    if nrb == 0:
        return kb
    ntr = nrb * (nrb + 1) // 2
    return ntr - 1 + nrb * (kb + 1)


def n_workers(G):
    return G - 1


def phase4_units(MP):
    """(n_tiles, n_beta, n_fwd, n_bwd) of the forward's phase 4."""
    nb = MP // TB
    return (nb * nb, MP // 32) + image_counts(MP)


def parts(MP, G):
    n_tiles, n_beta, n_fwd, n_bwd = phase4_units(MP)
    if n_fwd + n_bwd == 0:
        return 1
    p = int((G - n_tiles - n_beta) / (n_fwd + n_bwd))      # C division: truncates toward zero
    return min(max(p, 1), 8)


def bwd_items(MP):
    """Items of the backward's product phases: NH row parts of each of the nb^2 tiles."""
    nb = MP // TB
    return (2 if half_tiles(MP) else 1) * nb * nb


def stage_cta_cap(H, sms=B200_SMS):
    """ops._stage_cta_cap: the grid bound of each stage of a multi-output layer."""
    return 0 if H <= 1 else max(MIN_CTAS, sms // min(H, 16))


def critical_grids(M, D, sms=B200_SMS):
    """Grid bounds (max_ctas) that change the division of work of the stage at this shape, in [8, 148]."""
    MP = padded_m(M)
    n_tiles, n_beta, n_fwd, n_bwd = phase4_units(MP)
    g = {MIN_CTAS, stage_grid("fwd", M, D, 0, sms), stage_grid("bwd", M, D, 0, sms)}
    g |= {n_items(MP, 0) + i for i in (0, 1, 2)}                  # NW just below, equal to, above the first step
    thr = n_tiles + n_beta + 2 * (n_fwd + n_bwd)                   # parts: 1 below, 2 from here
    g |= {thr - 1, thr}
    g |= {bwd_items(MP) - 1, bwd_items(MP) + 1}
    g |= {stage_cta_cap(H, sms) for H in (2, 4, 17)}               # what multi-output layers run with
    return sorted(x for x in g if MIN_CTAS <= x <= CTA_LIMIT)


# (M, D, kind): every Mp class (128, 256, 512, 768, 1024) with RBF and a Matern kind, both backward tile heights
# (16 rows up to Mp = 256, 32 above), D from {5, 20, 64, 100, 128} with D = 5 (Dp = 16) reaching the thread-per-(i, d)
# branch of the backward's phase C.
SWEEP_CELLS = [(33, 5, "rbf"), (64, 100, "matern32"), (200, 20, "matern52"), (256, 128, "rbf"), (300, 5, "matern12"),
               (300, 64, "rbf"), (600, 20, "matern32"), (600, 100, "rbf"), (1024, 64, "rbf"), (1024, 20, "matern12")]
N_SWEEP = 333


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests of the mirror
# ---------------------------------------------------------------------------------------------------------------------
def test_grid_mirror_hand_checked_rows():
    # forward: nb^2 + nb + 3 (n_fwd + n_bwd), then max_ctas, the floor of 8 and the cap of 148
    assert image_counts(128) == (4, 4) and image_counts(256) == (8, 12) and image_counts(512) == (24, 40)
    assert stage_grid("fwd", 64, 20, 0) == 16 + 4 + 24 == 44
    assert stage_grid("fwd", 200, 20, 0) == 64 + 8 + 60 == 132
    assert stage_grid("fwd", 300, 20, 0) == 148 and stage_grid("fwd", 1024, 128, 0) == 148
    assert stage_grid("fwd", 256, 64, 74) == 74 and stage_grid("fwd", 256, 64, 9) == 9
    assert stage_grid("fwd", 256, 64, 5) == 8 and stage_grid("fwd", 64, 20, 200) == 44
    assert stage_grid("fwd", 32, 20, 0) == 1 and stage_grid("bwd", 3, 5, 9) == 1
    # backward: (2 | 1) nb^2, at least ceil(Mp Dp / 256), then max_ctas (raised to 8) and the cap of 148
    assert stage_grid("bwd", 64, 20, 0) == 32 and stage_grid("bwd", 64, 100, 0) == 64
    assert stage_grid("bwd", 256, 64, 0) == 128 and stage_grid("bwd", 300, 5, 0) == 148
    assert stage_grid("bwd", 1024, 64, 9) == 9 and stage_grid("bwd", 1024, 64, 5) == 8
    assert stage_grid("bwd", 64, 20, 200) == 32 and stage_grid("bwd", 64, 100, 40) == 40
    # phase 2: worker items per step and workers
    assert [n_items(128, kb) for kb in range(4)] == [8, 6, 3, 3]
    assert n_items(256, 0) == 34 and n_items(512, 0) == 134 and n_items(768, 0) == 298
    assert n_workers(8) == 7
    # phase 4: parts of the operand images
    assert phase4_units(128) == (16, 4, 4, 4) and phase4_units(256) == (64, 8, 8, 12)
    assert parts(128, 35) == 1 and parts(128, 36) == 2 and parts(128, 44) == 3 and parts(128, 8) == 1
    assert parts(256, 111) == 1 and parts(256, 112) == 2 and parts(256, 132) == 3 and parts(512, 148) == 1
    assert parts(128, 148) == 8
    # backward items NH nb^2 and the tile height (the dispatch matrix's mm_backward_kernel<16 | 32, .>)
    assert [bwd_items(mp) for mp in (128, 256, 512, 768, 1024)] == [32, 128, 256, 576, 1024]
    assert half_tiles(256) and not half_tiles(512)
    # ops._stage_cta_cap on 148 SMs, H = 1 ... 20
    assert [stage_cta_cap(H) for H in range(1, 21)] == [0, 74, 49, 37, 29, 24, 21, 18, 16, 14, 13, 12, 11, 10, 9, 9,
                                                         9, 9, 9, 9]


def test_stage_cta_cap_matches_ops(monkeypatch):
    from fine_grained_gaussian_process_forcasting_b200 import ops
    dev = torch.device("cuda", 97)                     # never opened: the SM count comes from the cache
    monkeypatch.setitem(ops._SM_COUNT, (dev.type, dev.index), B200_SMS)
    assert [ops._stage_cta_cap(dev, H) for H in range(1, 21)] == [stage_cta_cap(H) for H in range(1, 21)]


def test_critical_grids_cover_every_boundary():
    for M, D, _ in SWEEP_CELLS:
        MP = padded_m(M)
        g = set(critical_grids(M, D))
        n_tiles, n_beta, n_fwd, n_bwd = phase4_units(MP)
        thr = n_tiles + n_beta + 2 * (n_fwd + n_bwd)
        want = {MIN_CTAS, stage_grid("fwd", M, D, 0), stage_grid("bwd", M, D, 0)}
        want |= {n_items(MP, 0) + i for i in (0, 1, 2)} | {thr - 1, thr} | {bwd_items(MP) - 1, bwd_items(MP) + 1}
        want = {x for x in want if MIN_CTAS <= x <= CTA_LIMIT}
        assert want <= g, (M, D, sorted(want - g))
        assert all(MIN_CTAS <= x <= CTA_LIMIT for x in g)
        # the boundaries are what they claim to be
        if thr <= CTA_LIMIT:
            assert parts(MP, thr - 1) == 1 and parts(MP, thr) == 2
        k0 = n_items(MP, 0)
        if k0 + 2 <= CTA_LIMIT:
            assert [n_workers(k0 + i) - k0 for i in (0, 1, 2)] == [-1, 0, 1]
    # every Mp class and both backward tile heights appear, RBF and a Matern kind on each class, Dp = 16 on both
    classes = {padded_m(M) for M, _, _ in SWEEP_CELLS}
    assert classes == {128, 256, 512, 768, 1024}
    for mp in classes:
        kinds = {k for M, _, k in SWEEP_CELLS if padded_m(M) == mp}
        assert "rbf" in kinds and kinds - {"rbf"}, mp
    assert {half_tiles(padded_m(M)) for M, D, _ in SWEEP_CELLS if padded_d(D) == 16} == {True, False}
    assert {padded_d(D) for _, D, _ in SWEEP_CELLS} == {16, 32, 64, 128}
    # the Mp = 128 / 256 classes reach the phase-2 and phase-4 boundaries inside [8, 148]
    assert {8, 9, 10, 35, 36, 31, 33} <= set(critical_grids(64, 100))
    assert {34, 35, 36, 111, 112, 127, 129} <= set(critical_grids(256, 128))
    assert {134, 135, 136} <= set(critical_grids(300, 64))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: grid sweep
# ---------------------------------------------------------------------------------------------------------------------
SEED, OFFSET, STREAM, GKL = 4321, 19, 2, 0.37
MM_KERNELS = ("mm_forward_kernel", "mm_backward_kernel")


def _dev_args(p32, dev):
    args = [p32["inducing_points"], p32["raw_lengthscale"].reshape(-1), p32["raw_outputscale"].reshape(1),
            p32["variational_mean"], p32["variational_stddev"], p32["weights"].reshape(-1), p32["bias"]]
    return [t.to(dev).contiguous() for t in args]


def _stage_run(args, xd, M, kind, G, g_up, gkl, sgrad_in=None):
    """Stage at grid bound G, point forward + backward on it, stage backward (on `sgrad_in` first when given, then on
    the run's own stage gradient).  Outputs are zeroed before the calls, so that an element no kernel writes compares
    equal instead of holding whatever the allocation held."""
    from fine_grained_gaussian_process_forcasting_b200 import ops
    dev = xd.device
    N, D = xd.shape
    k = KIND_ID[kind]
    stage = torch.zeros(ops.param_stage_bytes(D, M), device=dev, dtype=torch.uint8)
    kl = torch.zeros(1, device=dev, dtype=torch.float32)
    info = torch.full((1,), -1, device=dev, dtype=torch.int32)
    ops.param_stage_raw(*args, out=(stage, kl, info), max_ctas=G, kind=k)
    mean, var, sample, ws = ops.point_forward_raw(stage, xd, M, SEED, OFFSET, STREAM, True, True, kind=k)
    dx = torch.zeros(N, D, device=dev, dtype=torch.float32)
    sgrad = torch.zeros(ops.stage_grad_doubles(D, M), device=dev, dtype=torch.float64)
    ops.point_backward_raw(xd, M, *g_up, var, SEED, OFFSET, STREAM, ws, dx=dx, sgrad=sgrad, stage=stage, kind=k)
    buckets = []
    for sg in ([] if sgrad_in is None else [sgrad_in]) + [sgrad]:
        b = torch.zeros(ops.grad_bucket_floats(D, M), device=dev, dtype=torch.float32)
        ops.param_stage_backward_raw(*args, sg, gkl, stage, bucket=b, max_ctas=G, kind=k)
        buckets.append(b)
    torch.cuda.synchronize()
    r = {"Kzz": ops.debug_fetch(2, 0, D, M, stage), "L": ops.debug_fetch(0, 0, D, M, stage),
         "Linv": ops.debug_fetch(1, 0, D, M, stage), "kl": kl, "info": info, "mean": mean, "var": var,
         "sample": sample, "dx": dx, "sgrad": sgrad, "buckets": buckets}
    return {key: ([b.cpu() for b in v] if isinstance(v, list) else v.cpu()) for key, v in r.items()}


def _launched_grids(trace_path):
    """{kernel family: [grid x of each launch, in launch order]} of the M x M stage kernels in a chrome trace."""
    with open(trace_path) as f:
        evs = json.load(f)["traceEvents"]
    out = {k: [] for k in MM_KERNELS}
    for e in sorted((e for e in evs if e.get("cat") == "kernel"), key=lambda e: e["ts"]):
        fam = kernel_id(e["name"]).split("<")[0]
        if fam in out:
            grid = e.get("args", {}).get("grid")
            assert grid is not None, ("this torch build records no grid in its kernel events", e)
            assert list(grid[1:]) == [1, 1], e
            out[fam].append(int(grid[0]))
    return out


BITWISE = ("Kzz", "L", "Linv", "kl", "info", "mean", "var", "sample", "dx", "sgrad")


def _assert_same(ref, r, what):
    for key in BITWISE:
        assert torch.equal(ref[key], r[key]), (what, key)
    for i, b in enumerate(r["buckets"]):
        assert torch.equal(ref["buckets"][-1], b), (what, "bucket", i)


def _oracle_errors(kind, p32, x32, gm, gv, gs, r):
    N, D = x32.shape
    M = p32["inducing_points"].shape[0]
    eps = torch.from_numpy(O.philox_normal(SEED, OFFSET, N, STREAM)).double()
    mo, vo, klo, dxo, go = oracle(kind, p32, x32, gm, gv, gs, eps, True)
    Kzz, Lc, Linv, _, _ = _stage_fp64(O.clone_params(p32, torch.float64), kind)
    errs = {"Kzz": rel(r["Kzz"][:M, :M], Kzz), "L": rel(torch.tril(r["L"][:M, :M]), Lc),
            "Linv": rel(torch.tril(r["Linv"][:M, :M]), Linv),
            "kl": abs(r["kl"].item() - klo.item()) / max(1.0, abs(klo.item())),
            "mean": rel(r["mean"], mo), "var": rel(r["var"], vo), "dx": rel(r["dx"], dxo)}
    from fine_grained_gaussian_process_forcasting_b200 import ops
    grads = {n: v.reshape(go[n].shape) for n, v in zip(NAMES, ops.split_bucket(r["buckets"][-1], D, M, True))}
    for n in NAMES:
        errs[n] = rel(grads[n], go[n])
    if errs["raw_outputscale"] >= 2e-4:
        # one number, a sum of terms of both signs: measured against the size of the terms (test_gpu_dispatch_matrix)
        scale = oracle(kind, p32, x32, gm.abs(), gv.abs(), gs.abs(), eps, True)[4]["raw_outputscale"].abs()
        errs["raw_outputscale"] = ((grads["raw_outputscale"].double().reshape(()) - go["raw_outputscale"]).abs()
                                   / torch.maximum(go["raw_outputscale"].abs(), scale)).item()
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("M,D,kind", SWEEP_CELLS, ids=["M%d-D%d-%s" % c for c in SWEEP_CELLS])
def test_stage_bitwise_across_grids(cuda, tmp_path, M, D, kind):
    """Stage, point calls and stage backward at every critical grid: launched grids as mirrored, results bit-identical
    to the default grid, the run at G = 8 against the float64 oracle, the smallest and largest G twice."""
    from torch.profiler import profile, ProfilerActivity
    sms = torch.cuda.get_device_properties(cuda).multi_processor_count
    N = N_SWEEP
    p32, x32, gm, gv, gs = _inputs(N, D, M, kind)
    args = _dev_args(p32, cuda)
    xd = x32.to(cuda).contiguous()
    g_up = [t.to(cuda) for t in (gm, gv, gs)]
    gkl = torch.tensor([GKL], device=cuda)
    grids = critical_grids(M, D, sms)
    runs = [0] + grids + [grids[0], grids[-1]]
    want = {"mm_forward_kernel": [], "mm_backward_kernel": []}
    res = []
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        time.sleep(0.02)            # the trace keeps kernels inside its window: a head start over the first launch
        ref = _stage_run(args, xd, M, kind, 0, g_up, gkl)
        want["mm_forward_kernel"].append(stage_grid("fwd", M, D, 0, sms))
        want["mm_backward_kernel"].append(stage_grid("bwd", M, D, 0, sms))
        for G in runs[1:]:
            res.append((G, _stage_run(args, xd, M, kind, G, g_up, gkl, sgrad_in=ref["sgrad"].to(cuda))))
            want["mm_forward_kernel"].append(stage_grid("fwd", M, D, G, sms))
            want["mm_backward_kernel"] += [stage_grid("bwd", M, D, G, sms)] * 2
        torch.cuda.synchronize()
    trace = str(tmp_path / "trace.json")
    prof.export_chrome_trace(trace)
    got = _launched_grids(trace)
    assert got == want, (got, want)
    assert int(ref["info"].item()) == 0
    for G, r in res:
        _assert_same(ref, r, f"G={G}")
    errs = _oracle_errors(kind, p32, x32, gm, gv, gs, next(r for G, r in res if G == MIN_CTAS))
    fwd_grids = sorted(set(want["mm_forward_kernel"]))
    bwd_grids = sorted(set(want["mm_backward_kernel"]))
    worst = max(errs, key=lambda k: errs[k])
    print(f"stage grid M={M} D={D} {kind}: max_ctas {grids} -> forward grids {fwd_grids}, backward grids {bwd_grids}; "
          f"oracle at G=8: worst {worst}={errs[worst]:.1e} | " + " ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    assert errs["Kzz"] < 1e-6 and errs["L"] < 1e-6 and errs["Linv"] < 1e-5, errs
    assert errs["kl"] < 1e-5, errs
    assert errs["mean"] < 1e-4 and errs["var"] < 1e-4, errs
    for k in ["dx"] + NAMES:
        assert errs[k] < 2e-4, (k, errs)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: multi-output layers as production runs them
# ---------------------------------------------------------------------------------------------------------------------
LAYER_CASES = [(M, H) for M in (64, 256) for H in (2, 5, 16, 17, 20)] + [(1024, 2)]
N_LAYER = 250


def _layer_dims(M):
    return {64: 20, 256: 64, 1024: 20}[M]


def _load_layer(layer, p):
    vs = layer.variational_strategy
    with torch.no_grad():
        vs.inducing_points.copy_(p["inducing_points"])
        layer.covar_module.base_kernel.raw_lengthscale.copy_(p["raw_lengthscale"])
        layer.covar_module.raw_outputscale.copy_(p["raw_outputscale"].reshape(layer.covar_module.raw_outputscale.shape))
        vs._variational_distribution.variational_mean.copy_(p["variational_mean"])
        vs._variational_distribution._variational_stddev.copy_(p["variational_stddev"])
        layer.mean_module.weights.copy_(p["weights"])
        layer.mean_module.bias.copy_(p["bias"])
        vs.variational_params_initialized.fill_(1)


@pytest.mark.gpu
@pytest.mark.parametrize("M,H", LAYER_CASES, ids=["M%d-H%d" % c for c in LAYER_CASES])
def test_multi_output_layer_matches_single_gps(cuda, M, H):
    """ToyDeepGPHiddenLayer(D, output_dims=H): H stages on side streams with ops._stage_cta_cap CTAs each (two stages
    per stream from H = 17 on).  GP h must give what GP h alone gives at the default grid, bit for bit; the shared
    LinearMean gets the fp32 sum over h of the single-GP gradients."""
    from fine_grained_gaussian_process_forcasting_b200 import gpcompat, ops
    from fine_grained_gaussian_process_forcasting_b200.DeepGP import ToyDeepGPHiddenLayer
    D, N = _layer_dims(M), N_LAYER
    p = O.init_params_hidden_layer(D, H, M, seed=M + H)
    g = torch.Generator().manual_seed(M * 100 + H)
    x = torch.randn(N, D, generator=g)
    gm, gv = torch.randn(1, N, H, generator=g), torch.randn(1, N, H, generator=g)
    layer = ToyDeepGPHiddenLayer(D, H, seed=0, num_inducing=M, mean_type="linear").to(cuda)
    _load_layer(layer, p)
    layer.set_rng(77, 5, stream=1)
    xd = x.to(cuda).requires_grad_(True)
    with gpcompat.num_likelihood_samples(1):
        dist = layer(xd)
        mean, var = dist.mean, dist.variance
        _, kl, info, _ = ops.svgp_param_stage(*layer._layer_params(), stage_cache=layer._stage_cache())
        loss = (gm.to(cuda) * mean).sum() + (gv.to(cuda) * var).sum()
        loss.backward()
    torch.cuda.synchronize()
    assert tuple(mean.shape) == (1, N, H) and torch.equal(info.cpu(), torch.zeros(H, dtype=torch.int32))
    vs = layer.variational_strategy
    vd = vs._variational_distribution
    lg = {"inducing_points": vs.inducing_points.grad, "raw_lengthscale": layer.covar_module.base_kernel.raw_lengthscale.grad,
          "raw_outputscale": layer.covar_module.raw_outputscale.grad, "variational_mean": vd.variational_mean.grad,
          "variational_stddev": vd._variational_stddev.grad}
    # GP h alone, one after the other on the current stream, default grid
    x2 = xd.detach()
    buckets = []
    for h in range(H):
        ph = {"inducing_points": p["inducing_points"][h], "raw_lengthscale": p["raw_lengthscale"][h],
              "raw_outputscale": p["raw_outputscale"][h], "variational_mean": p["variational_mean"][h],
              "variational_stddev": p["variational_stddev"][h], "weights": p["weights"], "bias": p["bias"]}
        args = _dev_args(ph, cuda)
        stage, kl1, info1 = ops.param_stage_raw(*args)
        m1, v1, _, ws = ops.point_forward_raw(stage, x2, M, 77, 5 + h * N, 1, True, True)
        _, sgrad = ops.point_backward_raw(x2, M, gm[0, :, h].to(cuda).contiguous(), gv[0, :, h].to(cuda).contiguous(),
                                          None, v1, 77, 5 + h * N, 1, ws, stage=stage)
        bucket = ops.param_stage_backward_raw(*args, sgrad, None, stage)
        torch.cuda.synchronize()
        assert int(info1.item()) == 0
        assert torch.equal(mean[0, :, h], m1) and torch.equal(var[0, :, h], v1), ("mean / var", h)
        assert torch.equal(kl[h:h + 1], kl1), ("kl", h)
        views = ops.split_bucket(bucket, D, M, True)
        for n, v in zip(NAMES[:5], views[:5]):
            assert torch.equal(lg[n][h].reshape(-1), v.reshape(-1)), (n, h)
        buckets.append(bucket)
    # the shared LinearMean: the sum over h that _ParamStageFunction._backward forms from the [H, bucket] buffer
    stacked = torch.stack(buckets)
    o = M * D + D + 1 + 2 * M
    assert torch.equal(layer.mean_module.weights.grad.reshape(-1), stacked[:, o:o + D].sum(0))
    assert torch.equal(layer.mean_module.bias.grad.reshape(-1), stacked[:, o + D:o + D + 1].sum(0))
    print(f"multi-output M={M} D={D} H={H}: {H} stages at max_ctas={stage_cta_cap(H)} bitwise equal to single GPs")
    if (M, H) == (64, 17):
        _layer_against_oracle(p, x, gm, gv, mean, var, layer, lg)


def _layer_against_oracle(p, x, gm, gv, mean, var, layer, lg):
    p64 = O.clone_params(p, torch.float64, requires_grad=True)
    mo, vo = O.hidden_layer_predict(p64, x.double().unsqueeze(0))
    ((gm.double() * mo).sum() + (gv.double() * vo).sum()).backward()
    got = dict(lg, weights=layer.mean_module.weights.grad, bias=layer.mean_module.bias.grad)
    errs = {"mean": rel(mean, mo), "var": rel(var, vo)}
    errs.update({n: rel(got[n].reshape(p64[n].shape), p64[n].grad) for n in NAMES})
    print("multi-output H=17 against the float64 oracle: " + " ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    assert errs["mean"] < 1e-4 and errs["var"] < 1e-4, errs
    for n in NAMES:
        assert errs[n] < 2e-4, (n, errs)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the Cholesky failure report
# ---------------------------------------------------------------------------------------------------------------------
INFO_CASES = [(M, k, G) for M in (256, 1024) for k in (0, 31, 32, 200, M - 1) for G in (0, 8)]
INFO_CASES += [(32, 0, 0), (32, 31, 0), (20, 19, 0), (20, 7, 0)]      # M <= 32: the one-CTA kernel


@pytest.mark.gpu
def test_nan_inducing_point_reports_its_pivot(cuda):
    """A NaN in inducing point k makes row and column k of Kzz NaN: the first non-positive pivot of the factorisation
    is k, and info is the 1-based LAPACK-style k + 1, from the cooperative stage at any grid and from the M <= 32
    kernel alike."""
    from fine_grained_gaussian_process_forcasting_b200 import ops
    D = 20
    got = {}
    for M, k, G in INFO_CASES:
        p32 = O.init_params_exercise(D, M, seed=M)
        p32["inducing_points"][k, 3] = float("nan")
        _, _, info = ops.param_stage_raw(*_dev_args(p32, cuda), max_ctas=G)
        got[(M, k, G)] = int(info.item())
    print("info per (M, k, max_ctas):", got)
    assert got == {c: c[1] + 1 for c in INFO_CASES}
