"""Every SVGP kernel instantiation that the dispatcher can reach, compared with the float64 oracle.

Which compiled specialisation runs depends on the padded inducing count Mp, the padded input width Dp, the kernel kind
and, on the FP32-FFMA path, N against the SM count.  `expected_kernels` restates the C++ dispatch rules
(csrc: padded_m / padded_d, tc_point_supported, dispatch_fwd_tn, dispatch_bwd_dp, launch_tc_point_*,
launch_tc_reductions, launch_reductions, launch_mm_*), and CELLS is a list of shapes whose kernels, taken together,
are exactly the reachable instantiations enumerated in REACHABLE.  The CPU tests hold that equality (and, when the
library is built, compare the instantiations compiled into it with REACHABLE + KNOB_ONLY + NOT_DISPATCHED), so a new
specialisation without a cell fails without a GPU.  The GPU tests run every cell under torch.profiler, check that the
launched kernels are the expected ones, and compare every output, the stage, the probed intermediates A and W, and
every gradient with the float64 closed form.

Metric: max|cuda - oracle| / max|oracle| (tests/test_gpu_parity.py), also on the last, ragged tile alone against that
tile's own scale, so that a wrong tail cannot hide behind larger values elsewhere.
"""
import json
import os
import re
import shutil
import subprocess
import sys
import time

import pytest
import torch

from oracle import gp_oracle as O
from oracle import matern_oracle as MO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ["rbf", "matern12", "matern32", "matern52"]
KIND_ID = {k: i for i, k in enumerate(KINDS)}          # GPBLUR_KERNEL_*
NAMES = ["inducing_points", "raw_lengthscale", "raw_outputscale", "variational_mean", "variational_stddev", "weights",
         "bias"]
TOL_FWD = 1e-5        # FP32 FFMA path
TOL_FWD_TC = 1e-4     # tcgen05 3xTF32 path
TOL_GRAD = 2e-4
B200_SMS = 148


# ---------------------------------------------------------------------------------------------------------------------
# Dispatch mirror
# ---------------------------------------------------------------------------------------------------------------------
K_THREADS, K_KS, K_SMEM_CAP, TC_TILE = 256, 16, 220 * 1024, 128


def padded_m(M):
    return 32 if M <= 32 else 128 if M <= 128 else (M + 255) // 256 * 256


def padded_d(D):
    return 16 if D <= 16 else 32 if D <= 32 else 64 if D <= 64 else 128


def tc_point_supported(MP, N, ffma_forced=False):
    return not ffma_forced and (MP == 128 or (MP >= 256 and MP % 256 == 0)) and N >= 1


def _ffma_tile_cfg(MP, TN):
    """TileCfg<PT, CT, CW> of the FFMA point kernels for an MP and a tile height (dispatch_fwd_tn / dispatch_bwd_dp)."""
    CT, CW = (4, 32) if MP == 32 else (4, 64) if MP == 64 else (8, 128)
    TYN = K_THREADS // (CW // CT)
    return TN // TYN, CT, CW


def fwd_smem_bytes(TN, DP, MP):
    CW = _ffma_tile_cfg(MP, TN)[2]
    return 4 * (TN * (DP + 4) + TN * (MP + 4) + 2 * K_KS * CW + 4 * TN)


def ffma_fwd_tile(N, DP, MP, sms):
    """dispatch_fwd_tn without the GPBLUR_FWD_TN override: the point tile height, or None (unsupported)."""
    smem = {tn: fwd_smem_bytes(tn, DP, MP) for tn in (32, 64, 128)}
    if 2 * smem[64] <= K_SMEM_CAP and N >= 64 * sms:
        return 64
    if smem[128] <= K_SMEM_CAP and N >= 128 * 2 * sms:
        return 128
    if smem[64] <= K_SMEM_CAP and N >= 64 * sms:
        return 64
    if smem[32] <= K_SMEM_CAP:
        return 32
    return None


def _cfg(t):
    return "TileCfg<%d,%d,%d>" % t


def expected_kernels(N, D, M, kind, training, sms=B200_SMS, ffma_forced=False):
    """Kernel ids (see kernel_id) that one param stage + point forward (+ point backward + stage backward when
    `training`) launch.  `ffma_forced`: the process runs with GPBLUR_TC=-1."""
    MP, DP, k = padded_m(M), padded_d(D), KIND_ID[kind]
    mat = "true" if k else "false"
    out = set()
    nb = MP // 32
    out.add(f"mm_small_forward_kernel<{mat}>" if nb == 1 else f"mm_forward_kernel<{mat}>")
    tc = tc_point_supported(MP, N, ffma_forced)
    if N >= 1:
        if tc:
            out.add(f"tc2_fwd_kernel<128,128,4,{k}>" if MP == 128 else f"tc2_fwd_kernel<128,256,3,{k}>")
        else:
            out.add(f"point_fwd_kernel<{_cfg(_ffma_tile_cfg(MP, ffma_fwd_tile(N, DP, MP, sms)))},{k}>")
    if not training:
        return out
    if N >= 1:
        if tc:
            dxw = 32 if DP <= 32 else DP
            out.add({32: f"tc2_bwd_kernel<128,32,3,4,{k}>", 64: f"tc2_bwd_kernel<128,64,3,4,{k}>",
                     128: f"tc2_bwd_kernel<128,128,2,3,{k}>"}[dxw])
            nt = 1 if MP == 128 else 2
            out.add(f"tc_reduce_kernel<{nt},{32 if DP <= 32 else DP},{'true' if MP >= 512 else 'false'}>")
        else:
            out.add(f"point_bwd_kernel<{_cfg(_ffma_tile_cfg(MP, 64))},{DP},{k}>")      # bwd_tile_points: TN = 64
            tp = MP if MP < 128 else 128
            out.add(f"reduce_gemm_kernel<{tp},{tp},true>")
            out.add(f"reduce_gemm_kernel<{tp},{DP},false>")
    out.add("stage_grad_reduce_kernel")
    if nb == 1:
        out.add(f"mm_small_backward_kernel<{mat}>")
    else:
        out.add(f"mm_backward_kernel<{16 if 2 * nb * nb <= 2 * 148 else 32},{mat}>")
    return out


def kernel_id(name):
    """Demangled kernel name (profiler or cu++filt spelling) -> 'name<args>' without namespaces, spaces or casts."""
    s = name.replace("(anonymous namespace)::", "").replace("<unnamed>::", "").replace("gpblur::", "")
    s = s.replace(" ", "").replace("(int)", "").replace("(bool)0", "false").replace("(bool)1", "true")
    if s.startswith("void"):
        s = s[4:]
    depth, out = 0, []
    for c in s:
        if c == "(" and depth == 0:
            break
        depth += c == "<"
        depth -= c == ">"
        out.append(c)
    return "".join(out)


KERNEL_FAMILIES = ("point_fwd_kernel", "point_bwd_kernel", "tc2_fwd_kernel", "tc2_bwd_kernel", "tc_reduce_kernel",
                   "reduce_gemm_kernel", "mm_small_forward_kernel", "mm_small_backward_kernel", "mm_forward_kernel",
                   "mm_backward_kernel", "stage_grad_reduce_kernel")


def svgp_kernel_ids(ids):
    return {i for i in ids if i.split("<")[0] in KERNEL_FAMILIES}


# Every instantiation a call can reach without a tuning knob.  K = kind (0 RBF, 1/2/3 Matern 1/2, 3/2, 5/2).
REACHABLE = set()
for _k in range(4):
    _m = "true" if _k else "false"
    REACHABLE |= {
        f"point_fwd_kernel<TileCfg<1,4,32>,{_k}>",        # M <= 32, N < 64 SMs: 32-point tiles
        f"point_fwd_kernel<TileCfg<2,4,32>,{_k}>",        # M <= 32, N >= 64 SMs: 64-point tiles, 2 CTAs / SM fit
        f"point_bwd_kernel<TileCfg<2,4,32>,16,{_k}>",     # M <= 32, D <= 16 (backward tile is always 64 points)
        f"point_bwd_kernel<TileCfg<2,4,32>,32,{_k}>",     # M <= 32, 16 < D <= 32
        f"point_bwd_kernel<TileCfg<2,4,32>,64,{_k}>",     # M <= 32, 32 < D <= 64
        f"point_bwd_kernel<TileCfg<2,4,32>,128,{_k}>",    # M <= 32, 64 < D <= 128
        f"tc2_fwd_kernel<128,128,4,{_k}>",                # 32 < M <= 128 (Mp = 128): one 128-column block
        f"tc2_fwd_kernel<128,256,3,{_k}>",                # M > 128 (Mp = 256 k): 256-column blocks
        f"tc2_bwd_kernel<128,32,3,4,{_k}>",               # M > 32, D <= 32: dx epilogue 32 wide
        f"tc2_bwd_kernel<128,64,3,4,{_k}>",               # M > 32, 32 < D <= 64
        f"tc2_bwd_kernel<128,128,2,3,{_k}>",              # M > 32, D > 64
    }
    if _k < 2:   # the M x M stage is templated on RBF / not RBF only
        REACHABLE |= {
            f"mm_small_forward_kernel<{_m}>",             # M <= 32: one 32 x 32 block, one CTA
            f"mm_small_backward_kernel<{_m}>",            # M <= 32
            f"mm_forward_kernel<{_m}>",                   # M > 32: cooperative blocked stage
            f"mm_backward_kernel<16,{_m}>",               # Mp <= 256 (2 nb^2 <= 296): 16-row tiles
            f"mm_backward_kernel<32,{_m}>",               # Mp >= 512: 32-row tiles
        }
REACHABLE |= {
    "reduce_gemm_kernel<32,32,true>",        # M <= 32: Gram A^T diag(g) A, one 32 x 32 tile
    "reduce_gemm_kernel<32,16,false>",       # M <= 32, D <= 16: W^T X
    "reduce_gemm_kernel<32,32,false>",       # M <= 32, 16 < D <= 32
    "reduce_gemm_kernel<32,64,false>",       # M <= 32, 32 < D <= 64
    "reduce_gemm_kernel<32,128,false>",      # M <= 32, D > 64
    "tc_reduce_kernel<1,32,false>",          # Mp = 128, D <= 32 (Dp 16 runs the 32-wide unit)
    "tc_reduce_kernel<1,64,false>",          # Mp = 128, 32 < D <= 64
    "tc_reduce_kernel<1,128,false>",         # Mp = 128, D > 64
    "tc_reduce_kernel<2,32,false>",          # Mp = 256 (one 256-wide band, no off-diagonal units), D <= 32
    "tc_reduce_kernel<2,64,false>",          # Mp = 256, 32 < D <= 64
    "tc_reduce_kernel<2,128,false>",         # Mp = 256, D > 64
    "tc_reduce_kernel<2,32,true>",           # Mp >= 512 (off-diagonal Gram units), D <= 32
    "tc_reduce_kernel<2,64,true>",           # Mp >= 512, 32 < D <= 64
    "tc_reduce_kernel<2,128,true>",          # Mp >= 512, D > 64
    "stage_grad_reduce_kernel",              # every backward
}

# Reachable only with GPBLUR_TC=-1 (FP32 FFMA kernels at Mp >= 128, RBF only): test_ffma_forced_by_knob runs them.
KNOB_ONLY = {f"point_fwd_kernel<TileCfg<{pt},8,128>,0>" for pt in (2, 4, 8)}
KNOB_ONLY |= {f"point_bwd_kernel<TileCfg<4,8,128>,{dp},0>" for dp in (16, 32, 64, 128)}
KNOB_ONLY |= {"reduce_gemm_kernel<128,128,true>"} | {f"reduce_gemm_kernel<128,{dp},false>" for dp in (16, 32, 64, 128)}

# Compiled but never dispatched without a tile-height override (GPBLUR_FWD_TN / GPBLUR_BWD_TN = 128) or at Mp = 64,
# which padded_m no longer produces (32 < M <= 64 is padded to 128 and runs on the tensor cores).
NOT_DISPATCHED = {f"point_fwd_kernel<TileCfg<4,4,32>,{k}>" for k in range(4)}
NOT_DISPATCHED |= {f"point_bwd_kernel<TileCfg<4,4,32>,{dp},{k}>" for dp in (16, 32, 64, 128) for k in range(4)}
NOT_DISPATCHED |= {f"point_bwd_kernel<TileCfg<8,8,128>,{dp},0>" for dp in (16, 32, 64, 128)}
NOT_DISPATCHED |= {f"point_fwd_kernel<TileCfg<{pt},4,64>,0>" for pt in (2, 4, 8)}
NOT_DISPATCHED |= {f"point_bwd_kernel<TileCfg<{pt},4,64>,{dp},0>" for pt in (4, 8) for dp in (16, 32, 64, 128)}
NOT_DISPATCHED |= {"reduce_gemm_kernel<64,64,true>"} | {f"reduce_gemm_kernel<64,{dp},false>" for dp in (16, 32, 64, 128)}


def _ffma_cells():
    # the full product D x M x kind x N on the FFMA path (M <= 32): D in {5, 32, 64, 100, 128} (Dp 16, 32, 64, 128 and
    # a padded 128), M in {3, 32}, N just below (9000) and above (9517, a ragged 45-point tail) the 64-point forward
    # tiles' threshold of 64 SMs (9472 points on 148 SMs)
    return [(N, D, M, kind) for kind in KINDS for D in (5, 32, 64, 100, 128) for M in (3, 32) for N in (9000, 9517)]


def _tc_cells():
    # every kind x Mp class (128 | 256 | >= 512) x dx-epilogue width (32 | 64 | 128); M and D rotate through their
    # classes so that Mp = 512, 768 and 1024 and the padded widths Dp = 32 (D = 20) and Dp = 128 (D = 100) all appear.
    m_class = {128: (64, 128), 256: (256, 200), 512: (600, 1024, 700, 300)}
    d_class = {32: (20, 32), 64: (64, 48), 128: (100, 128)}
    cells, r = [], 0
    for kind in KINDS:
        for mc in (128, 256, 512):
            for dw in (32, 64, 128):
                M = m_class[mc][r % len(m_class[mc])]
                D = d_class[dw][(r // 3) % len(d_class[dw])]
                N = 300 + 97 * (r % 11) if padded_m(M) >= 512 else 900 + 131 * (r % 7)
                cells.append((N, D, M, kind))
                r += 1
    return cells


# Large ragged N: most CTAs of the persistent tensor-core grid (one per SM) own two or more 128-point tiles.
BIG_N = 2 * TC_TILE * B200_SMS + 3 * 128 + 77
BIG_CELLS = [(BIG_N, 32, 128, "rbf"), (BIG_N, 20, 256, "matern52"), (BIG_N, 64, 300, "rbf"),
             (BIG_N, 20, 600, "matern32"), (BIG_N, 32, 1024, "matern12")]

CELLS = _ffma_cells() + _tc_cells() + BIG_CELLS


def _cell_id(c):
    return "N%d-D%d-M%d-%s" % c


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests of the mirror
# ---------------------------------------------------------------------------------------------------------------------
def test_cells_cover_every_reachable_instantiation():
    got = set()
    for N, D, M, kind in CELLS:
        got |= expected_kernels(N, D, M, kind, True)
    assert got == REACHABLE, (sorted(got - REACHABLE), sorted(REACHABLE - got))


def test_ffma_cells_are_the_full_product():
    """Every kind meets every D and M on the FFMA path at both forward tile heights."""
    ffma = {c for c in CELLS if c[2] <= 32}
    assert len(ffma) == 80
    for kind in KINDS:
        for D in (5, 32, 64, 100, 128):
            for M in (3, 32):
                ns = [c[0] for c in ffma if c[1:] == (D, M, kind)]
                assert min(ns) < 64 * B200_SMS <= max(ns), (D, M, kind)


def test_mirror_hand_checked_rows():
    e = expected_kernels(9500, 32, 32, "rbf", True)
    assert "point_fwd_kernel<TileCfg<2,4,32>,0>" in e and "point_bwd_kernel<TileCfg<2,4,32>,32,0>" in e
    assert "reduce_gemm_kernel<32,32,true>" in e and "mm_small_backward_kernel<false>" in e
    assert "point_fwd_kernel<TileCfg<1,4,32>,0>" in expected_kernels(9000, 32, 32, "rbf", False)
    # the C64 threshold follows the SM count
    assert "point_fwd_kernel<TileCfg<1,4,32>,2>" in expected_kernels(9500, 5, 3, "matern32", False, sms=150)
    e = expected_kernels(1000, 20, 600, "matern12", True)
    assert padded_m(600) == 768
    assert e == {"mm_forward_kernel<true>", "tc2_fwd_kernel<128,256,3,1>", "tc2_bwd_kernel<128,32,3,4,1>",
                 "tc_reduce_kernel<2,32,true>", "stage_grad_reduce_kernel", "mm_backward_kernel<32,true>"}
    e = expected_kernels(1000, 100, 100, "rbf", True)
    assert {"tc2_fwd_kernel<128,128,4,0>", "tc2_bwd_kernel<128,128,2,3,0>", "tc_reduce_kernel<1,128,false>",
            "mm_backward_kernel<16,false>"} <= e
    assert "tc_reduce_kernel<2,64,false>" in expected_kernels(5, 64, 256, "rbf", True)
    # GPBLUR_TC=-1: FFMA at Mp = 256; two 64-point CTAs do not fit at Dp = 128, so 32-point tiles unless N is large
    e = expected_kernels(1000, 100, 256, "rbf", True, ffma_forced=True)
    assert {"point_fwd_kernel<TileCfg<2,8,128>,0>", "point_bwd_kernel<TileCfg<4,8,128>,128,0>",
            "reduce_gemm_kernel<128,128,true>", "reduce_gemm_kernel<128,128,false>"} <= e
    assert 2 * fwd_smem_bytes(64, 128, 256) > K_SMEM_CAP
    assert "point_fwd_kernel<TileCfg<8,8,128>,0>" in expected_kernels(40000, 100, 256, "rbf", False, ffma_forced=True)
    assert "point_fwd_kernel<TileCfg<2,8,128>,0>" in expected_kernels(40000, 128, 1024, "rbf", False, ffma_forced=True)


def test_knob_cells_cover_every_knob_only_instantiation():
    got = set()
    for N, D, M, kind in KNOB_CELLS:
        got |= expected_kernels(N, D, M, kind, True, ffma_forced=True)
    assert got - REACHABLE == KNOB_ONLY, sorted(KNOB_ONLY ^ (got - REACHABLE))


def test_kernel_id_spellings():
    assert kernel_id("void gpblur::(anonymous namespace)::point_fwd_kernel<gpblur::TileCfg<2, 4, 32>, 0>"
                     "(gpblur::PointFwdArgs)") == "point_fwd_kernel<TileCfg<2,4,32>,0>"
    assert kernel_id("void gpblur::<unnamed>::tc_reduce_kernel<(int)2, (int)64, (bool)1>(gpblur::<unnamed>::A)") \
        == "tc_reduce_kernel<2,64,true>"
    assert kernel_id("gpblur::(anonymous namespace)::stage_grad_reduce_kernel(gpblur::SgReduceArgs)") \
        == "stage_grad_reduce_kernel"


def _compiled_kernel_ids():
    lib = os.path.join(ROOT, "fine_grained_gaussian_process_forcasting_b200", "libgpblur.so")
    cuda_bin = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")
    objdump = shutil.which("cuobjdump") or os.path.join(cuda_bin, "cuobjdump")
    filt = shutil.which("cu++filt") or os.path.join(cuda_bin, "cu++filt")
    if not (os.path.exists(lib) and os.path.exists(objdump) and os.path.exists(filt)):
        pytest.skip("library not built or CUDA binary utilities not found")
    syms = subprocess.run([objdump, "-symbols", lib], capture_output=True, text=True, timeout=120).stdout
    mangled = sorted(set(re.findall(r"_Z\w+", syms)))
    names = subprocess.run([filt], input="\n".join(mangled), capture_output=True, text=True, timeout=120).stdout
    return svgp_kernel_ids(kernel_id(n) for n in names.splitlines())


def test_compiled_instantiations_are_all_accounted_for():
    """Every SVGP point / reduction / stage kernel compiled into the library is reachable (and has a cell), reachable
    through GPBLUR_TC=-1 only, or listed as not dispatched; a new instantiation must be added to one of them."""
    compiled = _compiled_kernel_ids()
    listed = REACHABLE | KNOB_ONLY | NOT_DISPATCHED
    assert compiled - listed == set(), sorted(compiled - listed)
    assert listed - compiled == set(), sorted(listed - compiled)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: oracle parity per cell
# ---------------------------------------------------------------------------------------------------------------------
SEED, OFFSET, STREAM, GKL = 1234, 77, 3, 0.37


def _chunk(M, D):
    """Points per oracle chunk: the direct differences are [M, chunk, D] float64."""
    return max(128, min(4096, (1 << 25) // (M * D)))


def rel(a, b):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-300)).item()


def rel_rows(a, b, scale=None):
    """max|a - b| of each row against that row's own scale (max|b| of the row, or `scale` [rows]), worst row: a row of
    small values cannot hide behind larger rows of the same tile."""
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    s = b.abs().amax(1) if scale is None else scale
    return ((a - b).abs().amax(1) / (s + 1e-300)).max().item()


# A = k Linv^T cancels: |a_n| <= sqrt(os), while the terms it sums, |k| |Linv|^T, grow with the conditioning of Kzz.
# The 3xTF32 / FP32 error of a row follows the size of the terms (about 7e-7 of it on the tensor cores), so the row
# scale is max(max|a_n|, max(|k_n| |Linv|^T) / A_CANCEL).  Every cell has a term / value ratio <= 26 except
# N = 882, D = 20, M = 700 (700 inducing points in 20 dimensions, max|Linv| = 13), where it reaches 151 and the
# worst row, measured against max|a_n| alone, is off by 1.1e-4 on a B200.
A_CANCEL = 50


def _inputs(N, D, M, kind):
    seed = (N * 31 + D * 7 + M) * 4 + KIND_ID[kind]
    p32 = O.init_params_exercise(D, M, seed=seed)
    x32 = O.make_inputs(1, N, D, seed=seed + 1)[0].reshape(N, D)
    g = torch.Generator().manual_seed(seed + 2)
    gm, gv, gs = (torch.randn(N, generator=g) for _ in range(3))
    return p32, x32, gm, gv, gs


def _stage_fp64(p64, kind):
    Z = p64["inducing_points"].detach()
    M, D = Z.shape
    ell = O.softplus(p64["raw_lengthscale"].detach()).reshape(D)
    os_ = O.softplus(p64["raw_outputscale"].detach())
    Kzz = MO.scale_direct(Z, Z, ell, os_, kind) + O.JITTER * torch.eye(M, dtype=torch.float64)
    Lc = torch.linalg.cholesky(Kzz)
    Linv = torch.linalg.solve_triangular(Lc, torch.eye(M, dtype=torch.float64), upper=False)
    return Kzz, Lc, Linv, ell, os_


def oracle(kind, p32, x32, gm, gv, gs, eps, training):
    """float64 closed form (matern_oracle) of mean / var / sample and, when `training`, autograd of
    sum(gm mean + gv var + gs sample) + GKL kl.  Points are independent given the parameters, so the points are taken
    in chunks: the parameter gradients accumulate over the chunks, dx is per chunk."""
    N, D = x32.shape
    p64 = O.clone_params(p32, torch.float64, requires_grad=training)
    mean, var, dx = [], [], []
    chunk = _chunk(p32["inducing_points"].shape[0], D)
    for c in range(0, N, chunk):
        xc = x32[c:c + chunk].double().requires_grad_(training)
        with torch.set_grad_enabled(training):
            mo, vo = MO.svgp_predict_closed_form(p64, xc.reshape(1, -1, D), kernel=kind)
            mo, vo = mo.reshape(-1), vo.reshape(-1)
            if training:
                sl = slice(c, c + xc.shape[0])
                so = O.rsample(mo, vo, eps[sl])
                ((gm[sl].double() * mo).sum() + (gv[sl].double() * vo).sum() + (gs[sl].double() * so).sum()).backward()
                dx.append(xc.grad)
        mean.append(mo.detach())
        var.append(vo.detach())
    kl = O.kl_meanfield(p64)
    if training:
        (GKL * kl).backward()
    grads = {k: p64[k].grad for k in NAMES} if training else None
    return torch.cat(mean), torch.cat(var), kl.detach(), (torch.cat(dx) if training else None), grads


def _launched(prof):
    evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return svgp_kernel_ids(kernel_id(e.name) for e in evs)


def run_cuda(kind, p32, x32, gm, gv, gs, training):
    """The four split-form entry points (param stage, point forward, point backward, stage backward) on one cell, under
    torch.profiler.  Returns the outputs, the probes and the launched SVGP kernel ids."""
    from torch.profiler import profile, ProfilerActivity
    from fine_grained_gaussian_process_forcasting_b200 import ops
    dev = torch.device("cuda")
    N, D = x32.shape
    M = p32["inducing_points"].shape[0]
    k = KIND_ID[kind]
    args = [p32["inducing_points"], p32["raw_lengthscale"].reshape(-1), p32["raw_outputscale"].reshape(1),
            p32["variational_mean"], p32["variational_stddev"], p32["weights"].reshape(-1), p32["bias"]]
    args = [t.to(dev).contiguous() for t in args]
    xd = x32.to(dev)
    r = {}
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        # the trace keeps only kernels whose device timestamps fall inside its window: give the window a head start
        # over the first launch, which is the M x M stage
        time.sleep(0.02)
        stage, kl, info = ops.param_stage_raw(*args, kind=k)
        mean, var, sample, ws = ops.point_forward_raw(stage, xd, M, SEED, OFFSET, STREAM, True, True, kind=k)
        torch.cuda.synchronize()
        r["A"] = ops.debug_fetch(3, N, D, M, ws).cpu()
        if training:
            dx, sgrad = ops.point_backward_raw(xd, M, gm.to(dev), gv.to(dev), gs.to(dev), var, SEED, OFFSET, STREAM,
                                               ws, stage=stage, kind=k)
            bucket = ops.param_stage_backward_raw(*args, sgrad, torch.tensor([GKL], device=dev), stage, kind=k)
        torch.cuda.synchronize()
    assert int(info.item()) == 0
    r["launched"] = _launched(prof)
    r.update(mean=mean.cpu(), var=var.cpu(), sample=sample.cpu(), kl=kl.cpu())
    r["Kzz"], r["L"], r["Linv"] = (ops.debug_fetch(w, 0, D, M, stage).cpu()[:M, :M] for w in (2, 0, 1))
    if training:
        r["W"] = ops.debug_fetch(5, N, D, M, ws).cpu()
        r["g"] = ops.debug_fetch(6, N, D, M, ws).cpu()
        r["dx"] = dx.cpu()
        views = ops.split_bucket(bucket, D, M, True)
        r["grads"] = {n: v.cpu() for n, v in zip(NAMES, views)}
    return r


def _tile_rows(N, T):
    """Row ranges of the last (ragged) tile and of one interior tile of height T."""
    last0 = (N - 1) // T * T
    mid0 = (N // T // 2) * T
    return slice(last0, N), (slice(mid0, mid0 + T) if mid0 + T <= last0 else None)


def check_cell(N, D, M, kind):
    MP = padded_m(M)
    tc = tc_point_supported(MP, N)
    p32, x32, gm, gv, gs = _inputs(N, D, M, kind)
    eps = torch.from_numpy(O.philox_normal(SEED, OFFSET, N, STREAM)).double()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    r = run_cuda(kind, p32, x32, gm, gv, gs, True)
    want = expected_kernels(N, D, M, kind, True, sms=sms)
    assert r["launched"] == want, (sorted(r["launched"]), sorted(want))
    t0 = time.time()
    mo, vo, klo, dxo, go = oracle(kind, p32, x32, gm, gv, gs, eps, True)
    t_oracle = time.time() - t0
    so = O.rsample(mo, vo, eps)
    tile = TC_TILE if tc else ffma_fwd_tile(N, padded_d(D), MP, sms)
    tail, mid = _tile_rows(N, tile)
    errs = {"mean": rel(r["mean"], mo), "var": rel(r["var"], vo), "sample": rel(r["sample"], so),
            "mean_tail": rel(r["mean"][tail], mo[tail]), "var_tail": rel(r["var"][tail], vo[tail]),
            "kl": abs(r["kl"].item() - klo.item()) / max(1.0, abs(klo.item()))}
    # M x M stage
    Kzz, Lc, Linv, ell, os_ = _stage_fp64(O.clone_params(p32, torch.float64), kind)
    errs["Kzz"], errs["L"], errs["Linv"] = rel(r["Kzz"], Kzz), rel(torch.tril(r["L"]), Lc), rel(torch.tril(r["Linv"]), Linv)
    # A = k Linv^T, row by row on the tail tile and one interior tile; padded columns exactly zero
    A = r["A"]
    assert A.shape == (N, MP)
    if MP > M:
        assert A[:, M:].abs().max().item() == 0.0, "padded columns of A are not zero"
    Z64 = p32["inducing_points"].double()
    rows = {"tail": tail} if mid is None else {"tail": tail, "mid": mid}
    A64 = {}
    for nm, sl in rows.items():
        K, G = MO.scale_direct_kg(x32[sl].double(), Z64, ell, os_, kind)
        A64[nm] = (K @ Linv.t(), G)
        terms = (K.abs() @ Linv.abs().t()).amax(1)
        errs["A_" + nm] = rel_rows(A[sl, :M], A64[nm][0], torch.maximum(A64[nm][0].abs().amax(1), terms / A_CANCEL))
    tol = TOL_FWD_TC if tc else TOL_FWD
    # W = kbar o k (RBF) or kbar o g (Matern), kbar_n = Linv^T (g_mu,n m + 2 g_var,n (s^2 - 1) o a_n), from the
    # folded upstream gradients of probe 6
    mvec = p32["variational_mean"].double()
    s2m1 = p32["variational_stddev"].double() ** 2 - 1
    for nm, sl in rows.items():
        a64, G = A64[nm]
        gmu, gvar = r["g"][0, sl].double(), r["g"][1, sl].double()
        kbar = (gmu[:, None] * mvec + 2 * gvar[:, None] * s2m1 * a64) @ Linv
        errs["W_" + nm] = rel(r["W"][sl, :M], kbar * G)
    if MP > M:
        assert r["W"][:, M:].abs().max().item() == 0.0, "padded columns of W are not zero"
    errs["dx"] = rel(r["dx"], dxo)
    errs["dx_tail"] = rel(r["dx"][tail], dxo[tail])
    for n in NAMES:
        errs[n] = rel(r["grads"][n].reshape(go[n].shape), go[n])
    if errs["raw_outputscale"] >= TOL_GRAD:
        # one number, a sum of terms of both signs: measured against the size of the terms (test_gpu_matern)
        scale = oracle(kind, p32, x32, gm.abs(), gv.abs(), gs.abs(), eps, True)[4]["raw_outputscale"].abs()
        errs["raw_outputscale"] = ((r["grads"]["raw_outputscale"].double().reshape(()) - go["raw_outputscale"]).abs()
                                   / torch.maximum(go["raw_outputscale"].abs(), scale)).item()
    print(f"cell N={N} D={D} M={M} {kind} [{'tc' if tc else 'ffma'}, oracle {t_oracle:.1f}s] "
          f"{' '.join(sorted(r['launched']))} | " + " ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    for k in ("mean", "var", "sample", "mean_tail", "var_tail", "A_tail", "A_mid"):
        if k in errs:
            assert errs[k] < tol, (k, errs)
    assert errs["kl"] < 1e-5, errs
    assert errs["Kzz"] < 1e-6 and errs["L"] < 1e-6 and errs["Linv"] < 1e-5, errs
    for k in ("W_tail", "W_mid", "dx", "dx_tail") + tuple(NAMES):
        if k in errs:
            assert errs[k] < TOL_GRAD, (k, errs)


@pytest.mark.gpu
@pytest.mark.parametrize("N,D,M,kind", CELLS, ids=[_cell_id(c) for c in CELLS])
def test_cell_against_oracle(cuda, N, D, M, kind):
    check_cell(N, D, M, kind)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: segmented backward
# ---------------------------------------------------------------------------------------------------------------------
# (D, M, kind, segment sizes, segment without a sample gradient): boundaries at odd offsets inside the 64-point FFMA
# backward tiles / 128-point tensor-core tiles, one empty segment each.
SEG_CASES = [
    (32, 32, "rbf", (301, 0, 555, 144), 2),
    (100, 128, "matern52", (131, 0, 517, 353), 3),
    (20, 600, "matern32", (77, 389, 0, 435), 0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("D,M,kind,sizes,nosample", SEG_CASES, ids=["ffma", "tc128", "tc768"])
def test_segments_against_oracle(cuda, D, M, kind, sizes, nosample):
    """ops.svgp_predict_segments over 4 segments (one empty, one without a sample gradient): the whole backward
    against the float64 oracle of the same loss on the concatenated points."""
    from fine_grained_gaussian_process_forcasting_b200 import ops
    N = sum(sizes)
    p32, x32, gm, gv, gs = _inputs(N, D, M, kind)
    gs_used = gs.clone()
    starts = [sum(sizes[:i]) for i in range(len(sizes))]
    gs_used[starts[nosample]:starts[nosample] + sizes[nosample]] = 0.0
    dev = torch.device("cuda")
    pd = {k: p32[k].to(dev).requires_grad_(True) for k in NAMES}
    xd = x32.to(dev).requires_grad_(True)
    segs, kl, info = ops.svgp_predict_segments(xd, [(n,) for n in sizes], *(pd[k] for k in NAMES), SEED, OFFSET,
                                               STREAM, want_sample=True, kernel=kind)
    loss = GKL * kl.sum()
    for i, ((mean, var, sample), s0, n) in enumerate(zip(segs, starts, sizes)):
        sl = slice(s0, s0 + n)
        loss = loss + (gm[sl].to(dev) * mean).sum() + (gv[sl].to(dev) * var).sum()
        if i != nosample:
            loss = loss + (gs[sl].to(dev) * sample).sum()
    loss.backward()
    torch.cuda.synchronize()
    assert int(info.max().item()) == 0
    eps = torch.from_numpy(O.philox_normal(SEED, OFFSET, N, STREAM)).double()
    mo, vo, _, dxo, go = oracle(kind, p32, x32, gm, gv, gs_used, eps, True)
    mean = torch.cat([s[0].detach().cpu() for s in segs])
    errs = {"mean": rel(mean, mo), "dx": rel(xd.grad, dxo)}
    for i, (s0, n) in enumerate(zip(starts, sizes)):
        if n:
            errs[f"dx_seg{i}"] = rel(xd.grad[s0:s0 + n], dxo[s0:s0 + n])
    errs.update({k: rel(pd[k].grad.reshape(go[k].shape), go[k]) for k in NAMES})
    print(f"segments {sizes} D={D} M={M} {kind}: " + " ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    assert errs["mean"] < (TOL_FWD_TC if M > 32 else TOL_FWD), errs
    for k, v in errs.items():
        assert v < TOL_GRAD, (k, errs)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the FFMA kernels at Mp >= 128, reachable through GPBLUR_TC=-1 only (read once per process: a child process)
# ---------------------------------------------------------------------------------------------------------------------
# the tensor-core shapes M in {100, 256} x D in {20, 100}, plus the shapes that reach the other knob-only kernels:
# 64-point forward tiles with Dp = 16 and Dp = 64 (N >= 64 SMs), and 128-point forward tiles (N >= 256 SMs, where two
# 64-point CTAs do not fit: Mp = 256 with Dp = 128)
KNOB_CELLS = [(1000, 20, 100, "rbf"), (1000, 100, 256, "rbf"), (777, 100, 100, "rbf"), (777, 20, 256, "rbf"),
              (9600, 5, 100, "rbf"), (9601, 64, 128, "rbf"), (38000, 72, 200, "rbf")]

_CHILD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[2])
import test_gpu_dispatch_matrix as T
import torch
from oracle import gp_oracle as O
res = []
for N, D, M, kind in T.KNOB_CELLS:
    p32, x32, gm, gv, gs = T._inputs(N, D, M, kind)
    eps = torch.from_numpy(O.philox_normal(T.SEED, T.OFFSET, N, T.STREAM)).double()
    r = T.run_cuda(kind, p32, x32, gm, gv, gs, True)
    mo, vo, klo, dxo, go = T.oracle(kind, p32, x32, gm, gv, gs, eps, True)
    e = {"mean": T.rel(r["mean"], mo), "var": T.rel(r["var"], vo), "sample": T.rel(r["sample"], O.rsample(mo, vo, eps)),
         "dx": T.rel(r["dx"], dxo)}
    e.update({k: T.rel(r["grads"][k].reshape(go[k].shape), go[k]) for k in T.NAMES})
    res.append({"cell": [N, D, M, kind], "launched": sorted(r["launched"]), "errs": e,
                "sms": torch.cuda.get_device_properties(0).multi_processor_count})
print("RESULT " + json.dumps(res))
"""


@pytest.mark.gpu
def test_ffma_forced_by_knob(cuda):
    """GPBLUR_TC=-1 forces the FP32 FFMA point kernels at Mp >= 128: an independent second implementation at the
    shapes of the tensor-core cells, against the same oracle."""
    env = dict(os.environ, GPBLUR_TC="-1")
    p = subprocess.run([sys.executable, "-c", _CHILD, ROOT, os.path.dirname(os.path.abspath(__file__))], env=env,
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-4000:]
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    launched = set()
    for c in json.loads(line[len("RESULT "):]):
        launched |= set(c["launched"])
        N, D, M, kind = c["cell"]
        print(f"GPBLUR_TC=-1 N={N} D={D} M={M}: {' '.join(c['launched'])} | "
              + " ".join(f"{k}={v:.1e}" for k, v in c["errs"].items()))
        assert set(c["launched"]) == expected_kernels(N, D, M, kind, True, sms=c["sms"], ffma_forced=True)
        for k in ("mean", "var", "sample"):
            assert c["errs"][k] < TOL_FWD, (k, c)
        for k in ["dx"] + NAMES:
            assert c["errs"][k] < TOL_GRAD, (k, c)
    assert launched - REACHABLE == KNOB_ONLY
