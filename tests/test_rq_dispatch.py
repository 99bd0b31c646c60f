"""The rational quadratic point kernels compiled into libgpblur.so, against the dispatch rules.

The RQ instantiations of the point kernels are entry points of their own (point_fwd_rq_kernel, point_bwd_rq_kernel,
tc2_fwd_rq_kernel, tc2_bwd_rq_kernel) over the same templated bodies as the RBF / Matern kernels, which
tests/test_gpu_dispatch_matrix.py accounts for.  RQ takes the Matern routes (FP32-FFMA kernels for M <= 32 only,
tensor cores above; the M x M stage instantiation of the non-RBF kinds), so its reachable kernels are the Matern ones
renamed.  Every compiled RQ kernel must be reachable from some shape of that mirror or be a tile-height-override
instantiation, and every reachable one must be compiled.
"""
import re

import test_gpu_dispatch_matrix as T

RQ_FAMILIES = ("point_fwd_rq_kernel", "point_bwd_rq_kernel", "tc2_fwd_rq_kernel", "tc2_bwd_rq_kernel")


def rq_name(kid):
    """Kernel id of a Matern-kind (kind 1) instantiation -> the RQ kernel that the same shape launches."""
    m = re.fullmatch(r"(point_fwd_kernel|point_bwd_kernel|tc2_fwd_kernel|tc2_bwd_kernel)<(.*),1>", kid)
    if not m:
        return kid                                   # stage / reduction kernels: shared with the Matern kinds
    return m.group(1).replace("_kernel", "_rq_kernel") + "<" + m.group(2) + ">"


def expected_rq_kernels(N, D, M, training, sms=T.B200_SMS):
    return {rq_name(k) for k in T.expected_kernels(N, D, M, "matern12", training, sms=sms)}


REACHABLE_RQ = set()
for _c in T.CELLS:
    REACHABLE_RQ |= {k for k in expected_rq_kernels(_c[0], _c[1], _c[2], True) if k.split("<")[0] in RQ_FAMILIES}
# 128-point FFMA tiles at M <= 32: only with GPBLUR_FWD_TN / GPBLUR_BWD_TN = 128 (as for the other kinds)
NOT_DISPATCHED_RQ = {"point_fwd_rq_kernel<TileCfg<4,4,32>>"}
NOT_DISPATCHED_RQ |= {f"point_bwd_rq_kernel<TileCfg<4,4,32>,{dp}>" for dp in (16, 32, 64, 128)}


def test_rq_mirror_rows():
    e = expected_rq_kernels(9500, 32, 32, True)
    assert {"point_fwd_rq_kernel<TileCfg<2,4,32>>", "point_bwd_rq_kernel<TileCfg<2,4,32>,32>",
            "mm_small_forward_kernel<true>", "mm_small_backward_kernel<true>"} <= e
    e = expected_rq_kernels(1000, 20, 600, True)
    assert {"tc2_fwd_rq_kernel<128,256,3>", "tc2_bwd_rq_kernel<128,32,3,4>", "mm_forward_kernel<true>",
            "mm_backward_kernel<32,true>"} <= e
    assert len(REACHABLE_RQ) == 11


def test_compiled_rq_instantiations_are_all_accounted_for():
    import os
    import shutil
    import subprocess
    import pytest
    lib = os.path.join(T.ROOT, "fine_grained_gaussian_process_forcasting_b200", "libgpblur.so")
    cuda_bin = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")
    objdump = shutil.which("cuobjdump") or os.path.join(cuda_bin, "cuobjdump")
    filt = shutil.which("cu++filt") or os.path.join(cuda_bin, "cu++filt")
    if not (os.path.exists(lib) and os.path.exists(objdump) and os.path.exists(filt)):
        pytest.skip("library not built or CUDA binary utilities not found")
    syms = subprocess.run([objdump, "-symbols", lib], capture_output=True, text=True, timeout=120).stdout
    mangled = sorted(set(re.findall(r"_Z\w+", syms)))
    names = subprocess.run([filt], input="\n".join(mangled), capture_output=True, text=True, timeout=120).stdout
    compiled = {T.kernel_id(n) for n in names.splitlines()}
    compiled = {k for k in compiled if k.split("<")[0] in RQ_FAMILIES}
    listed = REACHABLE_RQ | NOT_DISPATCHED_RQ
    assert compiled == listed, (sorted(compiled - listed), sorted(listed - compiled))
