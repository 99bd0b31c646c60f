"""Prints the phase timestamps of the M x M kernels (debug probe 4) for a few M."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from fine_grained_gaussian_process_forcasting_b200 import ops
from oracle import gp_oracle as O
dev = torch.device("cuda")
for M in (32, 128, 256, 1024):
    D, B, L = 64, 64, 24
    p = {k: v.to(dev).requires_grad_(True) for k, v in O.init_params_exercise(D, M, 1).items()}
    x = torch.randn(B * L, D, device=dev)
    for it in range(int(os.environ.get("ITERS", "300"))):
        mean, var, sample, kl, info, ws = ops.svgp_forward_raw(x, p["inducing_points"].detach(), p["raw_lengthscale"].detach().reshape(-1),
            p["raw_outputscale"].detach().reshape(1), p["variational_mean"].detach(), p["variational_stddev"].detach(),
            p["weights"].detach().reshape(-1), p["bias"].detach(), 0, 0, 0, False, True)
        g = torch.ones_like(mean)
        dx, bucket = ops.svgp_backward_raw(x, p["inducing_points"].detach(), p["raw_lengthscale"].detach().reshape(-1),
            p["raw_outputscale"].detach().reshape(1), p["variational_mean"].detach(), p["variational_stddev"].detach(),
            p["weights"].detach().reshape(-1), p["bias"].detach(), g, g, None, None, var, 0, 0, 0, ws)
    torch.cuda.synchronize()
    t = ops.debug_fetch(4, B * L, D, M, ws).cpu().tolist()
    f = [(t[i + 1] - t[i]) / 1e3 for i in range(0, 7)]
    b = [(t[16 + i + 1] - t[16 + i]) / 1e3 for i in range(0, 4)]
    print(f"M={M}: fwd phases us [p0, p1 Kzz, p2 chol+inv, -, -, p4 fp32 operands, TF32 slab images] = {[round(v,1) for v in f]} total {sum(f):.1f}")
    print(f"        tail (not in the total): beta {(t[13]-t[7])/1e3:.1f} us, zn {(t[8]-t[13])/1e3:.1f} us")
    print(f"        first diagonal block: load {(t[10]-t[9])/1e3:.1f} us, chol32 {(t[11]-t[10])/1e3:.1f} us, trinv32 {(t[12]-t[11])/1e3:.1f} us")
    print(f"        bwd phases us [A Tm = P Linv, B sym(Kbar) + Wzz, C V = Wzz Z~, D bucket] = {[round(v,1) for v in b]} total {sum(b):.1f}")
