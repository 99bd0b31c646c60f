// Per-point fused forward of the whitened SVGP predictive (replaces, per DeepGPp.predict call,
// gpytorch's cat/expand + three batched kernel builds + fp64 trsm_batched + the small mean/variance
// kernels; /root/reference/denoising_model/DeepGP.py:56-73,94-99 via VariationalStrategy.forward):
//
//   stage A  k[n, m]  = os * exp(-1/2 |x~_n - z~_m|^2)          norm expansion, FP32 FFMA, Z~ tiles staged
//            (Matern / RQ kinds: os f of the same d2, gpblur_common.cuh: matern_kg / rq_kg)
//   stage B  a[n, :]  = Linv k[n, :]                             block-triangular GEMM, K resident in smem
//   epilogue mean = a.m + x.w + b ; var = max(os + jitter + sum (s^2-1) a^2, 1e-6) ;
//            sample = mean + sqrt(var) * PhiloxNormal(seed, offset + n)
// The cross-covariance tile K never leaves shared memory; A is written once for the backward when training.
#include "gpblur_tile.cuh"

namespace gpblur {

namespace {

// The body sits behind the entry points point_fwd_kernel (RBF, Matern) and point_fwd_rq_kernel (RQ).
template <class Cfg, int KIND>
__device__ __forceinline__ void point_fwd_body(const PointFwdArgs& a) {
  constexpr int PT = Cfg::PT, CT = Cfg::CT, CW = Cfg::CW, TN = Cfg::TN;
  extern __shared__ __align__(16) float smem[];
  const WsLayout& L = a.L;
  const int D = L.D, DP = L.DP, M = L.M, MP = L.MP;
  const long long N = L.N;
  const int ldx = DP + 4, ldk = MP + 4;
  float* Xs = smem;                       // [TN][ldx]
  float* Ks = Xs + TN * ldx;              // [TN][ldk]
  float* Bst = Ks + TN * ldk;             // [2][KS][CW]
  float* xn_s = Bst + 2 * kKS * CW;       // [TN] |x~|^2
  float* xw_s = xn_s + TN;                // [TN] linear mean
  float* mu_s = xw_s + TN;                // [TN]
  float* vv_s = mu_s + TN;                // [TN]

  const float* hyp = ws_cptr<float>(a.stage, L.hyp);
  const float* inv_ell = ws_cptr<float>(a.stage, L.inv_ell);
  const float* center = ws_cptr<float>(a.stage, L.center);
  const float* wl = ws_cptr<float>(a.stage, L.wl);
  const float* ZtT = ws_cptr<float>(a.stage, L.ZtT);
  const float* zn = ws_cptr<float>(a.stage, L.zn);
  const float* mvec = ws_cptr<float>(a.stage, L.mvec);
  const float* cvec = ws_cptr<float>(a.stage, L.cvec);
  const float* LinvT = ws_cptr<float>(a.stage, L.LinvT32);
  float* Ag = ws_ptr<float>(a.ws, L.A);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = Cfg::tx(), ty = Cfg::ty();
  const float os = hyp[H_OS], jit = hyp[H_JIT], cwb = hyp[H_CWB];
  const float alpha = KIND == GPBLUR_KERNEL_RQ ? hyp[H_ALPHA] : 0.f, i2a = KIND == GPBLUR_KERNEL_RQ ? hyp[H_I2A] : 0.f;

  for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
    const long long n0 = (long long)tile * TN;
    __syncthreads();
    stage_x_tile<TN>(Xs, ldx, a.x, n0, N, D, DP, center, inv_ell);
    __syncthreads();
    // row norms and linear mean
    for (int n = warp; n < TN; n += kThreads / 32) {
      float s2 = 0.f, sw = 0.f;
      for (int d = lane; d < DP; d += 32) {
        const float v = Xs[n * ldx + d];
        s2 = fmaf(v, v, s2);
        sw = fmaf(v, wl[d], sw);
      }
      s2 = warp_sum(s2);
      sw = warp_sum(sw);
      if (lane == 0) { xn_s[n] = s2; xw_s[n] = sw; }
    }
    __syncthreads();

    // ---- stage A: cross-covariance tile ----
    for (int mc = 0; mc < MP; mc += CW) {
      float acc[PT][CT];
#pragma unroll
      for (int e = 0; e < PT; ++e)
#pragma unroll
        for (int f = 0; f < CT; ++f) acc[e][f] = 0.f;
      gemm_resident_a<Cfg>(acc, Xs, ldx, ZtT, (size_t)MP, 0, DP, mc, Bst, tx, ty);
#pragma unroll
      for (int e = 0; e < PT; ++e) {
        const int n = ty * PT + e;
        const float xn = xn_s[n];
        float kv[CT];
#pragma unroll
        for (int f = 0; f < CT; ++f) {
          const int m = mc + Cfg::col(tx, f);
          const float d2 = fmaxf(xn + zn[m] - 2.0f * acc[e][f], 0.f);
          if constexpr (KIND == GPBLUR_KERNEL_RBF) {
            kv[f] = (m < M) ? os * expf(-0.5f * d2) : 0.f;
          } else if constexpr (KIND == GPBLUR_KERNEL_RQ) {
            float g, ka;
            rq_kg(d2, os, alpha, i2a, kv[f], g, ka);
            if (m >= M) kv[f] = 0.f;
          } else {
            float g;
            matern_kg<KIND>(d2, os, kv[f], g);
            if (m >= M) kv[f] = 0.f;
          }
        }
        *reinterpret_cast<float4*>(Ks + (size_t)n * ldk + mc + tx * 4) = make_float4(kv[0], kv[1], kv[2], kv[3]);
        if (CT == 8)
          *reinterpret_cast<float4*>(Ks + (size_t)n * ldk + mc + CW / 2 + tx * 4) =
              make_float4(kv[CT - 4], kv[CT - 3], kv[CT - 2], kv[CT - 1]);
      }
    }
    __syncthreads();

    // ---- stage B: whitening a = Linv k, fused mean / variance ----
    float mu_p[PT], vv_p[PT];
#pragma unroll
    for (int e = 0; e < PT; ++e) { mu_p[e] = 0.f; vv_p[e] = 0.f; }
    for (int ic = 0; ic < MP; ic += CW) {
      float acc[PT][CT];
#pragma unroll
      for (int e = 0; e < PT; ++e)
#pragma unroll
        for (int f = 0; f < CT; ++f) acc[e][f] = 0.f;
      gemm_resident_a<Cfg>(acc, Ks, ldk, LinvT, (size_t)MP, 0, ic + CW, ic, Bst, tx, ty);
      float mv[CT], cv[CT];
#pragma unroll
      for (int f = 0; f < CT; ++f) {
        const int i = ic + Cfg::col(tx, f);
        mv[f] = mvec[i];
        cv[f] = cvec[i];
      }
#pragma unroll
      for (int e = 0; e < PT; ++e) {
#pragma unroll
        for (int f = 0; f < CT; ++f) {
          const float av = acc[e][f];
          mu_p[e] = fmaf(av, mv[f], mu_p[e]);
          vv_p[e] = fmaf(cv[f] * av, av, vv_p[e]);
        }
        if (L.training) {
          const long long gn = n0 + ty * PT + e;
          if (gn < N) {
            float* row = Ag + (size_t)gn * MP + ic;
            *reinterpret_cast<float4*>(row + tx * 4) = make_float4(acc[e][0], acc[e][1], acc[e][2], acc[e][3]);
            if (CT == 8)
              *reinterpret_cast<float4*>(row + CW / 2 + tx * 4) =
                  make_float4(acc[e][CT - 4], acc[e][CT - 3], acc[e][CT - 2], acc[e][CT - 1]);
          }
        }
      }
    }
    // reduce the partial sums over the TXN lanes that share a point
#pragma unroll
    for (int e = 0; e < PT; ++e) {
#pragma unroll
      for (int o = Cfg::TXN / 2; o > 0; o >>= 1) {
        mu_p[e] += __shfl_xor_sync(0xffffffffu, mu_p[e], o);
        vv_p[e] += __shfl_xor_sync(0xffffffffu, vv_p[e], o);
      }
      if (tx == 0) { mu_s[ty * PT + e] = mu_p[e]; vv_s[ty * PT + e] = vv_p[e]; }
    }
    __syncthreads();
    for (int t = tid; t < TN; t += kThreads) {
      const long long gn = n0 + t;
      if (gn < N) {
        const float mean = mu_s[t] + xw_s[t] + cwb;
        const float var = fmaxf(os + jit + vv_s[t], kMinVariance);
        a.mean[gn] = mean;
        a.var[gn] = var;
        if (a.sample) {
          const float eps = philox_normal(a.seed, rng_offset(a.offset, a.offset_dev) + (uint64_t)gn, a.stream_id);
          a.sample[gn] = fmaf(sqrtf(var), eps, mean);
        }
      }
    }
  }
}

template <class Cfg, int KIND>
__global__ void __launch_bounds__(kThreads, Cfg::PT <= 4 ? 2 : 1) point_fwd_kernel(PointFwdArgs a) {
  point_fwd_body<Cfg, KIND>(a);
}
template <class Cfg>
__global__ void __launch_bounds__(kThreads, Cfg::PT <= 4 ? 2 : 1) point_fwd_rq_kernel(PointFwdArgs a) {
  point_fwd_body<Cfg, GPBLUR_KERNEL_RQ>(a);
}

template <class Cfg>
size_t fwd_smem_bytes(const WsLayout& L) {
  return sizeof(float) * ((size_t)Cfg::TN * (L.DP + 4) + (size_t)Cfg::TN * (L.MP + 4) + 2 * kKS * Cfg::CW +
                          4 * Cfg::TN);
}

template <class Cfg, int KIND>
int launch_fwd_kind(const PointFwdArgs& a0, cudaStream_t st) {
  PointFwdArgs a = a0;
  const size_t smem = fwd_smem_bytes<Cfg>(a.L);
  auto* kernel = [] {
    if constexpr (KIND == GPBLUR_KERNEL_RQ) return point_fwd_rq_kernel<Cfg>;
    else return point_fwd_kernel<Cfg, KIND>;
  }();
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   // per device
  a.ntiles = (int)((a.L.N + Cfg::TN - 1) / Cfg::TN);
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kThreads, smem);
  if (occ < 1) occ = 1;
  int grid = occ * num_sms();
  if (grid > a.ntiles) grid = a.ntiles;
  if (grid < 1) grid = 1;
  ProfScope ps(ST_POINT_FWD, st);
  kernel<<<grid, kThreads, smem, st>>>(a);
  note_launch();
  return check_launch("point_fwd");
}

template <class Cfg>
int launch_fwd_cfg(const PointFwdArgs& a, cudaStream_t st) {
  // the Matern / RQ kinds run on the FP32-FFMA kernels for MP = 32 only (MP >= 128 takes the tensor-core kernels)
  if constexpr (Cfg::CW != 32) {
    if (a.L.kind != GPBLUR_KERNEL_RBF) return GPBLUR_EUNSUPPORTED;
    return launch_fwd_kind<Cfg, GPBLUR_KERNEL_RBF>(a, st);
  } else {
    switch (a.L.kind) {
      case GPBLUR_KERNEL_MATERN12: return launch_fwd_kind<Cfg, GPBLUR_KERNEL_MATERN12>(a, st);
      case GPBLUR_KERNEL_MATERN32: return launch_fwd_kind<Cfg, GPBLUR_KERNEL_MATERN32>(a, st);
      case GPBLUR_KERNEL_MATERN52: return launch_fwd_kind<Cfg, GPBLUR_KERNEL_MATERN52>(a, st);
      case GPBLUR_KERNEL_RQ: return launch_fwd_kind<Cfg, GPBLUR_KERNEL_RQ>(a, st);
      default: return launch_fwd_kind<Cfg, GPBLUR_KERNEL_RBF>(a, st);
    }
  }
}

constexpr size_t kSmemCap = 220 * 1024;

template <int CT, int CW>
int dispatch_fwd_tn(const PointFwdArgs& a, cudaStream_t st) {
  constexpr int TYN = kThreads / (CW / CT);
  using C128 = TileCfg<128 / TYN, CT, CW>;
  using C64 = TileCfg<64 / TYN, CT, CW>;
  using C32 = TileCfg<32 / TYN, CT, CW>;
  const long long N = a.L.N;
  const int sms = num_sms();
  const int force = tile_override("GPBLUR_FWD_TN");
  if (force == 128 && fwd_smem_bytes<C128>(a.L) <= kSmemCap) return launch_fwd_cfg<C128>(a, st);
  if (force == 64 && fwd_smem_bytes<C64>(a.L) <= kSmemCap) return launch_fwd_cfg<C64>(a, st);
  if (force == 32 && fwd_smem_bytes<C32>(a.L) <= kSmemCap) return launch_fwd_cfg<C32>(a, st);
  // 64-point tiles with two CTAs per SM (16 warps) hide the shared-memory / barrier latency better than one
  // 128-point CTA (ncu r01a: 8 warps/SM, issue slots 61 % busy); fall back to whatever fits in shared memory.
  if (2 * fwd_smem_bytes<C64>(a.L) <= kSmemCap && N >= (long long)64 * sms) return launch_fwd_cfg<C64>(a, st);
  if (fwd_smem_bytes<C128>(a.L) <= kSmemCap && N >= (long long)128 * 2 * sms) return launch_fwd_cfg<C128>(a, st);
  if (fwd_smem_bytes<C64>(a.L) <= kSmemCap && N >= (long long)64 * sms) return launch_fwd_cfg<C64>(a, st);
  if (fwd_smem_bytes<C32>(a.L) <= kSmemCap) return launch_fwd_cfg<C32>(a, st);
  return GPBLUR_EUNSUPPORTED;
}

}  // namespace

int launch_point_forward(const WsLayout& L, const void* stage, void* ws, const float* x, float* mean, float* var,
                         float* sample, uint64_t seed, uint64_t offset, uint32_t stream_id,
                         const unsigned long long* offset_dev, cudaStream_t st) {
  if (L.N <= 0) return GPBLUR_OK;
  PointFwdArgs a{L, ws, stage, x, mean, var, sample, seed, offset, stream_id, 0, offset_dev};
  if (L.MP == 32) return dispatch_fwd_tn<4, 32>(a, st);
  if (L.MP == 64) return dispatch_fwd_tn<4, 64>(a, st);
  return dispatch_fwd_tn<8, 128>(a, st);
}

}  // namespace gpblur
