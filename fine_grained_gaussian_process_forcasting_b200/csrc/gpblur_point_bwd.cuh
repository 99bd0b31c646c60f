// Per-point fused backward of the whitened SVGP predictive (hand-written replacement for torch autograd
// through gpytorch's kernel / solve / matmul chain; SURVEY Appendix A):
//
//   g_mu, g_var  <- upstream (mean, variance, reparameterised sample folded, variance clamp respected)
//   k            <- recomputed from X and the staged Z~ tiles (stage A, as in the forward)
//   kbar[n, :]   = g_mu[n] beta + 2 g_var[n] (diag(c) Linv)^T a[n, :]        block-triangular GEMM on saved A
//   W            = kbar o k ;  r[n] = sum_m W ;  colsum[m] = sum_n W     (Matern / RQ kinds: W = kbar o g)
//   dx[n, :]     = ( W Z~ - r x~ ) / ell + g_mu w                             GEMM on the resident W chunk
// W is also written to HBM once: the N-reduction GEMMs (gpblur_reduce.cu) turn it into dZ / d lengthscale.
// Per-CTA vector partials (colsum, q = sum r x~^2, wbar, scalar sums) are reduced by the M x M stage.
#pragma once
#include "gpblur_tile.cuh"

namespace gpblur {

template <class Cfg, int DP>
struct BwdSmem {
  static constexpr int TN = Cfg::TN, CW = Cfg::CW;
  static constexpr int ldx = DP + 4, lda = kKS + 4, ldw = CW + 4;
  static constexpr int BZ = (CW > DP ? CW : DP);      // B-operand slice width (LC / ZtT slices or Zt slices)
  static constexpr size_t floats(int MP) {
    return (size_t)TN * ldx + 2 * TN * lda + 2 * kKS * BZ + (size_t)TN * ldw + (size_t)Cfg::TYN * CW + MP +
           5 * TN + 3 * DP + 256 + 16;
  }
};

// KIND (GPBLUR_KERNEL_*): for the Matern / RQ kinds the recomputed chunk holds d2 instead of k, and step (c) forms
// W = kbar o g and the sum of kbar o k (vector partial slot VS_KBK) from it; RQ also the sum of kbar o dk/dalpha
// (VS_KBA).  The body sits behind the entry points point_bwd_kernel (RBF, Matern) and point_bwd_rq_kernel (RQ).
template <class Cfg, int DP, int KIND>
__device__ __forceinline__ void point_bwd_body(const PointBwdArgs& a) {
  constexpr int PT = Cfg::PT, CT = Cfg::CT, CW = Cfg::CW, TN = Cfg::TN, TXN = Cfg::TXN, TYN = Cfg::TYN;
  using S = BwdSmem<Cfg, DP>;
  constexpr int ldx = S::ldx, lda = S::lda, ldw = S::ldw, BZ = S::BZ;
  constexpr int DPQ = DP / 4;                 // lanes along d in the dx GEMM
  constexpr int NG = kThreads / DPQ;          // point groups in the dx GEMM
  constexpr int PX = (TN >= NG) ? TN / NG : 1;
  constexpr int NPART = kThreads / DP;        // row partitions for the per-d reductions

  extern __shared__ __align__(16) float smem[];
  const WsLayout& L = a.L;
  const int D = L.D, M = L.M, MP = L.MP;
  const long long N = L.N;

  float* Xs = smem;                               // [TN][ldx]
  float* Ast = Xs + TN * ldx;                     // [2][TN][lda]
  float* Bst = Ast + 2 * TN * lda;                // [2][KS][BZ]
  float* Ws = Bst + 2 * kKS * BZ;                 // [TN][ldw]
  float* colpart = Ws + TN * ldw;                 // [TYN][CW]
  float* colsum_s = colpart + TYN * CW;           // [MP]
  float* xn_s = colsum_s + MP;                    // [TN]
  float* gmu_s = xn_s + TN;
  float* gvar_s = gmu_s + TN;
  float* rs_s = gvar_s + TN;
  float* spare_s = rs_s + TN;                     // [TN]
  float* q_s = spare_s + TN;                      // [DP] accumulators across tiles
  float* t1_s = q_s + DP;                         // [DP]
  float* dred = t1_s + DP;                        // [DP] unused pad
  float* dpart = dred + DP;                       // [NPART][DP] = 256 floats
  float* sc_s = dpart + 256;                   // [16] scalar accumulators

  const float* hyp = ws_cptr<float>(a.stage, L.hyp);
  const float* inv_ell = ws_cptr<float>(a.stage, L.inv_ell);
  const float* ellv = ws_cptr<float>(a.stage, L.ell);
  const float* center = ws_cptr<float>(a.stage, L.center);
  const float* wl = ws_cptr<float>(a.stage, L.wl);
  const float* Zt = ws_cptr<float>(a.stage, L.Zt);
  const float* ZtT = ws_cptr<float>(a.stage, L.ZtT);
  const float* zn = ws_cptr<float>(a.stage, L.zn);
  const float* beta = ws_cptr<float>(a.stage, L.beta);
  const float* LC = ws_cptr<float>(a.stage, L.LC32);
  const float* Ag = ws_cptr<float>(a.ws, L.A);
  float* Wg = ws_ptr<float>(a.ws, L.W);
  float* vecpart = ws_ptr<float>(a.ws, L.vecpart);
  float* gsc = ws_ptr<float>(a.ws, L.gsc);        // [2][N] folded g_mu, g_var for the Gram reduction

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = Cfg::tx(), ty = Cfg::ty();
  const int txd = tid % DPQ, tyd = tid / DPQ;
  const float os = hyp[H_OS];

  for (int i = tid; i < MP; i += kThreads) colsum_s[i] = 0.f;
  for (int i = tid; i < DP; i += kThreads) { q_s[i] = 0.f; t1_s[i] = 0.f; }
  if (tid < 16) sc_s[tid] = 0.f;
  float kbk_acc = 0.f;                            // Matern / RQ kinds: this thread's share of sum kbar o k
  float kba_acc = 0.f;                            // RQ: this thread's share of sum kbar o dk/dalpha
  const float alpha = KIND == GPBLUR_KERNEL_RQ ? hyp[H_ALPHA] : 0.f, i2a = KIND == GPBLUR_KERNEL_RQ ? hyp[H_I2A] : 0.f;

  for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
    const long long n0 = (long long)tile * TN;
    __syncthreads();
    stage_x_tile<TN>(Xs, ldx, a.x, n0, N, D, DP, center, inv_ell);
    // fold the upstream gradients of mean / variance / sample into (g_mu, g_var)
    for (int t = tid; t < TN; t += kThreads) {
      const long long gn = n0 + t;
      float gm = 0.f, gv = 0.f;
      if (gn < N) {
        float gs;
        bool has_gs;
        upstream_grads(a.seg, gn, gm, gv, gs, has_gs);
        const float v = a.var[gn];
        if (has_gs) {
          const float eps = philox_normal(a.seed, rng_offset(a.offset, a.offset_dev) + (uint64_t)gn, a.stream_id);
          gm += gs;
          gv = fmaf(gs * eps, 0.5f * rsqrtf(v), gv);
        }
        if (v <= kMinVariance) gv = 0.f;    // clamp active in the forward: no gradient through var
      }
      gmu_s[t] = gm;
      gvar_s[t] = gv;
      if (gn < N) { gsc[gn] = gm; gsc[N + gn] = gv; }
    }
    __syncthreads();
    for (int n = warp; n < TN; n += kThreads / 32) {
      float s2 = 0.f;
      for (int d = lane; d < DP; d += 32) {
        const float v = Xs[n * ldx + d];
        s2 = fmaf(v, v, s2);
      }
      s2 = warp_sum(s2);
      if (lane == 0) xn_s[n] = s2;
    }
    __syncthreads();

    float rsum_p[PT];
#pragma unroll
    for (int e = 0; e < PT; ++e) rsum_p[e] = 0.f;
    float xacc[PX][4];
#pragma unroll
    for (int e = 0; e < PX; ++e) { xacc[e][0] = xacc[e][1] = xacc[e][2] = xacc[e][3] = 0.f; }

    for (int jc = 0; jc < MP; jc += CW) {
      // ---- (a) recompute the cross-covariance chunk, park it in Ws ----
      {
        float acc[PT][CT];
#pragma unroll
        for (int e = 0; e < PT; ++e)
#pragma unroll
          for (int f = 0; f < CT; ++f) acc[e][f] = 0.f;
        // B slices are [KS][CW] dense inside the (possibly wider) staging buffer
        gemm_resident_a<Cfg>(acc, Xs, ldx, ZtT, (size_t)MP, 0, DP, jc, Bst, tx, ty);
#pragma unroll
        for (int e = 0; e < PT; ++e) {
          const int n = ty * PT + e;
          const float xn = xn_s[n];
          float kv[CT];
#pragma unroll
          for (int f = 0; f < CT; ++f) {
            const int m = jc + Cfg::col(tx, f);
            const float d2 = fmaxf(xn + zn[m] - 2.0f * acc[e][f], 0.f);
            if constexpr (KIND == GPBLUR_KERNEL_RBF) kv[f] = (m < M) ? os * expf(-0.5f * d2) : 0.f;
            else kv[f] = (m < M) ? d2 : 1e30f;   // padded columns: k = g = 0
          }
          *reinterpret_cast<float4*>(Ws + (size_t)n * ldw + tx * 4) = make_float4(kv[0], kv[1], kv[2], kv[3]);
          if (CT == 8)
            *reinterpret_cast<float4*>(Ws + (size_t)n * ldw + CW / 2 + tx * 4) =
                make_float4(kv[CT - 4], kv[CT - 3], kv[CT - 2], kv[CT - 1]);
        }
      }
      // ---- (b) kbar chunk: sum_{i >= jc} a[n][i] * LC[i][jc + col] with both operands streamed ----
      float acc[PT][CT];
#pragma unroll
      for (int e = 0; e < PT; ++e)
#pragma unroll
        for (int f = 0; f < CT; ++f) acc[e][f] = 0.f;
      {
        const int nsl = (MP - jc) / kKS;
        stage_points<TN>(Ast, Ag, (size_t)MP, n0, N, jc);
        stage_rows<CW>(Bst, LC, (size_t)MP, jc, jc);
        cp_async_commit();
        for (int s = 0; s < nsl; ++s) {
          if (s + 1 < nsl) {
            stage_points<TN>(Ast + ((s + 1) & 1) * TN * lda, Ag, (size_t)MP, n0, N, jc + (s + 1) * kKS);
            stage_rows<CW>(Bst + ((s + 1) & 1) * kKS * BZ, LC, (size_t)MP, jc + (s + 1) * kKS, jc);
            cp_async_commit();
            cp_async_wait<1>();
          } else {
            cp_async_wait<0>();
          }
          __syncthreads();
          mma_slice<Cfg>(acc, Ast + (s & 1) * TN * lda, lda, Bst + (s & 1) * kKS * BZ, CW, tx, ty);
          __syncthreads();
        }
      }
      // ---- (c) W = kbar o k ; row / column sums ; write W ----
      {
        float bet[CT], cpart[CT];
#pragma unroll
        for (int f = 0; f < CT; ++f) { bet[f] = beta[jc + Cfg::col(tx, f)]; cpart[f] = 0.f; }
#pragma unroll
        for (int e = 0; e < PT; ++e) {
          const int n = ty * PT + e;
          const float gm = gmu_s[n], gv2 = 2.0f * gvar_s[n];
          float4 k0 = *reinterpret_cast<const float4*>(Ws + (size_t)n * ldw + tx * 4);
          float kk[CT];
          kk[0] = k0.x; kk[1] = k0.y; kk[2] = k0.z; kk[3] = k0.w;
          if (CT == 8) {
            const float4 k1 = *reinterpret_cast<const float4*>(Ws + (size_t)n * ldw + CW / 2 + tx * 4);
            kk[CT - 4] = k1.x; kk[CT - 3] = k1.y; kk[CT - 2] = k1.z; kk[CT - 1] = k1.w;
          }
          float w[CT];
#pragma unroll
          for (int f = 0; f < CT; ++f) {
            const float kb = fmaf(gv2, acc[e][f], gm * bet[f]);
            if constexpr (KIND == GPBLUR_KERNEL_RBF) {
              w[f] = kb * kk[f];
            } else if constexpr (KIND == GPBLUR_KERNEL_RQ) {
              float kv, g, ka;
              rq_kg(kk[f], os, alpha, i2a, kv, g, ka);
              if (!(kk[f] < 1e20f)) { kv = 0.f; g = 0.f; ka = 0.f; }   // padded column (d2 = 1e30)
              w[f] = kb * g;
              kbk_acc = fmaf(kb, kv, kbk_acc);
              kba_acc = fmaf(kb, ka, kba_acc);
            } else {
              float kv, g;
              matern_kg<KIND>(kk[f], os, kv, g);
              w[f] = kb * g;
              kbk_acc = fmaf(kb, kv, kbk_acc);
            }
            rsum_p[e] += w[f];
            cpart[f] += w[f];
          }
          *reinterpret_cast<float4*>(Ws + (size_t)n * ldw + tx * 4) = make_float4(w[0], w[1], w[2], w[3]);
          if (CT == 8)
            *reinterpret_cast<float4*>(Ws + (size_t)n * ldw + CW / 2 + tx * 4) =
                make_float4(w[CT - 4], w[CT - 3], w[CT - 2], w[CT - 1]);
          const long long gn = n0 + n;
          if (gn < N) {
            float* row = Wg + (size_t)gn * MP + jc;
            *reinterpret_cast<float4*>(row + tx * 4) = make_float4(w[0], w[1], w[2], w[3]);
            if (CT == 8)
              *reinterpret_cast<float4*>(row + CW / 2 + tx * 4) =
                  make_float4(w[CT - 4], w[CT - 3], w[CT - 2], w[CT - 1]);
          }
        }
#pragma unroll
        for (int f = 0; f < CT; ++f) colpart[ty * CW + Cfg::col(tx, f)] = cpart[f];
      }
      __syncthreads();
      for (int c = tid; c < CW; c += kThreads) {
        float s = 0.f;
#pragma unroll 4
        for (int g = 0; g < TYN; ++g) s += colpart[g * CW + c];
        colsum_s[jc + c] += s;
      }
      // ---- (d) dx accumulators: xacc += W[:, chunk] * Z~[chunk, :] ----
      {
        constexpr int nsl = CW / kKS;
        stage_rows<DP>(Bst, Zt, (size_t)DP, jc, 0);
        cp_async_commit();
        for (int s = 0; s < nsl; ++s) {
          if (s + 1 < nsl) {
            stage_rows<DP>(Bst + ((s + 1) & 1) * kKS * BZ, Zt, (size_t)DP, jc + (s + 1) * kKS, 0);
            cp_async_commit();
            cp_async_wait<1>();
          } else {
            cp_async_wait<0>();
          }
          __syncthreads();
          if (tyd * PX < TN) {
            const float* Bs = Bst + (s & 1) * kKS * BZ;
#pragma unroll
            for (int k4 = 0; k4 < kKS; k4 += 4) {
              float4 a4[PX];
#pragma unroll
              for (int e = 0; e < PX; ++e)
                a4[e] = *reinterpret_cast<const float4*>(Ws + (size_t)(tyd * PX + e) * ldw + s * kKS + k4);
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                const float4 b = *reinterpret_cast<const float4*>(Bs + (k4 + kk) * DP + txd * 4);
#pragma unroll
                for (int e = 0; e < PX; ++e) {
                  const float av = kk == 0 ? a4[e].x : kk == 1 ? a4[e].y : kk == 2 ? a4[e].z : a4[e].w;
                  xacc[e][0] = fmaf(av, b.x, xacc[e][0]);
                  xacc[e][1] = fmaf(av, b.y, xacc[e][1]);
                  xacc[e][2] = fmaf(av, b.z, xacc[e][2]);
                  xacc[e][3] = fmaf(av, b.w, xacc[e][3]);
                }
              }
            }
          }
          __syncthreads();
        }
      }
    }  // chunks

    // ---- row sums of W over the TXN lanes sharing a point ----
#pragma unroll
    for (int e = 0; e < PT; ++e) {
#pragma unroll
      for (int o = TXN / 2; o > 0; o >>= 1) rsum_p[e] += __shfl_xor_sync(0xffffffffu, rsum_p[e], o);
      if (tx == 0) rs_s[ty * PT + e] = rsum_p[e];
    }
    __syncthreads();

    // ---- dx ----
    if (a.dx && tyd * PX < TN) {
      const int d = txd * 4;
      const float4 ie = *reinterpret_cast<const float4*>(inv_ell + d);
      const float4 wv = *reinterpret_cast<const float4*>(wl + d);
      const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.dx) & 15) == 0);
#pragma unroll
      for (int e = 0; e < PX; ++e) {
        const int n = tyd * PX + e;
        const long long gn = n0 + n;
        if (gn < N && d < D) {
          const float r = rs_s[n], gm = gmu_s[n];
          const float4 xv = *reinterpret_cast<const float4*>(Xs + (size_t)n * ldx + d);
          float4 o;
          o.x = (xacc[e][0] - r * xv.x) * ie.x + gm * (wv.x * ie.x);
          o.y = (xacc[e][1] - r * xv.y) * ie.y + gm * (wv.y * ie.y);
          o.z = (xacc[e][2] - r * xv.z) * ie.z + gm * (wv.z * ie.z);
          o.w = (xacc[e][3] - r * xv.w) * ie.w + gm * (wv.w * ie.w);
          float* row = a.dx + (size_t)gn * D;
          if (vec) {
            *reinterpret_cast<float4*>(row + d) = o;
          } else {
            row[d] = o.x;
            if (d + 1 < D) row[d + 1] = o.y;
            if (d + 2 < D) row[d + 2] = o.z;
            if (d + 3 < D) row[d + 3] = o.w;
          }
        }
      }
    }
    // ---- per-d reductions over the tile: q_d += sum_n r x~^2 ; t1_d += sum_n g_mu x~ ----
    {
      const int d = tid % DP, part = tid / DP;
      constexpr int ROWS = TN / NPART;
      float qs = 0.f, ts = 0.f;
      for (int n = part * ROWS; n < (part + 1) * ROWS; ++n) {
        const float v = Xs[(size_t)n * ldx + d];
        qs = fmaf(rs_s[n] * v, v, qs);
        ts = fmaf(gmu_s[n], v, ts);
      }
      dpart[part * DP + d] = qs;
      __syncthreads();
      if (part == 0) {
        float s = 0.f;
        for (int p2 = 0; p2 < NPART; ++p2) s += dpart[p2 * DP + d];
        q_s[d] += s;
      }
      __syncthreads();
      dpart[part * DP + d] = ts;
      __syncthreads();
      if (part == 0) {
        float s = 0.f;
        for (int p2 = 0; p2 < NPART; ++p2) s += dpart[p2 * DP + d];
        t1_s[d] += s;
      }
    }
    if (warp == 0) {
      float sg = 0.f, sr = 0.f, sv = 0.f;
      for (int n = lane; n < TN; n += 32) { sg += gmu_s[n]; sr += rs_s[n]; sv += gvar_s[n]; }
      sg = warp_sum(sg); sr = warp_sum(sr); sv = warp_sum(sv);
      if (lane == 0) { sc_s[VS_GMU] += sg; sc_s[VS_RSUM] += sr; sc_s[VS_GVAR] += sv; }
    }
  }  // tiles

  if constexpr (KIND != GPBLUR_KERNEL_RBF) {                // fixed order: lanes, then warps
    __syncthreads();
    const float s = warp_sum(kbk_acc);
    if (lane == 0) dpart[warp] = s;
    __syncthreads();
    if (tid == 0) {
      float t = 0.f;
      for (int w8 = 0; w8 < kThreads / 32; ++w8) t += dpart[w8];
      sc_s[VS_KBK] = t;
    }
  }
  if constexpr (KIND == GPBLUR_KERNEL_RQ) {
    __syncthreads();
    const float s = warp_sum(kba_acc);
    if (lane == 0) dpart[warp] = s;
    __syncthreads();
    if (tid == 0) {
      float t = 0.f;
      for (int w8 = 0; w8 < kThreads / 32; ++w8) t += dpart[w8];
      sc_s[VS_KBA] = t;
    }
  }
  __syncthreads();
  float* vp = vecpart + (size_t)blockIdx.x * L.vp_len;
  for (int i = tid; i < MP; i += kThreads) vp[i] = colsum_s[i];
  for (int d = tid; d < DP; d += kThreads) {
    vp[MP + d] = q_s[d];
    // wbar_d = sum_n g_mu x_nd = ell_d * sum_n g_mu x~_nd + c_d * sum_n g_mu
    vp[MP + DP + d] = (d < D) ? ellv[d] * t1_s[d] + center[d] * sc_s[VS_GMU] : 0.f;
  }
  if (tid < VS_PART) vp[MP + 2 * DP + tid] = sc_s[tid];
}

template <class Cfg, int DP, int KIND>
__global__ void __launch_bounds__(kThreads, Cfg::TN <= 64 ? 2 : 1) point_bwd_kernel(PointBwdArgs a) {
  point_bwd_body<Cfg, DP, KIND>(a);
}
template <class Cfg, int DP>
__global__ void __launch_bounds__(kThreads, Cfg::TN <= 64 ? 2 : 1) point_bwd_rq_kernel(PointBwdArgs a) {
  point_bwd_body<Cfg, DP, GPBLUR_KERNEL_RQ>(a);
}

// tile height used by the backward for a given problem (shared with the M x M stage, which needs the
// number of vector partials)
inline int bwd_tile_points(const WsLayout& L) {
  const int force = tile_override("GPBLUR_BWD_TN");
  if (force == 128 && L.DP != 128) return 128;
  if (force == 64) return 64;
  // 64-point tiles: <= 128 registers and ~90 KB shared memory -> two CTAs (16 warps) per SM
  return 64;
}

inline int bwd_persistent_grid(const WsLayout& L, int TN) {
  const long long nt = (L.N + TN - 1) / TN;
  return (int)(nt < kMaxPersist ? (nt < 1 ? 1 : nt) : kMaxPersist);
}

template <class Cfg, int DP, int KIND>
int launch_bwd_kind(const PointBwdArgs& a0, cudaStream_t st) {
  PointBwdArgs a = a0;
  const size_t smem = sizeof(float) * BwdSmem<Cfg, DP>::floats(a.L.MP);
  auto* kernel = [] {
    if constexpr (KIND == GPBLUR_KERNEL_RQ) return point_bwd_rq_kernel<Cfg, DP>;
    else return point_bwd_kernel<Cfg, DP, KIND>;
  }();
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   // per device
  a.ntiles = (int)((a.L.N + Cfg::TN - 1) / Cfg::TN);
  const int grid = bwd_persistent_grid(a.L, Cfg::TN);
  ProfScope ps(ST_POINT_BWD, st);
  kernel<<<grid, kThreads, smem, st>>>(a);
  note_launch();
  return check_launch("point_bwd");
}

template <class Cfg, int DP>
int launch_bwd_cfg(const PointBwdArgs& a, cudaStream_t st) {
  // the Matern / RQ kinds run on the FP32-FFMA kernels for MP = 32 only (MP >= 128 takes the tensor-core kernels)
  if constexpr (Cfg::CW != 32) {
    if (a.L.kind != GPBLUR_KERNEL_RBF) return GPBLUR_EUNSUPPORTED;
    return launch_bwd_kind<Cfg, DP, GPBLUR_KERNEL_RBF>(a, st);
  } else {
    switch (a.L.kind) {
      case GPBLUR_KERNEL_MATERN12: return launch_bwd_kind<Cfg, DP, GPBLUR_KERNEL_MATERN12>(a, st);
      case GPBLUR_KERNEL_MATERN32: return launch_bwd_kind<Cfg, DP, GPBLUR_KERNEL_MATERN32>(a, st);
      case GPBLUR_KERNEL_MATERN52: return launch_bwd_kind<Cfg, DP, GPBLUR_KERNEL_MATERN52>(a, st);
      case GPBLUR_KERNEL_RQ: return launch_bwd_kind<Cfg, DP, GPBLUR_KERNEL_RQ>(a, st);
      default: return launch_bwd_kind<Cfg, DP, GPBLUR_KERNEL_RBF>(a, st);
    }
  }
}

template <int DP>
int dispatch_bwd_dp(const PointBwdArgs& a, cudaStream_t st) {
  const int TN = bwd_tile_points(a.L);
  if (a.L.MP == 32) {
    if (TN == 128) return launch_bwd_cfg<TileCfg<4, 4, 32>, DP>(a, st);
    return launch_bwd_cfg<TileCfg<2, 4, 32>, DP>(a, st);
  }
  if (a.L.MP == 64) {
    if (TN == 128) return launch_bwd_cfg<TileCfg<8, 4, 64>, DP>(a, st);
    return launch_bwd_cfg<TileCfg<4, 4, 64>, DP>(a, st);
  }
  if (TN == 128) return launch_bwd_cfg<TileCfg<8, 8, 128>, DP>(a, st);
  return launch_bwd_cfg<TileCfg<4, 8, 128>, DP>(a, st);
}

}  // namespace gpblur
