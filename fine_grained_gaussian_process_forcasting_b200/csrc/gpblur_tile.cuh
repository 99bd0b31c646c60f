// Register-tiled FP32 FFMA GEMM core shared by the per-point kernels.
//
// Thread layout of a 256-thread CTA for an output tile [TN points] x [CW columns]:
//   TXN = CW / CT lanes along the columns, TYN = 256 / TXN groups along the points,
//   each thread owns PT consecutive points x CT columns (CT = 4: cols tx*4..+3;
//   CT = 8: cols tx*4..+3 and CW/2 + tx*4..+3, so that every LDS.128 of a warp is contiguous).
// A operands are POINT-major in shared memory ([n][k], read as float4 along k),
// B operands are K-major ([k][c], read as float4 along c).
#pragma once
#include "gpblur_common.cuh"

namespace gpblur {

template <int PT_, int CT_, int CW_>
struct TileCfg {
  static constexpr int PT = PT_, CT = CT_, CW = CW_;
  static constexpr int TXN = CW / CT;
  static constexpr int TYN = kThreads / TXN;
  static constexpr int TN = TYN * PT;
  static_assert(CT == 4 || CT == 8, "CT");
  static_assert(TXN * TYN == kThreads, "layout");
  __device__ static __forceinline__ int tx() { return threadIdx.x % TXN; }
  __device__ static __forceinline__ int ty() { return threadIdx.x / TXN; }
  // column (within the chunk) of micro-tile element f
  __device__ static __forceinline__ int col(int tx, int f) {
    return (CT == 4 || f < 4) ? tx * 4 + f : CW / 2 + tx * 4 + (f - 4);
  }
};

// acc[e][f] += sum_{k < KS} A[(ty*PT + e)][k] * B[k][col(f)]
template <class Cfg>
__device__ __forceinline__ void mma_slice(float (&acc)[Cfg::PT][Cfg::CT], const float* __restrict__ As,
                                          int lda, const float* __restrict__ Bs, int ldb, int tx, int ty) {
  constexpr int PT = Cfg::PT, CT = Cfg::CT, CW = Cfg::CW;
#pragma unroll
  for (int k4 = 0; k4 < kKS; k4 += 4) {
    float4 a4[PT];
#pragma unroll
    for (int e = 0; e < PT; ++e)
      a4[e] = *reinterpret_cast<const float4*>(As + (size_t)(ty * PT + e) * lda + k4);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      float b[CT];
      const float4 b0 = *reinterpret_cast<const float4*>(Bs + (size_t)(k4 + kk) * ldb + tx * 4);
      b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
      if (CT == 8) {
        const float4 b1 = *reinterpret_cast<const float4*>(Bs + (size_t)(k4 + kk) * ldb + CW / 2 + tx * 4);
        b[CT - 4] = b1.x; b[CT - 3] = b1.y; b[CT - 2] = b1.z; b[CT - 1] = b1.w;
      }
#pragma unroll
      for (int e = 0; e < PT; ++e) {
        const float av = kk == 0 ? a4[e].x : kk == 1 ? a4[e].y : kk == 2 ? a4[e].z : a4[e].w;
#pragma unroll
        for (int f = 0; f < CT; ++f) acc[e][f] = fmaf(av, b[f], acc[e][f]);
      }
    }
  }
}

// cp.async a [KS rows][W floats] slice of a row-major global matrix into dense shared memory [KS][W]
template <int W>
__device__ __forceinline__ void stage_rows(float* dst, const float* __restrict__ src, size_t ld,
                                           int row0, int col0) {
  constexpr int CH = W / 4;
  for (int idx = threadIdx.x; idx < kKS * CH; idx += kThreads) {
    const int r = idx / CH, cq = idx - r * CH;
    cp_async16(dst + r * W + cq * 4, src + (size_t)(row0 + r) * ld + col0 + cq * 4);
  }
}

// cp.async a [TN rows][KS floats] slice (rows = points, clamped to nmax-1) into shared [TN][KS + 4]
template <int TN>
__device__ __forceinline__ void stage_points(float* dst, const float* __restrict__ src, size_t ld,
                                             long long n0, long long nmax, int col0) {
  constexpr int CH = kKS / 4;
  for (int idx = threadIdx.x; idx < TN * CH; idx += kThreads) {
    const int r = idx / CH, cq = idx - r * CH;
    long long n = n0 + r;
    if (n >= nmax) n = nmax - 1;
    cp_async16(dst + r * (kKS + 4) + cq * 4, src + (size_t)n * ld + col0 + cq * 4);
  }
}

struct PointFwdArgs {
  WsLayout L;
  void* ws;
  const void* stage;   // parameter stage (== ws when the stage was built in the workspace)
  const float* x;
  float* mean;
  float* var;
  float* sample;
  uint64_t seed, offset;
  uint32_t stream_id;
  int ntiles;
  const unsigned long long* offset_dev;   // optional device-resident addend of `offset` (CUDA-graph replays)
};

// Upstream gradients of a point backward, given per SEGMENT of the point range (several activations of one training
// step evaluated in one call): segment s covers points [start[s], start[s + 1]) and brings its own (nullable)
// g_mean / g_var / g_sample arrays, indexed from the start of the segment.  1 <= nseg <= kMaxSegments, start[0] = 0.
constexpr int kMaxSegments = 4;
struct SegGrads {
  int nseg;
  long long start[kMaxSegments];
  const float* gm[kMaxSegments];
  const float* gv[kMaxSegments];
  const float* gs[kMaxSegments];
};
__device__ __forceinline__ void upstream_grads(const SegGrads& sg, long long gn, float& gm, float& gv, float& gsv,
                                               bool& has_gs) {
  // one segment (every single-call backward): the pointers are fixed kernel-parameter loads, no indexed lookup in
  // front of the gradient loads
  const float *pm = sg.gm[0], *pv = sg.gv[0], *ps = sg.gs[0];
  long long ln = gn;
  if (sg.nseg > 1) {
    int s = 0;
#pragma unroll
    for (int i = 1; i < kMaxSegments; ++i)
      if (i < sg.nseg && gn >= sg.start[i]) s = i;
    pm = sg.gm[s]; pv = sg.gv[s]; ps = sg.gs[s];
    ln = gn - sg.start[s];
  }
  gm = pm ? pm[ln] : 0.f;
  gv = pv ? pv[ln] : 0.f;
  has_gs = ps != nullptr;
  gsv = ps ? ps[ln] : 0.f;
}

struct PointBwdArgs {
  WsLayout L;
  void* ws;
  const void* stage;   // parameter stage (== ws when the stage was built in the workspace)
  const float* x;
  const float* var;
  uint64_t seed, offset;
  uint32_t stream_id;
  float* dx;
  int ntiles;
  const unsigned long long* offset_dev;
  SegGrads seg;
};

// Stage a [TN][DP] tile of X into shared memory, centred and scaled: Xs[n][d] = (x - c) / ell (0 beyond N, D).
template <int TN>
__device__ __forceinline__ void stage_x_tile(float* Xs, int ldx, const float* __restrict__ x, long long n0,
                                             long long N, int D, int DP, const float* __restrict__ center,
                                             const float* __restrict__ inv_ell) {
  const int dq_n = DP / 4;
  const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  for (int idx = threadIdx.x; idx < TN * dq_n; idx += kThreads) {
    const int n = idx / dq_n, d = (idx - n * dq_n) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const long long gn = n0 + n;
    if (gn < N && d < D) {
      const float* row = x + (size_t)gn * D;
      if (vec) {
        v = *reinterpret_cast<const float4*>(row + d);
      } else {
        v.x = row[d];
        if (d + 1 < D) v.y = row[d + 1];
        if (d + 2 < D) v.z = row[d + 2];
        if (d + 3 < D) v.w = row[d + 3];
      }
      const float4 c = *reinterpret_cast<const float4*>(center + d);
      const float4 ie = *reinterpret_cast<const float4*>(inv_ell + d);
      v.x = (v.x - c.x) * ie.x; v.y = (v.y - c.y) * ie.y;
      v.z = (v.z - c.z) * ie.z; v.w = (v.w - c.w) * ie.w;
    }
    *reinterpret_cast<float4*>(Xs + (size_t)n * ldx + d) = v;
  }
}

// K-loop of one output chunk with a double-buffered cp.async B operand (rows k0.. of `bsrc`, cols c0..c0+CW)
// and a resident point-major A operand in shared memory.
template <class Cfg>
__device__ __forceinline__ void gemm_resident_a(float (&acc)[Cfg::PT][Cfg::CT], const float* As, int lda,
                                                const float* __restrict__ bsrc, size_t ldb_g, int k0, int k1,
                                                int c0, float* Bst, int tx, int ty) {
  constexpr int CW = Cfg::CW;
  const int nsl = (k1 - k0) / kKS;
  stage_rows<CW>(Bst, bsrc, ldb_g, k0, c0);
  cp_async_commit();
  for (int s = 0; s < nsl; ++s) {
    if (s + 1 < nsl) {
      stage_rows<CW>(Bst + ((s + 1) & 1) * kKS * CW, bsrc, ldb_g, k0 + (s + 1) * kKS, c0);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    mma_slice<Cfg>(acc, As + k0 + s * kKS, lda, Bst + (s & 1) * kKS * CW, CW, tx, ty);
    __syncthreads();
  }
}

}  // namespace gpblur
