// Shared definitions for the gpblur sm_100a kernels: workspace layout, Philox, small device helpers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <math.h>

#include "../../include/gpblur.h"

namespace gpblur {

constexpr float kJitter = 1e-4f;        // gpytorch.settings.variational_cholesky_jitter (fp32)
constexpr float kMinVariance = 1e-6f;   // gpytorch.settings.min_variance (fp32)
constexpr float kNoiseLower = 1e-4f;    // GaussianLikelihood GreaterThan(1e-4)
constexpr int kThreads = 256;
constexpr int kKS = 16;                 // K-slice depth of the staged operand tiles
constexpr int kMaxPersist = 296;        // persistent CTAs of the backward point kernel (2 x 148 SMs)
constexpr int kMaxSplits = 148;          // split-K factor cap of the N-reduction GEMMs

// hyp (fp32) slots; H_ALPHA / H_I2A: alpha and 1 / (2 alpha) of the rational quadratic kind (hyp64: H_ALPHA only)
enum { H_OS = 0, H_JIT = 1, H_CWB = 2, H_KL = 3, H_ALPHA = 4, H_I2A = 5, H_COUNT = 8 };
constexpr int kStampSlots = 32;   // phase timestamps (globaltimer ns) of the M x M kernels: [0,16) forward, [16,32) backward
// per-CTA vector partial layout of the backward point kernels: [colsum MP | q DP | wbar DP | scalars VS_PART]
// VS_KBK = sum kbar o k: the outputscale gradient of the Matern and RQ kinds (for RBF, W = kbar o k and VS_RSUM is that
// sum); VS_KBA = sum kbar o dk/dalpha (RQ only).  The stage gradient keeps the first VS_COUNT scalars in its vector
// section (vec_len) and VS_KBA, for RQ only, as its last element (stage_grad_doubles), so that its layout is the same
// for every other kind.
enum { VS_GMU = 0, VS_RSUM = 1, VS_GVAR = 2, VS_KBK = 3, VS_COUNT = 4, VS_KBA = 4, VS_PART = 5 };

// ---- covariance functions (GPBLUR_KERNEL_*, include/gpblur.h) ----------------------------------------------------
// k = os f(r) with r = sqrt(max(d2, 1e-30)), and g = -2 os df/d(d2) = -os f'(r) / r: every distance gradient is the RBF
// one with W = kbar o g in place of kbar o k (for RBF g = k).  g = 0 where the clamp is active (d2 <= 1e-30).  Every
// kernel site evaluates the Matern and RQ kinds through these functions; the RBF sites keep their own exp.
// Rational quadratic (no clamp: d2 enters directly): u = d2 / (2 alpha), k = os (1 + u)^-alpha, g = k / (1 + u), and
// ka = dk/dalpha = k (u / (1 + u) - log1p(u)).
__host__ __device__ constexpr bool kernel_kind_valid(int kind) {
  return kind >= GPBLUR_KERNEL_RBF && kind <= GPBLUR_KERNEL_RQ;
}
__device__ __forceinline__ float ex2_fast(float v) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(v));
  return y;
}
// fp32, the kind a template argument so that the coefficients are immediates
template <int KIND>
__device__ __forceinline__ void matern_kg(float d2, float os, float& k, float& g) {
  static_assert(KIND == GPBLUR_KERNEL_MATERN12 || KIND == GPBLUR_KERNEL_MATERN32 || KIND == GPBLUR_KERNEL_MATERN52,
                "Matern kinds only");
  const float dc = fmaxf(d2, 1e-30f);
  const float ir = rsqrtf(dc), r = dc * ir;
  const bool live = d2 > 1e-30f;
  if constexpr (KIND == GPBLUR_KERNEL_MATERN12) {
    const float e = os * ex2_fast(-1.4426950408889634f * r);
    k = e;
    g = live ? e * ir : 0.f;
  } else if constexpr (KIND == GPBLUR_KERNEL_MATERN32) {
    const float s = 1.7320508075688772f * r, e = os * ex2_fast(-1.4426950408889634f * s);
    k = fmaf(s, e, e);
    g = live ? 3.0f * e : 0.f;
  } else {
    const float s = 2.2360679774997896f * r, e = os * ex2_fast(-1.4426950408889634f * s);
    const float p = 1.0f + s;
    k = fmaf(s * s * (1.0f / 3.0f), e, p * e);
    g = live ? (5.0f / 3.0f) * p * e : 0.f;
  }
}
// fp32 rational quadratic: alpha and i2a = 1 / (2 alpha) from hyp[H_ALPHA] / hyp[H_I2A].  log1pf, not log2(1 + u):
// near the RBF limit (alpha >~ 1e2, u ~ 1e-3) 1 + u rounds and would cost ~1e-4 relative in k.  The caller zeroes
// padded columns.
__device__ __forceinline__ void rq_kg(float d2, float os, float alpha, float i2a, float& k, float& g, float& ka) {
  const float u = d2 * i2a, lp = log1pf(u), q = __frcp_rn(1.0f + u);
  k = os * ex2_fast(-1.4426950408889634f * alpha * lp);
  g = k * q;
  ka = k * (u * q - lp);
}
// fp64 (the M x M stage): any kind; ka = dk/dalpha is set for RQ only (alpha is read for RQ only)
__device__ __forceinline__ void kernel_kg64(int kind, double d2, double os, double alpha, double& k, double& g,
                                            double& ka) {
  if (kind == GPBLUR_KERNEL_RBF) { k = os * exp(-0.5 * d2); g = k; return; }
  if (kind == GPBLUR_KERNEL_RQ) {
    const double u = d2 / (2.0 * alpha), lp = log1p(u), q = 1.0 / (1.0 + u);
    k = os * exp(-alpha * lp);
    g = k * q;
    ka = k * (u * q - lp);
    return;
  }
  const double r = sqrt(fmax(d2, 1e-30));
  const bool live = d2 > 1e-30;
  if (kind == GPBLUR_KERNEL_MATERN12) {
    const double e = os * exp(-r);
    k = e;
    g = live ? e / r : 0.0;
  } else if (kind == GPBLUR_KERNEL_MATERN32) {
    const double s = 1.7320508075688772 * r, e = os * exp(-s);
    k = (1.0 + s) * e;
    g = live ? 3.0 * e : 0.0;
  } else {
    const double s = 2.2360679774997896 * r, e = os * exp(-s);
    k = (1.0 + s + s * s / 3.0) * e;
    g = live ? (5.0 / 3.0) * (1.0 + s) * e : 0.0;
  }
}

__host__ __device__ inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
__host__ __device__ inline long long round_up_ll(long long a, long long b) { return (a + b - 1) / b * b; }

// padded inducing count: 32, 128, or a multiple of 256 (the column-block width of the tensor-core kernels)
__host__ __device__ inline int padded_m(int M) {
  if (M <= 32) return 32;
  // 32 < M <= 64 is padded to 128 and takes the tensor-core path: measured at B = 8192, L = 24, D = 64, M = 64 the
  // FP32-FFMA kernels (MP = 64) need 0.70 ms per step, the tcgen05 kernels on the zero / identity padded MP = 128
  // problem 0.47 ms (the FFMA instantiations for MP = 64 stay compiled but are not dispatched any more)
  if (M <= 128) return 128;
  return round_up(M, 256);
}
// padded input dim: 16, 32, 64 or 128
__host__ __device__ inline int padded_d(int D) {
  if (D <= 16) return 16;
  if (D <= 32) return 32;
  if (D <= 64) return 64;
  return 128;
}

struct WsLayout {
  long long N;
  int D, DP, M, MP;
  int training;
  int splitsS, splitsZ;     // split-K factors of the Gram (its diagonal bands on the tensor-core path) / W^T X
  int splitsO;              // tensor-core path: split-K factor of the off-diagonal Gram units (0: none, MP <= 256)
  int nvec;                 // number of per-CTA vector partials (persistent backward CTAs)
  int vec_len;              // doubles of the stage gradient's vector section: MP + 2 DP + VS_COUNT
  int vp_len;               // floats per vector partial: MP + 2 DP + VS_PART
  // byte offsets
  size_t hyp, hyp64, stamps, inv_ell, ell, center, wl, Zt, ZtT, zn, znc, mvec, cvec, svec, beta;
  size_t K64, L64, Linv64, T64, U64, LinvT32, LC32, Linv32, LCT32;
  size_t ZtU, LinvU, LCTU, ZtTU;   // constant operands pre-split (TF32 hi | lo) in UMMA slab layout (tensor-core path)
  size_t ZtQ;                      // Z~ images in row blocks of tc_bq(MP) (TS-form point kernels)
  size_t LCTQ;                     // (diag(c) Linv)^T images in row blocks of tc_bq(MP) (TS-form backward)
  size_t v64, t64;                 // fp64 scratch of the M x M backward (part of the parameter stage)
  size_t A, W, Spart, upart, WXpart, vecpart, gsc, rrow, cpart, sgrad;
  size_t total;
  size_t D2zz64;            // fp64 inducing-pair distances d2 of the Kzz build (Matern kinds: read by the backward)
  int kind;                 // covariance function (GPBLUR_KERNEL_*); make_layout leaves RBF, the entry points set it
};

// ---- UMMA slab images of the constant operands (tensor-core path) -------------------------------------------
// Every image is [hi plane | lo plane], a plane is [8 k-chunks][rows][4 floats] (64 * rows floats per image).
// The inducing dimension is processed in column blocks of width BW = min(MP, 256).
__host__ __device__ inline int tc_bw(int MP) { return MP >= 256 ? 256 : MP; }
// TS-form point kernels: the cross-covariance logits S are formed in column blocks of BQ = min(MP, 128) inducing points
__host__ __device__ inline int tc_bq(int MP) { return MP >= 128 ? 128 : MP; }
__host__ __device__ inline size_t tc_zq_image(int MP, int nds, int q, int ds) {
  return (size_t)(q * nds + ds) * 64 * tc_bq(MP);
}
// Z~ images: block q (rows m = q BW + r, r < BW), d-slab ds (k = d)
__host__ __device__ inline size_t tc_zt_image(int MP, int nds, int q, int ds) {
  return (size_t)(q * nds + ds) * 64 * tc_bw(MP);
}
// forward Linv images: output block p (rows i in block p), global k-slab s (k = j in [32 s, 32 s + 32)), s < (p + 1) BW / 32.
// rows i run from max(p BW, 32 s) to (p + 1) BW.  Returns the float offset, *rows the row count.
__host__ __device__ inline size_t tc_linv_image(int MP, int p, int s, int* rows) {
  const int BW = tc_bw(MP), spb = BW / 32;
  size_t off = 0;
  for (int pp = 0; pp < p; ++pp)
    off += (size_t)64 * ((size_t)pp * spb * BW + (size_t)BW * spb - (size_t)16 * spb * (spb - 1));
  for (int ss = 0; ss < s; ++ss) {
    const int lo = ss * 32 > p * BW ? ss * 32 : p * BW;
    off += (size_t)64 * ((p + 1) * BW - lo);
  }
  const int lo = s * 32 > p * BW ? s * 32 : p * BW;
  if (rows) *rows = (p + 1) * BW - lo;
  return off;
}
__host__ __device__ inline size_t tc_linv_total(int MP) { return tc_linv_image(MP, MP / tc_bw(MP), 0, nullptr); }
// backward (diag(c) Linv)^T images: column block p (rows j in [p BW, min((p + 1) BW, 32 (s + 1)))), k-slab s >= p BW / 32
__host__ __device__ inline size_t tc_lct_image(int MP, int p, int s, int* rows) {
  const int BW = tc_bw(MP), spb = BW / 32, nsl = MP / 32;
  size_t off = 0;
  for (int pp = 0; pp < p; ++pp) {
    // slabs of block pp itself: rows 32, 64, ..., BW ; slabs above it: BW rows each
    off += (size_t)64 * ((size_t)16 * spb * (spb + 1) + (size_t)(nsl - (pp + 1) * spb) * BW);
  }
  for (int ss = p * spb; ss < s; ++ss) {
    const int r = 32 * (ss + 1) - p * BW;
    off += (size_t)64 * (r < BW ? r : BW);
  }
  const int r = 32 * (s + 1) - p * BW;
  if (rows) *rows = r < BW ? r : BW;
  return off;
}
__host__ __device__ inline size_t tc_lct_total(int MP) { return tc_lct_image(MP, MP / tc_bw(MP), MP / 32, nullptr); }
__host__ __device__ inline size_t tc_slab_ztt(int dpt, int s) { return (size_t)s * 64 * dpt; }
// TS-form backward: (diag(c) Linv)^T images in column blocks of BT = tc_bq(MP): image (p, s), k-slab s >= p BT / 32,
// holds rows j = p BT + r, r < min(BT, 32 (s + 1) - p BT), k = i = 32 s + 4 c + e: value c_i Linv[i][j] (0 for j > i).
// Returns the float offset, *rows the row count.
__host__ __device__ inline size_t tc_lctq_image(int MP, int p, int s, int* rows) {
  const int BT = tc_bq(MP), spb = BT / 32, nsl = MP / 32;
  size_t off = 0;
  for (int pp = 0; pp < p; ++pp)      // slabs of block pp itself: rows 32, 64, ..., BT; slabs above it: BT rows each
    off += (size_t)64 * ((size_t)16 * spb * (spb + 1) + (size_t)(nsl - (pp + 1) * spb) * BT);
  for (int ss = p * spb; ss < s; ++ss) {
    const int r = 32 * (ss + 1) - p * BT;
    off += (size_t)64 * (r < BT ? r : BT);
  }
  const int r = 32 * (s + 1) - p * BT;
  if (rows) *rows = r < BT ? r : BT;
  return off;
}
__host__ __device__ inline size_t tc_lctq_total(int MP) { return tc_lctq_image(MP, MP / tc_bq(MP), MP / 32, nullptr); }

// Tile-major layout of the saved [N, MP] matrices A and W of the tensor-core path: per 128-point tile
// [MP / 4 column pieces][128 rows][4 floats].  A thread that owns one point (row) and 16 consecutive columns writes /
// reads 4 float4, and the 32 lanes of a warp (32 consecutive rows) touch 512 contiguous bytes per instruction instead
// of 32 different lines.  Returns the FLOAT index of element (n, m).
__host__ __device__ inline size_t tc_tiled_index(long long n, int m, int MP) {
  return ((((size_t)(n >> 7) * (size_t)(MP >> 2) + (size_t)(m >> 2)) << 7) + (size_t)(n & 127)) * 4 + (size_t)(m & 3);
}

// Gram partials of the tensor-core path: only the lower triangle of 128 x 128 blocks is computed and stored, packed,
// block (bi, bj), bi >= bj, at block index bi (bi + 1) / 2 + bj, each block row-major.  S is symmetric: an element
// of a block above the diagonal is the element of the mirrored block.  The Gram kernel writes through
// tc_gram_index, stage_grad_reduce reads through its inverse tc_gram_element.
__host__ __device__ inline size_t tc_gram_index(int i, int j) {
  if ((i >> 7) < (j >> 7)) { const int t = i; i = j; j = t; }
  const int bi = i >> 7, bj = j >> 7;
  return ((size_t)(bi * (bi + 1) / 2 + bj) << 14) + ((size_t)(i & 127) << 7) + (size_t)(j & 127);
}
// inverse of tc_gram_index on the stored (lower) blocks: packed float index -> (i, j)
__host__ __device__ inline void tc_gram_element(size_t idx, int* i, int* j) {
  const int b = (int)(idx >> 14);
  int bi = 0;
  while ((bi + 1) * (bi + 2) / 2 <= b) ++bi;
  *i = bi * 128 + (int)((idx >> 7) & 127);
  *j = (b - bi * (bi + 1) / 2) * 128 + (int)(idx & 127);
}
__host__ __device__ inline size_t tc_gram_floats(int MP) { const size_t nb = MP / 128; return nb * (nb + 1) / 2 * 16384; }
// the Gram units are 256-wide column bands (128 at MP = 128): a block inside the diagonal band belongs to that
// band's diagonal unit, every other block to an off-diagonal unit (their split counts differ)
__host__ __device__ inline bool tc_gram_diag_block(int MP, int bi, int bj) {
  const int bw = MP >= 256 ? 2 : 1;
  return bi / bw == bj / bw;
}

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

inline int choose_splits(long long N, int ntiles) {
  // enough CTAs to fill ~2 waves of 148 SMs, each split at least 64 rows deep (FP32-FFMA path, M <= 32: a split walks
  // its rows in 16-row slices behind a two-stage cp.async pipeline, ~0.8 us per slice - with 256-row splits the Gram of
  // configs[0] (6 144 points) ran on 24 CTAs for 19 us)
  long long want = (2 * 148 + ntiles - 1) / ntiles;
  long long maxs = (N + 63) / 64;
  long long s = want < maxs ? want : maxs;
  if (s < 1) s = 1;
  if (s > kMaxSplits) s = kMaxSplits;
  return (int)s;
}

// per-row cost of a W^T X unit per 128 rows of W, relative to one 128 x 128 Gram block, for the split choice below
// (measured at c2 on B200: 0.6 / 1.0 / 1.5 gave 0.362 / 0.351 / 0.359 ms per step)
constexpr double kWxCost = 1.0;

// "Stage gradient": everything the per-point backward of ONE call contributes to the parameter gradients, reduced
// over that call's points (fp64, fixed summation order).  It is linear in the upstream gradients, so the stage
// gradients of several calls that share one parameter stage are simply added before the M x M backward runs once.
//   [ u MP | vec vec_len (colsum MP, q DP, wbar DP, scalars) | S MP x MP (full, symmetric) | W^T X  MP x DP |
//     RQ only: sum kbar o dk/dalpha ]
__host__ __device__ inline size_t stage_grad_doubles(int MP, int DP, int kind) {
  return (size_t)MP + (size_t)(MP + 2 * DP + VS_COUNT) + (size_t)MP * MP + (size_t)MP * DP +
         (kind == GPBLUR_KERNEL_RQ ? 1 : 0);
}

inline WsLayout make_layout(long long N, int D, int M, int training) {
  WsLayout w;
  w.N = N; w.D = D; w.M = M; w.training = training; w.kind = GPBLUR_KERNEL_RBF;
  w.DP = padded_d(D); w.MP = padded_m(M);
  const size_t MP = w.MP, DP = w.DP;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes); return r; };
  w.hyp = take(H_COUNT * 4);
  w.hyp64 = take(H_COUNT * 8);
  w.stamps = take(kStampSlots * 8);
  w.inv_ell = take(DP * 4);
  w.ell = take(DP * 4);
  w.center = take(DP * 4);
  w.wl = take(DP * 4);
  w.Zt = take(MP * DP * 4);
  w.ZtT = take(DP * MP * 4);
  w.zn = take(MP * 4);
  w.znc = take(MP * 4);   // -1/2 log2(e) |z~_j|^2 + log2(os)  (-1e30 on padded columns): exponent offset of the tc kernels
  w.mvec = take(MP * 4);
  w.cvec = take(MP * 4);
  w.svec = take(MP * 4);
  w.beta = take(MP * 4);
  w.K64 = take(MP * MP * 8);
  w.L64 = take(MP * MP * 8);
  w.Linv64 = take(MP * MP * 8);
  w.T64 = take(MP * MP * 8);
  w.U64 = take(MP * MP * 8);
  w.LinvT32 = take(MP * MP * 4);
  w.LC32 = take(MP * MP * 4);
  w.Linv32 = take(MP * MP * 4);   // row-major Linv (tensor-core forward B operand)
  w.LCT32 = take(MP * MP * 4);    // (diag(c) Linv)^T (tensor-core backward B operand)
  {
    // UMMA slab images, see tc_slab_* helpers below.  Sizes in floats (hi + lo planes).
    const size_t nsl = MP / 32, nds = DP >= 32 ? DP / 32 : 1, dpt = DP < 32 ? 32 : DP;
    w.ZtU = take(nds * 64 * MP * 4);
    w.LinvU = take(tc_linv_total(w.MP) * 4);
    w.LCTU = take(tc_lct_total(w.MP) * 4);
    w.ZtTU = take(nsl * 64 * dpt * 4);
    w.ZtQ = take(nds * 64 * MP * 4);
    w.LCTQ = take(tc_lctq_total(w.MP) * 4);
  }
  const int tp = w.MP < 128 ? w.MP : 128;
  const int nt = w.MP / tp;
  w.splitsS = choose_splits(N, nt * (nt + 1) / 2);
  w.splitsZ = choose_splits(N, nt);
  w.splitsO = 0;
  if (w.MP >= 128) {
    // tensor-core reductions, ONE launch of about one wave of 148 SMs (gpblur_tc_reduce.cu): per band of BW = 256
    // inducing points (128 at MP = 128) one diagonal Gram unit (its 3 lower-triangle 128 x 128 blocks) and one W^T X
    // unit, plus a (row tile, column band) unit of 2 blocks per row tile and band below the diagonal.  The split
    // counts follow the per-row cost of a unit, in 128 x 128 Gram blocks: diagonal 3 (1 at MP = 128), off-diagonal 2,
    // W^T X kWxCost per band, so that all CTAs of the wave finish together.  Splits are >= 128 rows deep.
    const int nb = w.MP / tc_bw(w.MP);
    const double cd = w.MP >= 256 ? 3.0 : 1.0, co = 2.0, cz = kWxCost * (w.MP >= 256 ? 2 : 1);
    const double units = nb * cd + (double)nb * (nb - 1) * co + nb * cz;
    const double share = units / 148.0;   // cost per CTA
    const long long maxs = (N + 127) / 128;
    auto fit = [&](double c) {
      long long s = (long long)(c / share);
      if (s > maxs) s = maxs;
      return (int)(s < 1 ? 1 : s);
    };
    w.splitsS = fit(cd);
    w.splitsO = nb > 1 ? fit(co) : 0;
    w.splitsZ = fit(cz);
  }
  w.nvec = kMaxPersist;
  w.vec_len = w.MP + 2 * w.DP + VS_COUNT;
  w.vp_len = w.MP + 2 * w.DP + VS_PART;
  w.v64 = take((size_t)(3 * MP + w.vec_len) * 8);
  w.t64 = take((size_t)MP * DP * 8);
  w.D2zz64 = take(MP * MP * 8);      // last region of the parameter stage: the offsets before it do not depend on it
  if (training) {
    // the tensor-core kernels keep A and W TILE-major (see tc_tiled_index): whole 128-point tiles
    const size_t Nt = w.MP >= 128 ? (size_t)round_up_ll(N, 128) : (size_t)N;
    w.A = take(Nt * MP * 4);
    w.W = take(Nt * MP * 4);
    // [MP x MP] per split: the FFMA kernels (forced for MP >= 128 by GPBLUR_TC=-1) store full partials, the
    // tensor-core Gram writes only the first tc_gram_floats(MP) of each
    w.Spart = take((size_t)(w.splitsS > w.splitsO ? w.splitsS : w.splitsO) * MP * MP * 4);
    w.upart = take((size_t)w.splitsS * MP * 4);
    w.WXpart = take((size_t)w.splitsZ * MP * DP * 4);
    w.vecpart = take((size_t)w.nvec * w.vp_len * 4);
    w.gsc = take((size_t)2 * (N > 0 ? N : 1) * 4);   // folded upstream grads g_mu, g_var [N] each
    w.rrow = take((size_t)(N > 0 ? N : 1) * 4);           // row sums r[n] of W (tensor-core backward)
    w.cpart = take((size_t)w.splitsZ * MP * 4);           // column sums of W per split (tensor-core W^T X)
    w.sgrad = take(stage_grad_doubles(w.MP, w.DP, GPBLUR_KERNEL_RQ) * 8);   // the longest stage gradient
  } else {
    w.A = w.W = w.Spart = w.upart = w.WXpart = w.vecpart = w.gsc = w.rrow = w.cpart = w.sgrad = o;
  }
  w.total = o;
  return w;
}


template <typename T>
__host__ __device__ inline T* ws_ptr(void* ws, size_t off) {
  return reinterpret_cast<T*>(reinterpret_cast<char*>(ws) + off);
}
template <typename T>
__host__ __device__ inline const T* ws_cptr(const void* ws, size_t off) {
  return reinterpret_cast<const T*>(reinterpret_cast<const char*>(ws) + off);
}

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ double softplus64(double x) {
  return x > 30.0 ? x : log1p(exp(x));
}
__device__ __forceinline__ double sigmoid64(double x) { return 1.0 / (1.0 + exp(-x)); }

// Philox4x32-10 (Random123).  Counter layout documented in oracle/gp_oracle.py::philox_bits.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}
__device__ __forceinline__ uint4 philox_element(uint64_t seed, uint64_t e, uint32_t stream_id) {
  return philox4x32_10(make_uint4((uint32_t)e, (uint32_t)(e >> 32), stream_id, 0u),
                       make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}
__device__ __forceinline__ float philox_normal(uint64_t seed, uint64_t e, uint32_t stream_id) {
  const uint4 r = philox_element(seed, e, stream_id);
  const float u1 = ((float)(r.x >> 9) + 0.5f) * 1.1920928955078125e-07f;   // 2^-23
  const float u2 = ((float)(r.y >> 9) + 0.5f) * 1.1920928955078125e-07f;
  return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// host-side launch bookkeeping (defined in gpblur_api.cu)
enum Stage { ST_MM_FWD = 0, ST_POINT_FWD, ST_POINT_BWD, ST_GRAM, ST_WX, ST_MM_BWD, ST_ELBO_FWD, ST_ELBO_BWD,
             ST_OTHER, ST_SG_REDUCE, ST_COUNT };
// RAII: when profiling is enabled, brackets the launches issued in its scope with CUDA events on `st`
struct ProfScope {
  int stage; cudaStream_t st; void* rec;
  ProfScope(int stage, cudaStream_t st);
  ~ProfScope();
};
void note_launch(int n = 1);
// `offset_dev` (nullable): device-resident addend of the Philox offset, read when the kernel runs (CUDA-graph replays)
__device__ __forceinline__ uint64_t rng_offset(uint64_t offset, const unsigned long long* offset_dev) {
  return offset + (offset_dev ? (uint64_t)*offset_dev : 0ull);
}
int check_launch(const char* what);
long long* debug_trace_buffer();      // device buffer registered with gpblur_debug_set_trace (null: tracing off)
int num_sms();
int tile_override(const char* env);   // 0 = heuristic, else forced tile height (tuning knob)

// launchers implemented in the other translation units
int launch_mm_forward(const gpblur_svgp_params& p, const WsLayout& L, void* ws, float* kl, int* info,
                      cudaStream_t st, double extra_jitter = 0.0, int max_ctas = 0);
// stage: the parameter stage of the forward (its fp64 scratch regions are overwritten); sgrad: summed stage gradient
int launch_mm_backward(const gpblur_svgp_params& p, const WsLayout& L, void* stage, const double* sgrad,
                       const float* g_kl, float* grad_bucket, cudaStream_t st, int accumulate = 0, int max_ctas = 0);
// reduces the split partials left in `ws` by the point backward + N-reduction GEMMs into sgrad (fixed order, fp64)
int launch_stage_grad_reduce(const WsLayout& L, const void* ws, double* sgrad, cudaStream_t st);
struct SegGrads;   // per-segment upstream gradients of a point backward (gpblur_tile.cuh)
// The point launchers read the constant operands from `stage` (the parameter stage: the caller's workspace itself
// when the stage was built there) and write the per-call buffers into `ws`.
int launch_point_forward(const WsLayout& L, const void* stage, void* ws, const float* x, float* mean, float* var,
                         float* sample, uint64_t seed, uint64_t offset, uint32_t stream_id,
                         const unsigned long long* offset_dev, cudaStream_t st);
int launch_point_backward(const WsLayout& L, const void* stage, void* ws, const float* x, const SegGrads& seg,
                          const float* var, uint64_t seed, uint64_t offset, uint32_t stream_id,
                          const unsigned long long* offset_dev, float* dx, cudaStream_t st);
int launch_reductions(const WsLayout& L, void* ws, const float* x, cudaStream_t st);
// tensor-core (tcgen05 3xTF32) variants; *_supported() decides per problem shape
bool tc_point_supported(const WsLayout& L);
int launch_tc_point_forward(const WsLayout& L, const void* stage, void* ws, const float* x, float* mean, float* var,
                            float* sample, uint64_t seed, uint64_t offset, uint32_t stream_id,
                            const unsigned long long* offset_dev, cudaStream_t st);
int launch_tc_point_backward(const WsLayout& L, const void* stage, void* ws, const float* x, const SegGrads& seg,
                             const float* var, uint64_t seed, uint64_t offset, uint32_t stream_id,
                             const unsigned long long* offset_dev, float* dx, cudaStream_t st);
int tc_vector_partials(const WsLayout& L);

}  // namespace gpblur
