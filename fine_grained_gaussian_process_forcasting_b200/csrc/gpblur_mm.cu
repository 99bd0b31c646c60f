// Once-per-step M x M stage of the whitened SVGP, fp64, one cooperative launch each way.
//
// forward  (replaces gpytorch's B batched copies of: kernel(Z,Z) build, add_jitter, psd_safe_cholesky in
//           float64 and the triangular solve set-up; /root/reference/denoising_model/DeepGP.py:33-38,46-49
//           via VariationalStrategy.forward):
//   phase 0  hyper-parameters (softplus constraints), input centre, KL(q(u) || N(0, I))
//   phase 1  scaled/centred inducing points Zt, Kzz + jitter (fp64, direct differences)
//   phase 2  right-looking blocked Cholesky, 32 x 32 blocks staged in shared memory
//   phase 3  triangular inverse Linv = L^-1 by recursive doubling (all-GEMM, parallel over tiles)
//   phase 4  fp32 operands for the per-point kernels: Linv^T, diag(c) Linv, beta = Linv^T m
// backward (replaces LinalgCholeskyExBackward0 + kernel-matrix autograd):
//   Lbar = -tril(Linv^T X), X = m u^T + 2 diag(c) S ; Kbar = sym(Linv^T Phi(L^T Lbar) Linv), in closed form
//   sym(Kbar) = Linv^T P Linv with P = -1/2 (m_hi u_lo + 2 c_hi S_hi,lo) (two products, see PForm)
//   phase A  Tm = P Linv
//   phase B  sym(Kbar) = Linv^T Tm, Wzz = sym(Kbar) o (Kzz - jitter I) (Matern / RQ kinds: o g(d2)) in its epilogue
//   phase C  Kzz-path gradients of Z and the per-(i, d) lengthscale terms (V = Wzz Z~)
//   phase D  final parameter bucket
//
// All matrices are [MP, MP] row-major doubles with MP a multiple of 32 (identity padding).
#include <cooperative_groups.h>

#include <cstdlib>

#include "gpblur_common.cuh"

namespace cg = cooperative_groups;

namespace gpblur {

namespace {

constexpr int TB = 32;          // block size of the blocked algorithms
// "not yet written" marker of the diagonal blocks of L^-1 (a NaN payload no arithmetic produces)
constexpr long long kDinvSentinel = (long long)0xFFF7A5A5DEADBEEFull;
constexpr int TLD = TB + 1;     // padded leading dimension of a shared tile
typedef double Tile[TB][TLD];

struct MatRef {
  const double* p;
  int ld;
  bool trans;   // element(i, j) = trans ? p[j * ld + i] : p[i * ld + j]
  const float* pf = nullptr;   // fp32 source instead of p (widened on load; fetch_tile() only)
};

// dst[r][c] = M(r0 + r, c0 + c), coalesced for both orientations.  256 threads.
__device__ __forceinline__ void load_tile(Tile& dst, const MatRef& m, int r0, int c0) {
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = ty + 8 * i;
    if (!m.trans) dst[r][tx] = m.p[(size_t)(r0 + r) * m.ld + c0 + tx];
    else dst[tx][r] = m.p[(size_t)(c0 + r) * m.ld + r0 + tx];
  }
}

// register half of load_tile: fetch (global -> registers) now, park (registers -> shared) later
__device__ __forceinline__ void fetch_tile(double (&v)[4], const MatRef& m, int r0, int c0) {
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = ty + 8 * i;
    const size_t off = m.trans ? (size_t)(c0 + r) * m.ld + r0 + tx : (size_t)(r0 + r) * m.ld + c0 + tx;
    v[i] = m.pf ? (double)m.pf[off] : m.p[off];
  }
}
__device__ __forceinline__ void park_tile(Tile& dst, const double (&v)[4], bool trans) {
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = ty + 8 * i;
    if (!trans) dst[r][tx] = v[i];
    else dst[tx][r] = v[i];
  }
}

// fp64 tensor-core step D(8x8) += A(8x4) B(4x8): lane = 4 g + t holds A[g][t], B[t][g], C[g][2t], C[g][2t + 1]
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// Shared-memory scratch of tile_gemm: A as At[row][k] and B TRANSPOSED as Bt[col][k], pitch 34 doubles: the fragment
// loads of dmma884 (address 34 g + t + const) then hit every 8-byte bank exactly twice (the minimum for 256 bytes).
constexpr int GLD = TB + 2;
constexpr int kGemmScratchDoubles = 2 * TB * GLD;

// acc[i] (+)= sum_{k in [k0, k1)} A(r0 + ty + 8 i, k) * B(k, c0 + tx);  k0, k1 multiples of 32.
// The 32 x 32 x 32 products run on the FP64 tensor path (mma.sync m8n8k4): warp w owns rows 8 (w & 3) .. + 8 and
// columns 16 (w >> 2) .. + 16, i.e. two 8 x 8 accumulators sharing one A fragment - 3 shared-memory loads per 16
// FMAs per lane, where the FFMA-style loop needed 5 loads per 4 and was bound by them (phases of the backward M x M
// kernel: ~10 -> ~7.5 us at M = 256; neither a two-deep operand prefetch nor four accumulator chains changed that).  Software-pipelined: the global (L2) loads of k-step kk + 1 are in flight while
// step kk is multiplied.  The accumulators go back to the callers' (row ty + 8 i, column tx) mapping through `scratch`.
__device__ __forceinline__ void tile_gemm(double acc[4], const MatRef& A, int r0, const MatRef& B, int c0,
                                          int k0, int k1, double* scratch) {
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  if (k0 >= k1) return;
  double* At = scratch;
  double* Bt = scratch + TB * GLD;
  const int g = tx >> 2, t = tx & 3;
  const int rw = 8 * (ty & 3), cw = 16 * (ty >> 2);
  double c[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
  double ra[4], rb[4];
  fetch_tile(ra, A, r0, k0);
  fetch_tile(rb, B, k0, c0);
  for (int kk = k0; kk < k1; kk += TB) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = ty + 8 * i;
      // fetch_tile(): non-transposed -> element (row r, column tx), transposed -> element (row tx, column r)
      if (!A.trans) At[r * GLD + tx] = ra[i]; else At[tx * GLD + r] = ra[i];      // At[row = tile row][col = k]
      if (!B.trans) Bt[tx * GLD + r] = rb[i]; else Bt[r * GLD + tx] = rb[i];      // Bt[col = tile column][row = k]
    }
    __syncthreads();
    if (kk + TB < k1) {
      fetch_tile(ra, A, r0, kk + TB);
      fetch_tile(rb, B, kk + TB, c0);
    }
    const double* ap = At + (rw + g) * GLD + t;
    const double* bp0 = Bt + (cw + g) * GLD + t;
    const double* bp1 = bp0 + 8 * GLD;
#pragma unroll
    for (int k4 = 0; k4 < TB; k4 += 4) {
      const double a = ap[k4];
      dmma884(c[0][0], c[0][1], a, bp0[k4]);
      dmma884(c[1][0], c[1][1], a, bp1[k4]);
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    At[(rw + g) * GLD + cw + 8 * j + 2 * t] = c[j][0];
    At[(rw + g) * GLD + cw + 8 * j + 2 * t + 1] = c[j][1];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i] += At[(ty + 8 * i) * GLD + tx];
}

// ---- products of the backward M x M phases: 16 x 32 output tiles, the WHOLE k-range staged at once ----
// FP64 runs at 64 FMA / clk / SM on B200 whether issued as DFMA or as mma.m8n8k4 (measured: one mma per 4 cycles per
// SM, 26 cycles dependent): a 32 x 32 tile with K = 256 is 2.1 us of pure pipe time on the one SM that owns it, and
// the phases of the backward are chains of such products separated by grid barriers.  So (1) tiles are 16 x 32: at
// M = 256 a phase has up to 128 of them, one per SM; (2) every operand element of up to KW = 256 k-values is requested
// up front with 8-byte cp.async copies straight into shared memory (no registers: ~100 KB in flight per CTA), in commit
// groups of 64 k so that the mma loop starts when the first group has landed (tile_gemm() above pays one L2 round
// trip and two CTA barriers per 32 k).
constexpr int KW = 256;
constexpr int PW = KW + 2;                               // pitch (doubles): fragment loads hit every bank pair twice
// operand buffers + k-vectors [3][KW] (m / u / c of PForm) + row vectors [3][TB] of PForm
template <int RT>
constexpr size_t wide_bytes() { return ((size_t)(RT + TB) * PW + 3 * KW + 3 * TB) * sizeof(double); }

// A operand of the first backward product: the staged rows of the (exactly symmetric) stage gradient S become
//   P(r, k) = -1/2 (m_hi u_lo + 2 c_hi S(hi, lo)),  hi = max(r, k), lo = min(r, k),
// i.e. P = (Phi + Phi^T) / 2 with Phi = Phi(L^T Lbar) = -Phi(m u^T + 2 diag(c) S) (see mm_backward_kernel).
// m, c are 0 and u, S are 0 in the padding, so P is 0 there.
struct PForm {
  const float* m = nullptr;    // variational mean
  const double* u = nullptr;   // u of the stage gradient
  const float* c = nullptr;    // s^2 - 1
};

__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc)
               : "memory");
}
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// acc[i] += sum_{k in [k0, k1)} A(r0 + ty + 8 i, k) * B(k, c0 + tx), i < RT / 8;  k0, k1 multiples of 32.
// RT = 16 or 32 rows per tile (16: up to 128 tiles per phase at M = 256, one per SM; 32: half the operand traffic
// per flop, for the sizes where every SM has several tiles anyway).
//  * B may be an fp32 matrix (B.pf): staged as floats, widened when the fragment is read;
//  * rowsum != nullptr (RT doubles of shared memory): receives the row sums of the A block, fixed order;
//  * pform.m != nullptr: A (non-transposed) is S, and P (see PForm) is multiplied instead.
// `wide`: wide_bytes<RT>() of shared memory.
template <int RT>
__device__ __forceinline__ void wide_gemm(double (&acc)[RT / 8], const MatRef& A, int r0, const MatRef& B, int c0, int k0,
                                          int k1, double* wide, double* rowsum = nullptr, PForm pform = PForm{}) {
  if (k0 >= k1) return;
  constexpr int NCB = RT / 16;                           // 8-column blocks per warp
  const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
  double* Aw = wide;                                     // [RT rows][k]
  double* Bw = wide + RT * PW;                           // [32 cols][k]
  double* pm = Bw + TB * PW;                             // [k] m of the chunk (PForm)
  double* pu = pm + KW;                                  // [k] u of the chunk (PForm)
  double* pc = pu + KW;                                  // [k] c of the chunk (PForm)
  double* prow = pc + KW;                                // [3][RT] m, u, c of the tile rows (PForm)
  float* Bf = reinterpret_cast<float*>(Bw);              // fp32 B: [col][k], pitch 2 PW floats
  const int g = tx >> 2, t = tx & 3;
  const int rw = RT == 16 ? 8 * (ty & 1) : 8 * (ty & 3);
  const int cw = RT == 16 ? 8 * (ty >> 1) : 16 * (ty >> 2);
  double c[2][NCB][2] = {};                              // [even / odd k-step][column block][element]: two mma chains
  for (int kc = k0; kc < k1; kc += KW) {
    const int klen = (k1 - kc) < KW ? (k1 - kc) : KW;   // multiple of 32
    const int ngroups = (klen + 63) / 64;
    __syncthreads();                                     // previous chunk / previous user of `wide` is done
    if (pform.m) {
      for (int k = tid; k < klen; k += kThreads) {
        pm[k] = (double)pform.m[kc + k];
        pu[k] = pform.u[kc + k];
        pc[k] = (double)pform.c[kc + k];
      }
      if (tid < RT) {
        prow[tid] = (double)pform.m[r0 + tid];
        prow[RT + tid] = pform.u[r0 + tid];
        prow[2 * RT + tid] = (double)pform.c[r0 + tid];
      }
    }
    for (int gq = 0; gq < 4; ++gq) {
      if (gq < ngroups) {
        const int kg0 = gq * 64, kgl = (klen - kg0) < 64 ? (klen - kg0) : 64;   // 64 or 32
        const int sh = kgl == 64 ? 6 : 5;
        for (int e = tid; e < RT * kgl; e += kThreads) {
          int row, k;
          if (!A.trans) { row = e >> sh; k = kg0 + (e & (kgl - 1)); }
          else { k = kg0 + e / RT; row = e % RT; }
          const size_t off = A.trans ? (size_t)(kc + k) * A.ld + r0 + row : (size_t)(r0 + row) * A.ld + kc + k;
          cp_async8(Aw + row * PW + k, A.p + off);
        }
        for (int e = tid; e < TB * kgl; e += kThreads) {
          int col, k;
          if (B.trans) { col = e >> sh; k = kg0 + (e & (kgl - 1)); }
          else { k = kg0 + (e >> 5); col = e & 31; }
          const size_t off = B.trans ? (size_t)(c0 + col) * B.ld + kc + k : (size_t)(kc + k) * B.ld + c0 + col;
          if (B.pf) cp_async4(Bf + col * (2 * PW) + k, B.pf + off);
          else cp_async8(Bw + col * PW + k, B.p + off);
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");   // (empty groups keep the wait counts static)
    }
    for (int gq = 0; gq < ngroups; ++gq) {
      if (gq == 0) cp_async_wait<3>();
      else if (gq == 1) cp_async_wait<2>();
      else if (gq == 2) cp_async_wait<1>();
      else cp_async_wait<0>();
      __syncthreads();
      const int kg0 = gq * 64, kgl = (klen - kg0) < 64 ? (klen - kg0) : 64;
      if (pform.m) {
        // S(r, k) -> P(r, k) in place; S(r, k) = S(hi, lo) because S is exactly symmetric (stage_grad_reduce_kernel)
        const int sh = kgl == 64 ? 6 : 5;
        for (int e = tid; e < RT * kgl; e += kThreads) {
          const int row = e >> sh, k = kg0 + (e & (kgl - 1));
          double& s = Aw[row * PW + k];
          s = (kc + k >= r0 + row) ? -fma(pc[k], s, 0.5 * pm[k] * prow[RT + row])
                                   : -fma(prow[2 * RT + row], s, 0.5 * prow[row] * pu[k]);
        }
        __syncthreads();
      }
      if (rowsum) {
        // row sums of this k-group (rows ty, ty + 8, ...), fixed order: groups in sequence, shuffle tree inside
#pragma unroll
        for (int rr = 0; rr < RT / 8; ++rr) {
          const int row = ty + 8 * rr;
          double sacc = Aw[row * PW + kg0 + tx];
          if (kgl == 64) sacc += Aw[row * PW + kg0 + 32 + tx];
          sacc = warp_sum(sacc);
          if (tx == 0) rowsum[row] = ((kc == k0 && gq == 0) ? 0.0 : rowsum[row]) + sacc;
        }
      }
      const double* ap = Aw + (rw + g) * PW + t + kg0;
#pragma unroll 4
      for (int k4 = 0; k4 < kgl; k4 += 8) {
        double a0 = ap[k4], a1 = ap[k4 + 4];
#pragma unroll
        for (int cb = 0; cb < NCB; ++cb) {
          double b0, b1;
          if (!B.pf) {
            const double* bp = Bw + (cw + 8 * cb + g) * PW + t + kg0;
            b0 = bp[k4]; b1 = bp[k4 + 4];
          } else {
            const float* bp = Bf + (cw + 8 * cb + g) * (2 * PW) + t + kg0;
            b0 = (double)bp[k4]; b1 = (double)bp[k4 + 4];
          }
          dmma884(c[0][cb][0], c[0][cb][1], a0, b0);
          dmma884(c[1][cb][0], c[1][cb][1], a1, b1);
        }
      }
    }
  }
  __syncthreads();
  // fragments -> the callers' (row ty + 8 i, column tx) mapping through the (now free) A buffer
#pragma unroll
  for (int cb = 0; cb < NCB; ++cb) {
    Aw[(rw + g) * PW + cw + 8 * cb + 2 * t] = c[0][cb][0] + c[1][cb][0];
    Aw[(rw + g) * PW + cw + 8 * cb + 2 * t + 1] = c[0][cb][1] + c[1][cb][1];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < RT / 8; ++i) acc[i] += Aw[(ty + 8 * i) * PW + tx];
}

// decode t -> (i, j) with j <= i, t = i (i + 1) / 2 + j
__device__ __forceinline__ void tri_decode(int t, int& i, int& j) {
  int ii = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
  while ((ii + 1) * (ii + 2) / 2 <= t) ++ii;
  while (ii * (ii + 1) / 2 > t) --ii;
  i = ii;
  j = t - ii * (ii + 1) / 2;
}

// Grid-wide barrier on a monotonically increasing counter (zeroed by the host before the launch), for plain launches
// (GPBLUR_MM_COOP=0).  Measured: no faster and no slower than cooperative launches + grid.sync().
// All CTAs are co-resident (grid <= SM count x occupancy, checked by the launcher); a CTA that cannot be scheduled yet
// because an independent kernel holds its SM only delays the barrier.
__device__ __forceinline__ void counter_grid_sync(unsigned* cnt, unsigned& target, int G) {
  __syncthreads();
  if (G == 1) return;                         // a single CTA: its own global writes are visible after the CTA barrier
  if (threadIdx.x == 0) {
    target += (unsigned)G;
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(cnt) : "memory");
    unsigned v;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(cnt) : "memory");
    } while (v < target);
  }
  __syncthreads();
}

// 1 / sqrt(d) in double from the FP64 MUFU seed (MUFU.RSQ64H works on the high word: ~20 good bits, no conversions to
// and from fp32 on the pivot chain) and ONE third-order Newton step (error ~ (5/16) e^3, e ~ 2^-20 -> below 2^-60):
// 4 dependent FP64 operations instead of the library routine's special-case handling on the pivot critical path.
// d is a Cholesky pivot of a jittered kernel matrix: 1e-4 <~ d <~ outputscale, far from under/overflow.
__device__ __forceinline__ double fast_rsqrt64(double d) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  const double e = fma(-d * y, y, 1.0);
  return fma(y * e, fma(0.375, e, 0.5), y);
}

// Cholesky of a 32 x 32 block held one row per lane in registers, FUSED with the inverse of the factor (one warp).
// Per column c: pivot broadcast (shuffle), reciprocal square root, then the scaled column goes through a
// double-buffered shared-memory vector so that the trailing updates of a lane read their multipliers with broadcast
// loads (one 16-byte load per two columns) instead of two shuffles each.
//  * The NEXT pivot never waits for that shared-memory round trip: in lane c + 1 the multiplier of column c + 1 is the
//    lane's own l, so `piv = a[c + 1] - l * l` is formed locally and shuffled at the top of the next iteration (the
//    dependent chain per column is shuffle -> rsqrt -> 2 FP64 operations: 126 cycles measured).
//  * The same column broadcast drives one step of the column-oriented forward substitution X = L^-1 (lane = column
//    of X): x[c] = s[c] / L[c][c], then s[r] -= L[r][c] x[c] for r > c.
//  * No pivot test inside the loop (it cost 1000 of 6900 cycles): a non-positive pivot turns its reciprocal square
//    root, and with it the rest of the factor, into NaN / Inf; the caller finds the first bad diagonal entry afterwards.
// Measured alone (scripts/micro/chol32_bench.cu, B200): chain only 4000 cycles, + trailing update 5100, + inverse
// 5900 (3.0 us).  Two warps (factor | inverse, handshake through a shared-memory flag) were SLOWER: 7100 cycles with a
// polling consumer, 10000 with a fence per column.
// On exit a[c] = L[lane][c] (0 above the diagonal), x[r] = (L^-1)[r][lane].  `lcol`: 2 x 32 doubles, 16-byte aligned.
__device__ __forceinline__ void chol32_inv_warp(double (&a)[TB], double (&x)[TB], int lane, double* lcol) {
#pragma unroll
  for (int r = 0; r < TB; ++r) x[r] = (r == lane) ? 1.0 : 0.0;
  double d = __shfl_sync(0xffffffffu, a[0], 0);
  double rs = fast_rsqrt64(d);
#pragma unroll
  for (int c = 0; c < TB; ++c) {
    const double l = a[c] * rs;
    const double xc = (c >= lane) ? x[c] * rs : 0.0;
    // software pipelining by hand: the pivot of column c + 1 (meaningful in lane c + 1: a[c + 1] - l^2) is shuffled
    // and its reciprocal square root started BEFORE the trailing update of column c is issued
    if (c + 1 < TB) {
      const double piv = fma(-l, l, a[c + 1]);
      d = __shfl_sync(0xffffffffu, piv, c + 1);
      rs = fast_rsqrt64(d);
    }
    a[c] = (lane >= c) ? l : 0.0;
    x[c] = xc;
    double* buf = lcol + (c & 1) * TB;
    buf[lane] = l;
    __syncwarp();
    // branch-free trailing update: lanes above the diagonal (lane < c2) update entries that are never read
    // (they are overwritten with 0 when their column is processed), so no predicate is needed
    if ((c + 1) & 1) {
      if (c + 1 < TB) {
        const double m = buf[c + 1];
        a[c + 1] = fma(-l, m, a[c + 1]);
        x[c + 1] = fma(-m, xc, x[c + 1]);
      }
#pragma unroll
      for (int c2 = c + 2; c2 + 1 < TB; c2 += 2) {
        const double2 m2 = *reinterpret_cast<const double2*>(buf + c2);
        a[c2] = fma(-l, m2.x, a[c2]);
        a[c2 + 1] = fma(-l, m2.y, a[c2 + 1]);
        x[c2] = fma(-m2.x, xc, x[c2]);
        x[c2 + 1] = fma(-m2.y, xc, x[c2 + 1]);
      }
    } else {
#pragma unroll
      for (int c2 = c + 1; c2 + 1 < TB; c2 += 2) {
        const double2 m2 = *reinterpret_cast<const double2*>(buf + c2);
        a[c2] = fma(-l, m2.x, a[c2]);
        a[c2 + 1] = fma(-l, m2.y, a[c2 + 1]);
        x[c2] = fma(-m2.x, xc, x[c2]);
        x[c2 + 1] = fma(-m2.y, xc, x[c2 + 1]);
      }
    }
  }
}

// ---- 32 x 32 x 32 products with BOTH operands already in shared memory (FP64 tensor path), accumulators kept in the
// mma fragment layout: warp w owns rows 8 (w & 3) .. + 8 and columns 16 (w >> 2) .. + 16; lane = 4 g + t holds
// C[rw + g][cw + 8 j + 2 t], C[rw + g][cw + 8 j + 2 t + 1] for j = 0, 1.  Operand buffers: A as At[row][k], B TRANSPOSED
// as Bt[col][k], pitch GLD doubles.
struct Frag {
  double c[2][2];
};
__device__ __forceinline__ void frag_coords(int& row, int& col0) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  row = 8 * (w & 3) + (lane >> 2);
  col0 = 16 * (w >> 2) + 2 * (lane & 3);
}
__device__ __forceinline__ void smem_gemm32(Frag& f, const double* At, const double* Bt) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const double* ap = At + (8 * (w & 3) + g) * GLD + t;
  const double* bp0 = Bt + (16 * (w >> 2) + g) * GLD + t;
  const double* bp1 = bp0 + 8 * GLD;
#pragma unroll
  for (int k4 = 0; k4 < TB; k4 += 4) {
    const double av = ap[k4];
    dmma884(f.c[0][0], f.c[0][1], av, bp0[k4]);
    dmma884(f.c[1][0], f.c[1][1], av, bp1[k4]);
  }
}
// dst[row][col] = sign * f (row-major, pitch GLD): the layout of an A operand, and of a B operand read as B^T
__device__ __forceinline__ void frag_park(double* dst, const Frag& f, double sign) {
  int row, col0;
  frag_coords(row, col0);
#pragma unroll
  for (int j = 0; j < 2; ++j)
    *reinterpret_cast<double2*>(dst + row * GLD + col0 + 8 * j) = make_double2(sign * f.c[j][0], sign * f.c[j][1]);
}
// dst[col][row] = sign * f: the layout of a B operand read as B
__device__ __forceinline__ void frag_park_t(double* dst, const Frag& f, double sign) {
  int row, col0;
  frag_coords(row, col0);
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    dst[(col0 + 8 * j) * GLD + row] = sign * f.c[j][0];
    dst[(col0 + 8 * j + 1) * GLD + row] = sign * f.c[j][1];
  }
}
__device__ __forceinline__ void frag_load(Frag& f, const double* src, int ld, int r0, int c0) {
  int row, col0;
  frag_coords(row, col0);
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const double2 v = *reinterpret_cast<const double2*>(src + (size_t)(r0 + row) * ld + c0 + col0 + 8 * j);
    f.c[j][0] = v.x;
    f.c[j][1] = v.y;
  }
}
__device__ __forceinline__ void frag_store(double* dst, int ld, int r0, int c0, const Frag& f, double sign) {
  int row, col0;
  frag_coords(row, col0);
#pragma unroll
  for (int j = 0; j < 2; ++j)
    *reinterpret_cast<double2*>(dst + (size_t)(r0 + row) * ld + c0 + col0 + 8 * j) =
        make_double2(sign * f.c[j][0], sign * f.c[j][1]);
}
// registers of fetch_tile() -> operand buffer (pitch GLD); trans: dst[col][row]
__device__ __forceinline__ void park_operand(double* dst, const double (&v)[4], bool trans) {
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = ty + 8 * i;
    if (!trans) dst[r * GLD + tx] = v[i];
    else dst[tx * GLD + r] = v[i];
  }
}

// RQ: alpha (fp64 and fp32) and 1 / (2 alpha) (fp32) for the point kernels and the backward
__device__ __forceinline__ void set_alpha(float* hyp, double* hyp64, const float* raw_alpha) {
  const double alpha = softplus64((double)raw_alpha[0]);
  hyp64[H_ALPHA] = alpha;
  hyp[H_ALPHA] = (float)alpha;
  hyp[H_I2A] = (float)(0.5 / alpha);
}

struct MmFwdArgs {
  gpblur_svgp_params p;
  WsLayout L;
  void* ws;
  float* kl;
  int* info;
  double extra_jitter;   // added to the diagonal of Kzz on top of the variational jitter (psd_safe_cholesky retries)
  unsigned* bar;         // != nullptr: plain launch, counter_grid_sync() on this zeroed word; nullptr: cooperative launch
  int debug_stop;        // >= 0: every CTA returns after that phase (timing experiments; results are incomplete)
  unsigned* flags;       // two zeroed words: diagonal blocks published, worker arrivals (phase 2)
};

// MAT: any kind but RBF (L.kind, evaluated through kernel_kg64); the RBF instantiation carries none of that code
template <bool MAT>
__global__ void __launch_bounds__(kThreads) mm_forward_kernel(MmFwdArgs a) {
  cg::grid_group grid = cg::this_grid();
  unsigned bar_target = 0;
#define GPBLUR_GRID_SYNC() do { if (a.bar) counter_grid_sync(a.bar, bar_target, (int)gridDim.x); else grid.sync(); } while (0)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Tile* tiles = reinterpret_cast<Tile*>(smem_raw);
  Tile& As = tiles[0];
  Tile& Bs = tiles[1];
  double* gsm = reinterpret_cast<double*>(tiles + 11);   // tile_gemm scratch
  Tile* Cs = tiles + 2;   // 8 per-warp tiles
  Tile& Dg = tiles[10];   // factorised diagonal block of the current panel

  const WsLayout& L = a.L;
  const int D = L.D, DP = L.DP, M = L.M, MP = L.MP;
  const int nb = MP / TB;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = gridDim.x;
  const int gtid = blockIdx.x * kThreads + tid, gsize = G * kThreads;

  float* hyp = ws_ptr<float>(a.ws, L.hyp);
  double* hyp64 = ws_ptr<double>(a.ws, L.hyp64);
  float* inv_ell = ws_ptr<float>(a.ws, L.inv_ell);
  float* ellv = ws_ptr<float>(a.ws, L.ell);
  float* center = ws_ptr<float>(a.ws, L.center);
  float* wl = ws_ptr<float>(a.ws, L.wl);
  float* Zt = ws_ptr<float>(a.ws, L.Zt);
  float* ZtT = ws_ptr<float>(a.ws, L.ZtT);
  float* mvec = ws_ptr<float>(a.ws, L.mvec);
  float* cvec = ws_ptr<float>(a.ws, L.cvec);
  float* svec = ws_ptr<float>(a.ws, L.svec);
  float* beta = ws_ptr<float>(a.ws, L.beta);
  double* K64 = ws_ptr<double>(a.ws, L.K64);
  double* L64 = ws_ptr<double>(a.ws, L.L64);
  double* Li64 = ws_ptr<double>(a.ws, L.Linv64);
  double* T64 = ws_ptr<double>(a.ws, L.T64);
  double* W64 = ws_ptr<double>(a.ws, L.U64);   // forward only: trailing matrix of the Cholesky (the backward reuses it)
  double* D2 = ws_ptr<double>(a.ws, L.D2zz64);
  float* LinvT32 = ws_ptr<float>(a.ws, L.LinvT32);
  float* LC32 = ws_ptr<float>(a.ws, L.LC32);
  float* Linv32 = ws_ptr<float>(a.ws, L.Linv32);
  float* LCT32 = ws_ptr<float>(a.ws, L.LCT32);
  const float* Z = a.p.inducing_points;
  unsigned long long* stamps = ws_ptr<unsigned long long>(a.ws, L.stamps);
  int stamp_i = 0;
#define GPBLUR_STAMP() do { if (blockIdx.x == 0 && tid == 0) stamps[stamp_i] = global_ns(); ++stamp_i; } while (0)
  GPBLUR_STAMP();
  if (a.debug_stop == 0) return;
  if (blockIdx.x == 0 && tid == 0) *a.flags = 0u;   // worker-arrival counter of phase 2 (ordered by the phase-1 barrier)

  // ---------------- phase 1: Kzz (fp64, direct differences) | per-dimension hyper-parameters, centre, KL ----------------
  // CTA 0 takes no part when there are other CTAs: it spends the phase warming the instruction cache for the
  // factorisation (see phase 2)
  const int p1_id = G > 1 ? (int)blockIdx.x - 1 : 0, p1_n = G > 1 ? G - 1 : 1;
  // One barrier: the Kzz tiles take their 1 / lengthscale straight from the raw parameter (a softplus per thread), so
  // nothing here waits for the hyper-parameter block; everything derived from it (Z~, vectors, Z~ operand images) is
  // built by the worker CTAs of phase 2 while CTA 0 factorises the first diagonal block.
  {
    const double os = softplus64((double)a.p.raw_outputscale[0]);
    const double alpha = MAT && L.kind == GPBLUR_KERNEL_RQ ? softplus64((double)a.p.raw_alpha[0]) : 0.0;
    const int ntiles = nb * (nb + 1) / 2;
    const int tx = lane, ty = warp;
    for (int t = p1_id; t >= 0 && t < ntiles; t += p1_n) {
      int bi, bj;
      tri_decode(t, bi, bj);
      double acc[4] = {0.0, 0.0, 0.0, 0.0};
      // all the rows of both blocks are requested at once (D <= 128: 4 k-steps x 4 rows x 2 blocks per thread), and
      // the softplus of the lengthscales (a few hundred instructions) is evaluated while they are in flight
      constexpr int kMaxSteps = GPBLUR_MAX_D / TB;
      float za[kMaxSteps][4], zb[kMaxSteps][4];
      double ie[kMaxSteps];
#pragma unroll
      for (int st = 0; st < kMaxSteps; ++st) {
        const int d = st * TB + tx;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int ra = bi * TB + ty + 8 * i, rb = bj * TB + ty + 8 * i;
          za[st][i] = (d < D && ra < M) ? Z[(size_t)ra * D + d] : 0.f;
          zb[st][i] = (d < D && rb < M) ? Z[(size_t)rb * D + d] : 0.f;
        }
      }
#pragma unroll
      for (int st = 0; st < kMaxSteps; ++st) {
        const int d = st * TB + tx;
        ie[st] = d < D ? 1.0 / softplus64((double)a.p.raw_lengthscale[d]) : 0.0;
      }
#pragma unroll
      for (int st = 0; st < kMaxSteps; ++st) {
        if (st * TB < D) {
          __syncthreads();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            As[ty + 8 * i][tx] = (double)za[st][i] * ie[st];
            Bs[ty + 8 * i][tx] = (double)zb[st][i] * ie[st];
          }
          __syncthreads();
#pragma unroll 8
          for (int k = 0; k < TB; ++k) {
            const double b = Bs[tx][k];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const double df = As[ty + 8 * i][k] - b;
              acc[i] = fma(df, df, acc[i]);
            }
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int gi = bi * TB + ty + 8 * i, gj = bj * TB + tx;
        double kv;
        if (gi < M && gj < M) {
          if constexpr (!MAT) {
            kv = os * exp(-0.5 * acc[i]) + (gi == gj ? (double)kJitter + a.extra_jitter : 0.0);
          } else {
            double kk, g, ka;
            kernel_kg64(L.kind, acc[i], os, alpha, kk, g, ka);
            kv = kk + (gi == gj ? (double)kJitter + a.extra_jitter : 0.0);
            D2[(size_t)gi * MP + gj] = acc[i];
            D2[(size_t)gj * MP + gi] = acc[i];
          }
        } else {
          kv = (gi == gj) ? 1.0 : 0.0;
        }
        K64[(size_t)gi * MP + gj] = kv;
        K64[(size_t)gj * MP + gi] = kv;
        W64[(size_t)gi * MP + gj] = kv;                       // working copy (lower block triangle) of the factorisation
        if (bi == bj) Li64[(size_t)gi * MP + gj] = __longlong_as_double(kDinvSentinel);   // armed: see phase 2
        if (bi != bj) L64[(size_t)gj * MP + gi] = 0.0;        // L is written once per block; the upper block triangle is 0
      }
    }
  }
  // per-dimension hyper-parameters and the input centre: CTAs from the END of the grid first (the Kzz tiles start at 0)
  for (int d = p1_id >= 0 ? (p1_n - 1 - p1_id) * 8 + warp : DP; d < DP; d += p1_n * 8) {
    if (d < D) {
      const double ell = softplus64((double)a.p.raw_lengthscale[d]);
      double s = 0.0;
      for (int m = lane; m < M; m += 32) s += (double)Z[(size_t)m * D + d];
      s = warp_sum(s);
      if (lane == 0) {
        const float c = (float)(s / (double)M);
        center[d] = c;
        ellv[d] = (float)ell;
        inv_ell[d] = (float)(1.0 / ell);
        wl[d] = a.p.mean_weights ? (float)(ell * (double)a.p.mean_weights[d]) : 0.0f;
      }
    } else if (lane == 0) {
      center[d] = 0.f; ellv[d] = 1.f; inv_ell[d] = 0.f; wl[d] = 0.f;
    }
  }
  if (p1_id == p1_n - 1) {
    // KL( N(m, diag s^2) || N(0, I) ) = 1/2 [ sum s^2 + sum m^2 - M - sum log s^2 ]
    double part = 0.0;
    for (int m = tid; m < M; m += kThreads) {
      const double mm = (double)a.p.variational_mean[m];
      const double ss = (double)a.p.variational_stddev[m];
      part += ss * ss + mm * mm - 1.0 - log(ss * ss);
    }
    part = warp_sum(part);
    __shared__ double red[8];
    __syncthreads();
    if (lane == 0) red[warp] = part;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int i = 0; i < 8; ++i) t += red[i];
      const double os = softplus64((double)a.p.raw_outputscale[0]);
      hyp[H_OS] = (float)os;
      hyp[H_JIT] = kJitter;
      hyp64[H_JIT] = (double)kJitter + a.extra_jitter;      // diagonal actually added to Kzz (the backward removes it)
      hyp[H_KL] = (float)(0.5 * t);
      hyp64[H_OS] = os;
      hyp64[H_KL] = 0.5 * t;
      if (MAT && L.kind == GPBLUR_KERNEL_RQ) set_alpha(hyp, hyp64, a.p.raw_alpha);
      if (a.kl) a.kl[0] = (float)(0.5 * t);
      if (a.info) a.info[0] = 0;
    }
  }
  // (the barrier that ends phase 1 sits at the top of iteration kb = 0 of the phase-2 loop)

  // Everything that depends only on the hyper-parameter block: Z~, Z~^T, the variational vectors, the Z~ operand images
  // of the tensor-core kernels and the exponent offsets.  `part` of `nparts` CTAs.
  float* zn = ws_ptr<float>(a.ws, L.zn);
  float* znc = ws_ptr<float>(a.ws, L.znc);
  auto split_tf32 = [](float v, float& hi, float& lo) {
    uint32_t h;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(v));
    hi = __uint_as_float(h);
    lo = v - hi;
  };
  auto aux_operands = [&](int part, int nparts) {
    const int ptid = part * kThreads + tid, psize = nparts * kThreads;
    auto zt_of = [&](int m, int d) -> float {       // straight from the parameters: no dependence on the Zt array
      return (m < M && d < D) ? (Z[(size_t)m * D + d] - center[d]) * inv_ell[d] : 0.f;
    };
    for (int idx = ptid; idx < MP * DP; idx += psize) {
      const int m = idx / DP, d = idx - m * DP;
      const float v = zt_of(m, d);
      Zt[idx] = v;
      ZtT[(size_t)d * MP + m] = v;
    }
    for (int m = ptid; m < MP; m += psize) {
      const float mm = m < M ? a.p.variational_mean[m] : 0.f;
      const float ss = m < M ? a.p.variational_stddev[m] : 1.f;
      mvec[m] = mm;
      svec[m] = ss;
      cvec[m] = m < M ? ss * ss - 1.0f : 0.f;
    }
    if (part == 0 && warp == 0) {
      double sdot = 0.0;
      if (a.p.mean_weights)
        for (int d = lane; d < D; d += 32) sdot += (double)center[d] * (double)a.p.mean_weights[d];
      sdot = warp_sum(sdot);
      if (lane == 0) hyp[H_CWB] = (float)(sdot + (double)a.p.mean_bias[0]);
    }
    // |z~_j|^2 and the exponent offsets: one warp per inducing point
    {
      const float l2os = (float)(log(softplus64((double)a.p.raw_outputscale[0])) * 1.4426950408889634);
      for (int j = part * 8 + warp; j < MP; j += nparts * 8) {
        float z2 = 0.f;
        for (int d = lane; d < DP; d += 32) { const float v = zt_of(j, d); z2 = fmaf(v, v, z2); }
        z2 = warp_sum(z2);
        if (lane == 0) {
          zn[j] = z2;
          znc[j] = j < M ? fmaf(-0.72134752044448170f, z2, l2os) : -1e30f;
        }
      }
    }
    if (MP >= 128) {
      const int nsl = MP / 32, nds = DP >= 32 ? DP / 32 : 1, dpt = DP < 32 ? 32 : DP;
      float* ZtQ = ws_ptr<float>(a.ws, L.ZtQ);
      float* ZtTU = ws_ptr<float>(a.ws, L.ZtTU);
      // Z~ images (rows m of block q of BQ rows, k = d): element (c, r, e) of image (q, ds) = Zt[q BQ + r][32 ds + 4 c + e]
      const int BQ = tc_bq(MP), NQ = MP / BQ;
      for (int idx = ptid; idx < NQ * nds * 8 * BQ * 4; idx += psize) {
        const int e = idx & 3, r = (idx >> 2) % BQ, c = ((idx >> 2) / BQ) & 7, img = (idx >> 2) / (BQ * 8);
        const int q = img / nds, ds = img - q * nds;
        const int d = ds * 32 + c * 4 + e;
        const float v = (d < DP) ? zt_of(q * BQ + r, d) : 0.f;
        float hi, lo;
        split_tf32(v, hi, lo);
        float* base = ZtQ + tc_zq_image(MP, nds, q, ds);
        base[(c * BQ + r) * 4 + e] = hi;
        base[32 * BQ + (c * BQ + r) * 4 + e] = lo;
      }
      // Z~^T slabs (rows d, k = m): element (c, r, e) of slab s = Zt[32 s + 4 c + e][r]
      for (int idx = ptid; idx < nsl * 8 * dpt * 4; idx += psize) {
        const int e = idx & 3, r = (idx >> 2) % dpt, c = ((idx >> 2) / dpt) & 7, sl = (idx >> 2) / (dpt * 8);
        const int m = sl * 32 + c * 4 + e;
        const float v = (r < DP) ? zt_of(m, r) : 0.f;
        float hi, lo;
        split_tf32(v, hi, lo);
        float* base = ZtTU + tc_slab_ztt(dpt, sl);
        base[(c * dpt + r) * 4 + e] = hi;
        base[32 * dpt + (c * dpt + r) * 4 + e] = lo;
      }
    }
  };

  // ---------------- phase 2: blocked Cholesky (right-looking, look-ahead) + triangular inverse ----------------
  // CTA 0 owns the critical path: factorise the diagonal block (one warp, registers, 3 us) and invert it, publish
  // L_kk / Dinv, then update the NEXT diagonal block itself (2 small products) and go on factorising.  Every other CTA
  // is a worker one step behind: it waits for Dinv_kb, then does the trailing tiles and the triangular-inverse sums of
  // step kb.  With Dinv the panel solve is the product P_i = A_ik Dinv^T - cheap enough (32^3) to be REPEATED by every
  // CTA that needs it instead of being published through memory behind another barrier:
  //   trailing tile (i, j), kb < j <= i :  C_ij -= P_i P_j^T                       (3 small products, 2 CTA barriers)
  //   inverse sums  (i, j), i > kb >= j :  Y_ij += P_i X_kj,  X_kj = -Dinv Y_kj (j < kb) or Dinv (j = kb)
  // where Y_ij = sum_k L_ik X_kj accumulates in T64 and block row kb of X = L^-1 is X_kj above (the triangular inverse
  // costs no extra phase).  Synchronisation: Dinv_kb is its own flag (its block of Li64 is armed with a sentinel in phase
  // 1 and polled by the workers), and `wcnt` counts worker arrivals (a worker arrives once per step in which it had
  // tiles); nobody waits at a grid-wide barrier inside the loop.  The working matrix (W64) is only read in block column kb and only written in tiles (i, j > kb) owned by
  // one CTA per step; the factor L (L64: P_i, written by the owner of tile (i, kb + 1)) and the inverse (Li64: X_kj,
  // written by the owner of (kb + 1, j)) are write-once outputs.
  // Measured at M = 256 (us): round-1 scheme (redundant factorisation, 2 grid barriers per step) 82; one barrier per
  // step 61; look-ahead: see DESIGN.md.
  __shared__ __align__(16) double lcol[2 * TB];
  double* opbuf = reinterpret_cast<double*>(smem_raw);   // 7 operand buffers of 32 x GLD doubles (the Tile slots of other phases)
  double* sD = opbuf + 0 * TB * GLD;     // Dinv           [row][k]   (A operand of X_kj; B operand (as B^T) of P_i)
  double* sDT = opbuf + 1 * TB * GLD;    // Dinv^T         [col][row] (B operand when X_kj = Dinv)
  double* sA = opbuf + 2 * TB * GLD;     // A_ik           [row][k]
  double* sB = opbuf + 3 * TB * GLD;     // A_jk [row][k]  or Y_kj^T [col][k]
  double* sP = opbuf + 4 * TB * GLD;     // P_i            [row][k]
  double* sQ = opbuf + 5 * TB * GLD;     // P_j [row][k] (= B^T layout of P_j^T)  or X_kj^T [col][k]
  double* sL = opbuf + 6 * TB * GLD;     // diagonal block: A_kk before, L_kk after the factorisation, row-major
  static_assert(sizeof(Tile) * 11 >= sizeof(double) * 7 * TB * GLD, "operand buffers live in the Tile slots");
  unsigned* wcnt = a.flags;
  const int NW = G - 1;                                  // workers (nb > 1 implies G >= 4, see launch_mm_forward)
  unsigned w_arrived_prev = 0;                           // worker arrivals expected through step kb - 1
  auto wait_counter = [&](const unsigned* ctr, unsigned target) {
    if (tid == 0) {
      unsigned v;
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
      } while (v < target);
    }
    __syncthreads();
  };
  auto signal_counter = [&](unsigned* ctr) {             // after the CTA's global writes
    __syncthreads();
    if (tid == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
  };
  double* sL1 = opbuf + 7 * TB * GLD;    // second diagonal-block buffer (CTA 0 alternates: the next block is built while
                                         // the factor of the current one is still being written out)
  double* sC = sB;                       // CTA 0: the next diagonal block before its update
  // Iteration kb = -1 (CTA 0 only, DURING phase 1): the factorisation of an identity block, results discarded.  Its
  // 33 KB of straight-line code are then in the instruction cache when the first real block arrives: the first
  // factorisation took 6.4 us cold against 3.6 us warm.
  for (int kb = G > 1 ? -1 : 0; kb < nb; ++kb) {
    if (kb == 0) {
      GPBLUR_GRID_SYNC();                                 // end of phase 1
      GPBLUR_STAMP();
      GPBLUR_STAMP();
      if (a.debug_stop == 2) return;
      if (blockIdx.x == 0) {                              // first diagonal block: one coalesced round trip
        double dg4[4];
        fetch_tile(dg4, MatRef{W64, MP, false}, 0, 0);
        park_operand(sL, dg4, false);
      } else {
        aux_operands((int)blockIdx.x - 1, NW);            // hidden behind CTA 0's first factorisation
      }
    }
    if (kb < 0) {
      if (blockIdx.x != 0) continue;
      for (int e = tid; e < TB * GLD; e += kThreads) sL1[e] = (e / GLD == e % GLD) ? 1.0 : 0.0;
    }
    const int nrb = nb - kb - 1;
    const int ntr = nrb * (nrb + 1) / 2;                 // trailing tiles (tile 0 = the next diagonal block: CTA 0's)
    const int ny = nrb * (kb + 1);                       // inverse partial-sum tiles
    const int n_items = nrb > 0 ? ntr - 1 + ny : kb;     // worker tiles; last block column: only X[kb][j], j < kb
    if (blockIdx.x == 0) {
      // Critical path of the whole phase: factorisation -> 2 small products -> factorisation ...  Everything else CTA 0
      // does is moved off it: warps 1-7 fetch the operands of the look-ahead products WHILE warp 0 factorises, the
      // outputs of a step are plain stores, and the release that publishes them (a memory barrier: ~0.5 us) is issued
      // by a thread of warp 1 at the start of the NEXT step, under the next factorisation.
      double* cur = (kb & 1) ? sL1 : sL;
      double* nxt = (kb & 1) ? sL : sL1;
      __syncthreads();                                    // `cur` holds A_kk; the stores of step kb - 1 are issued
      if (kb == 0 && tid == 0) stamps[9] = global_ns();
      if (a.debug_stop == 9 && tid == 0 && kb >= 0 && kb < 8) stamps[16 + 2 * kb] = global_ns();   // per-step probe
      if (a.debug_stop == 8 && tid == 0 && kb == 2) stamps[16] = global_ns();
      if (a.debug_stop == 8 && tid == 0 && kb == 3) stamps[21] = global_ns();
      if (warp == 0) {
        double arow[TB];
#pragma unroll
        for (int c = 0; c < TB; c += 2) {
          const double2 v = *reinterpret_cast<const double2*>(cur + lane * GLD + c);
          arow[c] = v.x;
          arow[c + 1] = v.y;
        }
        if (kb == 0 && lane == 0) stamps[10] = global_ns() + (unsigned long long)(arow[0] == 12345.678);
        double xcol[TB];
        chol32_inv_warp(arow, xcol, lane, lcol);
        if (kb == 0 && lane == 0) stamps[11] = global_ns() + (unsigned long long)(xcol[31] == 12345.678);
#pragma unroll
        for (int c = 0; c < TB; ++c) {
          cur[lane * GLD + c] = arow[c];
          sD[c * GLD + lane] = xcol[c];        // xcol[r] = Dinv[r][lane]
        }
        if (a.info && kb >= 0) {
          // first non-positive pivot: its column (and everything after it) is NaN / Inf or non-positive on the diagonal
          const double dg = cur[lane * GLD + lane];   // own row: written by this lane
          const unsigned badmask = __ballot_sync(0xffffffffu, !(dg > 0.0) || !(dg < 1e300));
          if (badmask && lane == 0) atomicCAS(a.info, 0, kb * TB + __ffs(badmask));
        }
        if (kb == 0 && lane == 0) stamps[12] = global_ns() + (unsigned long long)(sD[0] == 12345.678);
      } else {
        if (nrb > 0 && kb >= 0) {
          // both tiles were last updated by workers in step kb - 1
          if (kb > 0 && tid == 32) {
            unsigned v;
            do {
              asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(wcnt) : "memory");
            } while (v < w_arrived_prev);
          }
          asm volatile("bar.sync 1, 224;" ::: "memory");
          const double* srcA = W64 + (size_t)(kb + 1) * TB * MP + kb * TB;
          const double* srcC = W64 + (size_t)(kb + 1) * TB * MP + (kb + 1) * TB;
          for (int e = tid - 32; e < TB * TB; e += 224) {
            const int r = e >> 5, c = e & 31;
            sA[r * GLD + c] = srcA[(size_t)r * MP + c];
            sC[r * GLD + c] = srcC[(size_t)r * MP + c];
          }
        }
      }
      __syncthreads();                                    // L_kk, Dinv, and the look-ahead operands are in shared memory
      if (a.debug_stop == 9 && tid == 0 && kb >= 0 && kb < 8) stamps[17 + 2 * kb] = global_ns();
      if (a.debug_stop == 8 && tid == 0 && kb == 2) stamps[17] = global_ns();
      if (kb < 0) continue;                               // warm-up iteration: nothing is published
#pragma unroll
      for (int i = 0; i < 4; ++i) {                       // write-once outputs: diagonal blocks of L and of L^-1
        const int r = warp + 8 * i;
        L64[(size_t)(kb * TB + r) * MP + kb * TB + lane] = cur[r * GLD + lane];
        // Dinv is its own flag: the workers poll this block until the sentinel is gone (8-byte stores are atomic), so
        // no release (a ~0.5 us memory barrier) sits between the factorisation and the look-ahead products
        *reinterpret_cast<volatile double*>(Li64 + (size_t)(kb * TB + r) * MP + kb * TB + lane) = sD[r * GLD + lane];
      }
      if (nrb > 0) {
        // look-ahead: the next diagonal block, C = A_(kb+1)(kb+1) - P P^T with P = A_(kb+1)(kb) Dinv^T = L_(kb+1)(kb)
        if (a.debug_stop == 8 && tid == 0 && kb == 2) stamps[18] = global_ns();
        Frag pfr = {};
        smem_gemm32(pfr, sA, sD);
        frag_park(sP, pfr, 1.0);
        frag_store(L64, MP, (kb + 1) * TB, kb * TB, pfr, 1.0);
        __syncthreads();
        if (a.debug_stop == 8 && tid == 0 && kb == 2) stamps[19] = global_ns();
        Frag u = {};
        smem_gemm32(u, sP, sP);
        int row, col0;
        frag_coords(row, col0);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const double2 cv = *reinterpret_cast<const double2*>(sC + row * GLD + col0 + 8 * j);
          *reinterpret_cast<double2*>(nxt + row * GLD + col0 + 8 * j) = make_double2(cv.x - u.c[j][0], cv.y - u.c[j][1]);
        }
        if (a.debug_stop == 8 && tid == 0 && kb == 2) stamps[20] = global_ns() + (unsigned long long)(u.c[0][0] == 12345.678);
      }
    } else if ((int)blockIdx.x - 1 < n_items) {
      const int w = (int)blockIdx.x - 1;
      auto item_decode = [&](int it, int& bi, int& bj, bool& trailing) {
        if (nrb == 0) { bi = kb; bj = it; trailing = false; return; }
        const int t = it + 1;                             // trailing tile 0 is CTA 0's
        if (t < ntr) {
          int ti, tj;
          tri_decode(t, ti, tj);
          bi = kb + 1 + ti; bj = kb + 1 + tj; trailing = true;
        } else {
          const int yi = (t - ntr) / (kb + 1);
          bi = kb + 1 + yi; bj = (t - ntr) - yi * (kb + 1); trailing = false;
        }
      };
      double preA[4] = {0.0, 0.0, 0.0, 0.0}, preB[4] = {0.0, 0.0, 0.0, 0.0};
      auto item_fetch = [&](int it) {
        int bi, bj; bool trailing;
        item_decode(it, bi, bj, trailing);
        if (nrb > 0) fetch_tile(preA, MatRef{W64, MP, false}, bi * TB, kb * TB);
        if (trailing) { if (bj != bi) fetch_tile(preB, MatRef{W64, MP, false}, bj * TB, kb * TB); }
        else if (bj != kb) fetch_tile(preB, MatRef{T64, MP, false}, kb * TB, bj * TB);
      };
      if (kb > 0) wait_counter(wcnt, w_arrived_prev);    // every tile of step kb - 1 is visible
      else __syncthreads();
      item_fetch(w);                                      // in flight while CTA 0 still factorises
      {
        // Dinv_kb: poll the block itself (volatile loads bypass L1) until CTA 0 has overwritten the sentinel
        double dv[4];
        const int tx = lane, ty = warp;
        const volatile long long* src =
            reinterpret_cast<const volatile long long*>(Li64 + (size_t)(kb * TB + ty) * MP + kb * TB + tx);
        long long b0, b1, b2, b3;
        do {                                      // the four loads of a thread travel together (one L2 round trip)
          b0 = src[0];
          b1 = src[(size_t)8 * MP];
          b2 = src[(size_t)16 * MP];
          b3 = src[(size_t)24 * MP];
        } while (b0 == kDinvSentinel || b1 == kDinvSentinel || b2 == kDinvSentinel || b3 == kDinvSentinel);
        dv[0] = __longlong_as_double(b0);
        dv[1] = __longlong_as_double(b1);
        dv[2] = __longlong_as_double(b2);
        dv[3] = __longlong_as_double(b3);
        park_operand(sD, dv, false);
        park_operand(sDT, dv, true);
      }
      for (int it = w; it < n_items; it += NW) {
        int bi, bj; bool trailing;
        item_decode(it, bi, bj, trailing);
        if (it != w) {
          __syncthreads();                      // the previous item's products are done with the operand buffers
          item_fetch(it);
        }
        if (nrb == 0) {
          // X[kb][bj] = -Dinv Y[kb][bj]
          park_operand(sB, preB, true);
          __syncthreads();
          Frag x = {};
          smem_gemm32(x, sD, sB);
          frag_store(Li64, MP, kb * TB, bj * TB, x, -1.0);
          continue;
        }
        park_operand(sA, preA, false);
        if (trailing) { if (bj != bi) park_operand(sB, preB, false); }
        else if (bj != kb) park_operand(sB, preB, true);
        Frag cfr = {};                          // C_ij or Y_ij, requested before the products
        if (trailing) frag_load(cfr, W64, MP, bi * TB, bj * TB);
        else if (bj != kb) frag_load(cfr, T64, MP, bi * TB, bj * TB);
        __syncthreads();
        Frag p = {};
        smem_gemm32(p, sA, sD);                 // P_i = A_ik Dinv^T  (B^T layout of Dinv^T is Dinv row-major)
        frag_park(sP, p, 1.0);
        const double* second = sQ;
        if (trailing) {
          if (bj != bi) {
            Frag q = {};
            smem_gemm32(q, sB, sD);
            frag_park(sQ, q, 1.0);
          } else {
            second = sP;
          }
          if (bj == kb + 1) frag_store(L64, MP, bi * TB, kb * TB, p, 1.0);      // L[bi][kb], write-once
        } else if (bj != kb) {
          Frag x = {};
          smem_gemm32(x, sD, sB);               // Dinv Y_kj
          frag_park_t(sQ, x, -1.0);             // X_kj = -(...) as a B operand: [col][k]
          if (bi == kb + 1) frag_store(Li64, MP, kb * TB, bj * TB, x, -1.0);    // X[kb][bj], write-once
        } else {
          second = sDT;
        }
        __syncthreads();
        Frag u = {};
        smem_gemm32(u, sP, second);
        if (trailing) {
#pragma unroll
          for (int j = 0; j < 2; ++j) { cfr.c[j][0] -= u.c[j][0]; cfr.c[j][1] -= u.c[j][1]; }
          frag_store(W64, MP, bi * TB, bj * TB, cfr, 1.0);
        } else {
#pragma unroll
          for (int j = 0; j < 2; ++j) { cfr.c[j][0] += u.c[j][0]; cfr.c[j][1] += u.c[j][1]; }
          frag_store(T64, MP, bi * TB, bj * TB, cfr, 1.0);
        }
      }
      signal_counter(wcnt);
    }
    w_arrived_prev += (unsigned)(n_items < NW ? n_items : NW);
  }
  if (NW == 0) aux_operands(0, 1);
  GPBLUR_GRID_SYNC();   // L, L^-1 and the auxiliary operands complete and visible

  GPBLUR_STAMP();   // (the slot of the former recursive-doubling inverse phase: now ~0)
  if (a.debug_stop == 3) return;
  GPBLUR_STAMP();
  GPBLUR_STAMP();
  // ---------------- phase 4: fp32 operands, TF32 operand images of Linv, beta - ONE pass over disjoint CTA groups -------
  // units: [nb^2 fp32 tiles | (n_fwd + n_bwd) * parts image parts | MP / 32 beta chunks]; a CTA takes units
  // blockIdx.x, + G, ...: with G >= the unit count (launch_mm_forward) every CTA has one, and the three kinds of work -
  // one L2 round trip each - overlap instead of queueing behind each other (they took 1.1 + 4.6 + 2.6 us in sequence).
  {
    const int nsl = MP / 32;
    const int BW = tc_bw(MP), NP = MP / BW, spb = BW / 32;
    const int BT = tc_bq(MP), NPT = MP / BT, spt = BT / 32;
    const int n_fwd = MP >= 128 ? spb * NP * (NP + 1) / 2 : 0;
    const int n_bwd = MP >= 128 ? NPT * nsl - spt * NPT * (NPT - 1) / 2 : 0;
    const int n_tiles = nb * nb, n_beta = MP / 32;
    int parts = n_fwd + n_bwd > 0 ? (G - n_tiles - n_beta) / (n_fwd + n_bwd) : 1;
    parts = parts < 1 ? 1 : (parts > 8 ? 8 : parts);
    const int n_img = (n_fwd + n_bwd) * parts;
    float* LinvU = ws_ptr<float>(a.ws, L.LinvU);
    float* LCTQ = ws_ptr<float>(a.ws, L.LCTQ);
    __shared__ double bred[8][32];
    for (int unit = blockIdx.x; unit < n_tiles + n_img + n_beta; unit += G) {
      if (unit < n_tiles) {
        const int bi = unit / nb, bj = unit - bi * nb;
        __syncthreads();
        if (bi >= bj) load_tile(As, MatRef{Li64, MP, false}, bi * TB, bj * TB);
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = warp + 8 * i;
          // LC32 tile (bi, bj): element (r, lane)
          const int gi = bi * TB + r, gj = bj * TB + lane;
          float v = 0.f;
          if (bi >= bj && gj <= gi) v = (float)As[r][lane];
          LC32[(size_t)gi * MP + gj] = v * cvec[gi];
          Linv32[(size_t)gi * MP + gj] = v;
          // LinvT32 tile (bj, bi): element (r, lane) = Linv[bi*TB + lane][bj*TB + r]
          const int ti = bi * TB + lane, tj = bj * TB + r;
          float vt = 0.f;
          if (bi >= bj && tj <= ti) vt = (float)As[lane][r];
          LinvT32[(size_t)tj * MP + ti] = vt;
          LCT32[(size_t)tj * MP + ti] = vt * cvec[ti];
        }
      } else if (unit < n_tiles + n_img) {
        // Linv images (forward): image (p, s) holds rows i = ilo + r, ilo = max(p BW, 32 s), k = j = 32 s + 4 c + e
        // (diag(c) Linv)^T images (backward): image (p, s) holds rows j = p BT + r, k = i = 32 s + 4 c + e
        const int iu = unit - n_tiles;
        const int img = iu / parts, part = iu - img * parts;
        const bool fwd_img = img < n_fwd;
        int rem = fwd_img ? img : img - n_fwd, pp = 0;
        while (true) {
          const int cnt = fwd_img ? (pp + 1) * spb : nsl - pp * spt;
          if (rem < cnt) break;
          rem -= cnt;
          ++pp;
        }
        const int sl = fwd_img ? rem : pp * spt + rem;
        int nr;
        float* base = fwd_img ? LinvU + tc_linv_image(MP, pp, sl, &nr) : LCTQ + tc_lctq_image(MP, pp, sl, &nr);
        const int ilo = (pp + 1) * BW - nr;
#pragma unroll 4
        for (int idx = part * kThreads + tid; idx < 8 * nr * 4; idx += parts * kThreads) {
          const int e = idx & 3, r = (idx >> 2) % nr, c = (idx >> 2) / nr;
          float v;
          if (fwd_img) {
            const int i = ilo + r, j = 32 * sl + 4 * c + e;
            v = (j <= i) ? (float)Li64[(size_t)i * MP + j] : 0.f;
          } else {
            const int i = 32 * sl + 4 * c + e, j = pp * BT + r;
            v = (j <= i) ? (float)Li64[(size_t)i * MP + j] * cvec[i] : 0.f;
          }
          float hi, lo;
          split_tf32(v, hi, lo);
          base[(c * nr + r) * 4 + e] = hi;
          base[32 * nr + (c * nr + r) * 4 + e] = lo;
        }
      } else {
        // beta = Linv^T m : one unit per 32-column chunk, lanes = columns (coalesced rows), the 8 warps split the rows
        const int cj = unit - n_tiles - n_img;
        const int j = cj * 32 + lane;
        double sacc = 0.0;
#pragma unroll 4
        for (int i = cj * 32 + warp; i < M; i += 8)
          if (i >= j) sacc = fma(Li64[(size_t)i * MP + j], (double)mvec[i], sacc);
        __syncthreads();
        bred[warp][lane] = sacc;
        __syncthreads();
        if (warp == 0) {
          double t = 0.0;
#pragma unroll
          for (int w = 0; w < 8; ++w) t += bred[w][lane];
          beta[j] = (float)t;
        }
      }
    }
  }
  GPBLUR_STAMP();
  GPBLUR_STAMP();
  if (blockIdx.x == 0 && tid == 0) stamps[13] = global_ns();
  GPBLUR_STAMP();
#undef GPBLUR_STAMP
}

// ==================================================================================================
// MP = 32 (M <= 32: configs[0]): the whole stage is ONE 32 x 32 block.  The general kernel above spends its time in
// grid barriers and L2 round trips between phases that have nothing to parallelise here (measured at M = 32: 16 us
// in-kernel warm, 26 us cold, 30 us with the cooperative launch around it), so this case gets ONE CTA that keeps
// everything in shared memory: no grid barrier, a plain launch, and the hyper-parameter vectors / Z~ operands are
// built by warps 1-7 WHILE warp 0 factorises.  Same arithmetic, same output regions of the stage.
constexpr int kSmallZs = TB * (GPBLUR_MAX_D + 1);     // doubles: scaled inducing points [32][DP + 1]
constexpr size_t kSmallFwdSmem = (size_t)(kSmallZs + 2 * TB * TLD + 2 * TB + GPBLUR_MAX_D) * sizeof(double) +
                                 (size_t)(2 * GPBLUR_MAX_D + 2 * TB) * sizeof(float);

template <bool MAT>
__global__ void __launch_bounds__(kThreads) mm_small_forward_kernel(MmFwdArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* Zs = reinterpret_cast<double*>(smem_raw);          // [32][DP + 1]  Z / ell (raw, not centred: differences)
  double* Ks = Zs + kSmallZs;                                // [32][33]      Kzz + jitter, then L
  double* Xs = Ks + TB * TLD;                                // [32][33]      L^-1
  double* lcol = Xs + TB * TLD;                              // [64]
  double* ie_s = lcol + 2 * TB;                              // [DP]          1 / ell (double)
  float* cen_s = reinterpret_cast<float*>(ie_s + GPBLUR_MAX_D);   // [DP]  input centre (float, as the point kernels use it)
  float* inv_s = cen_s + GPBLUR_MAX_D;                       // [DP]  1 / ell (float)
  float* m_s = inv_s + GPBLUR_MAX_D;                         // [32]  variational mean
  float* c_s = m_s + TB;                                     // [32]  s^2 - 1
  __shared__ double os_s;

  const WsLayout& L = a.L;
  const int D = L.D, DP = L.DP, M = L.M, MP = L.MP;          // MP == 32
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ZP = DP + 1;                                     // pitch of Zs
  float* hyp = ws_ptr<float>(a.ws, L.hyp);
  double* hyp64 = ws_ptr<double>(a.ws, L.hyp64);
  float* Zt = ws_ptr<float>(a.ws, L.Zt);
  float* ZtT = ws_ptr<float>(a.ws, L.ZtT);
  double* K64 = ws_ptr<double>(a.ws, L.K64);
  double* L64 = ws_ptr<double>(a.ws, L.L64);
  double* Li64 = ws_ptr<double>(a.ws, L.Linv64);
  const float* Z = a.p.inducing_points;
  unsigned long long* stamps = ws_ptr<unsigned long long>(a.ws, L.stamps);
  if (tid == 0) stamps[0] = global_ns();

  // ---- per-dimension hyper-parameters and the input centre (threads = dimensions); outputscale; KL (warp 7) ----
  if (tid < DP) {
    const int d = tid;
    float c = 0.f, e = 1.f, ie = 0.f, w = 0.f;
    double ied = 0.0;
    if (d < D) {
      const double ell = softplus64((double)a.p.raw_lengthscale[d]);
      double s = 0.0;
      for (int m = 0; m < M; ++m) s += (double)Z[(size_t)m * D + d];
      c = (float)(s / (double)M);
      e = (float)ell;
      ied = 1.0 / ell;
      ie = (float)ied;
      w = a.p.mean_weights ? (float)(ell * (double)a.p.mean_weights[d]) : 0.0f;
    }
    ws_ptr<float>(a.ws, L.center)[d] = c;
    ws_ptr<float>(a.ws, L.ell)[d] = e;
    ws_ptr<float>(a.ws, L.inv_ell)[d] = ie;
    ws_ptr<float>(a.ws, L.wl)[d] = w;
    cen_s[d] = c; inv_s[d] = ie; ie_s[d] = ied;
  }
  if (warp == 7) {
    const double os = softplus64((double)a.p.raw_outputscale[0]);
    double part = 0.0;
    if (lane < M) {
      const double mm = (double)a.p.variational_mean[lane], ss = (double)a.p.variational_stddev[lane];
      part = ss * ss + mm * mm - 1.0 - log(ss * ss);
    }
    part = warp_sum(part);
    if (lane == 0) {
      os_s = os;
      hyp[H_OS] = (float)os;
      hyp[H_JIT] = kJitter;
      hyp64[H_JIT] = (double)kJitter + a.extra_jitter;
      hyp[H_KL] = (float)(0.5 * part);
      hyp64[H_OS] = os;
      hyp64[H_KL] = 0.5 * part;
      if (MAT && L.kind == GPBLUR_KERNEL_RQ) set_alpha(hyp, hyp64, a.p.raw_alpha);
      if (a.kl) a.kl[0] = (float)(0.5 * part);
      if (a.info) a.info[0] = 0;
    }
  }
  if (tid < MP) {
    const float mm = tid < M ? a.p.variational_mean[tid] : 0.f;
    const float ss = tid < M ? a.p.variational_stddev[tid] : 1.f;
    const float cc = tid < M ? ss * ss - 1.0f : 0.f;
    ws_ptr<float>(a.ws, L.mvec)[tid] = mm;
    ws_ptr<float>(a.ws, L.svec)[tid] = ss;
    ws_ptr<float>(a.ws, L.cvec)[tid] = cc;
    m_s[tid] = mm; c_s[tid] = cc;
  }
  __syncthreads();
  // ---- Z / ell in double (rows m >= M and columns d >= D are zero) ----
  for (int idx = tid; idx < MP * DP; idx += kThreads) {
    const int m = idx / DP, d = idx - m * DP;
    Zs[m * ZP + d] = (m < M && d < D) ? (double)Z[(size_t)m * D + d] * ie_s[d] : 0.0;
  }
  __syncthreads();
  // ---- Kzz + jitter (direct differences, fp64), identity padding ----
  {
    const double os = os_s;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int gi = warp + 8 * i, gj = lane;
      double acc = 0.0;
      for (int d = 0; d < DP; ++d) {
        const double df = Zs[gi * ZP + d] - Zs[gj * ZP + d];
        acc = fma(df, df, acc);
      }
      double kv;
      if (gi < M && gj < M) {
        if constexpr (!MAT) {
          kv = os * exp(-0.5 * acc) + (gi == gj ? (double)kJitter + a.extra_jitter : 0.0);
        } else {
          double kk, g, ka;
          kernel_kg64(L.kind, acc, os, hyp64[H_ALPHA], kk, g, ka);
          kv = kk + (gi == gj ? (double)kJitter + a.extra_jitter : 0.0);
          ws_ptr<double>(a.ws, L.D2zz64)[(size_t)gi * MP + gj] = acc;
        }
      } else {
        kv = (gi == gj) ? 1.0 : 0.0;
      }
      K64[(size_t)gi * MP + gj] = kv;
      Ks[gi * TLD + gj] = kv;
    }
  }
  __syncthreads();
  if (warp == 0) {
    // ---- Cholesky + inverse of the one block (registers, one row per lane) ----
    double arow[TB], xcol[TB];
#pragma unroll
    for (int c = 0; c < TB; ++c) arow[c] = Ks[lane * TLD + c];
    chol32_inv_warp(arow, xcol, lane, lcol);
#pragma unroll
    for (int c = 0; c < TB; ++c) {
      L64[(size_t)lane * MP + c] = arow[c];
      Li64[(size_t)c * MP + lane] = xcol[c];            // xcol[r] = Linv[r][lane]
      Xs[c * TLD + lane] = xcol[c];
      Ks[lane * TLD + c] = arow[c];                     // L (row `lane` is this lane's own)
    }
    if (a.info) {
      const double dg = Ks[lane * TLD + lane];          // (a dynamic index into arow would push it out of registers)
      const unsigned badmask = __ballot_sync(0xffffffffu, !(dg > 0.0) || !(dg < 1e300));
      if (badmask && lane == 0) a.info[0] = __ffs(badmask);
    }
  } else {
    // ---- meanwhile: Z~ (centred, scaled; fp32 exactly as the point kernels evaluate it), |z~|^2, exponent offsets ----
    const int t7 = tid - 32;
    auto zt_of = [&](int m, int d) -> float {
      return (m < M && d < D) ? (Z[(size_t)m * D + d] - cen_s[d]) * inv_s[d] : 0.f;
    };
    for (int idx = t7; idx < MP * DP; idx += kThreads - 32) {
      const int m = idx / DP, d = idx - m * DP;
      const float v = zt_of(m, d);
      Zt[idx] = v;
      ZtT[(size_t)d * MP + m] = v;
    }
    float* zn = ws_ptr<float>(a.ws, L.zn);
    float* znc = ws_ptr<float>(a.ws, L.znc);
    const float l2os = (float)(log(os_s) * 1.4426950408889634);
    for (int j = warp - 1; j < MP; j += 7) {
      float z2 = 0.f;
      for (int d = lane; d < DP; d += 32) { const float v = zt_of(j, d); z2 = fmaf(v, v, z2); }
      z2 = warp_sum(z2);
      if (lane == 0) {
        zn[j] = z2;
        znc[j] = j < M ? fmaf(-0.72134752044448170f, z2, l2os) : -1e30f;
      }
    }
    if (warp == 1) {
      double sdot = 0.0;
      if (a.p.mean_weights)
        for (int d = lane; d < D; d += 32) sdot += (double)cen_s[d] * (double)a.p.mean_weights[d];
      sdot = warp_sum(sdot);
      if (lane == 0) hyp[H_CWB] = (float)(sdot + (double)a.p.mean_bias[0]);
    }
  }
  __syncthreads();
  // ---- fp32 operands of the point kernels and beta = Linv^T m ----
  {
    float* LinvT32 = ws_ptr<float>(a.ws, L.LinvT32);
    float* LC32 = ws_ptr<float>(a.ws, L.LC32);
    float* Linv32 = ws_ptr<float>(a.ws, L.Linv32);
    float* LCT32 = ws_ptr<float>(a.ws, L.LCT32);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = warp + 8 * i;
      const float v = lane <= r ? (float)Xs[r * TLD + lane] : 0.f;       // Linv[r][lane]
      LC32[(size_t)r * MP + lane] = v * c_s[r];
      Linv32[(size_t)r * MP + lane] = v;
      const float vt = r <= lane ? (float)Xs[lane * TLD + r] : 0.f;      // Linv[lane][r]
      LinvT32[(size_t)r * MP + lane] = vt;
      LCT32[(size_t)r * MP + lane] = vt * c_s[lane];
    }
    if (warp == 0) {
      double t = 0.0;
      for (int i = lane; i < M; ++i) t = fma(Xs[i * TLD + lane], (double)m_s[i], t);
      ws_ptr<float>(a.ws, L.beta)[lane] = (float)t;
    }
  }
  if (tid == 0) { stamps[1] = stamps[0]; stamps[7] = global_ns(); for (int k = 2; k < 7; ++k) stamps[k] = stamps[7]; stamps[13] = stamps[7]; }
}

// ==================================================================================================
struct MmBwdArgs {
  gpblur_svgp_params p;
  WsLayout L;
  void* ws;               // parameter stage (fp64 scratch regions T64 / U64 / v64 / t64 are overwritten)
  const double* sgrad;    // summed stage gradient [u | vec | S | W^T X (| RQ: sum kbar o dk/dalpha)], stage_grad_doubles()
  const float* g_kl;
  float* bucket;
  int accumulate;         // != 0: add into `bucket` (it is the caller's live gradient buffer) instead of overwriting it
  unsigned* bar;          // see MmFwdArgs
};
#define GPBLUR_PUT(ptr, val) do { float* p_ = (ptr); const float v_ = (val); *p_ = a.accumulate ? *p_ + v_ : v_; } while (0)

// Per-call reduction of the split partials into the stage gradient (fixed order => bit-deterministic).
struct SgReduceArgs {
  WsLayout L;
  const void* ws;
  double* sgrad;
  int nvec_used;
  int ncpart;   // > 0: column sums of W come as [ncpart][MP] partials from the tensor-core W^T X kernel
};

__global__ void __launch_bounds__(kThreads, 6) stage_grad_reduce_kernel(SgReduceArgs a) {   // latency-bound: occupancy matters
  const WsLayout& L = a.L;
  const int MP = L.MP, DP = L.DP;
  const float* Spart = ws_cptr<float>(a.ws, L.Spart);
  const float* upart = ws_cptr<float>(a.ws, L.upart);
  const float* WXpart = ws_cptr<float>(a.ws, L.WXpart);
  const float* vecpart = ws_cptr<float>(a.ws, L.vecpart);
  const float* cpart = ws_cptr<float>(a.ws, L.cpart);
  const bool tc = a.ncpart > 0;
  // S region: the FFMA Gram holds only the lower tile triangle (tiles of min(MP, 128)) of full [MP x MP] partials, read in
  // output order (upper elements transposed); the tensor-core Gram packed lower-triangle 128 x 128 blocks, read in
  // packed order (coalesced), lower elements only, each written to (i, j) and its mirror (j, i).
  // Both paths sum the partials of the LOWER element for (i, j) and (j, i), so S is exactly symmetric: the Gram
  // computes the two elements of a pair inside a diagonal block separately, and mm_backward_kernel's first product
  // reads S(i, k) as S(max, min).
  const size_t n_u = MP, n_vec = L.vec_len, n_S = tc ? tc_gram_floats(MP) : (size_t)MP * MP, n_WX = (size_t)MP * DP;
  const size_t n_kba = L.kind == GPBLUR_KERNEL_RQ ? 1 : 0;   // RQ: sum kbar o dk/dalpha, after W^T X
  const size_t total = n_u + n_vec + n_S + n_WX + n_kba;
  const size_t s_out = n_u + n_vec;   // first S element of the stage gradient
  // A CTA owns 32 consecutive input elements per iteration (lanes, coalesced); warp g sums partials g, g + 8, ...
  // and the 8 warp sums are folded in fixed order through shared memory (bit-deterministic), which keeps 8x more
  // loads in flight than one thread per element.
  __shared__ double red[8][32];
  const int g = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t nchunks = (total + 31) / 32;
  for (size_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const size_t e = ch * 32 + lane;
    size_t dst = e, mirror = 0;   // output element(s); mirror 0: none
    bool skip = false;            // upper element of a diagonal block (tensor-core Gram): written by its mirror
    if (e >= s_out + n_S) dst = e - n_S + (size_t)MP * MP;
    double s = 0.0;
    if (e >= s_out && e < s_out + n_S) {
      const size_t idx = e - s_out;
      int i, j;
      const float* src;
      size_t pstride;
      int nsp = L.splitsS;
      if (tc) {
        tc_gram_element(idx, &i, &j);
        src = Spart + idx;
        pstride = tc_gram_floats(MP);
        if (!tc_gram_diag_block(MP, i >> 7, j >> 7)) nsp = L.splitsO;
        skip = i < j;
        if (i > j) mirror = s_out + (size_t)j * MP + i;
      } else {
        i = (int)(idx / MP); j = (int)(idx - (size_t)i * MP);
        const bool lower = i >= j;
        src = Spart + (size_t)(lower ? i : j) * MP + (lower ? j : i);
        pstride = (size_t)MP * MP;
      }
      dst = s_out + (size_t)i * MP + j;
      if (L.N > 0 && !skip) {
        // loads batched 4 deep before the (ordered) adds: independent requests in flight
        int sp = g;
        for (; sp + 24 < nsp; sp += 32) {
          const float v0 = src[(size_t)sp * pstride], v1 = src[(size_t)(sp + 8) * pstride];
          const float v2 = src[(size_t)(sp + 16) * pstride], v3 = src[(size_t)(sp + 24) * pstride];
          s += (double)v0; s += (double)v1; s += (double)v2; s += (double)v3;
        }
        for (; sp < nsp; sp += 8) s += (double)src[(size_t)sp * pstride];
      }
    } else if (e < total && L.N > 0) {
      if (e < n_u) {
        for (int sp = g; sp < L.splitsS; sp += 8) s += (double)upart[(size_t)sp * MP + e];
      } else if (e < n_u + n_vec) {
        const size_t k = e - n_u;
        for (int c = g; c < a.nvec_used; c += 8) s += (double)vecpart[(size_t)c * L.vp_len + k];
        if (tc && k < (size_t)MP)
          for (int c = g; c < a.ncpart; c += 8) s += (double)cpart[(size_t)c * MP + k];
      } else if (e < s_out + n_S + n_WX) {
        const size_t idx = e - s_out - n_S;
        for (int sp = g; sp < L.splitsZ; sp += 8) s += (double)WXpart[(size_t)sp * MP * DP + idx];
      } else {
        for (int c = g; c < a.nvec_used; c += 8) s += (double)vecpart[(size_t)c * L.vp_len + L.vec_len];   // VS_KBA
      }
    }
    __syncthreads();
    red[g][lane] = s;
    __syncthreads();
    if (g == 0 && e < total && !skip) {
      double t = 0.0;
#pragma unroll
      for (int w = 0; w < 8; ++w) t += red[w][lane];
      a.sgrad[dst] = t;
      if (mirror) a.sgrad[mirror] = t;
    }
  }
}

template <int RT, bool MAT>
__global__ void __launch_bounds__(kThreads) mm_backward_kernel(MmBwdArgs a) {
  constexpr int NH = TB / RT;   // row parts of a 32 x 32 tile
  constexpr int NR = RT / 8;    // rows per thread
  cg::grid_group grid = cg::this_grid();
  unsigned bar_target = 0;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* gsm = reinterpret_cast<double*>(smem_raw);      // tile_gemm scratch

  const WsLayout& L = a.L;
  const int D = L.D, DP = L.DP, M = L.M, MP = L.MP;
  const int nb = MP / TB;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = gridDim.x;
  const int gtid = blockIdx.x * kThreads + tid, gsize = G * kThreads;

  const float* hyp = ws_cptr<float>(a.ws, L.hyp);
  double* hyp64 = ws_ptr<double>(a.ws, L.hyp64);
  const float* inv_ell = ws_cptr<float>(a.ws, L.inv_ell);
  const float* center = ws_cptr<float>(a.ws, L.center);
  const float* Zt = ws_cptr<float>(a.ws, L.Zt);
  const float* mvec = ws_cptr<float>(a.ws, L.mvec);
  const float* cvec = ws_cptr<float>(a.ws, L.cvec);
  const float* svec = ws_cptr<float>(a.ws, L.svec);
  const double* K64 = ws_cptr<double>(a.ws, L.K64);
  const double* Li64 = ws_cptr<double>(a.ws, L.Linv64);
  double* T64 = ws_ptr<double>(a.ws, L.T64);
  double* U64 = ws_ptr<double>(a.ws, L.U64);
  // stage gradient (read-only): [u MP | vec vec_len | S MP x MP | W^T X MP x DP | RQ: sum kbar o dk/dalpha]
  const double* u64 = a.sgrad;
  const double* vec64 = a.sgrad + MP;
  const double* S64 = vec64 + L.vec_len;
  const double* WX64 = S64 + (size_t)MP * MP;
  // fp64 vector scratch: [per-item sums of sym(Kb) o (Kzz - jitter I) (Matern / RQ kinds; NH nb^2 <= MP items) |
  // per-item sums of sym(Kb) o dKzz/dalpha (RQ; in vec_len >= MP) | unused MP | rz MP]
  double* v64 = ws_ptr<double>(a.ws, L.v64);
  double* kbk64 = v64;
  double* kba64 = v64 + MP;
  double* rz64 = v64 + 2 * MP + L.vec_len;
  double* t64 = ws_ptr<double>(a.ws, L.t64);   // [MP, DP] per-(i, d) terms of d lengthscale

  unsigned long long* stamps = ws_ptr<unsigned long long>(a.ws, L.stamps) + 16;
  int stamp_i = 0;
#define GPBLUR_STAMP() do { if (blockIdx.x == 0 && tid == 0) stamps[stamp_i] = global_ns(); ++stamp_i; } while (0)
  GPBLUR_STAMP();

  // Work items of the product phases: item t -> tile t / NH = (bi, bj), rows bi * 32 + RT (t % NH) .. + RT.
  // ---------------- phase A: Tm = P Linv -> T64 (full) ----------------
  // P = sym(Phi(L^T Lbar)) in closed form (PForm): the lower triangle of L^T Lbar reads only the lower triangle of
  // Lbar = -tril(Linv^T X), X = m u^T + 2 diag(c) S, and L^T Linv^T = I, so Phi(L^T Lbar) = -Phi(X); and
  // sym(Linv^T Phi Linv) = Linv^T P Linv.  Linv is lower triangular: k runs from the column block up.
  for (int t = blockIdx.x; t < NH * nb * nb; t += G) {
    const int tile = t / NH, bi = tile / nb, bj = tile - bi * nb, r0 = bi * TB + RT * (t % NH);
    double acc[NR] = {};
    wide_gemm<RT>(acc, MatRef{S64, MP, false}, r0, MatRef{Li64, MP, false}, bj * TB, bj * TB, MP, gsm, nullptr,
                  PForm{mvec, u64, cvec});
#pragma unroll
    for (int i = 0; i < NR; ++i) T64[(size_t)(r0 + warp + 8 * i) * MP + bj * TB + lane] = acc[i];
  }
  GPBLUR_GRID_SYNC();

  GPBLUR_STAMP();
  // ---------------- phase B: sym(Kb) = Linv^T Tm ; Wzz = sym(Kb) o (Kzz - jitter I) -> U64 ----------------
  // Matern / RQ kinds: Wzz = sym(Kb) o g(d2) from the distances the forward kept; the outputscale term
  // sum sym(Kb) o (Kzz - jitter I) is no longer sum Wzz: one partial per item -> kbk64[t], added in fixed order in D.
  // RQ: likewise the alpha term sum sym(Kb) o dKzz/dalpha -> kba64[t].
  {
    const double zz_jitter = hyp64[H_JIT];
    const double os = hyp64[H_OS];
    const bool rq = MAT && L.kind == GPBLUR_KERNEL_RQ;
    const double alpha = rq ? hyp64[H_ALPHA] : 0.0;
    const double* D2 = ws_cptr<double>(a.ws, L.D2zz64);
    __shared__ double kred[8], ared[8];
    for (int t = blockIdx.x; t < NH * nb * nb; t += G) {
      const int tile = t / NH, bi = tile / nb, bj = tile - bi * nb, r0 = bi * TB + RT * (t % NH);
      // operands of the epilogue, requested before the product
      double e_k[NR];
      [[maybe_unused]] double e_d2[NR];
#pragma unroll
      for (int i = 0; i < NR; ++i) {
        const size_t idx = (size_t)(r0 + warp + 8 * i) * MP + bj * TB + lane;
        e_k[i] = K64[idx];
        if constexpr (MAT) e_d2[i] = D2[idx];
      }
      double acc[NR] = {};
      wide_gemm<RT>(acc, MatRef{Li64, MP, true}, r0, MatRef{T64, MP, false}, bj * TB, bi * TB, MP, gsm);
      double kbk = 0.0, kba = 0.0;
#pragma unroll
      for (int i = 0; i < NR; ++i) {
        const int gi = r0 + warp + 8 * i, gj = bj * TB + lane;
        double v = 0.0;
        if (gi < M && gj < M) {
          const double kz = e_k[i] - (gi == gj ? zz_jitter : 0.0);
          if constexpr (MAT) {
            double kk, g, ka = 0.0;
            kernel_kg64(L.kind, e_d2[i], os, alpha, kk, g, ka);
            v = acc[i] * g;
            kbk += acc[i] * kz;
            kba += acc[i] * ka;
          } else {
            v = acc[i] * kz;
          }
        }
        U64[(size_t)gi * MP + gj] = v;
      }
      if constexpr (MAT) {
        kbk = warp_sum(kbk);
        if (lane == 0) kred[warp] = kbk;
        if (rq) {
          kba = warp_sum(kba);
          if (lane == 0) ared[warp] = kba;
        }
        __syncthreads();
        if (tid == 0) {
          double s = 0.0, sa = 0.0;
#pragma unroll
          for (int w8 = 0; w8 < 8; ++w8) s += kred[w8];
          kbk64[t] = s;
          if (rq) {
#pragma unroll
            for (int w8 = 0; w8 < 8; ++w8) sa += ared[w8];
            kba64[t] = sa;
          }
        }
      }
    }
  }
  GPBLUR_GRID_SYNC();

  GPBLUR_STAMP();
  // ---------------- phase C: Kzz-path + a-space gradients of Z; per-(i, d) terms of d ell -------
  // V = Wzz Z~ is an [MP, MP] x [MP, DP] product: 16 x 32 tiles on the FP64 tensor path (a thread-per-(i, d) loop over
  // j exposed one L2 round trip per few terms: 16 us at M = 256, 166 us at M = 1024); the row sums of Wzz come from
  // the staged operand with a fixed shuffle tree.
  auto zgrad_terms = [&](int i, int d, double V, double rz, double wx, double z, double csum) {
    const double ie = (double)inv_ell[d];
    const double wxt = (wx - csum * (double)center[d]) * ie;          // (W^T Xtilde)_id
    const double dz = (wxt - csum * z) * ie + 2.0 * (V - rz * z) * ie;
    GPBLUR_PUT(&a.bucket[(size_t)i * D + d], (float)dz);
    return -2.0 * z * wxt + csum * z * z + 2.0 * rz * z * z - 2.0 * z * V;
  };
  if (DP >= TB) {
    __shared__ double rz_s[RT];
    __shared__ double tred[8][32];
    const int ndt = DP / TB;
    for (int t = blockIdx.x; t < NH * nb * ndt; t += G) {
      const int tile = t / NH, bi = tile / ndt, bd = tile - bi * ndt, r0 = bi * TB + RT * (t % NH);
      // operands of the epilogue, requested before the product
      double e_wx[NR], e_z[NR], e_cs[NR];
#pragma unroll
      for (int r2 = 0; r2 < NR; ++r2) {
        const int i = r0 + warp + 8 * r2, d = bd * TB + lane;
        e_wx[r2] = WX64[(size_t)i * DP + d];
        e_z[r2] = (double)Zt[(size_t)i * DP + d];
        e_cs[r2] = vec64[i];
      }
      double acc[NR] = {};
      wide_gemm<RT>(acc, MatRef{U64, MP, false}, r0, MatRef{nullptr, DP, false, Zt}, bd * TB, 0, MP, gsm, rz_s);
      double tsum = 0.0;
#pragma unroll
      for (int r2 = 0; r2 < NR; ++r2) {
        const int i = r0 + warp + 8 * r2, d = bd * TB + lane;
        if (i < M && d < D) {
          const double rz = rz_s[warp + 8 * r2];
          if (d == 0) rz64[i] = rz;
          tsum += zgrad_terms(i, d, acc[r2], rz, e_wx[r2], e_z[r2], e_cs[r2]);
        }
      }
      // column sums over the RT rows of the item (fixed order) -> t64[item row block][d]; phase D adds the NH nb blocks
      __syncthreads();
      tred[warp][lane] = tsum;
      __syncthreads();
      if (warp == 0) {
        double tt = 0.0;
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) tt += tred[w8][lane];
        t64[(size_t)(NH * bi + (t % NH)) * DP + bd * TB + lane] = tt;
      }
    }
  } else {
    // DP = 16: thread per (i, d)
    for (int idx = gtid; idx < MP * DP; idx += gsize) {
      const int i = idx / DP, d = idx - i * DP;
      double tval = 0.0;
      if (i < M && d < D) {
        double V = 0.0, rz = 0.0;
        for (int j = 0; j < M; ++j) {
          const double w = U64[(size_t)i * MP + j];
          V = fma(w, (double)Zt[(size_t)j * DP + d], V);
          rz += w;
        }
        if (d == 0) rz64[i] = rz;
        tval = zgrad_terms(i, d, V, rz, WX64[(size_t)i * DP + d], (double)Zt[(size_t)i * DP + d], vec64[i]);
      }
      t64[idx] = tval;
    }
  }
  GPBLUR_GRID_SYNC();

  GPBLUR_STAMP();
  // ---------------- phase D: final bucket (block 0) ----------------
  if (blockIdx.x == 0) {
    const double os = hyp64[H_OS];
    const double gkl = a.g_kl ? (double)a.g_kl[0] : 0.0;
    float* b_ell = a.bucket + (size_t)M * D;
    float* b_os = b_ell + D;
    float* b_m = b_os + 1;
    float* b_s = b_m + M;
    float* b_w = b_s + M;
    float* b_b = b_w + D;
    const double* q = vec64 + MP;
    const double* wbar = vec64 + MP + DP;
    const double* sc = vec64 + MP + 2 * DP;
    // column sums of the per-(i, d) terms: NPART row partitions per column, combined in fixed order
    {
      __shared__ double colred[kThreads];
      const int npart = kThreads / DP;           // DP in {16, 32, 64, 128}
      const int d = tid % DP, part = tid / DP;
      double s = 0.0;
#pragma unroll 8
      const int trows = DP >= TB ? NH * nb : M;   // phase C leaves per-item column sums (DP >= 32) or the full terms
      for (int i = part; i < trows; i += npart) s += t64[(size_t)i * DP + d];
      colred[tid] = s;
      __syncthreads();
      if (part == 0 && d < D) {
        double tot = q[d];
        for (int p2 = 0; p2 < npart; ++p2) tot += colred[p2 * DP + d];
        const double dell = tot * (double)inv_ell[d];
        GPBLUR_PUT(&b_ell[d], (float)(dell * sigmoid64((double)a.p.raw_lengthscale[d])));
        GPBLUR_PUT(&b_w[d], a.p.mean_weights ? (float)wbar[d] : 0.f);
      }
    }
    for (int m = tid; m < M; m += kThreads) {
      const double mm = (double)mvec[m], ss = (double)svec[m];
      GPBLUR_PUT(&b_m[m], (float)(u64[m] + gkl * mm));
      GPBLUR_PUT(&b_s[m], (float)(2.0 * ss * S64[(size_t)m * MP + m] + gkl * (ss - 1.0 / ss)));
    }
    if (warp == 0) {
      // sum sym(Kb) o (Kzz - jitter I) + sum kbar o k: for RBF both are the sums of the W matrices
      constexpr bool rbf = !MAT;
      const double* parts = rbf ? rz64 : kbk64;    // row sums of Wzz | per-item sums of phase B
      const int nparts = rbf ? M : NH * nb * nb;
      double s = 0.0;
      for (int i = lane; i < nparts; i += 32) s += parts[i];
      s = warp_sum(s);
      if (lane == 0) {
        const double dos = (s + sc[rbf ? VS_RSUM : VS_KBK]) / os + sc[VS_GVAR];
        GPBLUR_PUT(&b_os[0], (float)(dos * sigmoid64((double)a.p.raw_outputscale[0])));
        GPBLUR_PUT(&b_b[0], (float)sc[VS_GMU]);
      }
    }
    if (MAT && L.kind == GPBLUR_KERNEL_RQ && warp == 1) {
      // d raw_alpha: sum sym(Kb) o dKzz/dalpha (per-item sums of phase B, fixed order) + sum kbar o dk/dalpha
      double s = 0.0;
      for (int i = lane; i < NH * nb * nb; i += 32) s += kba64[i];
      s = warp_sum(s);
      if (lane == 0) {
        const double da = s + WX64[(size_t)MP * DP];
        GPBLUR_PUT(&b_b[1], (float)(da * sigmoid64((double)a.p.raw_alpha[0])));
      }
    }
  }
  GPBLUR_STAMP();
#undef GPBLUR_STAMP
  (void)hyp;
}

// MP = 32: the backward of the one-block stage in ONE CTA (see mm_small_forward_kernel).  All operands (S, L^-1, Kzz,
// Z~, W^T X: < 60 KB) are fetched into shared memory in one round trip; the two 32 x 32 x 32 products of sym(Kbar),
// the Kzz-path terms and the final bucket then run between CTA barriers instead of grid barriers + L2 round trips
// (general kernel at M = 32: 23 us in-kernel, 45 us with the cooperative launch around it).
constexpr size_t kSmallBwdSmem = (size_t)(5 * TB * TLD + 2 * TB * (GPBLUR_MAX_D + 1) + 6 * TB + GPBLUR_MAX_D + 8) * sizeof(double);

template <bool MAT>
__global__ void __launch_bounds__(kThreads) mm_small_backward_kernel(MmBwdArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* Ss = reinterpret_cast<double*>(smem_raw);   // [32][33] S (stage gradient), later Wzz
  double* Li = Ss + TB * TLD;                         // L^-1
  double* Kz = Li + TB * TLD;                         // Kzz + jitter
  double* Us = Kz + TB * TLD;                         // P, then sym(Kbar) o (Kzz - jitter I) (Matern / RQ kinds)
  double* Ts = Us + TB * TLD;                         // Tm, then sym(Kbar) o dKzz/dalpha (RQ)
  double* Zd = Ts + TB * TLD;                         // [32][DP + 1] Z~ (double)
  double* Wx = Zd + TB * (GPBLUR_MAX_D + 1);          // [32][DP + 1] W^T X (stage gradient)
  double* u_s = Wx + TB * (GPBLUR_MAX_D + 1);         // [32]
  double* m_s = u_s + TB;                             // [32]
  double* c_s = m_s + TB;                             // [32]
  double* cs_s = c_s + TB;                            // [32] colsum(W)
  double* rz_s = cs_s + TB;                           // [32] row sums of Wzz
  double* tcol = rz_s + TB;                           // [DP] column sums of the lengthscale terms

  const WsLayout& L = a.L;
  const int D = L.D, DP = L.DP, M = L.M, MP = L.MP;   // MP == 32
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ZP = DP + 1;
  const double* hyp64 = ws_cptr<double>(a.ws, L.hyp64);
  const float* inv_ell = ws_cptr<float>(a.ws, L.inv_ell);
  const float* center = ws_cptr<float>(a.ws, L.center);
  const float* Zt = ws_cptr<float>(a.ws, L.Zt);
  const float* mvec = ws_cptr<float>(a.ws, L.mvec);
  const float* cvec = ws_cptr<float>(a.ws, L.cvec);
  const float* svec = ws_cptr<float>(a.ws, L.svec);
  const double* K64 = ws_cptr<double>(a.ws, L.K64);
  const double* Li64 = ws_cptr<double>(a.ws, L.Linv64);
  const double* u64 = a.sgrad;
  const double* vec64 = a.sgrad + MP;
  const double* S64 = vec64 + L.vec_len;
  const double* WX64 = S64 + (size_t)MP * MP;
  unsigned long long* stamps = ws_ptr<unsigned long long>(a.ws, L.stamps) + 16;
  if (tid == 0) stamps[0] = global_ns();

  // ---- one round trip: everything into shared memory ----
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = warp + 8 * i;
    Ss[r * TLD + lane] = S64[(size_t)r * MP + lane];
    Li[r * TLD + lane] = Li64[(size_t)r * MP + lane];
    Kz[r * TLD + lane] = K64[(size_t)r * MP + lane];
  }
  for (int idx = tid; idx < MP * DP; idx += kThreads) {
    const int m = idx / DP, d = idx - m * DP;
    Zd[m * ZP + d] = (double)Zt[idx];
    Wx[m * ZP + d] = WX64[idx];
  }
  if (tid < MP) {
    u_s[tid] = u64[tid];
    m_s[tid] = (double)mvec[tid];
    c_s[tid] = (double)cvec[tid];
    cs_s[tid] = vec64[tid];
  }
  if (tid < DP) tcol[tid] = 0.0;
  __syncthreads();

  // out(r, lane) for r = warp + 8 i:  sum_k A(r, k) B(k, lane), A / B given as element functions of shared memory
  // ---- phase A: P = sym(Phi(L^T Lbar)) = -1/2 (m_hi u_lo + 2 c_hi S_hi,lo) -> Us (see PForm); Tm = P Linv -> Ts ----
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = warp + 8 * i;
    const int hi = r > lane ? r : lane, lo = r > lane ? lane : r;
    Us[r * TLD + lane] = -fma(c_s[hi], Ss[hi * TLD + lo], 0.5 * m_s[hi] * u_s[lo]);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = warp + 8 * i;
    double acc = 0.0;
    for (int k = 0; k < TB; ++k) acc = fma(Us[r * TLD + k], Li[k * TLD + lane], acc);
    Ts[r * TLD + lane] = acc;
  }
  __syncthreads();
  // ---- phase B: sym(Kbar) = Linv^T Tm ; Wzz = sym(Kbar) o (Kzz - jitter I) -> Ss ; row sums ----
  // (Matern / RQ kinds: Wzz = sym(Kbar) o g(d2); the products sym(Kbar) o (Kzz - jitter I) of the outputscale term are
  //  parked in Us, free since phase A, and summed into kbk; RQ: the products sym(Kbar) o dKzz/dalpha go to Ts once
  //  every thread has read Tm, and are summed in phase D)
  constexpr bool rbf = !MAT;
  const bool rq = MAT && L.kind == GPBLUR_KERNEL_RQ;
  double kbk = 0.0;
  double ua[4] = {0.0, 0.0, 0.0, 0.0};
  {
    const double zz_jitter = hyp64[H_JIT];
    const double os = hyp64[H_OS];
    const double alpha = rq ? hyp64[H_ALPHA] : 0.0;
    const double* D2 = ws_cptr<double>(a.ws, L.D2zz64);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = warp + 8 * i;
      double kb = 0.0;
      for (int k = 0; k < TB; ++k) kb = fma(Li[k * TLD + r], Ts[k * TLD + lane], kb);
      double v = 0.0;
      if (rbf) {
        if (r < M && lane < M) v = kb * (Kz[r * TLD + lane] - (r == lane ? zz_jitter : 0.0));
      } else {
        double u = 0.0;
        if (r < M && lane < M) {
          double kk, g, ka = 0.0;
          kernel_kg64(L.kind, D2[(size_t)r * MP + lane], os, alpha, kk, g, ka);
          v = kb * g;
          u = kb * (Kz[r * TLD + lane] - (r == lane ? zz_jitter : 0.0));
          ua[i] = kb * ka;
        }
        Us[r * TLD + lane] = u;
      }
      Ss[r * TLD + lane] = v;
    }
  }
  __syncthreads();
  if (rq) {
#pragma unroll
    for (int i = 0; i < 4; ++i) Ts[(warp + 8 * i) * TLD + lane] = ua[i];
  }
  if (tid < MP) {
    double rz = 0.0;
    for (int j = 0; j < TB; ++j) rz += Ss[tid * TLD + j];
    rz_s[tid] = rz;
  }
  if (!rbf && warp == 7) {
    for (int r = 0; r < M; ++r) kbk += Us[r * TLD + lane];
    kbk = warp_sum(kbk);
  }
  __syncthreads();
  // (diag(S) of the stage gradient is needed in phase D and Ss now holds Wzz: it is re-read from global memory there)
  // ---- phase C: V = Wzz Z~ ; Kzz-path + a-space gradients of Z ; per-(i, d) lengthscale terms ----
  for (int d0 = 0; d0 < DP; d0 += TB) {
    const int d = d0 + lane;
    double tsum = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = warp + 8 * i;
      double V = 0.0;
      for (int k = 0; k < TB; ++k) V = fma(Ss[r * TLD + k], Zd[k * ZP + d], V);
      if (r < M && d < D) {
        const double ie = (double)inv_ell[d], z = Zd[r * ZP + d], csum = cs_s[r], rz = rz_s[r];
        const double wxt = (Wx[r * ZP + d] - csum * (double)center[d]) * ie;
        const double dz = (wxt - csum * z) * ie + 2.0 * (V - rz * z) * ie;
        GPBLUR_PUT(&a.bucket[(size_t)r * D + d], (float)dz);
        tsum += -2.0 * z * wxt + csum * z * z + 2.0 * rz * z * z - 2.0 * z * V;
      }
    }
    // column sums over the 32 rows: 8 warps x 4 rows each -> shared, added in warp order
    __syncthreads();
    double* part = Us;                     // [8][33] scratch (Us is free now)
    part[warp * TLD + lane] = tsum;
    __syncthreads();
    if (warp == 0) {
      double t = 0.0;
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) t += part[w8 * TLD + lane];
      tcol[d] = t;
    }
    __syncthreads();
  }
  // ---- phase D: final bucket ----
  {
    const double os = hyp64[H_OS];
    const double gkl = a.g_kl ? (double)a.g_kl[0] : 0.0;
    float* b_ell = a.bucket + (size_t)M * D;
    float* b_os = b_ell + D;
    float* b_m = b_os + 1;
    float* b_s = b_m + M;
    float* b_w = b_s + M;
    float* b_b = b_w + D;
    const double* q = vec64 + MP;
    const double* wbar = vec64 + MP + DP;
    const double* sc = vec64 + MP + 2 * DP;
    if (tid < D) {
      const double dell = (q[tid] + tcol[tid]) * (double)inv_ell[tid];
      GPBLUR_PUT(&b_ell[tid], (float)(dell * sigmoid64((double)a.p.raw_lengthscale[tid])));
      GPBLUR_PUT(&b_w[tid], a.p.mean_weights ? (float)wbar[tid] : 0.f);
    }
    if (tid >= 128 && tid < 128 + M) {
      const int m = tid - 128;
      const double mm = (double)mvec[m], ss = (double)svec[m];
      GPBLUR_PUT(&b_m[m], (float)(u_s[m] + gkl * mm));
      GPBLUR_PUT(&b_s[m], (float)(2.0 * ss * S64[(size_t)m * MP + m] + gkl * (ss - 1.0 / ss)));
    }
    if (warp == 7) {
      double s = lane < M ? rz_s[lane] : 0.0;
      s = rbf ? warp_sum(s) : kbk;
      if (lane == 0) {
        const double dos = (s + sc[rbf ? VS_RSUM : VS_KBK]) / os + sc[VS_GVAR];
        GPBLUR_PUT(&b_os[0], (float)(dos * sigmoid64((double)a.p.raw_outputscale[0])));
        GPBLUR_PUT(&b_b[0], (float)sc[VS_GMU]);
      }
    }
    if (rq && warp == 6) {
      // d raw_alpha: column sums of the parked products (rows in order), lanes by the shuffle tree, + sum kbar o dk/dalpha
      double s = 0.0;
      for (int r = 0; r < M; ++r) s += Ts[r * TLD + lane];
      s = warp_sum(s);
      if (lane == 0)
        GPBLUR_PUT(&b_b[1], (float)((s + WX64[(size_t)MP * DP]) * sigmoid64((double)a.p.raw_alpha[0])));
    }
  }
  if (tid == 0) { const unsigned long long t = global_ns(); for (int k = 1; k < 5; ++k) stamps[k] = t; }
}

// Cooperative launches + cg grid.sync() by default.  GPBLUR_MM_COOP=0: plain launches + a counter barrier on a word
// that a memset node zeroes before every launch - the kernels run equally fast, but each memset is one more graph node
// (~3.5 us) on the critical path of a step.
bool mm_cooperative() {
  static const int v = [] { const char* e = getenv("GPBLUR_MM_COOP"); return e ? atoi(e) : 1; }();
  return v != 0;
}

int coop_grid(const void* func, int want, size_t smem) {
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, func, kThreads, smem);
  if (occ < 1) occ = 1;
  const int cap = occ * num_sms();
  if (want < 1) want = 1;
  return want < cap ? want : cap;
}

}  // namespace

// max_ctas > 0: an upper bound on the grid (>= 8): the H independent stages of a multi-output layer are launched on H
// streams with 148 / H CTAs each so that they run CONCURRENTLY (a cooperative grid of ~130 CTAs owns the GPU alone; the
// stage is a latency-bound chain, so ten stages side by side finish in little more than the time of one).
int launch_mm_forward(const gpblur_svgp_params& p, const WsLayout& L, void* ws, float* kl, int* info,
                      cudaStream_t st, double extra_jitter, int max_ctas) {
  const size_t smem = sizeof(Tile) * 11 + kGemmScratchDoubles * sizeof(double);
  const bool mat = L.kind != GPBLUR_KERNEL_RBF;
  const void* fwd = mat ? (const void*)mm_forward_kernel<true> : (const void*)mm_forward_kernel<false>;
  // per-DEVICE attribute: set on every launch (cheap) instead of a process-wide flag
  cudaFuncSetAttribute(fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const int nb = L.MP / TB;
  if (nb == 1) {   // M <= 32: one CTA, no grid barrier, plain launch
    const void* small = mat ? (const void*)mm_small_forward_kernel<true> : (const void*)mm_small_forward_kernel<false>;
    cudaFuncSetAttribute(small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmallFwdSmem);
    MmFwdArgs args{p, L, ws, kl, info, extra_jitter, nullptr, -1, nullptr};
    ProfScope ps(ST_MM_FWD, st);
    void* kargs[] = {&args};
    cudaLaunchKernel(small, dim3(1), dim3(kThreads), kargs, kSmallFwdSmem, st);
    note_launch();
    return check_launch("mm_small_forward");
  }
  // CTA 0 (the factorisation chain) + workers, and enough CTAs that the final pass (fp32 tiles | operand images | beta
  // chunks) gives each of them one unit
  int n_img = 0;
  if (L.MP >= 128) {
    const int nsl = L.MP / 32, BW = tc_bw(L.MP), NP = L.MP / BW, spb = BW / 32, BT = tc_bq(L.MP), NPT = L.MP / BT, spt = BT / 32;
    n_img = spb * NP * (NP + 1) / 2 + NPT * nsl - spt * NPT * (NPT - 1) / 2;
  }
  int want = nb * nb + nb + 3 * n_img;
  if (max_ctas > 0 && want > max_ctas) want = max_ctas;
  if (want < 8) want = 8;
  if (want > 148) want = 148;
  const int grid = coop_grid(fwd, want, smem);
#ifdef GPBLUR_TRACE   // developer builds only (scripts/mm_only.py, mm_step_probe.py): the kernel returns after a phase
  static const int dbg_stop = [] { const char* e = getenv("GPBLUR_MM_STOP"); return e ? atoi(e) : -1; }();
#else
  const int dbg_stop = -1;
#endif
  unsigned* sync_words = reinterpret_cast<unsigned*>(ws_ptr<unsigned long long>(ws, L.stamps) + 14);   // 4 words
  MmFwdArgs args{p, L, ws, kl, info, extra_jitter, nullptr, dbg_stop, sync_words + 1};
  ProfScope ps(ST_MM_FWD, st);
  if (!mm_cooperative()) {
    args.bar = sync_words;
    cudaMemsetAsync(sync_words, 0, sizeof(unsigned), st);
    void* kargs[] = {&args};
    cudaLaunchKernel(fwd, dim3(grid), dim3(kThreads), kargs, smem, st);
    note_launch();
    return check_launch("mm_forward");
  }
  void* kargs[] = {&args};
  cudaError_t e = cudaLaunchCooperativeKernel(fwd, dim3(grid), dim3(kThreads),
                                              kargs, smem, st);
  note_launch();
  if (e != cudaSuccess) return check_launch("mm_forward");
  return GPBLUR_OK;
}

int launch_mm_backward(const gpblur_svgp_params& p, const WsLayout& L, void* stage, const double* sgrad,
                       const float* g_kl, float* grad_bucket, cudaStream_t st, int accumulate, int max_ctas) {
  const int nb = L.MP / TB;
  const bool mat = L.kind != GPBLUR_KERNEL_RBF;
  if (nb == 1) {   // M <= 32: one CTA, everything in shared memory, plain launch
    const void* small = mat ? (const void*)mm_small_backward_kernel<true> : (const void*)mm_small_backward_kernel<false>;
    cudaFuncSetAttribute(small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmallBwdSmem);
    MmBwdArgs args{p, L, stage, sgrad, g_kl, grad_bucket, accumulate, nullptr};
    ProfScope ps(ST_MM_BWD, st);
    void* kargs[] = {&args};
    cudaLaunchKernel(small, dim3(1), dim3(kThreads), kargs, kSmallBwdSmem, st);
    note_launch();
    return check_launch("mm_small_backward");
  }
  // 16-row tiles while that still gives every SM at most two of them (one CTA for a single 32 x 32 block, with CTA
  // barriers instead of grid barriers, was tried: 29 us against 21 us on 8 CTAs - the elementwise phases want the threads)
  const bool half = 2 * nb * nb <= 2 * 148;
  const size_t smem = half ? wide_bytes<16>() : wide_bytes<32>();
  const void* func = mat ? (half ? (const void*)mm_backward_kernel<16, true> : (const void*)mm_backward_kernel<32, true>)
                         : (half ? (const void*)mm_backward_kernel<16, false> : (const void*)mm_backward_kernel<32, false>);
  cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   // per device
  int want = (half ? 2 : 1) * nb * nb;
  const int dwant = (L.MP * L.DP + kThreads - 1) / kThreads;
  if (want < dwant) want = dwant;
  if (max_ctas > 0 && want > max_ctas) want = max_ctas < 8 ? 8 : max_ctas;
  if (want > 148) want = 148;
  const int grid = coop_grid(func, want, smem);
  MmBwdArgs args{p, L, stage, sgrad, g_kl, grad_bucket, accumulate, nullptr};
  ProfScope ps(ST_MM_BWD, st);
  void* kargs[] = {&args};
  if (!mm_cooperative()) {
    args.bar = reinterpret_cast<unsigned*>(ws_ptr<unsigned long long>(stage, L.stamps) + 31);
    cudaMemsetAsync(args.bar, 0, sizeof(unsigned), st);
    cudaError_t e = cudaLaunchKernel(func, dim3(grid), dim3(kThreads), kargs, smem, st);
    note_launch();
    if (e != cudaSuccess) return check_launch("mm_backward");
    return check_launch("mm_backward");
  }
  cudaError_t e = cudaLaunchCooperativeKernel(func, dim3(grid), dim3(kThreads), kargs, smem, st);
  note_launch();
  if (e != cudaSuccess) return check_launch("mm_backward");
  return GPBLUR_OK;
}

int stage_grad_reduce_impl(const WsLayout& L, const void* ws, double* sgrad, int nvec_used, int ncpart,
                           cudaStream_t st) {
  const size_t total = stage_grad_doubles(L.MP, L.DP, L.kind);   // at most the elements the kernel reads
  int grid = (int)((total + 31) / 32);
  if (grid > 16 * 148) grid = 16 * 148;
  SgReduceArgs args{L, ws, sgrad, nvec_used, ncpart};
  ProfScope ps(ST_SG_REDUCE, st);
  stage_grad_reduce_kernel<<<grid, kThreads, 0, st>>>(args);
  note_launch();
  return check_launch("stage_grad_reduce");
}

}  // namespace gpblur
