// tcgen05 3xTF32 N-reduction GEMMs of the backward (tensor-core replacement of reduce_gemm_kernel for M >= 128):
//   Gram  : S[p][q]  = sum_n A[n][p] * (g_var[n] A[n][q])      (+ u[p] = sum_n g_mu[n] A[n][p], for free in the loader)
//   W^T X : WX[m][d] = sum_n W[n][m] * X[n][d]                 (+ the column sums of W)
// Both run in ONE launch (tc_reduce_kernel): the Gram is bound by tensor-core time and loader issue, W^T X by memory,
// and neither needs the other's result, so their CTAs share the wave.  The work is cut into units per band of
// BW = min(MP, 256) inducing points, each split over N across CTAs (the split counts come from make_layout):
//   * diagonal Gram unit (band r): ONLY the lower-triangle 128 x 128 blocks of the band (3 at BW = 256: row tile 0
//     with N = 128, row tile 1 with N = 256).  Every 16-byte piece of A is fetched, transposed and split ONCE: the
//     unscaled value goes to the TMEM A operand, the g_var-scaled value to the shared-memory B operand;
//   * off-diagonal Gram unit (MP >= 512): one 128-row tile x one 256-column band strictly below the diagonal band;
//   * W^T X unit (band r): both row tiles of the band against the same x slab, so x is read once per band.
// Operands are "MN-major" in memory (the reduction index n is the slow one): the loader threads gather 4 consecutive
// n per 16-byte k-chunk, split every value into TF32 hi/lo planes and write the canonical K-major no-swizzle UMMA
// tiles.  A and W arrive TILE-major from the point kernels (tc_tiled_index: per 128-point tile [MP / 4 column pieces]
// [128 rows][4 floats]): the 4 lanes that own the 4 columns of a piece load the float4 of 4 consecutive rows and
// transpose 4 x 4 among themselves with 4 shuffles; one elected thread issues tcgen05.mma.kind::tf32 (M = 128, K = 8)
// into TMEM accumulators, completion is tracked with tcgen05.commit -> mbarrier, the epilogue reads TMEM with
// tcgen05.ld.  Partials are reduced in fixed order by stage_grad_reduce.
#include "gpblur_tc.cuh"

namespace gpblur {

namespace {

// 16 producer warps: the producers are bound by instruction latency (gather, TF32 split, stores), not by bandwidth,
// and with the A operand in tensor memory a thread needs few enough registers for 4 warps per scheduler
constexpr int kProd = 512;
constexpr int kIssuerWarp = kProd / 32;           // warp 16: dedicated MMA issuer
constexpr int kBlockThreads = kProd + 32;
constexpr int kSplitRows = 32;                    // split boundaries are multiples of every unit's slab depth
__device__ __forceinline__ void prod_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}

struct TcReduceArgs {
  const float* A;      // tile-major [N, MP] saved a
  const float* W;      // tile-major [N, MP]
  const float* x;      // row-major [N][D]
  const float* gmu;    // [N] weights of u
  const float* gvar;   // [N] row scale of the Gram
  float* S;            // [splits][tc_gram_floats(MP)] packed lower-triangle blocks (tc_gram_index)
  float* u;            // [splitsS][MP]
  float* WX;           // [splitsZ][MP][DP]
  float* c;            // [splitsZ][MP] column sums of W
  long long N;
  int MP, D, DP;
  int splitsS, splitsO, splitsZ, rowsS, rowsO, rowsZ;
  int ndiag, noff;     // Gram units: ndiag diagonal bands, then noff (row tile, column band) units
};

enum Role { GRAM_DIAG, GRAM_OFF, WX_UNIT };

// in-register 4 x 4 transpose among the 4 lanes l = 4 j + e of a quad: lane e holds row e = (m0, m1, m2, m3) and ends
// up with column e = (row 0, row 1, row 2, row 3)[e]
__device__ __forceinline__ float4 quad_transpose(float4 v, int lane) {
  {
    const bool odd = lane & 1;
    const float s0 = odd ? v.x : v.y, s1 = odd ? v.z : v.w;
    const float r0 = __shfl_xor_sync(0xffffffffu, s0, 1), r1 = __shfl_xor_sync(0xffffffffu, s1, 1);
    if (odd) { v.x = r0; v.z = r1; } else { v.y = r0; v.w = r1; }
  }
  {
    const bool up = lane & 2;
    const float s0 = up ? v.x : v.z, s1 = up ? v.y : v.w;
    const float r0 = __shfl_xor_sync(0xffffffffu, s0, 2), r1 = __shfl_xor_sync(0xffffffffu, s1, 2);
    if (up) { v.x = r0; v.y = r1; } else { v.z = r0; v.w = r1; }
  }
  return v;
}

// NT row tiles of 128 (A operand in TMEM), B operand of TB rows in shared memory
template <Role R, int NT, int TQ>
struct Cfg {
  // the diagonal unit at BW = 256 holds 384 accumulator columns: its A ring of 2 stages x 2 tiles fits the 512 TMEM
  // columns only with 16-row slabs
  static constexpr int KT = (R == GRAM_DIAG && NT == 2) ? 16 : 32;
  static constexpr int KC = KT / 4;                              // 16-byte k-chunks per row and slab
  static constexpr int TB = R == GRAM_DIAG ? 128 * NT : TQ;      // rows of the B image
  static constexpr int NA = NT * KC / 4;                         // A pieces per producer thread and slab
  static constexpr int BG0 = kProd / TB > 0 ? kProd / TB : 1;
  static constexpr int BG = BG0 > KC ? KC : BG0;                 // thread groups along the B chunks
  static constexpr int BCH = R == GRAM_DIAG ? 1 : KC / BG;       // B chunks per thread (unused on the diagonal)
  static constexpr int DC = TQ < 32 ? 32 : TQ;
  // MMA N of row tile t: the diagonal unit stops at the diagonal (tile t covers columns [0, 128 (t + 1)))
  __host__ __device__ static constexpr int ncols(int t) { return R == GRAM_DIAG ? 128 * (t + 1) : DC; }
  __host__ __device__ static constexpr int acc_col(int t) { return R == GRAM_DIAG ? 64 * t * (t + 1) : t * DC; }
  static constexpr int ACC = acc_col(NT);
  static constexpr int A_COLS = 2 * KT;                          // hi | lo of one tile and stage
  static constexpr int USED = ACC + 2 * NT * A_COLS;
  static_assert(USED <= 512, "TMEM budget");
  static constexpr uint32_t TMEM_COLS = USED <= 256 ? 256 : 512;
  static constexpr int B_PLANE = KC * TB * 4;                    // floats
  static constexpr int STAGE = 2 * B_PLANE;
  static constexpr size_t smem = (size_t)2 * STAGE * 4;
};

struct RedShared {
  alignas(16) float scs[4][kSplitRows];   // row scales g_var / weights g_mu, read as float4
  alignas(16) float gms[4][kSplitRows];
  float ured[4][256];
  alignas(8) uint64_t bars[4];            // [0..1] mma_done (tcgen05.commit), [2..3] a_ready (512 producers)
  uint32_t tmem_slot;
};

template <Role R, int NT, int TQ>
__device__ __forceinline__ void reduce_unit(const TcReduceArgs& a, int unit, int split, float* stage_base,
                                            RedShared& sh) {
  using C = Cfg<R, NT, TQ>;
  constexpr int KT = C::KT, KC = C::KC, TB = C::TB, BG = C::BG, BCH = C::BCH;
  constexpr bool GRAM = R != WX_UNIT;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int MP = a.MP;

  int p0, q0 = 0;                 // first output row / column of the unit
  if (R == GRAM_DIAG) {
    p0 = q0 = unit * 128 * NT;
  } else if (R == GRAM_OFF) {     // row tile pt of band r >= 1, column band q < r: r-major, then tile, then q
    int r = 1, u = unit;
    while (u >= 2 * r) { u -= 2 * r; ++r; }
    p0 = r * 256 + (u / r) * 128;
    q0 = (u % r) * 256;
  } else {
    p0 = unit * 128 * NT;
  }
  const int rps = R == GRAM_DIAG ? a.rowsS : R == GRAM_OFF ? a.rowsO : a.rowsZ;
  const long long r0 = (long long)split * rps;
  long long r1 = r0 + rps;
  if (r1 > a.N) r1 = a.N;
  const int nsl = r1 > r0 ? (int)((r1 - r0 + KT - 1) / KT) : 0;

  if (warp == 0) tc::tmem_alloc(&sh.tmem_slot, C::TMEM_COLS);
  if (tid == 0) {
    tc::mbar_init(&sh.bars[0], 1);
    tc::mbar_init(&sh.bars[1], 1);
    tc::mbar_init(&sh.bars[2], kProd);
    tc::mbar_init(&sh.bars[3], kProd);
    tc::fence_barrier_init();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_d = sh.tmem_slot;
  uint64_t* bars = sh.bars;

  if (warp == kIssuerWarp) {
    // ---------------- issuer warp: one thread fires the MMAs as soon as a slab's operands are published ----------------
    if (lane == 0) {
      uint32_t iuses[2] = {0, 0};
      for (int s = 0; s < nsl; ++s) {
        const int st = s & 1;
        float* b_hi = stage_base + st * C::STAGE;
        float* b_lo = b_hi + C::B_PLANE;
        tc::mbar_wait(&bars[2 + st], iuses[st] & 1);
        tc::tc_fence_after();
        const uint32_t bh = tc::smem_u32(b_hi), bl = tc::smem_u32(b_lo);
#pragma unroll
        for (int t = 0; t < NT; ++t) {
          const uint32_t idesc = tc::make_idesc_tf32(128, C::ncols(t));
          const uint32_t d = tmem_d + C::acc_col(t);
          const uint32_t a_hi_t = tmem_d + C::ACC + (st * NT + t) * C::A_COLS, a_lo_t = a_hi_t + KT;
#pragma unroll
          for (int j = 0; j < KT / 8; ++j) {
            const uint64_t dbh = tc::make_smem_desc(bh + 2 * j * TB * 16, TB * 16, 128);
            const uint64_t dbl = tc::make_smem_desc(bl + 2 * j * TB * 16, TB * 16, 128);
            tc::umma_tf32_ts(d, a_lo_t + 8 * j, dbh, idesc, (s == 0 && j == 0) ? 0u : 1u);   // small cross terms first
            tc::umma_tf32_ts(d, a_hi_t + 8 * j, dbl, idesc, 1u);
            tc::umma_tf32_ts(d, a_hi_t + 8 * j, dbh, idesc, 1u);
          }
        }
        tc::umma_commit(&bars[st]);
        iuses[st] += 1;
      }
    }
  } else {
    // ---- loader thread mapping: A row `ar` (= TMEM lane) of every tile, chunks acg, acg + 4 ----
    const int ar = tid & 127, acg = tid >> 7;
    const int bq = tid % TB, bcg = (tid / TB) % BG;      // B (separate source): row, chunk group
    const float* asrc = R == WX_UNIT ? a.W : a.A;
    struct Regs { float4 a[C::NA]; float4 b[BCH]; };
    float usum[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) usum[t] = 0.f;

    // the gathered operands of TWO slabs are in flight per thread (two register sets): with one, the global-load
    // latency of slab s + 1 was exposed between the split / store of consecutive slabs
    // Addresses: n0 is a multiple of KT, so the rows of a slab never cross a 128-point tile: element (n0 + k, col) of
    // a tile-major matrix sits at slab_base(n0) + (col >> 2) * 512 + k * 4 (+ col & 3) - one 64-bit base per slab plus
    // thread-constant offsets (the generic index cost ~15 integer instructions per load in an issue-bound loop).
    const uint32_t a_off0 = (uint32_t)(((p0 + ar) >> 2) * 512 + (4 * acg + (lane & 3)) * 4);
    const uint32_t b_off_t = (uint32_t)(((q0 + bq) >> 2) * 512 + (4 * bcg + (lane & 3)) * 4);
    const bool b_col_ok = q0 + bq < (GRAM ? MP : a.D);
    const bool b_thread = R != GRAM_DIAG && (TB >= kProd || tid < TB * BG);
    const size_t x_off = (size_t)(4 * bcg) * a.D + q0 + bq;                                            // W^T X: row 4 bcg
    auto prefetch = [&](Regs& rg, int s) {
      const long long n0 = r0 + (long long)s * KT;
      const bool full = n0 + KT <= r1;
      const float* ubase = asrc + (size_t)(n0 >> 7) * (size_t)MP * 128 + (size_t)(n0 & 127) * 4;
#pragma unroll
      for (int t = 0; t < NT; ++t)
#pragma unroll
        for (int i = 0; i < KC / 4; ++i) {
          // rows n0 + 4 c .. + 3, column p0 + 128 t + ar: this lane fetches row n0 + 4 c + (lane & 3) of its piece
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (full || n0 + 4 * (acg + 4 * i) + (lane & 3) < r1)
            v = *reinterpret_cast<const float4*>(ubase + a_off0 + t * (32 * 512) + i * 64);
          rg.a[t * (KC / 4) + i] = v;   // raw: the 4 x 4 transpose happens in produce(), two slabs later (a dependent
                                        // shuffle here would stall the prefetch on its own HBM round trip)
        }
      if (b_thread) {
        if (GRAM) {
#pragma unroll
          for (int i = 0; i < BCH; ++i) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (b_col_ok && (full || n0 + 4 * (bcg + BG * i) + (lane & 3) < r1))
              v = *reinterpret_cast<const float4*>(ubase + b_off_t + i * (BG * 16));
            rg.b[i] = v;   // raw (see above)
          }
        } else {
          const float* xbase = a.x + (size_t)n0 * a.D + x_off;
#pragma unroll
          for (int i = 0; i < BCH; ++i) {
            float v[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int k = 4 * (bcg + BG * i) + e;
              v[e] = (b_col_ok && (full || n0 + k < r1)) ? xbase[(size_t)(4 * BG * i + e) * a.D] : 0.f;
            }
            rg.b[i] = make_float4(v[0], v[1], v[2], v[3]);
          }
        }
      }
    };
    // per-row scales of slab s go through shared memory (4 buffers: staged two slabs ahead, before the producer
    // barrier of the iteration, which orders the write against the reads two iterations later)
    auto stage_scales = [&](int s) {
      if (GRAM && tid < KT) {       // W^T X has neither a row scale nor weights for its column sums
        const long long n = r0 + (long long)s * KT + tid;
        sh.scs[s & 3][tid] = (n < r1) ? a.gvar[n] : 0.f;
        if (R == GRAM_DIAG) sh.gms[s & 3][tid] = (n < r1) ? a.gmu[n] : 0.f;
      }
    };

    uint32_t uses[2] = {0, 0};
    auto produce = [&](const Regs& rg, int s) {
      const int st = s & 1, sb = s & 3;
      float* b_hi = stage_base + st * C::STAGE;
      float* b_lo = b_hi + C::B_PLANE;
      if (uses[st] > 0) {                                               // MMAs of slab s-2 are done with this stage
        tc::mbar_wait(&bars[st], (uses[st] - 1) & 1);
        tc::tc_fence_after();
      }
      // ---- A operand: this thread owns output row `ar` (TMEM lane) of every tile; its chunks go to tensor memory ----
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        const uint32_t a_hi_t = tmem_d + C::ACC + (st * NT + t) * C::A_COLS + ((uint32_t)((warp & 3) * 32) << 16);
        const uint32_t a_lo_t = a_hi_t + KT;
#pragma unroll
        for (int i = 0; i < KC / 4; ++i) {
          const int c = acg + 4 * i;
          const float4 av = quad_transpose(rg.a[t * (KC / 4) + i], lane);
          float4 h, l;
          tc::split_tf32(av.x, h.x, l.x); tc::split_tf32(av.y, h.y, l.y);
          tc::split_tf32(av.z, h.z, l.z); tc::split_tf32(av.w, h.w, l.w);
          tc::tmem_st4(a_hi_t + 4 * c, h);
          tc::tmem_st4(a_lo_t + 4 * c, l);
          if (R == GRAM_DIAG) {
            const float4 gw = *reinterpret_cast<const float4*>(&sh.gms[sb][4 * c]);
            usum[t] = fmaf(gw.x, av.x, usum[t]);
            usum[t] = fmaf(gw.y, av.y, usum[t]);
            usum[t] = fmaf(gw.z, av.z, usum[t]);
            usum[t] = fmaf(gw.w, av.w, usum[t]);
            // the same values, scaled by g_var, are the B operand (column q = 128 t + ar)
            const float4 sw = *reinterpret_cast<const float4*>(&sh.scs[sb][4 * c]);
            tc::store_split(b_hi, b_lo, tc::op_off<TB>(128 * t + ar, c),
                            make_float4(av.x * sw.x, av.y * sw.y, av.z * sw.z, av.w * sw.w));
          } else if (R == WX_UNIT) {   // plain column sums of W (rows beyond the split are zero)
            usum[t] += av.x; usum[t] += av.y; usum[t] += av.z; usum[t] += av.w;
          }
        }
      }
      if (b_thread) {
#pragma unroll
        for (int i = 0; i < BCH; ++i) {
          const int c = bcg + BG * i;
          float4 v = GRAM ? quad_transpose(rg.b[i], lane) : rg.b[i];
          if (GRAM) {
            const float4 sw = *reinterpret_cast<const float4*>(&sh.scs[sb][4 * c]);
            v.x *= sw.x; v.y *= sw.y; v.z *= sw.z; v.w *= sw.w;
          }
          tc::store_split(b_hi, b_lo, tc::op_off<TB>(bq, c), v);
        }
      }
      tc::tmem_st_wait();          // the tensor-memory stores of this thread have landed
      tc::tc_fence_before();
      tc::fence_async_smem();      // generic-proxy writes of B -> visible to the tensor core (async proxy)
      mbar_arrive(&bars[2 + st]);  // the issuer warp fires the MMAs once all 512 producers have arrived
      uses[st] += 1;
    };

    Regs rg0, rg1;
    if (0 < nsl) { prefetch(rg0, 0); stage_scales(0); }
    if (1 < nsl) { prefetch(rg1, 1); stage_scales(1); }
    prod_sync();
    for (int s = 0; s < nsl; s += 2) {
      if (s + 2 < nsl) stage_scales(s + 2);
      produce(rg0, s);
      if (s + 2 < nsl) prefetch(rg0, s + 2);
      prod_sync();                 // orders the staged scales (and the reuse of their buffers) among producers
      if (s + 1 >= nsl) break;
      if (s + 3 < nsl) stage_scales(s + 3);
      produce(rg1, s + 1);
      if (s + 3 < nsl) prefetch(rg1, s + 3);
      prod_sync();
    }

    // ---- epilogue: warp (quadrant warp & 3) reads 32-column chunks warp >> 2, + 4, ... of every tile ----
    const int row = (warp & 3) * 32 + lane;
    if (nsl > 0) {
      const int last = (nsl - 1) & 1;
      tc::mbar_wait(&bars[last], (uses[last] - 1) & 1);
      tc::tc_fence_after();
    }
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      const int i_out = p0 + 128 * t + row;
      for (int cc = warp >> 2; cc < C::ncols(t) / 32; cc += 4) {
        const int col = cc * 32;
        float v[32];
        if (nsl > 0) {
          tc::tmem_ld32(tmem_d + C::acc_col(t) + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)col, v);
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0.f;
        }
        if (GRAM) {
          float* dst = a.S + (size_t)split * tc_gram_floats(MP) + tc_gram_index(i_out, q0 + col);
#pragma unroll
          for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        } else {
          float* dst = a.WX + ((size_t)split * MP + i_out) * a.DP + col;
#pragma unroll
          for (int i = 0; i < 32; i += 4)
            if (col + i < a.DP) *reinterpret_cast<float4*>(dst + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
      }
    }
    if (R != GRAM_OFF) {
#pragma unroll
      for (int t = 0; t < NT; ++t) sh.ured[acg][t * 128 + ar] = usum[t];
      prod_sync();
      float* out = R == GRAM_DIAG ? a.u : a.c;
      if (tid < NT * 128)
        out[(size_t)split * MP + p0 + tid] = (sh.ured[0][tid] + sh.ured[1][tid]) + (sh.ured[2][tid] + sh.ured[3][tid]);
    }
  }   // producer warps
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_d, C::TMEM_COLS);
}

// one launch: CTAs [0, nG) are Gram units (diagonal bands first), the rest W^T X units.  NT = BW / 128 row tiles per
// band, TQW = W^T X output columns (DP, at least 32), OFF: MP >= 512 (off-diagonal Gram units exist)
template <int NT, int TQW, bool OFF>
__global__ void __launch_bounds__(kBlockThreads, 1) tc_reduce_kernel(TcReduceArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ __align__(16) RedShared sh;
  float* stage_base = reinterpret_cast<float*>(smem_raw);
  int b = blockIdx.x;
  const int nd = a.ndiag * a.splitsS, no = a.noff * a.splitsO;
  if (b < nd) {
    reduce_unit<GRAM_DIAG, NT, 128 * NT>(a, b / a.splitsS, b % a.splitsS, stage_base, sh);
    return;
  }
  b -= nd;
  if constexpr (OFF) {
    if (b < no) {
      reduce_unit<GRAM_OFF, 1, 256>(a, b / a.splitsO, b % a.splitsO, stage_base, sh);
      return;
    }
    b -= no;
  }
  reduce_unit<WX_UNIT, NT, TQW>(a, b / a.splitsZ, b % a.splitsZ, stage_base, sh);
}

template <int NT, int TQW, bool OFF>
int launch_tc_reduce(const TcReduceArgs& a, int grid, cudaStream_t st) {
  size_t smem = Cfg<GRAM_DIAG, NT, 128 * NT>::smem;
  if (Cfg<WX_UNIT, NT, TQW>::smem > smem) smem = Cfg<WX_UNIT, NT, TQW>::smem;
  if (OFF && Cfg<GRAM_OFF, 1, 256>::smem > smem) smem = Cfg<GRAM_OFF, 1, 256>::smem;
  // the attribute is per DEVICE: set on every launch (cheap) instead of a process-wide flag
  cudaFuncSetAttribute(tc_reduce_kernel<NT, TQW, OFF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  ProfScope ps(ST_GRAM, st);   // Gram and W^T X share the launch: reported as the "gram" stage
  tc_reduce_kernel<NT, TQW, OFF><<<grid, kBlockThreads, smem, st>>>(a);
  note_launch();
  return check_launch("tc_reduce");
}

template <int NT, bool OFF>
int launch_tc_reduce_dp(const TcReduceArgs& a, int grid, cudaStream_t st) {
  switch (a.DP) {
    case 16:   // N = 32 MMA with the upper 16 columns zero (columns >= D), only DP = 16 columns are stored
    case 32: return launch_tc_reduce<NT, 32, OFF>(a, grid, st);
    case 64: return launch_tc_reduce<NT, 64, OFF>(a, grid, st);
    default: return launch_tc_reduce<NT, 128, OFF>(a, grid, st);
  }
}

}  // namespace

bool tc_reductions_supported(const WsLayout& L) { return tc_point_supported(L); }

int launch_tc_reductions(const WsLayout& L, void* ws, const float* x, cudaStream_t st) {
  const int MP = L.MP;
  const float* gsc = ws_cptr<float>(ws, L.gsc);
  auto rows = [&](int splits) {
    if (splits < 1) return 0;
    long long r = (L.N + splits - 1) / splits;
    return (int)round_up_ll(r, kSplitRows);
  };
  TcReduceArgs a{};
  a.A = ws_cptr<float>(ws, L.A); a.W = ws_cptr<float>(ws, L.W); a.x = x;
  a.gmu = gsc; a.gvar = gsc + L.N;
  a.S = ws_ptr<float>(ws, L.Spart); a.u = ws_ptr<float>(ws, L.upart);
  a.WX = ws_ptr<float>(ws, L.WXpart); a.c = ws_ptr<float>(ws, L.cpart);
  a.N = L.N; a.MP = MP; a.D = L.D; a.DP = L.DP;
  a.splitsS = L.splitsS; a.splitsO = L.splitsO; a.splitsZ = L.splitsZ;
  a.rowsS = rows(L.splitsS); a.rowsO = rows(L.splitsO); a.rowsZ = rows(L.splitsZ);
  const int nb = MP / tc_bw(MP);
  a.ndiag = nb;
  a.noff = nb * (nb - 1);
  const int grid = nb * L.splitsS + a.noff * L.splitsO + nb * L.splitsZ;
  if (MP == 128) return launch_tc_reduce_dp<1, false>(a, grid, st);
  if (MP == 256) return launch_tc_reduce_dp<2, false>(a, grid, st);
  return launch_tc_reduce_dp<2, true>(a, grid, st);
}

}  // namespace gpblur
