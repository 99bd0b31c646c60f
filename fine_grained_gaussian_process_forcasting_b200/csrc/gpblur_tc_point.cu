// Per-point forward / backward of the whitened SVGP on the 5th-gen tensor cores, TS form (tcgen05.mma with the A
// operand in TENSOR MEMORY): replaces, per DeepGPp.predict call, gpytorch's batched kernel build + fp64
// trsm_batched + predictive mean / variance kernels (/root/reference/denoising_model/DeepGP.py:56-73, 94-99) and
// their autograd backward.
//
// One CTA owns a tile of 128 points = the M dimension of the MMA and the 128 TMEM lanes.  A producer thread owns
// ONE point (lane) and 16 of the 32 k-values of a pipeline slab, so every A operand - the scaled inputs x~, the
// exp()'d cross-covariance k, the saved whitened a, W = kbar o k - goes from registers straight into tensor memory
// with tcgen05.st (hi plane | lo plane of the 3xTF32 split): no shared-memory stores, no proxy fences, and the
// tensor core reads only the constant B operand (pre-split slab images pulled by cp.async.bulk) from shared memory.
// The round-1 SS-form kernels spent 80 KB of shared-memory traffic per slab on the A planes and were bound by it
// (DESIGN.md section 5).
//
// TMEM columns (fp32):  [ S : BQ | ACC : BWO | A operand ring : 64 per stage (hi 32 | lo 32) ]
//   forward : S = X~ Z~[q]^T for a block of BQ = min(MP, 128) inducing points; ACC = whitened product for an
//             output block of BWO = min(MP, 256) columns: every whitening MMA of the blocks below the diagonal
//             has N = BWO, the cross-covariance of a block is exponentiated exactly once per output block.
// Pipeline: slab g uses A stage g & 1 and B stage g % NSTB; every wait is on a barrier whose NEXT phase cannot
// complete without the waiter's own arrival (or is signalled once per block for exactly one waiting group), so a
// parity can never be observed two phases late.
#include "gpblur_tc.cuh"
#include "gpblur_tile.cuh"

// clock64 event trace of CTA 0 (scripts/tc2_trace.py): compiled out of release builds (GPBLUR_TRACE=1 python -m ...build)
#ifndef GPBLUR_TRACE
#define GPBLUR_TRACE 0
#endif
#if GPBLUR_TRACE
#define TRACE_PTR(cond, expr) ((cond) ? (expr) : nullptr)
#else
#define TRACE_PTR(cond, expr) (static_cast<long long*>(nullptr))
#endif

namespace gpblur {

namespace {

constexpr int KT = 32;          // k-values per pipeline slab (4 UMMA k-steps)
constexpr int TNP = 128;        // points per tile (MMA M)
constexpr int kGroup = 256;     // threads per producer group (8 warps: 4 lane quadrants x 2 k-halves)
constexpr int kProducers = 2 * kGroup;
constexpr int kIssuerWarp = kProducers / 32;
constexpr int kCtaThreads = kProducers + 128;   // + the issuer warpgroup: warp 16 issues, warps 17..19 only donate registers
constexpr int kRegsIssuer = 32, kRegsProducer = 112;   // setmaxnreg: 512 x 112 + 128 x 32 = 61440 = 640 x 96 (the launch allocation)
constexpr int kMaxDs = 4;       // d-slabs of the x tile (D <= 128)

struct Tc2Args {
  WsLayout L;
  void* ws;
  const void* stage;   // parameter stage (== ws when the stage was built in the workspace)
  const float* x;
  float* mean;
  float* var;
  float* sample;
  SegGrads seg;          // per-segment upstream gradients (backward)
  const float* var_in;
  float* dx;
  uint64_t seed, offset;
  const unsigned long long* offset_dev;   // optional device-resident addend of `offset` (CUDA-graph replays)
  uint32_t stream_id;
  int ntiles;
  long long* trace;   // optional clock64 event trace of CTA 0 (gpblur_debug_set_trace; null in production)
};

// One pipeline slab = one K = 32 step of one GEMM of the tile.  The sequence is the same for every tile: tabulated
// once per CTA in shared memory, walked by the issuer warp.
struct Slab {
  const float* img;    // B image in global memory: [hi plane | lo plane], a plane is [8 k-chunks][rows][4 floats]
  int rows;            // B rows = MMA N
  uint32_t tmem_off;   // accumulator column offset inside the CTA's TMEM allocation
  uint32_t flags;      // SF_* | (1 + chunk barrier index) << 8
};
constexpr uint32_t SF_FIRST = 1u;    // the first MMA overwrites the accumulator
constexpr uint32_t SF_SIG_S = 2u;    // commit onto s_full: S of this pass is complete once the slab retires
constexpr uint32_t SF_SIG_DX = 4u;   // commit onto dx_full (backward): the dx accumulator of the tile is complete
constexpr uint32_t SF_GRP_E = 8u;    // (backward) the A operand comes from the row-owner group's private stage

struct Bars {
  uint64_t a_ready[3];   // producers -> issuer: the A operand of the slab in this stage is in tensor memory
  uint64_t mma_done[3];  // tcgen05.commit: the MMAs that read this A stage have retired
  uint64_t b_full[6];    // cp.async.bulk complete_tx: the B image of this stage has landed
  uint64_t b_empty[6];   // tcgen05.commit: the MMAs that read this B stage have retired
  uint64_t s_full;       // the S block of the current pass is complete
  uint64_t chunk[8];     // accumulator chunk c of the current output block is final
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
// all 512 producer threads (the issuer warp never joins)
__device__ __forceinline__ void producers_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

__device__ __forceinline__ float4 ldg4(const float* p) { return *reinterpret_cast<const float4*>(p); }
// global load that stays where it is written: the compiler treats plain loads through the (read-only) kernel
// arguments as invariant and sinks a prefetch down to its first use, which puts the L2 / HBM latency back on the
// critical path (trace: 1.2k cycles per first-pass x~ slab)
__device__ __forceinline__ float4 ldg4_pinned(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ldg1_pinned(const float* p) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}

// wait for two barriers with one shared-memory round trip per poll: even lanes poll (barA, parA), odd lanes (barB, parB)
__device__ __forceinline__ void mbar_wait2(uint64_t* barA, uint32_t parA, uint64_t* barB, uint32_t parB) {
  const bool odd = threadIdx.x & 1;
  const uint32_t addr = tc::smem_u32(odd ? barB : barA), parity = odd ? parB : parA;
  for (uint32_t tries = 0;; ++tries) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    if (__all_sync(0xffffffffu, ok != 0)) break;
    if (tries > (1u << 24)) asm volatile("trap;");
  }
}

// ---- B loader (warp 17): streams the pre-split slab images into the B ring with cp.async.bulk; a stage is refilled
// as soon as the issuer's commit on b_empty says that the MMAs which read it have retired ----
template <int NSTB>
__device__ __noinline__ void tc2_loader(unsigned char* bbase, uint32_t stage_bytes, Bars* bars, const Slab* tab,
                                        int nslabs, int ntiles_mine) {
  if (ntiles_mine <= 0 || nslabs <= 0) return;
  const int total = nslabs * ntiles_mine;
  int i = 0, stB = 0;
  uint32_t ephase = 1;                                      // parity of the PREVIOUS use of the stage (first round: none)
  for (int g = 0; g < total; ++g) {
    const float* img = reinterpret_cast<const float*>(tc::uniform_u64(reinterpret_cast<uint64_t>(tab[i].img)));
    const uint32_t rows = tc::uniform_u32((uint32_t)tab[i].rows);
    if (g >= NSTB) tc::mbar_wait(&bars->b_empty[stB], ephase);
    if (tc::elect_one()) {
      const uint32_t bytes = rows * 256u;                   // hi + lo planes: 2 x 8 k-chunks x rows x 16 B, contiguous
      tc::mbar_expect_tx(&bars->b_full[stB], bytes);
      tc::bulk_g2s(bbase + (size_t)stB * stage_bytes, img, bytes, &bars->b_full[stB]);
    }
    __syncwarp();
    if (++i == nslabs) i = 0;
    if (++stB == NSTB) { stB = 0; ephase ^= 1u; }
  }
}

// ---- MMA issuer (warp 16): the whole warp walks the slab table with warp-uniform values, one elected lane executes
// the tcgen05.mma / commit instructions.  The next slab's table entry is fetched while this slab's operands are
// awaited, both operand barriers are polled in the same shared-memory round trip ----
// SPLIT (backward): the two producer groups do not alternate, so they own SEPARATE A stages - the loaders the ring
// [0, NSTA - 1), the row owners stage NSTA - 1 - and every stage barrier is only ever awaited by the group whose own
// arrival gates its next phase.  (On a shared ring a group that skips the other group's slabs can poll a barrier two
// phases early, where the parity test aliases: it then overwrites an operand that is still being read.)
template <int NSTA, int NSTB, bool SPLIT = false>
__device__ __noinline__ void tc2_issuer(unsigned char* bbase, uint32_t stage_bytes, Bars* bars, uint32_t tmem_base,
                                        uint32_t aop_col, const Slab* tab, int nslabs, int ntiles_mine,
                                        long long* trace, uint64_t* dx_full = nullptr) {
  if (ntiles_mine <= 0 || nslabs <= 0) return;
  nslabs = (int)tc::uniform_u32((uint32_t)nslabs);
  const int total = (int)tc::uniform_u32((uint32_t)(nslabs * ntiles_mine));
  tmem_base = tc::uniform_u32(tmem_base);
  const uint32_t b0 = tc::uniform_u32(tc::smem_u32(bbase));
  constexpr uint64_t kDescHi = ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);   // SBO = 128 B, version 1
  int i = 0, stB = 0, stA = 0;
  uint32_t bphase = 0, aphase = 0;
  uint32_t cnt_l = 0, cnt_e = 0;                            // (SPLIT) slabs issued so far per producer group
  uint32_t n_rows = (uint32_t)tab[0].rows, n_off = tab[0].tmem_off, n_flags = tab[0].flags;
  for (int g = 0; g < total; ++g) {
    const uint32_t rows = tc::uniform_u32(n_rows);
    const uint32_t tmem_d = tmem_base + tc::uniform_u32(n_off);
    const uint32_t flags = tc::uniform_u32(n_flags);
    {
      const int in = (i + 1 == nslabs) ? 0 : i + 1;         // table entry of the next slab: in flight during the waits
      n_rows = (uint32_t)tab[in].rows; n_off = tab[in].tmem_off; n_flags = tab[in].flags;
    }
    const uint32_t idesc = tc::make_idesc_tf32(TNP, (int)rows);
    if (SPLIT) {
      if (flags & SF_GRP_E) { stA = NSTA - 1; aphase = cnt_e & 1u; ++cnt_e; }
      else { stA = (int)(cnt_l % (uint32_t)(NSTA - 1)); aphase = (cnt_l / (uint32_t)(NSTA - 1)) & 1u; ++cnt_l; }
    }
    const uint32_t a_hi_t = tmem_base + aop_col + (uint32_t)stA * 64u, a_lo_t = a_hi_t + 32u;
    const uint32_t bh = b0 + (uint32_t)stB * stage_bytes, bl = bh + rows * 128u;
    const uint64_t dbh0 = kDescHi | ((uint64_t)rows << 16) | (uint64_t)(bh >> 4);   // LBO = rows * 16 B
    const uint64_t dbl0 = kDescHi | ((uint64_t)rows << 16) | (uint64_t)(bl >> 4);
    long long* tr = TRACE_PTR(trace && g < 96 && (threadIdx.x & 31) == 0, trace + g * 8);
    if (tr) tr[0] = clock64();
    mbar_wait2(&bars->a_ready[stA], aphase, &bars->b_full[stB], bphase);
    if (tr) tr[2] = clock64();
    tc::tc_fence_after();
    if (tc::elect_one()) {
#pragma unroll
      for (int j = 0; j < KT / 8; ++j) {
        const uint64_t dbh = dbh0 + (uint64_t)(2 * j) * rows, dbl = dbl0 + (uint64_t)(2 * j) * rows;
        tc::umma_tf32_ts(tmem_d, a_lo_t + 8 * j, dbh, idesc, ((flags & SF_FIRST) && j == 0) ? 0u : 1u);   // small terms first
        tc::umma_tf32_ts(tmem_d, a_hi_t + 8 * j, dbl, idesc, 1u);
        tc::umma_tf32_ts(tmem_d, a_hi_t + 8 * j, dbh, idesc, 1u);
      }
      tc::umma_commit(&bars->mma_done[stA]);
      tc::umma_commit(&bars->b_empty[stB]);
      if (flags & SF_SIG_S) tc::umma_commit(&bars->s_full);
      if (flags & SF_SIG_DX) tc::umma_commit(dx_full);
      if (flags >> 8) tc::umma_commit(&bars->chunk[(flags >> 8) - 1]);
    }
    __syncwarp();
    if (tr) { tr[3] = clock64(); tr[5] = rows; }
    if (++i == nslabs) i = 0;
    if (++stB == NSTB) { stB = 0; bphase ^= 1u; }
    if (!SPLIT) { if (++stA == NSTA) { stA = 0; aphase ^= 1u; } }
  }
}

// producer side of one slab: wait until the MMAs that last read A stage (g % NSTA) have retired, then the caller
// stores its operand columns and publishes
template <int NSTA>
__device__ __forceinline__ void stage_acquire(Bars* bars, int g, bool known_free = false) {
  if (g >= NSTA && !known_free) {
    tc::mbar_wait(&bars->mma_done[g % NSTA], (uint32_t)(g / NSTA - 1) & 1u);
    tc::tc_fence_after();
  }
}
template <int NSTA>
__device__ __forceinline__ void stage_publish(Bars* bars, int g) {
  tc::tmem_st_wait();
  tc::tc_fence_before();
  mbar_arrive(&bars->a_ready[g % NSTA]);
}

// producer side of a PRIVATE ring of `nst` stages starting at stage `st0` (backward): `cnt` = slabs this group has
// produced so far
__device__ __forceinline__ int ring_acquire(Bars* bars, uint32_t cnt, int st0, int nst) {
  const int st = st0 + (int)(cnt % (uint32_t)nst);
  if (cnt >= (uint32_t)nst) {
    tc::mbar_wait(&bars->mma_done[st], (cnt / (uint32_t)nst - 1u) & 1u);
    tc::tc_fence_after();
  }
  return st;
}
__device__ __forceinline__ void ring_publish(Bars* bars, int st) {
  tc::tmem_st_wait();
  tc::tc_fence_before();
  mbar_arrive(&bars->a_ready[st]);
}

// split 16 values into the TF32 hi / lo planes of A stage `st`: columns [kofs, kofs + 16) of the slab
__device__ __forceinline__ void store_operand16(uint32_t aop_lane_base, int st, int kofs, const float (&v)[16]) {
  float h[16], l[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) tc::split_tf32(v[i], h[i], l[i]);
  tc::tmem_st16(aop_lane_base + (uint32_t)(st * 64 + kofs), h);
  tc::tmem_st16(aop_lane_base + (uint32_t)(st * 64 + 32 + kofs), l);
}

// 16 input dimensions [d0, d0 + 16) of point gn: raw loads only (a prefetch does not stall on its own data)
struct XRow16 { float4 v[4]; };
__device__ __forceinline__ void load_x16(XRow16& r, const float* x, long long gn, long long N, int D, int d0, bool vec) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int d = d0 + 4 * i;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gn < N && d < D) {
      const float* p = x + (size_t)gn * D + d;
      if (vec) v = ldg4_pinned(p);
      else {
        v.x = ldg1_pinned(p);
        if (d + 1 < D) v.y = ldg1_pinned(p + 1);
        if (d + 2 < D) v.z = ldg1_pinned(p + 2);
        if (d + 3 < D) v.w = ldg1_pinned(p + 3);
      }
    }
    r.v[i] = v;
  }
}
// centre / scale (padded dimensions: centre 0, 1 / ell 0 => 0) + the row-statistic partials of these 16 dimensions
__device__ __forceinline__ void transform_x16(const XRow16& r, float (&o)[16], int d0, int DP, const float* center,
                                              const float* inv_ell, const float* wl, float& pn, float& pw) {
  pn = 0.f; pw = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int d = d0 + 4 * i;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (d < DP) {
      const float4 c = ldg4(center + d), ie = ldg4(inv_ell + d), w4 = ldg4(wl + d);
      v.x = (r.v[i].x - c.x) * ie.x; v.y = (r.v[i].y - c.y) * ie.y;
      v.z = (r.v[i].z - c.z) * ie.z; v.w = (r.v[i].w - c.w) * ie.w;
      // explicit FMA chains: the outputs must not depend on how the compiler contracts (shard invariance is tested
      // bit-exactly)
      pn = fmaf(v.w, v.w, fmaf(v.z, v.z, fmaf(v.y, v.y, fmaf(v.x, v.x, pn))));
      pw = fmaf(v.w, w4.w, fmaf(v.z, w4.z, fmaf(v.y, w4.y, fmaf(v.x, w4.x, pw))));
    }
    o[4 * i + 0] = v.x; o[4 * i + 1] = v.y; o[4 * i + 2] = v.z; o[4 * i + 3] = v.w;
  }
}

// Store of a [32 rows x 16 columns] half chunk held one row per lane (16 consecutive floats), without staging:
// neighbouring lanes exchange two 16-byte pieces, so that every store instruction writes 32 contiguous bytes per lane
// pair - complete sectors - instead of half sectors of 32 different rows.  `dst` = global address of (row 0 of the
// warp, first column), `ld` = row pitch in floats, `nvalid` rows exist.
__device__ __forceinline__ void warp_store_rows16(float* dst, size_t ld, const float (&v)[16], int lane, int nvalid) {
  const bool odd = lane & 1;
  float sx[8], rx[8];
#pragma unroll
  for (int i = 0; i < 4; ++i) {          // even lanes send pieces 1 and 3, odd lanes pieces 0 and 2
    sx[i] = odd ? v[i] : v[4 + i];
    sx[4 + i] = odd ? v[8 + i] : v[12 + i];
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) rx[i] = __shfl_xor_sync(0xffffffffu, sx[i], 1);
  const int row_a = lane & ~1, row_b = row_a + 1;
  float* pa = dst + (size_t)row_a * ld + (odd ? 4 : 0);
  float* pb = dst + (size_t)row_b * ld + (odd ? 4 : 0);
  if (row_a < nvalid) {
    *reinterpret_cast<float4*>(pa) = odd ? make_float4(rx[0], rx[1], rx[2], rx[3]) : make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(pa + 8) =
        odd ? make_float4(rx[4], rx[5], rx[6], rx[7]) : make_float4(v[8], v[9], v[10], v[11]);
  }
  if (row_b < nvalid) {
    *reinterpret_cast<float4*>(pb) = odd ? make_float4(v[4], v[5], v[6], v[7]) : make_float4(rx[0], rx[1], rx[2], rx[3]);
    *reinterpret_cast<float4*>(pb + 8) =
        odd ? make_float4(v[12], v[13], v[14], v[15]) : make_float4(rx[4], rx[5], rx[6], rx[7]);
  }
}

// ---- forward slab table: for every output block P, for every S block q below or on it: nds phase-A slabs, then the
// BQ / 32 whitening slabs of block q ----
template <int BQ, int BWO>
__device__ __forceinline__ int fwd_table(Slab* tab, const Tc2Args& a, int nthreads) {
  const WsLayout& L = a.L;
  const int MP = L.MP, NPO = MP / BWO, SPQ = BQ / KT, QPB = BWO / BQ;
  const int nds = L.DP >= KT ? L.DP / KT : 1;
  const float* ZtQ = ws_cptr<float>(a.stage, L.ZtQ);
  const float* LinvU = ws_cptr<float>(a.stage, L.LinvU);
  const int per = nds + SPQ;
  const int total = QPB * NPO * (NPO + 1) / 2 * per;
  for (int i = threadIdx.x; i < total; i += nthreads) {
    const int pass = i / per, j = i - pass * per;
    int P = 0;
    while (QPB * (P + 1) * (P + 2) / 2 <= pass) ++P;      // passes before block P: QPB * P (P + 1) / 2
    const int q = pass - QPB * P * (P + 1) / 2;
    Slab d;
    if (j < nds) {
      d.img = ZtQ + tc_zq_image(MP, nds, q, j);
      d.rows = BQ; d.tmem_off = 0;
      d.flags = (j == 0 ? SF_FIRST : 0u) | (j == nds - 1 ? SF_SIG_S : 0u);
    } else {
      const int sl = j - nds, sg = q * SPQ + sl;
      int rows;
      d.img = LinvU + tc_linv_image(MP, P, sg, &rows);
      d.rows = rows; d.tmem_off = (uint32_t)(BQ + BWO - rows);
      d.flags = (q == 0 && sl == 0) ? SF_FIRST : 0u;
      const int c = sg - P * (BWO / KT);                    // this slab is the last one that touches chunk c of block P
      if (c >= 0) d.flags |= (uint32_t)(c + 1) << 8;
    }
    tab[i] = d;
  }
  return total;
}

constexpr int kMaxFwdSlabs = 20 * 8;   // MP = 1024: 20 passes x (4 d-slabs + 4 whitening slabs)

// =================================================================================================
// forward
// =================================================================================================
// Warp roles (544 threads): two producer groups (warps 0..7, 8..15) own ALTERNATE pipeline slabs (group = slab
// parity = A stage), so the latency chain of a slab (TMEM load -> exp -> stage acquire -> tcgen05.st -> arrive) has
// two slab times; warp 16 issues.  Accumulator chunk c is read out (mean / variance partials, A saved for the
// backward) by group c & 1 as soon as the issuer's commit on chunk[c] says that its last slab has retired.
// Matern / RQ epilogue of a cross-covariance element.  t = min(log2e (S + xnc' + znc'), log2 os) = log2 os - 1/2 log2e d2
// is the RBF exponent (RBF: k = 2^t).  The other kinds recover d2 = 2 ln2 (log2 os - t) >= 0 and evaluate k = os f,
// g and (RQ) ka = dk/dalpha through matern_kg / rq_kg; a padded column (znc = -1e30) gives d2 ~ 1e30 and exactly
// k = g = ka = 0 (RQ: (1 + u)^-alpha is not 0 there, so the column is masked on d2).  hp: alpha, 1 / (2 alpha) (RQ).
struct RqHyp { float alpha, i2a; };
template <int KIND>
__device__ __forceinline__ void tc_kg(float t, float l2os, float os, RqHyp hp, float& k, float& g, float& ka) {
  const float d2 = (l2os - t) * 1.3862943611198906f;
  if constexpr (KIND == GPBLUR_KERNEL_RQ) {
    rq_kg(d2, os, hp.alpha, hp.i2a, k, g, ka);
    if (!(d2 < 1e20f)) { k = 0.f; g = 0.f; ka = 0.f; }
  } else {
    matern_kg<KIND>(d2, os, k, g);
    ka = 0.f;
  }
}

// The point kernels are __device__ bodies templated on the kind behind __global__ entry points: tc2_fwd_kernel /
// tc2_bwd_kernel for RBF and the Matern kinds, tc2_fwd_rq_kernel / tc2_bwd_rq_kernel for RQ, so that each kernel family
// of the compiled library covers a fixed set of kinds (tests/test_gpu_dispatch_matrix.py, tests/test_rq_dispatch.py).
template <int BQ, int BWO, int NSTB, int KIND>
__device__ __forceinline__ void tc2_fwd_body(const Tc2Args& a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) Bars bars;
  __shared__ uint32_t tmem_slot;
  __shared__ Slab tab[kMaxFwdSlabs];
  __shared__ int tab_n;
  __shared__ float part_n[kMaxDs][2][TNP], part_w[kMaxDs][2][TNP];   // row-statistic partials per d-slab / k-half
  __shared__ float mu_s[4][TNP], vv_s[4][TNP];                      // mean / variance partials per (group, k-half)
  constexpr int NSTA = 2;
  constexpr uint32_t S_COL = 0, ACC_COL = BQ, AOP_COL = BQ + BWO;
  constexpr uint32_t USED_COLS = BQ + BWO + NSTA * 64;
  constexpr uint32_t TMEM_COLS = USED_COLS <= 256 ? 256 : 512;
  static_assert(USED_COLS <= 512, "tensor memory budget");
  constexpr uint32_t STAGE_BYTES = BWO * 256;
  constexpr int SPQ = BQ / KT, QPB = BWO / BQ, CPB = BWO / KT;

  const WsLayout& L = a.L;
  const int MP = L.MP, NPO = MP / BWO;
  const long long N = L.N;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* hyp = ws_cptr<float>(a.stage, L.hyp);
  float* Ag = ws_ptr<float>(a.ws, L.A);
  const float* znc_g = ws_cptr<float>(a.stage, L.znc);
  const float* mvec_g = ws_cptr<float>(a.stage, L.mvec);
  const float* cvec_g = ws_cptr<float>(a.stage, L.cvec);
  const float* center = ws_cptr<float>(a.stage, L.center);
  const float* inv_ell = ws_cptr<float>(a.stage, L.inv_ell);
  const float* wl = ws_cptr<float>(a.stage, L.wl);
  const int DP = L.DP, D = L.D;
  const int nds = DP >= KT ? DP / KT : 1;

  // the small constant vectors live in shared memory behind the B ring: with ~200 KB of shared memory carved out
  // the L1 keeps nothing, and every one of these (warp-uniform) reads was an L2 round trip on the producers' critical
  // path (trace: 700 - 2700 cycles per epilogue chunk)
  float* cst = reinterpret_cast<float*>(smem_raw + (size_t)NSTB * STAGE_BYTES);
  float* znc_s = cst;                // [MP] exponent offsets
  float* mvec_s = znc_s + MP;        // [MP] variational mean
  float* cvec_s = mvec_s + MP;       // [MP] s^2 - 1
  float* cen_s = cvec_s + MP;        // [DP] centre
  float* iel_s = cen_s + DP;         // [DP] 1 / ell
  float* wl_s = iel_s + DP;          // [DP] ell * w
  for (int i = tid; i < MP; i += kCtaThreads) { znc_s[i] = znc_g[i]; mvec_s[i] = mvec_g[i]; cvec_s[i] = cvec_g[i]; }
  for (int i = tid; i < DP; i += kCtaThreads) { cen_s[i] = center[i]; iel_s[i] = inv_ell[i]; wl_s[i] = wl[i]; }
  if (warp == 0) tc::tmem_alloc(&tmem_slot, TMEM_COLS);
  if (tid == 32) {
    for (int i = 0; i < 3; ++i) { tc::mbar_init(&bars.a_ready[i], kGroup); tc::mbar_init(&bars.mma_done[i], 1); }
    for (int i = 0; i < 6; ++i) { tc::mbar_init(&bars.b_full[i], 1); tc::mbar_init(&bars.b_empty[i], 1); }
    tc::mbar_init(&bars.s_full, 1);
    for (int i = 0; i < 8; ++i) tc::mbar_init(&bars.chunk[i], 1);
    tc::fence_barrier_init();
  }
  {
    const int n = fwd_table<BQ, BWO>(tab, a, kCtaThreads);
    if (tid == 0) tab_n = n;
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const int tiles_mine = a.ntiles > (int)blockIdx.x ? (a.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  if (warp >= kIssuerWarp) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsIssuer));
    if (warp == kIssuerWarp)
      tc2_issuer<NSTA, NSTB>(smem_raw, STAGE_BYTES, &bars, tmem_base, AOP_COL, tab, tab_n, tiles_mine,
                             blockIdx.x == 0 ? a.trace : nullptr);
    else if (warp == kIssuerWarp + 1)
      tc2_loader<NSTB>(smem_raw, STAGE_BYTES, &bars, tab, tab_n, tiles_mine);
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsProducer));
    const int g = warp >> 3;                              // producer group = parity of the slabs it produces
    const int quad = warp & 3, half = (warp >> 2) & 1;   // TMEM lane quadrant / k-half of this warp
    const int row = quad * 32 + lane;                     // the point this thread owns
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const uint32_t tmem_s = tmem_base + lane_base + S_COL, tmem_acc = tmem_base + lane_base + ACC_COL;
    const uint32_t aop_base = tmem_base + lane_base + AOP_COL;
    const float os = hyp[H_OS], jit = hyp[H_JIT], cwb = hyp[H_CWB];
    const float l2os = log2f(os);
    const RqHyp hp = KIND == GPBLUR_KERNEL_RQ ? RqHyp{hyp[H_ALPHA], hyp[H_I2A]} : RqHyp{0.f, 0.f};
    const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.x) & 15) == 0);
    const int slabs_per_tile = tab_n;
    int gs = 0;                                           // global slab counter (identical in every producer thread)
    uint32_t pass_ctr = 0, blk_ctr = 0;                   // phases of s_full / chunk[]

    // Slab ownership is fixed: group g produces the d-slabs ds with (ds & 1) == g and the whitening slabs sl with
    // (sl & 1) == g, whatever A stage (gs % NSTA) they fall on - the stage barriers are functions of gs alone.
    // x of the group's first own d-slab of a TILE is requested one tile ahead (the L1 left beside 200 KB of shared
    // memory keeps nothing: every reload is an L2 / HBM round trip); the scaled values xt[] stay in registers for
    // the later passes of the tile (up to two d-slabs, D <= 64; a third / fourth d-slab is reloaded).
    XRow16 xr;
    const bool own_x = g < nds;
    if (own_x) load_x16(xr, a.x, (long long)blockIdx.x * TNP + row, N, D, g * KT + half * 16, vec);
    float xt[16];

    bool have_prev = false;                               // deferred mean / variance / sample of the previous tile
    long long prev_gn = 0;
    float xw_prev = 0.f;
    float mu = 0.f, vv = 0.f;                             // partials of the tile whose chunks are being read out
    auto finalize_prev = [&]() {
      if (g == 0 && half == 0 && have_prev && prev_gn < N) {
        const float mean = mu_s[0][row] + mu_s[1][row] + mu_s[2][row] + mu_s[3][row] + xw_prev + cwb;
        const float var = fmaxf(os + jit + vv_s[0][row] + vv_s[1][row] + vv_s[2][row] + vv_s[3][row], kMinVariance);
        a.mean[prev_gn] = mean;
        a.var[prev_gn] = var;
        if (a.sample)
          a.sample[prev_gn] = fmaf(sqrtf(var), philox_normal(a.seed, rng_offset(a.offset, a.offset_dev) + (uint64_t)prev_gn, a.stream_id), mean);
      }
    };
    // read-out of chunk c (32 columns; 16 per k-half) of output block P of tile `etile`: mean / variance partials, A
    // saved for the backward in the tile-major layout (tc_tiled_index): 512 contiguous bytes per warp and instruction
    int epi_ctr = 0;
    auto epi_chunk = [&](int P, int c, uint32_t par, int etile) {
      long long* et = TRACE_PTR(a.trace && blockIdx.x == 0 && (tid & 255) == 0 && epi_ctr < 24, a.trace + 3072 + (g * 24 + epi_ctr) * 8);
      ++epi_ctr;
      if (et) { et[0] = clock64(); et[6] = c; }
      tc::mbar_wait(&bars.chunk[c], par);
      tc::tc_fence_after();
      if (et) et[1] = clock64();
      const int col = c * KT + half * 16;
      float v[16];
      tc::tmem_ld16(tmem_acc + (uint32_t)col, v);
      if (et) et[2] = clock64();
      const float* mp = mvec_s + P * BWO + col;
      const float* cp = cvec_s + P * BWO + col;
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        const float4 m4 = ldg4(mp + i), c4 = ldg4(cp + i);
        mu = fmaf(v[i + 0], m4.x, mu); vv = fmaf(c4.x * v[i + 0], v[i + 0], vv);
        mu = fmaf(v[i + 1], m4.y, mu); vv = fmaf(c4.y * v[i + 1], v[i + 1], vv);
        mu = fmaf(v[i + 2], m4.z, mu); vv = fmaf(c4.z * v[i + 2], v[i + 2], vv);
        mu = fmaf(v[i + 3], m4.w, mu); vv = fmaf(c4.w * v[i + 3], v[i + 3], vv);
      }
      if (et) et[3] = clock64() + (long long)(mu == 12345.f);
      if (L.training) {
        float4* At = reinterpret_cast<float4*>(Ag) + ((size_t)etile * (size_t)(MP >> 2) + (size_t)((P * BWO + col) >> 2)) * TNP + row;
#pragma unroll
        for (int i = 0; i < 4; ++i) At[(size_t)i * TNP] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
      if (et) et[4] = clock64();
    };
    // The last two chunks a pass finalises are read out later: after the next pass's x~ operands have been published
    // and - unless that pass starts a new output block, whose first whitening slab overwrites ACC - after this
    // group's first whitening slab of that pass, so that the tensor core always has queued work meanwhile
    int pend_n = 0, pend_ca = 0, pend_P = 0, pend_tile = 0;
    uint32_t pend_par = 0;
    auto run_pending = [&]() {
      if (pend_n) {
        epi_chunk(pend_P, ((pend_ca & 1) == g) ? pend_ca : pend_ca + 1, pend_par, pend_tile);
        pend_n = 0;
      }
    };

    for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
      const long long n0 = (long long)tile * TNP;
      const long long gn = n0 + row;
      const bool more_tiles = tile + (int)gridDim.x < a.ntiles;
      float xnc = 0.f;
      bool first_pass = true;
      for (int P = 0; P < NPO; ++P, ++blk_ctr) {
        const int nq = (P + 1) * QPB;
        for (int q = 0; q < nq; ++q, ++pass_ctr) {
          const bool last_pass = (P == NPO - 1) && (q == nq - 1);
          // ---- phase A: S[128, BQ] = X~ Z~[block q]^T, the d-slabs alternate between the groups ----
          for (int ds = 0; ds < nds; ++ds, ++gs) {
            if ((ds & 1) != g) continue;
            long long* ptr = TRACE_PTR(a.trace && blockIdx.x == 0 && (tid & 255) == 0 && gs < 96, a.trace + 1024 + gs * 8);
            if (ptr) { ptr[0] = clock64(); ptr[1] = ptr[0]; }
            float v[16];
            if (ds == g && !first_pass) {
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] = xt[i];
            } else {
              XRow16 xs;
              if (ds == g) xs = xr;
              else load_x16(xs, a.x, gn, N, D, ds * KT + half * 16, vec);
              float pn, pw;
              transform_x16(xs, v, ds * KT + half * 16, DP, cen_s, iel_s, wl_s, pn, pw);
              if (first_pass) { part_n[ds][half][row] = pn; part_w[ds][half][row] = pw; }
              if (ds == g) {
#pragma unroll
                for (int i = 0; i < 16; ++i) xt[i] = v[i];
              }
            }
            if (ptr) ptr[2] = clock64() + (long long)(v[0] == 12345.f);
            stage_acquire<NSTA>(&bars, gs);
            if (ptr) ptr[3] = clock64();
            store_operand16(aop_base, gs % NSTA, half * 16, v);
            stage_publish<NSTA>(&bars, gs);
            if (ptr) ptr[4] = clock64();
          }
          if (last_pass && more_tiles && own_x)           // next tile's x: in flight during this pass
            load_x16(xr, a.x, gn + (long long)gridDim.x * TNP, N, D, g * KT + half * 16, vec);
          const bool defer_more = q > 0;                   // ACC is not overwritten by this pass: read-out can wait
          if (!defer_more) run_pending();                 // last chunks of the previous pass
          bool do_finalize = false;
          if (first_pass) {
            if (have_prev) { mu_s[g * 2 + half][row] = mu; vv_s[g * 2 + half][row] = vv; }   // previous tile complete
            mu = 0.f; vv = 0.f;
          }
          // every producer has (a) read the previous output block out of ACC - the first whitening slab of a block
          // overwrites it -, (b) published its row-statistic partials and the partials of the previous tile
          tc::tc_fence_before();
          producers_sync();
          tc::tc_fence_after();
          float xw_new = 0.f;
          if (first_pass) {
            float n2 = 0.f, xw = 0.f;
            for (int ds = 0; ds < nds; ++ds) {            // fixed order (bit-deterministic)
              n2 += part_n[ds][0][row] + part_n[ds][1][row];
              xw += part_w[ds][0][row] + part_w[ds][1][row];
            }
            xnc = -0.72134752044448170f * n2;
            xw_new = xw;
            do_finalize = true;                           // (after this group's first slab: off the S -> k chain)
            first_pass = false;
          }
          // ---- S of block q complete ----
          long long* st = TRACE_PTR(a.trace && blockIdx.x == 0 && (tid & 255) == 0 && pass_ctr < 32, a.trace + 2048 + pass_ctr * 4 + g * 2);
          if (st) st[0] = clock64();
          tc::mbar_wait(&bars.s_full, pass_ctr & 1u);
          tc::tc_fence_after();
          if (st) st[1] = clock64();
          // ---- whitening: ACC[:, j >= 32 sg] += k[:, slab sg] Linv[j, slab sg]^T ----
          const float* znq = znc_s + q * BQ;
          const int c0 = q * SPQ - P * CPB;               // chunk finalised by slab sl of this pass: c0 + sl (if >= 0)
#pragma unroll 1
          for (int sl = 0; sl < SPQ; ++sl, ++gs) {
            // ONE read-out site per iteration: the deferred chunk of the previous pass (group 1, whose first slab is
            // needed one slab time later, BEFORE its first slab - which also leaves the special-function unit to
            // group 0 for the slab the tensor core is waiting for -, group 0 after its first slab), or the chunk that
            // became final two slabs ago (group c & 1)
            {
              int rc = -1, rP = P, rt = tile;
              uint32_t rpar = blk_ctr & 1u;
              const int c = c0 + sl - 2;
              if (sl >= 2 && c >= 0 && (c & 1) == g) rc = c;
              else if (defer_more && pend_n && sl == 1 - g) {
                rc = ((pend_ca & 1) == g) ? pend_ca : pend_ca + 1; rP = pend_P; rt = pend_tile; rpar = pend_par;
                pend_n = 0;
              }
              if (rc >= 0) epi_chunk(rP, rc, rpar, rt);
              if (do_finalize && sl == 1) {
                finalize_prev();
                if (g == 0 && half == 0) xw_prev = xw_new;
                do_finalize = false;
              }
            }
            if ((sl & 1) == g) {
              const int col0 = sl * KT + half * 16;
              long long* ptr = TRACE_PTR(a.trace && blockIdx.x == 0 && (tid & 255) == 0 && gs < 96, a.trace + 1024 + gs * 8);
              if (ptr) ptr[0] = clock64();
              float v[16];
              tc::tmem_ld16(tmem_s + (uint32_t)col0, v);
              if (ptr) ptr[1] = clock64();
#pragma unroll
              for (int j = 0; j < 16; j += 4) {
                const float4 z4 = ldg4(znq + col0 + j);
                if constexpr (KIND == GPBLUR_KERNEL_RBF) {
                  v[j + 0] = tc::ex2_approx(fminf(fmaf(v[j + 0], 1.4426950408889634f, xnc + z4.x), l2os));
                  v[j + 1] = tc::ex2_approx(fminf(fmaf(v[j + 1], 1.4426950408889634f, xnc + z4.y), l2os));
                  v[j + 2] = tc::ex2_approx(fminf(fmaf(v[j + 2], 1.4426950408889634f, xnc + z4.z), l2os));
                  v[j + 3] = tc::ex2_approx(fminf(fmaf(v[j + 3], 1.4426950408889634f, xnc + z4.w), l2os));
                } else {
                  float g, ka;
                  tc_kg<KIND>(fminf(fmaf(v[j + 0], 1.4426950408889634f, xnc + z4.x), l2os), l2os, os, hp, v[j + 0], g, ka);
                  tc_kg<KIND>(fminf(fmaf(v[j + 1], 1.4426950408889634f, xnc + z4.y), l2os), l2os, os, hp, v[j + 1], g, ka);
                  tc_kg<KIND>(fminf(fmaf(v[j + 2], 1.4426950408889634f, xnc + z4.z), l2os), l2os, os, hp, v[j + 2], g, ka);
                  tc_kg<KIND>(fminf(fmaf(v[j + 3], 1.4426950408889634f, xnc + z4.w), l2os), l2os, os, hp, v[j + 3], g, ka);
                }
              }
              if (ptr) ptr[2] = clock64() + (long long)(v[0] == 12345.f);
              // s_full (a commit: every earlier MMA has retired) already covers the stages of the first two slabs
              stage_acquire<NSTA>(&bars, gs, sl < NSTA);
              if (ptr) ptr[3] = clock64();
              store_operand16(aop_base, gs % NSTA, half * 16, v);
              stage_publish<NSTA>(&bars, gs);
              if (ptr) ptr[4] = clock64();
            }
          }
          if (do_finalize) {                              // (SPQ < 2 never happens: BQ >= 64)
            finalize_prev();
            if (g == 0 && half == 0) xw_prev = xw_new;
          }
          if (c0 + SPQ - 2 >= 0) {                        // the last two chunks finalised by this pass: deferred
            pend_n = 2; pend_ca = c0 + SPQ - 2; pend_P = P; pend_par = blk_ctr & 1u; pend_tile = tile;
          }
        }
      }
      have_prev = true;
      prev_gn = gn;
    }
    run_pending();
    if (have_prev) { mu_s[g * 2 + half][row] = mu; vv_s[g * 2 + half][row] = vv; }
    tc::tc_fence_before();
    producers_sync();
    finalize_prev();
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_slot, TMEM_COLS);
}

// =================================================================================================
// backward: W = kbar o k, its row sums, dx and the per-dimension reductions in ONE kernel (W never leaves the chip on
// its way into the dx GEMM)
// =================================================================================================
//   S  = X~ Z~[p]^T                                   (column block p of BT = min(MP, 128) inducing points)
//   T  = a (diag(c) Linv)[:, block p]                 (slabs of the saved a in DEcreasing order: the first MMA
//                                                      initialises every column, chunk c is final after slab p SPB + c)
//   W  = (g_mu beta + 2 g_var T) o k,  r = rowsum(W)  (thread = point; W is saved tile-major for the W^T X reduction)
//   DX += W[:, chunk] Z~[chunk]                        (A operand = W straight from the epilogue registers)
//   dx = (DX - r x~) / ell + g_mu w                   (staged through shared memory: coalesced row-major stores)
// TMEM columns: [ S : BT | T : BT | DX : DXW | A operand ring : 64 per stage ].
// Warp roles (640 threads): warps 0..7 LOADERS (saved-a slabs: tile-major loads three slabs ahead -> tcgen05.st; x~ slabs
// from the shared x~ tile), warps 8..15 ROW OWNERS (x tile -> shared memory, chunk epilogues, W operand of the dx GEMM,
// dx epilogue), warp 16 MMA issuer, warp 17 B loader.  Slab g uses A stage g % NSTA whoever produces it.
struct BwdBars {
  Bars b;
  uint64_t dx_full;      // the DX accumulator of the tile is complete
  uint64_t x_ready;      // the row owners have put the x~ tile of the current tile into shared memory
};

// slab order of one tile (see the kernel header); returns the slab count.  `kind`: 0 = saved-a slab, 1 = x~ slab,
// 2 = W slab (the producers walk the same order)
template <int BT, int DXW>
__device__ __forceinline__ int bwd_table(Slab* tab, const Tc2Args& a, int nthreads) {
  const WsLayout& L = a.L;
  const int MP = L.MP, NP = MP / BT, SPB = BT / KT, NSL = MP / KT;
  const int nds = L.DP >= KT ? L.DP / KT : 1;
  const float* ZtQ = ws_cptr<float>(a.stage, L.ZtQ);
  const float* LCTQ = ws_cptr<float>(a.stage, L.LCTQ);
  const float* ZtTU = ws_cptr<float>(a.stage, L.ZtTU);
  int total = 0;
  for (int p = 0; p < NP; ++p) total += (NSL - p * SPB) + nds + SPB;
  for (int i = threadIdx.x; i < total; i += nthreads) {
    int p = 0, base = 0;
    while (true) {
      const int cnt = (NSL - p * SPB) + nds + SPB;
      if (i < base + cnt) break;
      base += cnt;
      ++p;
    }
    const int j = i - base;
    const int ndense = NSL - (p + 1) * SPB;               // slabs above block p: BT rows each
    Slab d;
    if (j < ndense || (j >= ndense + nds && j < ndense + nds + SPB)) {
      const int t = j < ndense ? j : j - nds;             // index among the T slabs of the block (decreasing s)
      const int sg = NSL - 1 - t;
      int rows;
      d.img = LCTQ + tc_lctq_image(MP, p, sg, &rows);
      d.rows = rows; d.tmem_off = (uint32_t)BT;
      d.flags = (t == 0 ? SF_FIRST : 0u);
      const int c = sg - p * SPB;
      if (c < SPB) d.flags |= (uint32_t)(c + 1) << 8;
    } else if (j < ndense + nds) {
      const int ds = j - ndense;
      d.img = ZtQ + tc_zq_image(MP, nds, p, ds);
      d.rows = BT; d.tmem_off = 0;
      d.flags = (ds == 0 ? SF_FIRST : 0u) | (ds == nds - 1 ? SF_SIG_S : 0u);
    } else {
      const int c = SPB - 1 - (j - ndense - nds - SPB);   // W chunks in the order they become final
      d.img = ZtTU + tc_slab_ztt(DXW, p * SPB + c);
      d.rows = DXW; d.tmem_off = (uint32_t)(2 * BT);
      d.flags = SF_GRP_E | ((p == 0 && c == SPB - 1) ? SF_FIRST : 0u) | ((p == NP - 1 && c == 0) ? SF_SIG_DX : 0u);
    }
    tab[i] = d;
  }
  return total;
}
constexpr int kMaxBwdSlabs = (32 + 28 + 24 + 20 + 16 + 12 + 8 + 4) + 8 * (4 + 4);   // MP = 1024, BT = 128, D = 128

// sum over the 32 lanes of v[i] for 16 values at once ("transpose-reduce": 16 shuffles instead of 80); afterwards lane l
// holds the total of value index ((l >> 4) & 1) * 8 + ((l >> 3) & 1) * 4 + ((l >> 2) & 1) * 2 + ((l >> 1) & 1)
__device__ __forceinline__ float warp_reduce16(float (&v)[16], int lane) {
  {
    const bool up = lane & 16;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float send = up ? v[i] : v[i + 8], keep = up ? v[i + 8] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
  }
  {
    const bool up = lane & 8;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float send = up ? v[i] : v[i + 4], keep = up ? v[i + 4] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
  }
  {
    const bool up = lane & 4;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float send = up ? v[i] : v[i + 2], keep = up ? v[i + 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
  }
  {
    const bool up = lane & 2;
    const float send = up ? v[0] : v[1], keep = up ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}
__device__ __forceinline__ int warp_reduce16_index(int lane) {
  return ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
}

template <int BT, int DXW, int NSTA, int NSTB, int KIND>
__device__ __forceinline__ void tc2_bwd_body(const Tc2Args& a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) BwdBars bb;
  __shared__ uint32_t tmem_slot;
  __shared__ Slab tab[kMaxBwdSlabs];
  __shared__ int tab_n;
  __shared__ float r_s[2][TNP];                   // row sums of W per k-half
  __shared__ float vec_s[2][4][2 * 128];          // [k-half][quadrant][q (DXW / 2) | t1 (DXW / 2)] per-warp partials
  __shared__ float sc_s[8][VS_PART];              // per-warp scalar sums
  constexpr uint32_t S_COL = 0, T_COL = BT, DX_COL = 2 * BT, AOP_COL = 2 * BT + DXW;
  constexpr uint32_t USED_COLS = 2 * BT + DXW + NSTA * 64;
  constexpr uint32_t TMEM_COLS = USED_COLS <= 256 ? 256 : 512;
  static_assert(USED_COLS <= 512, "tensor memory budget");
  constexpr uint32_t BROWS = BT > DXW ? BT : DXW;
  constexpr uint32_t STAGE_BYTES = BROWS * 256;
  constexpr int SPB = BT / KT;
  constexpr int HW = DXW / 2;                     // dx columns per k-half
  constexpr int NPIECE = HW / 16;                 // 16-column pieces per row owner
  constexpr int XP = DXW + 4;                     // pitch (floats) of the x~ tile: conflict-free 16-byte row reads
  constexpr int SP = 20;                          // pitch of a [32 rows x 16 columns] dx staging tile

  const WsLayout& L = a.L;
  const int MP = L.MP, NP = MP / BT, NSL = MP / KT;
  const long long N = L.N;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* hyp = ws_cptr<float>(a.stage, L.hyp);
  const float* Ag = ws_cptr<float>(a.ws, L.A);
  float* Wg = ws_ptr<float>(a.ws, L.W);
  float* gsc = ws_ptr<float>(a.ws, L.gsc);
  float* vecpart = ws_ptr<float>(a.ws, L.vecpart);
  const int DP = L.DP, D = L.D;
  const int nds = DP >= KT ? DP / KT : 1;

  // shared memory behind the B ring: constants, the x~ tile, the dx staging tiles of the 8 row-owner warps
  float* cst = reinterpret_cast<float*>(smem_raw + (size_t)NSTB * STAGE_BYTES);
  float* znc_s = cst;                // [MP] exponent offsets
  float* beta_s = znc_s + MP;        // [MP] Linv^T m
  float* cen_s = beta_s + MP;        // [DXW] centre
  float* iel_s = cen_s + DXW;        // [DXW] 1 / ell
  float* wl_s = iel_s + DXW;         // [DXW] ell * w
  float* xt_s = wl_s + DXW;          // [128][XP] scaled inputs of the tile
  float* stg_s = xt_s + TNP * XP;    // [8][32][SP]
  {
    const float* znc_g = ws_cptr<float>(a.stage, L.znc);
    const float* beta_g = ws_cptr<float>(a.stage, L.beta);
    const float* center = ws_cptr<float>(a.stage, L.center);
    const float* inv_ell = ws_cptr<float>(a.stage, L.inv_ell);
    const float* wl = ws_cptr<float>(a.stage, L.wl);
    for (int i = tid; i < MP; i += kCtaThreads) { znc_s[i] = znc_g[i]; beta_s[i] = beta_g[i]; }
    for (int i = tid; i < DXW; i += kCtaThreads) {
      const bool ok = i < DP;
      cen_s[i] = ok ? center[i] : 0.f; iel_s[i] = ok ? inv_ell[i] : 0.f; wl_s[i] = ok ? wl[i] : 0.f;
    }
  }
  if (warp == 0) tc::tmem_alloc(&tmem_slot, TMEM_COLS);
  if (tid == 32) {
    for (int i = 0; i < 3; ++i) { tc::mbar_init(&bb.b.a_ready[i], kGroup); tc::mbar_init(&bb.b.mma_done[i], 1); }
    for (int i = 0; i < 6; ++i) { tc::mbar_init(&bb.b.b_full[i], 1); tc::mbar_init(&bb.b.b_empty[i], 1); }
    tc::mbar_init(&bb.b.s_full, 1);
    for (int i = 0; i < 8; ++i) tc::mbar_init(&bb.b.chunk[i], 1);
    tc::mbar_init(&bb.dx_full, 1);
    tc::mbar_init(&bb.x_ready, kGroup);
    tc::fence_barrier_init();
  }
  {
    const int n = bwd_table<BT, DXW>(tab, a, kCtaThreads);
    if (tid == 0) tab_n = n;
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const int tiles_mine = a.ntiles > (int)blockIdx.x ? (a.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  Bars* bars = &bb.b;

  if (warp >= kIssuerWarp) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsIssuer));
    if (warp == kIssuerWarp) {
      // the issuer's extra commit: SF_SIG_DX rides on the s_full slot of the generic issuer via a wrapper table flag
      tc2_issuer<NSTA, NSTB, true>(smem_raw, STAGE_BYTES, bars, tmem_base, AOP_COL, tab, tab_n, tiles_mine,
                                   blockIdx.x == 0 ? a.trace : nullptr, &bb.dx_full);
    } else if (warp == kIssuerWarp + 1) {
      tc2_loader<NSTB>(smem_raw, STAGE_BYTES, bars, tab, tab_n, tiles_mine);
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsProducer));
    const int grp = warp >> 3;                            // 0 = loaders, 1 = row owners
    const int quad = warp & 3, half = (warp >> 2) & 1;   // TMEM lane quadrant / k-half of this warp
    const int row = quad * 32 + lane;                     // the point this thread owns
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    const uint32_t aop_base = tmem_base + lane_base + AOP_COL;
    uint32_t tile_ctr = 0;

    if (grp == 0) {
      // =================== loaders ===================
      uint32_t cnt = 0;                                   // slabs produced by this group (private ring [0, NSTA - 1))
      // three saved-a slabs in flight (rotating register sets), requested in the order of the table
      float4 ra[3][4];
      auto load_a = [&](float4 (&r)[4], int tile, int sg) {
        const float4* At = reinterpret_cast<const float4*>(Ag) +
                           ((size_t)tile * (size_t)(MP >> 2) + (size_t)((sg * KT + half * 16) >> 2)) * TNP + row;
#pragma unroll
        for (int i = 0; i < 4; ++i) r[i] = ldg4_pinned(reinterpret_cast<const float*>(At + (size_t)i * TNP));
      };
      // the sequence of saved-a slabs of this CTA: (tile, p, t) -> slab sg = NSL - 1 - t, t < NSL - p SPB
      int pf_tile = blockIdx.x, pf_p = 0, pf_t = 0;       // next slab to request
      auto pf_advance = [&]() {
        if (++pf_t == NSL - pf_p * SPB) { pf_t = 0; if (++pf_p == NP) { pf_p = 0; pf_tile += gridDim.x; } }
      };
      int slot_w = 0, slot_r = 0;
      for (int i = 0; i < 3; ++i) {
        if (pf_tile < a.ntiles) { load_a(ra[slot_w], pf_tile, NSL - 1 - pf_t); pf_advance(); }
        slot_w = slot_w == 2 ? 0 : slot_w + 1;
      }
      for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x, ++tile_ctr) {
        for (int p = 0; p < NP; ++p) {
          const int ndense = NSL - (p + 1) * SPB;
          const int nt = NSL - p * SPB;
          for (int t = 0; t < nt; ++t) {
            if (t == ndense) {
              // ---- x~ slabs of S block p (from the shared x~ tile the row owners publish once per tile) ----
              if (p == 0) tc::mbar_wait(&bb.x_ready, tile_ctr & 1u);
              for (int ds = 0; ds < nds; ++ds, ++cnt) {
                float v[16];
                const float* xr = xt_s + row * XP + ds * KT + half * 16;
#pragma unroll
                for (int i = 0; i < 16; i += 4) {
                  const float4 x4 = *reinterpret_cast<const float4*>(xr + i);
                  v[i] = x4.x; v[i + 1] = x4.y; v[i + 2] = x4.z; v[i + 3] = x4.w;
                }
                const int st = ring_acquire(bars, cnt, 0, NSTA - 1);
                store_operand16(aop_base, st, half * 16, v);
                ring_publish(bars, st);
              }
            }
            // ---- saved-a slab sg = NSL - 1 - t ----
            {
              float v[16];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float4 x4 = slot_r == 0 ? ra[0][i] : (slot_r == 1 ? ra[1][i] : ra[2][i]);
                v[4 * i] = x4.x; v[4 * i + 1] = x4.y; v[4 * i + 2] = x4.z; v[4 * i + 3] = x4.w;
              }
              const int st = ring_acquire(bars, cnt, 0, NSTA - 1);
              store_operand16(aop_base, st, half * 16, v);
              ring_publish(bars, st);
              ++cnt;
              // refill the slot with the slab three ahead
              if (pf_tile < a.ntiles) {
                if (slot_r == 0) load_a(ra[0], pf_tile, NSL - 1 - pf_t);
                else if (slot_r == 1) load_a(ra[1], pf_tile, NSL - 1 - pf_t);
                else load_a(ra[2], pf_tile, NSL - 1 - pf_t);
                pf_advance();
              }
              slot_r = slot_r == 2 ? 0 : slot_r + 1;
            }
          }
        }
      }
    } else {
      // =================== row owners ===================
      const float os = hyp[H_OS], l2os = log2f(os);
      const RqHyp hp = KIND == GPBLUR_KERNEL_RQ ? RqHyp{hyp[H_ALPHA], hyp[H_I2A]} : RqHyp{0.f, 0.f};
      const uint32_t tmem_s = tmem_base + lane_base + S_COL, tmem_t = tmem_base + lane_base + T_COL;
      const uint32_t tmem_dx = tmem_base + lane_base + DX_COL;
      const int et = tid - kGroup;                        // thread index within the group
      const int ew = warp - 8;                            // warp index within the group
      float* stg = stg_s + ew * 32 * SP;
      const bool vec = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.x) & 15) == 0);
      const bool vec_dx = a.dx && (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.dx) & 15) == 0);
      uint32_t pass_ctr = 0;
      float qacc[NPIECE], tacc[NPIECE];                   // per-dimension reductions of this warp (lane-distributed)
#pragma unroll
      for (int i = 0; i < NPIECE; ++i) { qacc[i] = 0.f; tacc[i] = 0.f; }
      float s_gm = 0.f, s_r = 0.f, s_gv = 0.f;           // scalar sums (k-half 0 threads)
      float s_kbk = 0.f;                                  // sum kbar o k of the Matern / RQ kinds (every thread)
      float s_kba = 0.f;                                  // sum kbar o dk/dalpha of RQ (every thread)
      uint32_t cnt = 0;                                   // W slabs produced so far (private stage NSTA - 1)
      // x rows of a tile go global -> shared memory with cp.async (coalesced: 16 bytes per thread and request, no
      // registers), one tile ahead: issued after the previous tile's dx epilogue, awaited at the tile head
      constexpr int XREQ = TNP * (DXW / 4) / kGroup;      // requests per thread
      auto request_x_tile = [&](long long n0) {
        if (!vec) return;                                 // (unaligned / D % 4 != 0: loaded synchronously below)
#pragma unroll 4
        for (int i = 0; i < XREQ; ++i) {
          const int idx = et + i * kGroup;
          const int r = idx / (DXW / 4), c4 = (idx % (DXW / 4)) * 4;
          if (n0 + r < N && c4 < D) cp_async16(xt_s + r * XP + c4, a.x + (size_t)(n0 + r) * D + c4);
        }
        cp_async_commit();
      };
      request_x_tile((long long)blockIdx.x * TNP);
      for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x, ++tile_ctr) {
        const long long n0 = (long long)tile * TNP;
        const long long gn = n0 + row;
        const bool live = gn < N;
        // ---- upstream gradients of this thread's point (requested early) ----
        float gm = 0.f, gv = 0.f;
        if (live) {
          float gsv;
          bool has_gs;
          upstream_grads(a.seg, gn, gm, gv, gsv, has_gs);
          const float vr = a.var_in[gn];
          if (has_gs) {
            const float eps = philox_normal(a.seed, rng_offset(a.offset, a.offset_dev) + (uint64_t)gn, a.stream_id);
            gm += gsv;
            gv = fmaf(gsv * eps, 0.5f * rsqrtf(vr), gv);
          }
          if (vr <= kMinVariance) gv = 0.f;
          if (half == 0) { gsc[gn] = gm; gsc[N + gn] = gv; }
        }
        // ---- x~ tile: centre / scale in place (every thread transforms the pieces it requested itself) ----
        if (vec) cp_async_wait<0>();
#pragma unroll 4
        for (int i = 0; i < XREQ; ++i) {
          const int idx = et + i * kGroup;
          const int r = idx / (DXW / 4), c4 = (idx % (DXW / 4)) * 4;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (n0 + r < N && c4 < D) {
            if (vec) v = *reinterpret_cast<const float4*>(xt_s + r * XP + c4);
            else {
              const float* p = a.x + (size_t)(n0 + r) * D + c4;
              v.x = p[0];
              if (c4 + 1 < D) v.y = p[1];
              if (c4 + 2 < D) v.z = p[2];
              if (c4 + 3 < D) v.w = p[3];
            }
            const float4 c = *reinterpret_cast<const float4*>(cen_s + c4), ie = *reinterpret_cast<const float4*>(iel_s + c4);
            v.x = (v.x - c.x) * ie.x; v.y = (v.y - c.y) * ie.y; v.z = (v.z - c.z) * ie.z; v.w = (v.w - c.w) * ie.w;
          }
          *reinterpret_cast<float4*>(xt_s + r * XP + c4) = v;
        }
        asm volatile("bar.sync 2, 256;" ::: "memory");
        mbar_arrive(&bb.x_ready);
        float xnc;
        {
          float n2 = 0.f;
          const float* xr = xt_s + row * XP;
#pragma unroll 4
          for (int i = 0; i < DXW; i += 4) {
            const float4 x4 = *reinterpret_cast<const float4*>(xr + i);
            n2 = fmaf(x4.w, x4.w, fmaf(x4.z, x4.z, fmaf(x4.y, x4.y, fmaf(x4.x, x4.x, n2))));
          }
          xnc = -0.72134752044448170f * n2;
        }
        float rsum = 0.f;
        for (int p = 0; p < NP; ++p, ++pass_ctr) {
          tc::mbar_wait(&bars->s_full, pass_ctr & 1u);    // S block p complete
          tc::tc_fence_after();
#pragma unroll 1
          for (int c = SPB - 1; c >= 0; --c, ++cnt) {
            // chunk c of T is final once slab p SPB + c has retired (the slabs run in decreasing order)
            tc::mbar_wait(&bars->chunk[c], pass_ctr & 1u);
            tc::tc_fence_after();
            const int col = c * KT + half * 16;
            uint32_t kr[16], tr[16];
            tc::tmem_ld16_issue(tmem_s + (uint32_t)col, kr);
            tc::tmem_ld16_issue(tmem_t + (uint32_t)col, tr);
            tc::tmem_ld16_wait(kr);
            tc::tmem_ld16_wait(tr);
            float w[16];
            const float* zp = znc_s + p * BT + col;
            const float* bp = beta_s + p * BT + col;
            const float gv2 = 2.0f * gv;
            if constexpr (KIND == GPBLUR_KERNEL_RBF) {
#pragma unroll
              for (int i = 0; i < 16; i += 4) {
                const float4 z4 = *reinterpret_cast<const float4*>(zp + i), b4 = *reinterpret_cast<const float4*>(bp + i);
                const float k0 = tc::ex2_approx(fminf(fmaf(__uint_as_float(kr[i + 0]), 1.4426950408889634f, xnc + z4.x), l2os));
                const float k1 = tc::ex2_approx(fminf(fmaf(__uint_as_float(kr[i + 1]), 1.4426950408889634f, xnc + z4.y), l2os));
                const float k2 = tc::ex2_approx(fminf(fmaf(__uint_as_float(kr[i + 2]), 1.4426950408889634f, xnc + z4.z), l2os));
                const float k3 = tc::ex2_approx(fminf(fmaf(__uint_as_float(kr[i + 3]), 1.4426950408889634f, xnc + z4.w), l2os));
                w[i + 0] = fmaf(gv2, __uint_as_float(tr[i + 0]), gm * b4.x) * k0;
                w[i + 1] = fmaf(gv2, __uint_as_float(tr[i + 1]), gm * b4.y) * k1;
                w[i + 2] = fmaf(gv2, __uint_as_float(tr[i + 2]), gm * b4.z) * k2;
                w[i + 3] = fmaf(gv2, __uint_as_float(tr[i + 3]), gm * b4.w) * k3;
              }
            } else {
#pragma unroll
              for (int i = 0; i < 16; i += 4) {
                const float4 z4 = *reinterpret_cast<const float4*>(zp + i), b4 = *reinterpret_cast<const float4*>(bp + i);
                const float zz[4] = {z4.x, z4.y, z4.z, z4.w}, bb4[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  float k, g, ka;
                  tc_kg<KIND>(fminf(fmaf(__uint_as_float(kr[i + e]), 1.4426950408889634f, xnc + zz[e]), l2os), l2os, os, hp,
                              k, g, ka);
                  const float kb = fmaf(gv2, __uint_as_float(tr[i + e]), gm * bb4[e]);
                  w[i + e] = kb * g;
                  s_kbk = fmaf(kb, k, s_kbk);
                  if constexpr (KIND == GPBLUR_KERNEL_RQ) s_kba = fmaf(kb, ka, s_kba);
                }
              }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) rsum += w[i];
            // the W operand of the dx GEMM first (the tensor core is waiting for it), then the tile-major copy for W^T X
            {
              const int st = ring_acquire(bars, cnt, NSTA - 1, 1);
              store_operand16(aop_base, st, half * 16, w);
              ring_publish(bars, st);
            }
            {
              float4* Wt = reinterpret_cast<float4*>(Wg) + ((size_t)tile * (size_t)(MP >> 2) + (size_t)((p * BT + col) >> 2)) * TNP + row;
#pragma unroll
              for (int i = 0; i < 4; ++i) Wt[(size_t)i * TNP] = make_float4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
            }
          }
        }
        // ---- row sums: the two k-halves of a point ----
        r_s[half][row] = rsum;
        asm volatile("bar.sync 2, 256;" ::: "memory");
        const float rtot = r_s[0][row] + r_s[1][row];
        if (half == 0 && live) { s_gm += gm; s_r += rtot; s_gv += gv; }
        // ---- dx epilogue ----
        tc::mbar_wait(&bb.dx_full, tile_ctr & 1u);
        tc::tc_fence_after();
#pragma unroll
        for (int pc = 0; pc < NPIECE; ++pc) {
          const int col = half * HW + pc * 16;
          float v[16], qv[16], tv[16];
          tc::tmem_ld16(tmem_dx + (uint32_t)col, v);
          const float* xr = xt_s + row * XP + col;
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const float4 x4 = *reinterpret_cast<const float4*>(xr + i);
            const float4 ie = *reinterpret_cast<const float4*>(iel_s + col + i), w4 = *reinterpret_cast<const float4*>(wl_s + col + i);
            const float xs[4] = {x4.x, x4.y, x4.z, x4.w}, ies[4] = {ie.x, ie.y, ie.z, ie.w}, ws4[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              v[i + e] = (v[i + e] - rtot * xs[e]) * ies[e] + gm * (ws4[e] * ies[e]);
              qv[i + e] = rtot * xs[e] * xs[e];
              tv[i + e] = gm * xs[e];
            }
          }
          // per-dimension sums over the 32 points of the warp (fixed shuffle tree: deterministic)
          qacc[pc] += warp_reduce16(qv, lane);
          tacc[pc] += warp_reduce16(tv, lane);
          if (a.dx) {
            // [32 rows x 16 columns] through the warp's staging tile: 8 rows x 64 contiguous bytes per store instruction
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 16; i += 4)
              *reinterpret_cast<float4*>(stg + lane * SP + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
            __syncwarp();
            const int c4 = (lane & 3) * 4, rsub = lane >> 2;
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              const int rr = it * 8 + rsub;
              const long long gr = n0 + quad * 32 + rr;
              const int d = col + c4;
              if (gr < N && d < D) {
                const float4 o = *reinterpret_cast<const float4*>(stg + rr * SP + c4);
                float* dst = a.dx + (size_t)gr * D + d;
                if (vec_dx) *reinterpret_cast<float4*>(dst) = o;
                else {
                  dst[0] = o.x;
                  if (d + 1 < D) dst[1] = o.y;
                  if (d + 2 < D) dst[2] = o.z;
                  if (d + 3 < D) dst[3] = o.w;
                }
              }
            }
          }
        }
        // the DX reads of this tile are done before this group publishes the next tile's first W slab; the x~ tile may be
        // overwritten (every slab of this tile has retired: dx_full)
        tc::tc_fence_before();
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (tile + (int)gridDim.x < a.ntiles) request_x_tile(n0 + (long long)gridDim.x * TNP);
      }
      // ---- per-CTA vector partial: [colsum MP (from the W^T X kernel) | q DP | wbar DP | scalars] ----
      if ((lane & 1) == 0) {
        const int idx = warp_reduce16_index(lane);
#pragma unroll
        for (int pc = 0; pc < NPIECE; ++pc) {
          vec_s[half][quad][pc * 16 + idx] = qacc[pc];
          vec_s[half][quad][HW + pc * 16 + idx] = tacc[pc];
        }
      }
      {
        const float sg = warp_sum(s_gm), sr = warp_sum(s_r), sv = warp_sum(s_gv);
        const float sk = KIND == GPBLUR_KERNEL_RBF ? 0.f : warp_sum(s_kbk);
        const float sa = KIND == GPBLUR_KERNEL_RQ ? warp_sum(s_kba) : 0.f;
        if (lane == 0) {
          sc_s[ew][VS_GMU] = sg; sc_s[ew][VS_RSUM] = sr; sc_s[ew][VS_GVAR] = sv; sc_s[ew][VS_KBK] = sk;
          sc_s[ew][VS_KBA] = sa;
        }
      }
      asm volatile("bar.sync 2, 256;" ::: "memory");
      float* vp = vecpart + (size_t)blockIdx.x * L.vp_len;
      const float* ellv = ws_cptr<float>(a.stage, L.ell);
      float sgm = 0.f;
      for (int w = 0; w < 4; ++w) sgm += sc_s[w][VS_GMU];                 // k-half 0 warps, fixed order
      for (int i = et; i < MP; i += kGroup) vp[i] = 0.f;
      for (int d = et; d < DP; d += kGroup) {
        float q = 0.f, t1 = 0.f;
        if (d < DXW) {
          const int hf = d / HW, within = d % HW;
          for (int qd = 0; qd < 4; ++qd) { q += vec_s[hf][qd][within]; t1 += vec_s[hf][qd][HW + within]; }
        }
        vp[MP + d] = q;
        vp[MP + DP + d] = d < D ? ellv[d] * t1 + cen_s[d < DXW ? d : 0] * sgm : 0.f;
      }
      if (et < VS_PART) {
        float sum = 0.f;
        if (et < 3) for (int w = 0; w < 4; ++w) sum += sc_s[w][et];
        else if (et == VS_KBK ? KIND != GPBLUR_KERNEL_RBF : KIND == GPBLUR_KERNEL_RQ)
          for (int w = 0; w < 8; ++w) sum += sc_s[w][et];   // VS_KBK / VS_KBA: both k-halves
        vp[MP + 2 * DP + et] = sum;
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_slot, TMEM_COLS);
}

template <int BQ, int BWO, int NSTB, int KIND>
__global__ void __launch_bounds__(kCtaThreads, 1) tc2_fwd_kernel(Tc2Args a) { tc2_fwd_body<BQ, BWO, NSTB, KIND>(a); }
template <int BQ, int BWO, int NSTB>
__global__ void __launch_bounds__(kCtaThreads, 1) tc2_fwd_rq_kernel(Tc2Args a) {
  tc2_fwd_body<BQ, BWO, NSTB, GPBLUR_KERNEL_RQ>(a);
}
template <int BT, int DXW, int NSTA, int NSTB, int KIND>
__global__ void __launch_bounds__(kCtaThreads, 1) tc2_bwd_kernel(Tc2Args a) { tc2_bwd_body<BT, DXW, NSTA, NSTB, KIND>(a); }
template <int BT, int DXW, int NSTA, int NSTB>
__global__ void __launch_bounds__(kCtaThreads, 1) tc2_bwd_rq_kernel(Tc2Args a) {
  tc2_bwd_body<BT, DXW, NSTA, NSTB, GPBLUR_KERNEL_RQ>(a);
}

int tc2_grid(const WsLayout& L) {
  const long long nt = (L.N + TNP - 1) / TNP;
  const int sms = num_sms();
  return (int)(nt < sms ? (nt < 1 ? 1 : nt) : sms);
}

// cudaFuncSetAttribute is per device: set it on every launch (cheap) rather than caching per process
template <class K>
void set_smem(K kernel, size_t bytes) {
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

template <int BQ, int BWO, int NSTB, int KIND>
void launch_fwd_kind(const Tc2Args& a, int grid, cudaStream_t st) {
  const size_t smem = (size_t)NSTB * BWO * 256 + (size_t)(3 * a.L.MP + 3 * a.L.DP) * sizeof(float);
  auto* kernel = [] {
    if constexpr (KIND == GPBLUR_KERNEL_RQ) return tc2_fwd_rq_kernel<BQ, BWO, NSTB>;
    else return tc2_fwd_kernel<BQ, BWO, NSTB, KIND>;
  }();
  set_smem(kernel, smem);
  kernel<<<grid, kCtaThreads, smem, st>>>(a);
}

template <int BQ, int BWO, int NSTB>
int launch_fwd(const Tc2Args& a, int grid, cudaStream_t st) {
  switch (a.L.kind) {
    case GPBLUR_KERNEL_MATERN12: launch_fwd_kind<BQ, BWO, NSTB, GPBLUR_KERNEL_MATERN12>(a, grid, st); break;
    case GPBLUR_KERNEL_MATERN32: launch_fwd_kind<BQ, BWO, NSTB, GPBLUR_KERNEL_MATERN32>(a, grid, st); break;
    case GPBLUR_KERNEL_MATERN52: launch_fwd_kind<BQ, BWO, NSTB, GPBLUR_KERNEL_MATERN52>(a, grid, st); break;
    case GPBLUR_KERNEL_RQ: launch_fwd_kind<BQ, BWO, NSTB, GPBLUR_KERNEL_RQ>(a, grid, st); break;
    default: launch_fwd_kind<BQ, BWO, NSTB, GPBLUR_KERNEL_RBF>(a, grid, st);
  }
  return 0;
}

template <int BT, int DXW, int NSTA, int NSTB, int KIND>
void launch_bwd_kind(const Tc2Args& a, int grid, cudaStream_t st) {
  constexpr size_t brows = BT > DXW ? BT : DXW;
  const size_t smem = (size_t)NSTB * brows * 256 +
                      (size_t)(2 * a.L.MP + 3 * DXW + TNP * (DXW + 4) + 8 * 32 * 20) * sizeof(float);
  auto* kernel = [] {
    if constexpr (KIND == GPBLUR_KERNEL_RQ) return tc2_bwd_rq_kernel<BT, DXW, NSTA, NSTB>;
    else return tc2_bwd_kernel<BT, DXW, NSTA, NSTB, KIND>;
  }();
  set_smem(kernel, smem);
  kernel<<<grid, kCtaThreads, smem, st>>>(a);
}

template <int BT, int DXW, int NSTA, int NSTB>
int launch_bwd(const Tc2Args& a, int grid, cudaStream_t st) {
  switch (a.L.kind) {
    case GPBLUR_KERNEL_MATERN12: launch_bwd_kind<BT, DXW, NSTA, NSTB, GPBLUR_KERNEL_MATERN12>(a, grid, st); break;
    case GPBLUR_KERNEL_MATERN32: launch_bwd_kind<BT, DXW, NSTA, NSTB, GPBLUR_KERNEL_MATERN32>(a, grid, st); break;
    case GPBLUR_KERNEL_MATERN52: launch_bwd_kind<BT, DXW, NSTA, NSTB, GPBLUR_KERNEL_MATERN52>(a, grid, st); break;
    case GPBLUR_KERNEL_RQ: launch_bwd_kind<BT, DXW, NSTA, NSTB, GPBLUR_KERNEL_RQ>(a, grid, st); break;
    default: launch_bwd_kind<BT, DXW, NSTA, NSTB, GPBLUR_KERNEL_RBF>(a, grid, st);
  }
  return 0;
}

}  // namespace

bool tc_point_supported(const WsLayout& L) {
  if (tile_override("GPBLUR_TC") < 0) return false;       // GPBLUR_TC=-1 forces the FP32 FFMA kernels (tests)
  return (L.MP == 128 || (L.MP >= 256 && L.MP % 256 == 0)) && L.N >= 1;
}

int tc_vector_partials(const WsLayout& L) { return tc2_grid(L); }

int launch_tc_point_forward(const WsLayout& L, const void* stage, void* ws, const float* x, float* mean, float* var,
                            float* sample, uint64_t seed, uint64_t offset, uint32_t stream_id,
                            const unsigned long long* offset_dev, cudaStream_t st) {
  Tc2Args a{};
  a.L = L; a.ws = ws; a.stage = stage; a.x = x; a.mean = mean; a.var = var; a.sample = sample;
  a.seed = seed; a.offset = offset; a.offset_dev = offset_dev; a.stream_id = stream_id;
  a.ntiles = (int)((L.N + TNP - 1) / TNP);
  a.trace = debug_trace_buffer();
  const int grid = tc2_grid(L);
  ProfScope ps(ST_POINT_FWD, st);
  if (L.MP == 128) launch_fwd<128, 128, 4>(a, grid, st);
  else launch_fwd<128, 256, 3>(a, grid, st);
  note_launch();
  return check_launch("tc_point_fwd");
}

int launch_tc_point_backward(const WsLayout& L, const void* stage, void* ws, const float* x, const SegGrads& seg,
                             const float* var, uint64_t seed, uint64_t offset, uint32_t stream_id,
                             const unsigned long long* offset_dev, float* dx, cudaStream_t st) {
  Tc2Args a{};
  a.L = L; a.ws = ws; a.stage = stage; a.x = x; a.seg = seg; a.var_in = var; a.dx = dx;
  a.seed = seed; a.offset = offset; a.offset_dev = offset_dev; a.stream_id = stream_id;
  a.ntiles = (int)((L.N + TNP - 1) / TNP);
  a.trace = debug_trace_buffer();
  const int grid = tc2_grid(L);
  ProfScope ps(ST_POINT_BWD, st);
  if (L.DP <= 32) launch_bwd<128, 32, 3, 4>(a, grid, st);
  else if (L.DP == 64) launch_bwd<128, 64, 3, 4>(a, grid, st);
  else launch_bwd<128, 128, 2, 3>(a, grid, st);
  note_launch();
  return check_launch("tc_point_bwd");
}

}  // namespace gpblur
