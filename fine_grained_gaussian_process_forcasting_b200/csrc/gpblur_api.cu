// extern "C" entry points (see include/gpblur.h) + the small elementwise kernels: ELBO, Philox probes,
// reparameterised sample, dense RBF covariance.
#include <atomic>
#include <mutex>
#include <vector>
#include <cstdio>
#include <cstring>
#include <cstdlib>

#include "gpblur_common.cuh"
#include "gpblur_tile.cuh"

namespace gpblur {

static std::atomic<unsigned long long> g_launches{0};
static thread_local char g_err[256] = "";

// ---- optional per-stage timing (bench.py roofline): events are recorded on the launching stream ----
struct ProfRec { int stage; cudaEvent_t a, b; };
static std::atomic<int> g_prof_on{0};
static std::mutex g_prof_mu;
static std::vector<ProfRec*> g_prof_recs;

ProfScope::ProfScope(int stage_, cudaStream_t st_) : stage(stage_), st(st_), rec(nullptr) {
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  ProfRec* r = new ProfRec{stage, nullptr, nullptr};
  cudaEventCreate(&r->a);
  cudaEventCreate(&r->b);
  cudaEventRecord(r->a, st);
  rec = r;
}
ProfScope::~ProfScope() {
  if (!rec) return;
  ProfRec* r = static_cast<ProfRec*>(rec);
  cudaEventRecord(r->b, st);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_recs.push_back(r);
}

static std::atomic<long long*> g_trace{nullptr};
long long* debug_trace_buffer() { return g_trace.load(std::memory_order_relaxed); }

void note_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return GPBLUR_OK;
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return GPBLUR_ELAUNCH;
}

int num_sms() {
  static int cache[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (cache[dev] == 0) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    cache[dev] = n > 0 ? n : 148;
  }
  return cache[dev];
}

// Tuning knobs (tile heights, GPBLUR_TC=-1): the environment is read ONCE per knob, not on every launch.  Callers
// pass string literals: a handful of distinct pointers, cached in a small table.
int tile_override(const char* env) {
  static std::mutex mu;
  static const char* names[8];
  static int values[8];
  static int n = 0;
  std::lock_guard<std::mutex> lk(mu);
  for (int i = 0; i < n; ++i)
    if (names[i] == env) return values[i];
  const char* v = getenv(env);
  const int val = v ? atoi(v) : 0;
  if (n < 8) { names[n] = env; values[n] = val; ++n; }
  return val;
}

int bwd_vector_partials(const WsLayout& L);
int stage_grad_reduce_impl(const WsLayout& L, const void* ws, double* sgrad, int nvec_used, int ncpart,
                           cudaStream_t st);

namespace {

// ---------------------------------------------------------------------------------------------
// ELBO (GaussianLikelihood.expected_log_prob summed over the event dim / L, minus KL / num_data)
// ---------------------------------------------------------------------------------------------
__global__ void elbo_fwd_kernel(const float* __restrict__ mean, const float* __restrict__ var,
                                const float* __restrict__ y, const float* __restrict__ raw_noise,
                                const float* __restrict__ kl, float num_data, long long B, int L,
                                float* __restrict__ elbo) {
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const float rn = raw_noise[0];
  const float noise = (rn > 20.f ? rn : log1pf(expf(rn))) + kNoiseLower;
  const float inv = 1.0f / noise, lg = logf(noise) + 1.8378770664093453f;   // log(2 pi)
  float s = 0.f;
  for (int l = lane; l < L; l += 32) {
    const size_t i = (size_t)b * L + l;
    const float d = y[i] - mean[i];
    s += -0.5f * (fmaf(d, d, var[i]) * inv + lg);
  }
  s = warp_sum(s);
  if (lane == 0) elbo[b] = s / (float)L - kl[0] / num_data;
}

__global__ void elbo_bwd_kernel(const float* __restrict__ mean, const float* __restrict__ var,
                                const float* __restrict__ y, const float* __restrict__ raw_noise,
                                const float* __restrict__ g_elbo, long long B, int L,
                                float* __restrict__ g_mean, float* __restrict__ g_var,
                                float* __restrict__ scratch) {
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const float rn = raw_noise[0];
  const float noise = (rn > 20.f ? rn : log1pf(expf(rn))) + kNoiseLower;
  const float inv = 1.0f / noise;
  const float ge = g_elbo[b] / (float)L;
  float s = 0.f;
  for (int l = lane; l < L; l += 32) {
    const size_t i = (size_t)b * L + l;
    const float d = y[i] - mean[i];
    g_mean[i] = ge * d * inv;
    g_var[i] = -0.5f * ge * inv;
    s += 0.5f * (fmaf(d, d, var[i]) * inv * inv - inv);
  }
  s = warp_sum(s);
  if (lane == 0) scratch[b] = ge * s;
}

// final reduction over the windows, fixed order (one block; volatile reads: the values come from other blocks)
__device__ __forceinline__ void elbo_bwd_finish(const float* scratch, const float* g_elbo, const float* raw_noise,
                                                float num_data, long long B, float* g_raw_noise, float* g_kl) {
  __shared__ double r1[32], r2[32];
  double s1 = 0.0, s2 = 0.0;
  for (long long b = threadIdx.x; b < B; b += blockDim.x) {
    s1 += (double)*reinterpret_cast<const volatile float*>(scratch + b);
    s2 += (double)g_elbo[b];
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { r1[warp] = s1; r2[warp] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { t1 += r1[i]; t2 += r2[i]; }
    const double rn = (double)raw_noise[0];
    if (g_raw_noise) g_raw_noise[0] = (float)(t1 * sigmoid64(rn));
    if (g_kl) g_kl[0] = (float)(-t2 / (double)num_data);
  }
}

// elbo_bwd_kernel + the final reduction in ONE launch: the block that takes the last ticket (a self-resetting
// atomicInc on a caller-provided zeroed word) reduces the per-window partials - one graph node less per step.
__global__ void elbo_bwd_fused_kernel(const float* __restrict__ mean, const float* __restrict__ var,
                                      const float* __restrict__ y, const float* __restrict__ raw_noise,
                                      const float* __restrict__ g_elbo, float num_data, long long B, int L,
                                      float* __restrict__ g_mean, float* __restrict__ g_var,
                                      float* __restrict__ scratch, float* __restrict__ g_raw_noise,
                                      float* __restrict__ g_kl, unsigned* __restrict__ ticket) {
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b < B) {
    const float rn = raw_noise[0];
    const float noise = (rn > 20.f ? rn : log1pf(expf(rn))) + kNoiseLower;
    const float inv = 1.0f / noise;
    const float ge = g_elbo[b] / (float)L;
    float s = 0.f;
    for (int l = lane; l < L; l += 32) {
      const size_t i = (size_t)b * L + l;
      const float d = y[i] - mean[i];
      g_mean[i] = ge * d * inv;
      g_var[i] = -0.5f * ge * inv;
      s += 0.5f * (fmaf(d, d, var[i]) * inv * inv - inv);
    }
    s = warp_sum(s);
    if (lane == 0) scratch[b] = ge * s;
  }
  __shared__ bool last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicInc(ticket, gridDim.x - 1) == gridDim.x - 1;     // wraps to 0: ready for the next launch
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  elbo_bwd_finish(scratch, g_elbo, raw_noise, num_data, B, g_raw_noise, g_kl);
}

__global__ void elbo_bwd_finish_kernel(const float* __restrict__ scratch, const float* __restrict__ g_elbo,
                                       const float* __restrict__ raw_noise, float num_data, long long B,
                                       float* __restrict__ g_raw_noise, float* __restrict__ g_kl) {
  __shared__ double r1[32], r2[32];
  double s1 = 0.0, s2 = 0.0;
  for (long long b = threadIdx.x; b < B; b += blockDim.x) {
    s1 += (double)scratch[b];
    s2 += (double)g_elbo[b];
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { r1[warp] = s1; r2[warp] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t1 = 0.0, t2 = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { t1 += r1[i]; t2 += r2[i]; }
    const double rn = (double)raw_noise[0];
    if (g_raw_noise) g_raw_noise[0] = (float)(t1 * sigmoid64(rn));
    if (g_kl) g_kl[0] = (float)(-t2 / (double)num_data);
  }
}

// ---------------------------------------------------------------------------------------------
__global__ void philox_bits_kernel(uint64_t seed, uint64_t offset, uint32_t stream_id, long long n,
                                   uint32_t* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint4 r = philox_element(seed, offset + (uint64_t)i, stream_id);
  reinterpret_cast<uint4*>(out)[i] = r;
}

__global__ void philox_normal_kernel(uint64_t seed, uint64_t offset, uint32_t stream_id, long long n,
                                     float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = philox_normal(seed, offset + (uint64_t)i, stream_id);
}

__global__ void rsample_fwd_kernel(const float* __restrict__ mean, const float* __restrict__ var, long long n,
                                   uint64_t seed, uint64_t offset, uint32_t stream_id,
                                   float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = fmaf(sqrtf(var[i]), philox_normal(seed, offset + (uint64_t)i, stream_id), mean[i]);
}

__global__ void rsample_bwd_kernel(const float* __restrict__ var, const float* __restrict__ g_out, long long n,
                                   uint64_t seed, uint64_t offset, uint32_t stream_id,
                                   float* __restrict__ g_mean, float* __restrict__ g_var) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float g = g_out[i];
  g_mean[i] = g;
  g_var[i] = g * philox_normal(seed, offset + (uint64_t)i, stream_id) * 0.5f * rsqrtf(var[i]);
}

// dense ScaleKernel(RBF | Matern | RQ): 16 x 16 output tile per CTA, direct differences
template <int KIND>
__global__ void rbf_cov_kernel(const float* __restrict__ x1, const float* __restrict__ x2, long long n1,
                               long long n2, int D, const float* __restrict__ raw_ell, int ard,
                               const float* __restrict__ raw_os, const float* __restrict__ raw_alpha,
                               float* __restrict__ out) {
  __shared__ float a[16][33], b[16][33], ie[32];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const long long i0 = (long long)blockIdx.y * 16, j0 = (long long)blockIdx.x * 16;
  float acc = 0.f;
  for (int d0 = 0; d0 < D; d0 += 32) {
    __syncthreads();
    if (threadIdx.x < 32) {
      const int d = d0 + threadIdx.x;
      float v = 0.f;
      if (d < D) {
        const float r = raw_ell[ard ? d : 0];
        v = 1.0f / (r > 20.f ? r : log1pf(expf(r)));
      }
      ie[threadIdx.x] = v;
    }
    for (int idx = threadIdx.x; idx < 16 * 32; idx += blockDim.x) {
      const int r = idx >> 5, c = idx & 31;
      const int d = d0 + c;
      a[r][c] = (i0 + r < n1 && d < D) ? x1[(size_t)(i0 + r) * D + d] : 0.f;
      b[r][c] = (j0 + r < n2 && d < D) ? x2[(size_t)(j0 + r) * D + d] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int c = 0; c < 32; ++c) {
      const float df = (a[ty][c] - b[tx][c]) * ie[c];
      acc = fmaf(df, df, acc);
    }
  }
  const long long i = i0 + ty, j = j0 + tx;
  if (i < n1 && j < n2) {
    const float r = raw_os[0];
    const float os = r > 20.f ? r : log1pf(expf(r));
    if constexpr (KIND == GPBLUR_KERNEL_RBF) {
      out[(size_t)i * n2 + j] = os * expf(-0.5f * acc);
    } else if constexpr (KIND == GPBLUR_KERNEL_RQ) {
      const float ra = raw_alpha[0], alpha = ra > 20.f ? ra : log1pf(expf(ra));
      float k, g, ka;
      rq_kg(acc, os, alpha, 0.5f / alpha, k, g, ka);
      out[(size_t)i * n2 + j] = k;
    } else {
      float k, g;
      matern_kg<KIND>(acc, os, k, g);
      out[(size_t)i * n2 + j] = k;
    }
  }
}

inline int ew_grid(long long n, int block) { return (int)((n + block - 1) / block); }

}  // namespace

int dispatch_point_forward(const WsLayout& L, const void* stage, void* ws, const float* x, float* mean, float* var,
                           float* sample, uint64_t seed, uint64_t offset, uint32_t stream_id,
                           const unsigned long long* offset_dev, cudaStream_t st) {
  if (tc_point_supported(L))
    return launch_tc_point_forward(L, stage, ws, x, mean, var, sample, seed, offset, stream_id, offset_dev, st);
  return launch_point_forward(L, stage, ws, x, mean, var, sample, seed, offset, stream_id, offset_dev, st);
}

int launch_stage_grad_reduce(const WsLayout& L, const void* ws, double* sgrad, cudaStream_t st) {
  if (tc_point_supported(L)) return stage_grad_reduce_impl(L, ws, sgrad, tc_vector_partials(L), L.splitsZ, st);
  return stage_grad_reduce_impl(L, ws, sgrad, bwd_vector_partials(L), 0, st);
}

}  // namespace gpblur

using namespace gpblur;

extern "C" {

size_t gpblur_svgp_grad_bucket_floats(int D, int M) { return (size_t)M * D + 2 * (size_t)M + 2 * (size_t)D + 2; }

size_t gpblur_svgp_grad_bucket_floats_kind(int D, int M, int kind) {
  if (!kernel_kind_valid(kind)) return 0;
  return gpblur_svgp_grad_bucket_floats(D, M) + (kind == GPBLUR_KERNEL_RQ ? 1 : 0);
}

size_t gpblur_svgp_workspace_bytes(long long N, int D, int M, int training) {
  if (N < 0 || D < 1 || M < 1 || D > GPBLUR_MAX_D || M > GPBLUR_MAX_M) return 0;
  return make_layout(N, D, M, training).total;
}

static bool aligned256(const void* p) { return p && !(reinterpret_cast<uintptr_t>(p) & 255); }

static int check_shape(long long N, int D, int M) {
  if (N < 0 || D < 1 || M < 1) return GPBLUR_EINVAL;
  return (D > GPBLUR_MAX_D || M > GPBLUR_MAX_M) ? GPBLUR_EUNSUPPORTED : GPBLUR_OK;
}

static int validate(const gpblur_svgp_params* p, long long N, int D, int M) {
  if (!p) return GPBLUR_EINVAL;
  const int rc = check_shape(N, D, M);
  if (rc) return rc;
  if (!p->inducing_points || !p->raw_lengthscale || !p->raw_outputscale || !p->variational_mean ||
      !p->variational_stddev || !p->mean_bias)
    return GPBLUR_EINVAL;
  return GPBLUR_OK;
}

// Arguments of the M x M stage and of its backward: parameters, kind and the stage buffer.  Fills the stage layout.
static int check_stage(const gpblur_svgp_params* p, int D, int M, int kind, const void* stage, size_t stage_bytes,
                       WsLayout* L) {
  const int rc = validate(p, 0, D, M);
  if (rc) return rc;
  if (!kernel_kind_valid(kind) || !aligned256(stage)) return GPBLUR_EINVAL;
  if (kind == GPBLUR_KERNEL_RQ && !p->raw_alpha) return GPBLUR_EINVAL;
  *L = make_layout(0, D, M, 0);
  L->kind = kind;
  return stage_bytes < L->total ? GPBLUR_EWORKSPACE : GPBLUR_OK;
}

// Arguments of the point forward and backward: shape, kind, the stage they read and the workspace.  Fills the layout
// of the call.
static int check_point(const void* stage, long long N, int D, int M, int kind, int training, const void* ws,
                       size_t ws_bytes, WsLayout* L) {
  const int rc = check_shape(N, D, M);
  if (rc) return rc;
  if (!kernel_kind_valid(kind) || !aligned256(stage) || !aligned256(ws)) return GPBLUR_EINVAL;
  *L = make_layout(N, D, M, training);
  L->kind = kind;
  return ws_bytes < L->total ? GPBLUR_EWORKSPACE : GPBLUR_OK;
}

int gpblur_svgp_forward(const gpblur_svgp_params* p, const float* x, long long N, int D, int M, float* mean,
                        float* var, float* sample, uint64_t seed, uint64_t offset, uint32_t stream_id,
                        float* kl, int* info, int training, void* ws, size_t ws_bytes, void* stream) {
  int rc = validate(p, N, D, M);
  if (rc) return rc;
  if (N > 0 && (!x || !mean || !var)) return GPBLUR_EINVAL;
  if (!aligned256(ws)) return GPBLUR_EINVAL;
  const WsLayout L = make_layout(N, D, M, training ? 1 : 0);
  if (ws_bytes < L.total) return GPBLUR_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  rc = launch_mm_forward(*p, L, ws, kl, info, st);
  if (rc) return rc;
  if (N == 0) return GPBLUR_OK;
  return dispatch_point_forward(L, ws, ws, x, mean, var, sample, seed, offset, stream_id, nullptr, st);
}

size_t gpblur_svgp_param_stage_bytes(int D, int M) {
  if (D < 1 || M < 1 || D > GPBLUR_MAX_D || M > GPBLUR_MAX_M) return 0;
  return make_layout(0, D, M, 0).total;   // the inference layout is exactly the parameter stage
}

size_t gpblur_svgp_stage_grad_doubles(int D, int M) { return gpblur_svgp_stage_grad_doubles_kind(D, M, GPBLUR_KERNEL_RBF); }

size_t gpblur_svgp_stage_grad_doubles_kind(int D, int M, int kind) {
  if (D < 1 || M < 1 || D > GPBLUR_MAX_D || M > GPBLUR_MAX_M || !kernel_kind_valid(kind)) return 0;
  return stage_grad_doubles(padded_m(M), padded_d(D), kind);
}

int gpblur_svgp_param_stage(const gpblur_svgp_params* p, int D, int M, int kind, double extra_jitter, int max_ctas,
                            float* kl, int* info, void* stage, size_t stage_bytes, void* stream) {
  WsLayout L;
  const int rc = check_stage(p, D, M, kind, stage, stage_bytes, &L);
  if (rc) return rc;
  if (!(extra_jitter >= 0.0) || max_ctas < 0) return GPBLUR_EINVAL;
  return launch_mm_forward(*p, L, stage, kl, info, (cudaStream_t)stream, extra_jitter, max_ctas);
}

int gpblur_svgp_param_stage_backward(const gpblur_svgp_params* p, int D, int M, int kind, const double* stage_grad,
                                     const float* g_kl, float* grad_bucket, int accumulate, int max_ctas,
                                     void* stage, size_t stage_bytes, void* stream) {
  WsLayout L;
  const int rc = check_stage(p, D, M, kind, stage, stage_bytes, &L);
  if (rc) return rc;
  if (!stage_grad || !grad_bucket || max_ctas < 0) return GPBLUR_EINVAL;
  return launch_mm_backward(*p, L, stage, stage_grad, g_kl, grad_bucket, (cudaStream_t)stream, accumulate ? 1 : 0,
                            max_ctas);
}

int gpblur_svgp_point_forward(const void* param_stage, const float* x, long long N, int D, int M, int kind,
                              float* mean, float* var, float* sample, uint64_t seed, uint64_t offset,
                              uint32_t stream_id, const unsigned long long* offset_dev, int training, void* ws,
                              size_t ws_bytes, void* stream) {
  WsLayout L;
  const int rc = check_point(param_stage, N, D, M, kind, training ? 1 : 0, ws, ws_bytes, &L);
  if (rc) return rc;
  if (N == 0) return GPBLUR_OK;
  if (!x || !mean || !var) return GPBLUR_EINVAL;
  return dispatch_point_forward(L, param_stage, ws, x, mean, var, sample, seed, offset, stream_id, offset_dev,
                                (cudaStream_t)stream);
}

int gpblur_svgp_point_backward(const void* param_stage, const float* x, long long N, int D, int M, int kind,
                               int nseg, const long long* seg_start, const float* const* g_mean,
                               const float* const* g_var, const float* const* g_sample, const float* var,
                               uint64_t seed, uint64_t offset, uint32_t stream_id, const unsigned long long* offset_dev,
                               float* dx, double* stage_grad, void* ws, size_t ws_bytes, void* stream) {
  const void* stage = param_stage ? param_stage : ws;
  WsLayout L;
  int rc = check_point(stage, N, D, M, kind, 1, ws, ws_bytes, &L);
  if (rc) return rc;
  if (!stage_grad || (N > 0 && (!x || !var))) return GPBLUR_EINVAL;
  if (nseg < 1 || nseg > kMaxSegments || !seg_start || seg_start[0] != 0) return GPBLUR_EINVAL;
  SegGrads sg{};
  sg.nseg = nseg;
  for (int i = 0; i < nseg; ++i) {
    if (seg_start[i] < 0 || seg_start[i] > N || (i > 0 && seg_start[i] < seg_start[i - 1])) return GPBLUR_EINVAL;
    sg.start[i] = seg_start[i];
    sg.gm[i] = g_mean ? g_mean[i] : nullptr;
    sg.gv[i] = g_var ? g_var[i] : nullptr;
    sg.gs[i] = g_sample ? g_sample[i] : nullptr;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (N > 0) {
    if (tc_point_supported(L))
      rc = launch_tc_point_backward(L, stage, ws, x, sg, var, seed, offset, stream_id, offset_dev, dx, st);
    else
      rc = launch_point_backward(L, stage, ws, x, sg, var, seed, offset, stream_id, offset_dev, dx, st);
    if (rc) return rc;
    rc = launch_reductions(L, ws, x, st);
    if (rc) return rc;
  }
  return launch_stage_grad_reduce(L, ws, stage_grad, st);
}

int gpblur_svgp_backward(const gpblur_svgp_params* p, const float* x, long long N, int D, int M,
                         const float* g_mean, const float* g_var, const float* g_sample, const float* g_kl,
                         const float* var, uint64_t seed, uint64_t offset, uint32_t stream_id, float* dx,
                         float* grad_bucket, void* ws, size_t ws_bytes, void* stream) {
  int rc = validate(p, N, D, M);
  if (rc) return rc;
  if (!grad_bucket || !aligned256(ws)) return GPBLUR_EINVAL;
  const WsLayout L = make_layout(N, D, M, 1);
  if (ws_bytes < L.total) return GPBLUR_EWORKSPACE;
  double* sgrad = ws_ptr<double>(ws, L.sgrad);
  const long long start = 0;
  rc = gpblur_svgp_point_backward(nullptr, x, N, D, M, GPBLUR_KERNEL_RBF, 1, &start, &g_mean, &g_var, &g_sample, var,
                                  seed, offset, stream_id, nullptr, dx, sgrad, ws, ws_bytes, stream);
  if (rc) return rc;
  return launch_mm_backward(*p, L, ws, sgrad, g_kl, grad_bucket, (cudaStream_t)stream);
}

int gpblur_elbo_forward(const float* mean, const float* var, const float* y, const float* raw_noise,
                        const float* kl, float num_data, long long B, int L, float* elbo, void* stream) {
  if (B < 0 || L < 1 || !raw_noise || !kl) return GPBLUR_EINVAL;
  if (B == 0) return GPBLUR_OK;
  if (!mean || !var || !y || !elbo) return GPBLUR_EINVAL;
  ProfScope ps(ST_ELBO_FWD, (cudaStream_t)stream);
  elbo_fwd_kernel<<<ew_grid(B, 8), 256, 0, (cudaStream_t)stream>>>(mean, var, y, raw_noise, kl, num_data, B, L,
                                                                   elbo);
  note_launch();
  return check_launch("elbo_fwd");
}

int gpblur_elbo_backward_fused(const float* mean, const float* var, const float* y, const float* raw_noise,
                               const float* g_elbo, float num_data, long long B, int L, float* g_mean, float* g_var,
                               float* g_raw_noise, float* g_kl, float* scratch, unsigned* ticket, void* stream) {
  if (B < 1 || L < 1 || !raw_noise || !ticket) return GPBLUR_EINVAL;
  if (!mean || !var || !y || !g_elbo || !g_mean || !g_var || !scratch) return GPBLUR_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope ps(ST_ELBO_BWD, st);
  elbo_bwd_fused_kernel<<<ew_grid(B, 8), 256, 0, st>>>(mean, var, y, raw_noise, g_elbo, num_data, B, L, g_mean, g_var,
                                                       scratch, g_raw_noise, g_kl, ticket);
  note_launch();
  return check_launch("elbo_bwd");
}

int gpblur_elbo_backward(const float* mean, const float* var, const float* y, const float* raw_noise,
                         const float* g_elbo, float num_data, long long B, int L, float* g_mean, float* g_var,
                         float* g_raw_noise, float* g_kl, float* scratch, void* stream) {
  if (B < 0 || L < 1 || !raw_noise) return GPBLUR_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope ps(ST_ELBO_BWD, st);
  if (B > 0) {
    if (!mean || !var || !y || !g_elbo || !g_mean || !g_var || !scratch) return GPBLUR_EINVAL;
    elbo_bwd_kernel<<<ew_grid(B, 8), 256, 0, st>>>(mean, var, y, raw_noise, g_elbo, B, L, g_mean, g_var,
                                                   scratch);
    note_launch();
  }
  elbo_bwd_finish_kernel<<<1, 1024, 0, st>>>(scratch, g_elbo, raw_noise, num_data, B, g_raw_noise, g_kl);
  note_launch();
  return check_launch("elbo_bwd");
}

int gpblur_philox_bits(uint64_t seed, uint64_t offset, uint32_t stream_id, long long n, uint32_t* out,
                       void* stream) {
  if (n < 0 || (n > 0 && !out)) return GPBLUR_EINVAL;
  if (n == 0) return GPBLUR_OK;
  philox_bits_kernel<<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(seed, offset, stream_id, n, out);
  note_launch();
  return check_launch("philox_bits");
}

int gpblur_philox_normal(uint64_t seed, uint64_t offset, uint32_t stream_id, long long n, float* out,
                         void* stream) {
  if (n < 0 || (n > 0 && !out)) return GPBLUR_EINVAL;
  if (n == 0) return GPBLUR_OK;
  philox_normal_kernel<<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(seed, offset, stream_id, n, out);
  note_launch();
  return check_launch("philox_normal");
}

int gpblur_rsample_forward(const float* mean, const float* var, long long n, uint64_t seed, uint64_t offset,
                           uint32_t stream_id, float* out, void* stream) {
  if (n < 0 || (n > 0 && (!mean || !var || !out))) return GPBLUR_EINVAL;
  if (n == 0) return GPBLUR_OK;
  rsample_fwd_kernel<<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(mean, var, n, seed, offset, stream_id,
                                                                       out);
  note_launch();
  return check_launch("rsample_fwd");
}

int gpblur_rsample_backward(const float* var, const float* g_out, long long n, uint64_t seed, uint64_t offset,
                            uint32_t stream_id, float* g_mean, float* g_var, void* stream) {
  if (n < 0 || (n > 0 && (!var || !g_out || !g_mean || !g_var))) return GPBLUR_EINVAL;
  if (n == 0) return GPBLUR_OK;
  rsample_bwd_kernel<<<ew_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(var, g_out, n, seed, offset, stream_id,
                                                                       g_mean, g_var);
  note_launch();
  return check_launch("rsample_bwd");
}

int gpblur_covariance(const float* x1, const float* x2, long long n1, long long n2, int D, int kind,
                      const float* raw_lengthscale, int ard, const float* raw_outputscale, float* out, void* stream) {
  return gpblur_covariance_alpha(x1, x2, n1, n2, D, kind, raw_lengthscale, ard, raw_outputscale, nullptr, out, stream);
}

int gpblur_covariance_alpha(const float* x1, const float* x2, long long n1, long long n2, int D, int kind,
                            const float* raw_lengthscale, int ard, const float* raw_outputscale, const float* raw_alpha,
                            float* out, void* stream) {
  if (n1 < 0 || n2 < 0 || D < 1 || !raw_lengthscale || !raw_outputscale || !kernel_kind_valid(kind)) return GPBLUR_EINVAL;
  if (kind == GPBLUR_KERNEL_RQ && !raw_alpha) return GPBLUR_EINVAL;
  if (n1 == 0 || n2 == 0) return GPBLUR_OK;
  if (!x1 || !x2 || !out) return GPBLUR_EINVAL;
  dim3 grid((unsigned)((n2 + 15) / 16), (unsigned)((n1 + 15) / 16));
  cudaStream_t st = (cudaStream_t)stream;
  switch (kind) {
    case GPBLUR_KERNEL_MATERN12:
      rbf_cov_kernel<GPBLUR_KERNEL_MATERN12><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, out);
      break;
    case GPBLUR_KERNEL_MATERN32:
      rbf_cov_kernel<GPBLUR_KERNEL_MATERN32><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, out);
      break;
    case GPBLUR_KERNEL_MATERN52:
      rbf_cov_kernel<GPBLUR_KERNEL_MATERN52><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, out);
      break;
    case GPBLUR_KERNEL_RQ:
      rbf_cov_kernel<GPBLUR_KERNEL_RQ><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, out);
      break;
    default:
      rbf_cov_kernel<GPBLUR_KERNEL_RBF><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, out);
  }
  note_launch();
  return check_launch("rbf_cov");
}

int gpblur_debug_fetch(int which, long long N, int D, int M, const void* ws, void* out, size_t out_bytes,
                       int* mp, void* stream) {
  if (!ws || !out || D < 1 || M < 1 || D > GPBLUR_MAX_D || M > GPBLUR_MAX_M) return GPBLUR_EINVAL;
  const WsLayout L = make_layout(N, D, M, 1);
  if (mp) *mp = L.MP;
  size_t off = 0, bytes = 0;
  const size_t mm8 = (size_t)L.MP * L.MP * 8;
  switch (which) {
    case 0: off = L.L64; bytes = mm8; break;
    case 1: off = L.Linv64; bytes = mm8; break;
    case 2: off = L.K64; bytes = mm8; break;
    case 3: off = L.A; bytes = (size_t)(L.MP >= 128 ? round_up_ll(N, 128) : N) * L.MP * 4; break;   // tile-major if MP >= 128
    case 4: off = L.stamps; bytes = kStampSlots * 8; break;
    case 5: off = L.W; bytes = (size_t)(L.MP >= 128 ? round_up_ll(N, 128) : N) * L.MP * 4; break;   // W = kbar o k (after a backward)
    case 6: off = L.gsc; bytes = (size_t)2 * (N > 0 ? N : 1) * 4; break;   // folded g_mu, g_var (after a backward)
    default: return GPBLUR_EINVAL;
  }
  if (out_bytes < bytes) return GPBLUR_EWORKSPACE;
  cudaMemcpyAsync(out, ws_cptr<char>(ws, off), bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
  return check_launch("debug_fetch");
}

int gpblur_debug_set_trace(void* device_buffer) {
  g_trace.store(static_cast<long long*>(device_buffer));
  return GPBLUR_OK;
}

int gpblur_profile_enable(int on) {
  g_prof_on.store(on ? 1 : 0);
  return GPBLUR_OK;
}

int gpblur_profile_collect(double* ms, unsigned long long* counts, int n) {
  if (!ms || !counts || n < ST_COUNT) return GPBLUR_EINVAL;
  for (int i = 0; i < n; ++i) { ms[i] = 0.0; counts[i] = 0; }
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (ProfRec* r : g_prof_recs) {
    cudaEventSynchronize(r->b);
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r->a, r->b) == cudaSuccess) { ms[r->stage] += (double)t; counts[r->stage] += 1; }
    cudaEventDestroy(r->a);
    cudaEventDestroy(r->b);
    delete r;
  }
  g_prof_recs.clear();
  return GPBLUR_OK;
}

unsigned long long gpblur_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
const char* gpblur_last_cuda_error(void) { return g_err; }
const char* gpblur_version(void) { return "gpblur 0.2 (sm_100a)"; }

}  // extern "C"
