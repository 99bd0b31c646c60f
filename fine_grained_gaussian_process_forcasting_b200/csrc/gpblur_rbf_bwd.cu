// Backward of the dense ScaleKernel(RBF) covariance (gpblur_covariance): what torch autograd computes through
// gpytorch's kernel evaluation when an exact GP is trained (/root/reference/denoising_model/GPModel.py:4-13 builds
// MultivariateNormal(mean, ScaleKernel(RBF)(x)); the marginal log likelihood differentiates the covariance w.r.t. the
// raw lengthscale / outputscale and the inputs).  With W = G o K (G = upstream gradient of the covariance):
//   g_x1[i, d] = -sum_j W_ij (x1_id - x2_jd) / l_d^2          g_x2[j, d] = +sum_i W_ij (x1_id - x2_jd) / l_d^2
//   g_l_d      =  sum_ij W_ij (x1_id - x2_jd)^2 / l_d^3        g_os = sum_ij W_ij / os
// and the chain rule through softplus (sigmoid of the raw value); an isotropic kernel sums g_l over d.
// Matern and RQ kinds: W = G o g (gpblur_common.cuh: matern_kg / rq_kg) in the distance gradients, and
// g_os = sum_ij G_ij K_ij / os from a second matrix Wk = G o K.  RQ: g_alpha = sum_ij G_ij dK_ij/dalpha from a third
// matrix Wa, summed per row as one more row statistic.
// Three launches: W (tile kernel, as the forward) -> row pass (g_x1, per-row lengthscale / W sums) and column pass
// (g_x2) -> one CTA adds the per-row sums in row order (bit-deterministic).  O(n1 n2 D) work, exact-GP sizes.
#include "gpblur_common.cuh"

namespace gpblur {

namespace {

__device__ __forceinline__ float softplus_f(float r) { return r > 20.f ? r : log1pf(expf(r)); }
__device__ __forceinline__ float sigmoid_f(float r) { return 1.0f / (1.0f + expf(-r)); }

// W[i, j] = G[i, j] * os * exp(-1/2 sum_d ((x1_id - x2_jd) / l_d)^2): 16 x 16 tile per CTA, direct differences
template <int KIND>
__global__ void rbf_w_kernel(const float* __restrict__ x1, const float* __restrict__ x2, long long n1, long long n2, int D,
                             const float* __restrict__ raw_ell, int ard, const float* __restrict__ raw_os,
                             const float* __restrict__ raw_alpha, const float* __restrict__ g_out,
                             float* __restrict__ W, float* __restrict__ Wk, float* __restrict__ Wa) {
  __shared__ float a[16][33], b[16][33], ie[32];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const long long i0 = (long long)blockIdx.y * 16, j0 = (long long)blockIdx.x * 16;
  float acc = 0.f;
  for (int d0 = 0; d0 < D; d0 += 32) {
    __syncthreads();
    if (threadIdx.x < 32) {
      const int d = d0 + threadIdx.x;
      ie[threadIdx.x] = d < D ? 1.0f / softplus_f(raw_ell[ard ? d : 0]) : 0.f;
    }
    for (int idx = threadIdx.x; idx < 16 * 32; idx += blockDim.x) {
      const int r = idx >> 5, c = idx & 31, d = d0 + c;
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
    if constexpr (KIND == GPBLUR_KERNEL_RBF) {
      W[(size_t)i * n2 + j] = g_out[(size_t)i * n2 + j] * softplus_f(raw_os[0]) * expf(-0.5f * acc);
    } else if constexpr (KIND == GPBLUR_KERNEL_RQ) {
      const float alpha = softplus_f(raw_alpha[0]);
      float k, g, ka;
      rq_kg(acc, softplus_f(raw_os[0]), alpha, 0.5f / alpha, k, g, ka);
      const float go = g_out[(size_t)i * n2 + j];
      W[(size_t)i * n2 + j] = go * g;
      Wk[(size_t)i * n2 + j] = go * k;
      Wa[(size_t)i * n2 + j] = go * ka;
    } else {
      float k, g;
      matern_kg<KIND>(acc, softplus_f(raw_os[0]), k, g);
      const float go = g_out[(size_t)i * n2 + j];
      W[(size_t)i * n2 + j] = go * g;
      Wk[(size_t)i * n2 + j] = go * k;
    }
  }
}

// one CTA per row i of x1: threads = dimensions (d < D <= 128), loop over j.
//   g_x1[i, d] ; rowstat[i, d] = sum_j W_ij (x1_id - x2_jd)^2 ; rowstat[i, D] = sum_j Wos_ij   (double)
//   (Wos: W for RBF, Wk for the Matern and RQ kinds); RQ (Wa non-null): rowstat[i, D + 1] = sum_j Wa_ij.
//   Row stride rs = D + 1, D + 2 for RQ.
__global__ void rbf_row_kernel(const float* __restrict__ x1, const float* __restrict__ x2, long long n2, int D,
                               const float* __restrict__ raw_ell, int ard, const float* __restrict__ W,
                               const float* __restrict__ Wos, const float* __restrict__ Wa, int rs,
                               float* __restrict__ g_x1, double* __restrict__ rowstat) {
  const long long i = blockIdx.x;
  const int d = threadIdx.x;
  const float* wr = W + (size_t)i * n2;
  if (d < D) {
    const float ell = softplus_f(raw_ell[ard ? d : 0]);
    const float xi = x1[(size_t)i * D + d];
    double s1 = 0.0, s2 = 0.0;
    for (long long j = 0; j < n2; ++j) {
      const float w = wr[j], df = xi - x2[(size_t)j * D + d];
      s1 += (double)(w * df);
      s2 += (double)(w * df * df);
    }
    if (g_x1) g_x1[(size_t)i * D + d] = (float)(-s1 / ((double)ell * ell));
    rowstat[(size_t)i * rs + d] = s2;
  } else if (d == D || (d == D + 1 && Wa)) {
    const float* wo = (d == D ? Wos : Wa) + (size_t)i * n2;
    double s = 0.0;
    for (long long j = 0; j < n2; ++j) s += (double)wo[j];
    rowstat[(size_t)i * rs + d] = s;
  }
}

// one CTA per column j: g_x2[j, d] = + sum_i W_ij (x1_id - x2_jd) / l_d^2
__global__ void rbf_col_kernel(const float* __restrict__ x1, const float* __restrict__ x2, long long n1, long long n2,
                               int D, const float* __restrict__ raw_ell, int ard, const float* __restrict__ W,
                               float* __restrict__ g_x2) {
  const long long j = blockIdx.x;
  const int d = threadIdx.x;
  if (d >= D) return;
  const float ell = softplus_f(raw_ell[ard ? d : 0]);
  const float xj = x2[(size_t)j * D + d];
  double s1 = 0.0;
  for (long long i = 0; i < n1; ++i) s1 += (double)(W[(size_t)i * n2 + j] * (x1[(size_t)i * D + d] - xj));
  g_x2[(size_t)j * D + d] = (float)(s1 / ((double)ell * ell));
}

// rows added in row order: g_raw_ell [D] (ard) or [1], g_raw_os [1], RQ (rs = D + 2): g_raw_alpha [1]
__global__ void rbf_finish_kernel(const double* __restrict__ rowstat, long long n1, int D, int rs,
                                  const float* __restrict__ raw_ell, int ard, const float* __restrict__ raw_os,
                                  const float* __restrict__ raw_alpha, float* __restrict__ g_raw_ell,
                                  float* __restrict__ g_raw_os, float* __restrict__ g_raw_alpha) {
  __shared__ double iso[129];
  const int d = threadIdx.x;
  double t = 0.0;
  if (d < rs)
    for (long long i = 0; i < n1; ++i) t += rowstat[(size_t)i * rs + d];
  if (d < D) {
    const float r = raw_ell[ard ? d : 0];
    const double ell = (double)softplus_f(r);
    const double gl = t / (ell * ell * ell) * (double)sigmoid_f(r);
    if (ard) g_raw_ell[d] = (float)gl;
    iso[d] = gl;
  } else if (d == D) {
    const float r = raw_os[0];
    g_raw_os[0] = (float)(t / (double)softplus_f(r) * (double)sigmoid_f(r));
  } else if (d == D + 1 && d < rs) {
    g_raw_alpha[0] = (float)(t * (double)sigmoid_f(raw_alpha[0]));
  }
  __syncthreads();
  if (!ard && d == 0) {
    double s = 0.0;
    for (int k = 0; k < D; ++k) s += iso[k];
    g_raw_ell[0] = (float)s;
  }
}

}  // namespace

}  // namespace gpblur

using namespace gpblur;

// W matrices of a kind (W; W, Wk; W, Wk, Wa for RQ) and the row-statistic stride
static int cov_wmats(int kind) { return kind == GPBLUR_KERNEL_RBF ? 1 : kind == GPBLUR_KERNEL_RQ ? 3 : 2; }
static int cov_rowstride(int D, int kind) { return D + (kind == GPBLUR_KERNEL_RQ ? 2 : 1); }

extern "C" size_t gpblur_covariance_backward_scratch_bytes(long long n1, long long n2, int D, int kind) {
  if (n1 < 0 || n2 < 0 || D < 1 || !kernel_kind_valid(kind)) return 0;
  const size_t wb = align_up((size_t)n1 * (size_t)n2 * 4);
  return cov_wmats(kind) * wb + (size_t)n1 * (size_t)cov_rowstride(D, kind) * 8;
}

extern "C" int gpblur_covariance_backward(const float* x1, const float* x2, long long n1, long long n2, int D, int kind,
                                          const float* raw_lengthscale, int ard, const float* raw_outputscale,
                                          const float* g_out, float* g_x1, float* g_x2, float* g_raw_lengthscale,
                                          float* g_raw_outputscale, void* scratch, size_t scratch_bytes, void* stream) {
  return gpblur_covariance_backward_alpha(x1, x2, n1, n2, D, kind, raw_lengthscale, ard, raw_outputscale, nullptr,
                                          g_out, g_x1, g_x2, g_raw_lengthscale, g_raw_outputscale, nullptr, scratch,
                                          scratch_bytes, stream);
}

extern "C" int gpblur_covariance_backward_alpha(const float* x1, const float* x2, long long n1, long long n2, int D,
                                                int kind, const float* raw_lengthscale, int ard,
                                                const float* raw_outputscale, const float* raw_alpha,
                                                const float* g_out, float* g_x1, float* g_x2, float* g_raw_lengthscale,
                                                float* g_raw_outputscale, float* g_raw_alpha, void* scratch,
                                                size_t scratch_bytes, void* stream) {
  if (n1 < 1 || n2 < 1 || D < 1 || D > GPBLUR_MAX_D || !kernel_kind_valid(kind)) return GPBLUR_EINVAL;
  if (!x1 || !x2 || !raw_lengthscale || !raw_outputscale || !g_out || !g_raw_lengthscale || !g_raw_outputscale || !scratch)
    return GPBLUR_EINVAL;
  if (kind == GPBLUR_KERNEL_RQ && (!raw_alpha || !g_raw_alpha)) return GPBLUR_EINVAL;
  if ((reinterpret_cast<uintptr_t>(scratch) & 255) ||
      scratch_bytes < gpblur_covariance_backward_scratch_bytes(n1, n2, D, kind))
    return GPBLUR_EWORKSPACE;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const size_t wb = align_up((size_t)n1 * (size_t)n2 * 4);
  const bool rbf = kind == GPBLUR_KERNEL_RBF, rq = kind == GPBLUR_KERNEL_RQ;
  float* W = static_cast<float*>(scratch);
  float* Wk = rbf ? W : reinterpret_cast<float*>(static_cast<char*>(scratch) + wb);
  float* Wa = rq ? reinterpret_cast<float*>(static_cast<char*>(scratch) + 2 * wb) : nullptr;
  double* rowstat = reinterpret_cast<double*>(static_cast<char*>(scratch) + cov_wmats(kind) * wb);
  const int rs = cov_rowstride(D, kind);
  const int threads = round_up(rs, 32);
  ProfScope ps(ST_OTHER, st);
  dim3 grid((unsigned)((n2 + 15) / 16), (unsigned)((n1 + 15) / 16));
  switch (kind) {
    case GPBLUR_KERNEL_MATERN12:
      rbf_w_kernel<GPBLUR_KERNEL_MATERN12><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, g_out, W, Wk, Wa);
      break;
    case GPBLUR_KERNEL_MATERN32:
      rbf_w_kernel<GPBLUR_KERNEL_MATERN32><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, g_out, W, Wk, Wa);
      break;
    case GPBLUR_KERNEL_MATERN52:
      rbf_w_kernel<GPBLUR_KERNEL_MATERN52><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, g_out, W, Wk, Wa);
      break;
    case GPBLUR_KERNEL_RQ:
      rbf_w_kernel<GPBLUR_KERNEL_RQ><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, g_out, W, Wk, Wa);
      break;
    default:
      rbf_w_kernel<GPBLUR_KERNEL_RBF><<<grid, 256, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, raw_outputscale, raw_alpha, g_out, W, Wk, Wa);
  }
  rbf_row_kernel<<<(unsigned)n1, threads, 0, st>>>(x1, x2, n2, D, raw_lengthscale, ard, W, Wk, Wa, rs, g_x1, rowstat);
  if (g_x2) rbf_col_kernel<<<(unsigned)n2, threads, 0, st>>>(x1, x2, n1, n2, D, raw_lengthscale, ard, W, g_x2);
  rbf_finish_kernel<<<1, threads, 0, st>>>(rowstat, n1, D, rs, raw_lengthscale, ard, raw_outputscale, raw_alpha,
                                           g_raw_lengthscale, g_raw_outputscale, g_raw_alpha);
  note_launch(g_x2 ? 4 : 3);
  return check_launch("rbf_cov_backward");
}
