/*
 * gpblur.h - C ABI of the B200 (sm_100a) GP blur / corruption hot path.
 *
 * The reference (SepKfr/Fine_grained_Gaussian_Process_Forcasting) has no FFI of its own: the path sits
 * behind Python classes that call gpytorch.  Each entry point below replaces the gpytorch call chain
 * cited next to it; the Python package binds them with ctypes (see INTEGRATION.md for the stub).
 *
 * Conventions
 *   - all tensor arguments are DEVICE pointers to contiguous fp32 unless stated; they are borrowed,
 *     never freed, never reallocated;  `stream` is a cudaStream_t passed as void*.
 *   - no entry point allocates device memory or synchronises; scratch comes from the caller as
 *     (`ws`, `ws_bytes`), sized by gpblur_svgp_workspace_bytes().  The SAME workspace must be
 *     handed to the matching backward call (it carries the saved whitened cross-covariances).
 *   - return value: 0 on success, negative GPBLUR_E* code on argument / launch errors.  Numerical
 *     failure of the Cholesky (non-PD Kzz) is reported asynchronously through the device int `info`
 *     (0 = ok, k>0 = pivot k was not positive), like LAPACK potrf.
 *   - thread-safe and re-entrant: no global mutable state except a per-device immutable
 *     attribute cache.
 */
#ifndef GPBLUR_H_
#define GPBLUR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPBLUR_OK 0
#define GPBLUR_EINVAL -1     /* bad shape / null pointer */
#define GPBLUR_EWORKSPACE -2 /* workspace too small */
#define GPBLUR_ELAUNCH -3    /* CUDA launch failure (see gpblur_last_cuda_error) */
#define GPBLUR_EUNSUPPORTED -4

#define GPBLUR_MAX_D 128
#define GPBLUR_MAX_M 1024

/* Covariance function of a layer (the `kind` argument of the entry points below).  With x~ = (x - c) / ell,
 * d2 = |x~ - z~|^2 and r = sqrt(max(d2, 1e-30)) (gpytorch's covar_dist), k = os f:
 *   RBF         f = exp(-d2 / 2)                         (gpblur_svgp_forward / gpblur_svgp_backward)
 *   MATERN12    f = exp(-r)                              (gpytorch MaternKernel(nu=0.5))
 *   MATERN32    f = (1 + sqrt3 r) exp(-sqrt3 r)          (nu=1.5)
 *   MATERN52    f = (1 + sqrt5 r + 5/3 r^2) exp(-sqrt5 r) (nu=2.5)
 *   RQ          f = (1 + d2 / (2 alpha))^-alpha          (gpytorch RQKernel; d2 unclamped, alpha = softplus(raw_alpha))
 *               df/dalpha = f (u / (1 + u) - log1p(u)), u = d2 / (2 alpha)
 * An unknown kind returns GPBLUR_EINVAL.  A parameter stage must be consumed (point forward / backward, stage backward)
 * with the kind it was built with; nothing on the device checks this. */
#define GPBLUR_KERNEL_RBF 0
#define GPBLUR_KERNEL_MATERN12 1
#define GPBLUR_KERNEL_MATERN32 2
#define GPBLUR_KERNEL_MATERN52 3
#define GPBLUR_KERNEL_RQ 4

/* Parameters of one whitened sparse variational GP layer.
 * Replaces the parameter set created by ToyDeepGPHiddenLayer.__init__
 * (/root/reference/denoising_model/DeepGP.py:15-49) for output_dims=None. */
typedef struct gpblur_svgp_params {
  const float* inducing_points;    /* [M, D]   VariationalStrategy.inducing_points        */
  const float* raw_lengthscale;    /* [D]      covar_module.base_kernel.raw_lengthscale   */
  const float* raw_outputscale;    /* [1]      covar_module.raw_outputscale               */
  const float* variational_mean;   /* [M]      _variational_distribution.variational_mean */
  const float* variational_stddev; /* [M]      _variational_distribution._variational_stddev */
  const float* mean_weights;       /* [D] LinearMean.weights, or NULL for ConstantMean    */
  const float* mean_bias;          /* [1] LinearMean.bias / ConstantMean constant         */
  const float* raw_alpha;          /* [1], read only for GPBLUR_KERNEL_RQ (NULL then: GPBLUR_EINVAL)
                                      covar_module.base_kernel.raw_alpha                 */
} gpblur_svgp_params;

/* Number of floats in the flat parameter-gradient bucket written by gpblur_svgp_backward:
 *   [ dZ (M*D) | d raw_lengthscale (D) | d raw_outputscale (1) | d variational_mean (M) |
 *     d variational_stddev (M) | d mean_weights (D) | d mean_bias (1) ]
 * This bucket is what data-parallel training all-reduces. */
size_t gpblur_svgp_grad_bucket_floats(int D, int M);
/* The bucket of a layer of kind `kind`: for GPBLUR_KERNEL_RQ one more trailing float, d raw_alpha. */
size_t gpblur_svgp_grad_bucket_floats_kind(int D, int M, int kind);

/* Scratch bytes for N input points.  `training` != 0 reserves room for the saved whitened
 * cross-covariance A [N, Mp] and the backward intermediates. */
size_t gpblur_svgp_workspace_bytes(long long N, int D, int M, int training);

/* Whitened SVGP predictive.
 * Replaces DeepGPp.forward / ToyDeepGPHiddenLayer.__call__ -> gpytorch
 * VariationalStrategy.forward (/root/reference/denoising_model/DeepGP.py:56-73, 90-92):
 *   Kzz build + jitter, fp64 blocked Cholesky, explicit whitening, predictive mean / variance,
 *   optional fused Philox reparameterised sample, KL(q(u)||p(u)).
 *   x [N, D] -> mean [N], var [N], sample [N] (nullable), kl [1], info [1].
 * sample_n = mean_n + sqrt(var_n) * eps_n, eps_n = BoxMuller(Philox4x32-10(counter = (offset + n,
 * stream_id), key = seed)).  With training != 0 the workspace keeps what the backward needs. */
int gpblur_svgp_forward(const gpblur_svgp_params* p, const float* x, long long N, int D, int M,
                        float* mean, float* var, float* sample, uint64_t seed, uint64_t offset,
                        uint32_t stream_id, float* kl, int* info, int training, void* ws,
                        size_t ws_bytes, void* stream);

/* Bytes at the start of a workspace that hold the once-per-parameter-update M x M stage (Kzz, L, Linv and the
 * fp32 operands derived from them).  They depend only on the parameters, not on x. */
size_t gpblur_svgp_param_stage_bytes(int D, int M);

/* Backward of gpblur_svgp_forward (replaces torch autograd through gpytorch, incl.
 * LinalgCholeskyExBackward0 / LinalgSolveTriangularBackward0).
 * Upstream gradients g_mean, g_var, g_sample [N] (each nullable) and g_kl [1] (nullable);
 * `var` is the forward output (needed for the variance clamp and the sample path).
 * Writes dx [N, D] (nullable) and the flat bucket described above. */
int gpblur_svgp_backward(const gpblur_svgp_params* p, const float* x, long long N, int D, int M,
                         const float* g_mean, const float* g_var, const float* g_sample,
                         const float* g_kl, const float* var, uint64_t seed, uint64_t offset,
                         uint32_t stream_id, float* dx, float* grad_bucket, void* ws,
                         size_t ws_bytes, void* stream);

/* ---- split form: one parameter stage shared by several calls -------------------------------------------
 * The reference evaluates the SAME GP on the encoder and on the decoder activations of one training step
 * (/root/reference/denoising_model/denoise_model_2.py:50-51) and gpytorch factorises Kzz (and differentiates the
 * factorisation) once per call and per batch element.  Here the once-per-parameter-update M x M work is its own
 * pair of entry points, and each call contributes a "stage gradient" that is LINEAR in its upstream gradients:
 *
 *   gpblur_svgp_param_stage          params -> stage (Kzz, L, Linv, fp32 / UMMA operand images), kl, info
 *   gpblur_svgp_point_forward        (stage, x) -> mean, var, sample              [any number of calls]
 *   gpblur_svgp_point_backward       upstream grads -> dx, stage_grad (fp64)      [one per forward call]
 *   gpblur_svgp_param_stage_backward (stage, SUM of the stage_grads, g_kl) -> flat parameter-gradient bucket
 *
 * stage_grad holds gpblur_svgp_stage_grad_doubles_kind(D, M, kind) doubles:
 *   [ u (Mp) | colsum(W) (Mp), q (Dp), wbar (Dp), scalars (4) | S = sum g_var a a^T (Mp x Mp) | W^T X (Mp x Dp) |
 *     GPBLUR_KERNEL_RQ only: sum kbar o dk/dalpha (1) ]
 * gpblur_svgp_forward / gpblur_svgp_backward above are the single-call compositions of these four (RBF, the stage
 * built in `ws`).  All four calls on one stage take the same `kind` (GPBLUR_KERNEL_*). */
size_t gpblur_svgp_stage_grad_doubles(int D, int M);   /* every kind but RQ */
size_t gpblur_svgp_stage_grad_doubles_kind(int D, int M, int kind);

/* Parameters -> M x M stage in `stage` (256-byte aligned, gpblur_svgp_param_stage_bytes(D, M) bytes), kl [1], info [1].
 * `extra_jitter` >= 0 is added to the diagonal of Kzz on top of the variational jitter 1e-4.  It replaces the retry
 * loop of gpytorch's psd_safe_cholesky (called from VariationalStrategy.forward,
 * /root/reference/denoising_model/DeepGP.py:33-38): when `info` reports a non-positive pivot the host retries with
 * 1e-6, 1e-5, 1e-4 and raises NotPSDError after that.  The jitter of the data-side diagonal diag(Kxx) stays 1e-4.
 * `max_ctas` bounds the cooperative grid (0 = none, else >= 8).  A multi-output layer (DeepGP.py:21-26: H independent
 * GPs) launches its H stages on H streams with (SM count / H) CTAs each, so that they run side by side. */
int gpblur_svgp_param_stage(const gpblur_svgp_params* p, int D, int M, int kind, double extra_jitter, int max_ctas,
                            float* kl, int* info, void* stage, size_t stage_bytes, void* stream);

/* (stage, x [N, D]) -> mean [N], var [N], sample [N] (nullable), as gpblur_svgp_forward.  The kernels read their
 * constant operands in place from `param_stage` (non-null, 256-byte aligned), which must stay unchanged until the
 * matching backward call has run.  `ws` (gpblur_svgp_workspace_bytes(N, D, M, training)) holds the per-call buffers;
 * with training != 0 hand the same `ws` to gpblur_svgp_point_backward.
 * `offset_dev` (nullable): device-resident uint64 added to `offset` when the kernel runs, so that a step captured in
 * a CUDA graph draws fresh Philox counters on every replay (the host bumps the device word between replays). */
int gpblur_svgp_point_forward(const void* param_stage, const float* x, long long N, int D, int M, int kind,
                              float* mean, float* var, float* sample, uint64_t seed, uint64_t offset, uint32_t stream_id,
                              const unsigned long long* offset_dev, int training, void* ws, size_t ws_bytes, void* stream);

/* Backward of gpblur_svgp_point_forward, with the forward's `ws`, RNG arguments and `var` output: writes dx [N, D]
 * (nullable) and stage_grad.  `param_stage` is the stage the forward read, or null when the stage lives in `ws`.
 * The upstream gradients come per segment, so that several activations evaluated as one call (the reference blurs the
 * encoder and the decoder activations with the same GP) keep them where autograd produced them: segment s covers
 * points [seg_start[s], seg_start[s + 1]) (nseg in [1, 4], seg_start[0] = 0, non-decreasing, <= N), and g_mean[s] /
 * g_var[s] / g_sample[s] (host arrays of nullable device pointers, or null arrays) are indexed from the start of the
 * segment.  One segment covers all N points. */
int gpblur_svgp_point_backward(const void* param_stage, const float* x, long long N, int D, int M, int kind,
                               int nseg, const long long* seg_start, const float* const* g_mean,
                               const float* const* g_var, const float* const* g_sample, const float* var,
                               uint64_t seed, uint64_t offset, uint32_t stream_id, const unsigned long long* offset_dev,
                               float* dx, double* stage_grad, void* ws, size_t ws_bytes, void* stream);

/* (stage, summed stage_grad, g_kl [1] nullable) -> flat parameter-gradient bucket.  `stage` is the buffer filled by
 * gpblur_svgp_param_stage; its fp64 scratch regions are overwritten.  `accumulate` != 0 ADDS the gradients to
 * `grad_bucket`, which then is the caller's live flat gradient buffer (what the data-parallel all-reduce operates on):
 * no intermediate bucket and no per-parameter accumulation kernels on the framework side.  `max_ctas` as for
 * gpblur_svgp_param_stage. */
int gpblur_svgp_param_stage_backward(const gpblur_svgp_params* p, int D, int M, int kind, const double* stage_grad,
                                     const float* g_kl, float* grad_bucket, int accumulate, int max_ctas,
                                     void* stage, size_t stage_bytes, void* stream);

/* Expected log-likelihood part of the ELBO.
 * Replaces DeepApproximateMLL(VariationalELBO(likelihood, model, num_data))(dist, y) built at
 * /root/reference/forecast_denoising.py:87-89 (GaussianLikelihood.expected_log_prob, sum over the
 * event dim / L, minus KL / num_data):
 *   elbo[b] = (1/L) sum_l -1/2 [ ((y-mean)^2 + var)/noise + log noise + log 2pi ] - kl / num_data
 * mean, var, y [B, L]; raw_noise [1]; kl [1] -> elbo [B]. */
int gpblur_elbo_forward(const float* mean, const float* var, const float* y, const float* raw_noise,
                        const float* kl, float num_data, long long B, int L, float* elbo,
                        void* stream);

/* Backward of gpblur_elbo_forward: g_elbo [B] -> g_mean, g_var [B, L], g_raw_noise [1], g_kl [1].
 * `scratch` must hold at least B floats. */
int gpblur_elbo_backward(const float* mean, const float* var, const float* y, const float* raw_noise,
                         const float* g_elbo, float num_data, long long B, int L, float* g_mean,
                         float* g_var, float* g_raw_noise, float* g_kl, float* scratch,
                         void* stream);

/* The same in ONE launch: the block that takes the last ticket does the final reduction.  `ticket`: a device word that
 * is 0 before the first call; the kernel leaves it at 0 (concurrent calls need distinct words).  B >= 1. */
int gpblur_elbo_backward_fused(const float* mean, const float* var, const float* y, const float* raw_noise,
                               const float* g_elbo, float num_data, long long B, int L, float* g_mean,
                               float* g_var, float* g_raw_noise, float* g_kl, float* scratch,
                               unsigned* ticket, void* stream);

/* Raw Philox4x32-10 words for elements offset .. offset+n-1 (bit-exactness probe): out [n, 4]. */
int gpblur_philox_bits(uint64_t seed, uint64_t offset, uint32_t stream_id, long long n,
                       uint32_t* out, void* stream);
/* Standard normals with the sampler's counter layout: out [n]. */
int gpblur_philox_normal(uint64_t seed, uint64_t offset, uint32_t stream_id, long long n,
                         float* out, void* stream);

/* Elementwise reparameterised sample used between DeepGP layers
 * (gpytorch DeepGPLayer: Normal(mean, var.sqrt()).rsample()): out = mean + sqrt(var) * eps. */
int gpblur_rsample_forward(const float* mean, const float* var, long long n, uint64_t seed,
                           uint64_t offset, uint32_t stream_id, float* out, void* stream);
int gpblur_rsample_backward(const float* var, const float* g_out, long long n, uint64_t seed,
                            uint64_t offset, uint32_t stream_id, float* g_mean, float* g_var,
                            void* stream);

/* Dense ScaleKernel covariance of kind `kind` for the exact-GP model (/root/reference/denoising_model/GPModel.py:10-13):
 * x1 [n1, D], x2 [n2, D], raw_lengthscale [D] (ard != 0) or [1] -> out [n1, n2].  gpblur_covariance_alpha also takes
 * raw_alpha [1], read only for GPBLUR_KERNEL_RQ (NULL then: GPBLUR_EINVAL); gpblur_covariance passes NULL. */
int gpblur_covariance(const float* x1, const float* x2, long long n1, long long n2, int D, int kind,
                      const float* raw_lengthscale, int ard, const float* raw_outputscale, float* out, void* stream);
int gpblur_covariance_alpha(const float* x1, const float* x2, long long n1, long long n2, int D, int kind,
                            const float* raw_lengthscale, int ard, const float* raw_outputscale, const float* raw_alpha,
                            float* out, void* stream);

/* Backward of gpblur_covariance (what autograd computes through the kernel evaluation when the exact GP of
 * /root/reference/denoising_model/GPModel.py:4-13 is trained): g_out [n1, n2] -> g_x1 [n1, D] (nullable), g_x2 [n2, D]
 * (nullable; when x2 is the same tensor as x1 the caller adds the two), g_raw_lengthscale [D] (ard) or [1],
 * g_raw_outputscale [1].  `scratch`: gpblur_covariance_backward_scratch_bytes(n1, n2, D, kind) bytes, 256-byte
 * aligned. */
size_t gpblur_covariance_backward_scratch_bytes(long long n1, long long n2, int D, int kind);
int gpblur_covariance_backward(const float* x1, const float* x2, long long n1, long long n2, int D, int kind,
                               const float* raw_lengthscale, int ard, const float* raw_outputscale,
                               const float* g_out, float* g_x1, float* g_x2, float* g_raw_lengthscale,
                               float* g_raw_outputscale, void* scratch, size_t scratch_bytes, void* stream);
/* The same with raw_alpha [1] and g_raw_alpha [1] (both read / written only for GPBLUR_KERNEL_RQ, which needs them). */
int gpblur_covariance_backward_alpha(const float* x1, const float* x2, long long n1, long long n2, int D, int kind,
                                     const float* raw_lengthscale, int ard, const float* raw_outputscale,
                                     const float* raw_alpha, const float* g_out, float* g_x1, float* g_x2,
                                     float* g_raw_lengthscale, float* g_raw_outputscale, float* g_raw_alpha,
                                     void* scratch, size_t scratch_bytes, void* stream);

/* Debug / test probes into the workspace of the last forward on (ws): copies device-to-device.
 * which: 0 = L (fp64 [Mp,Mp]), 1 = Linv (fp64 [Mp,Mp]), 2 = Kzz+jitter (fp64 [Mp,Mp]),
 *        3 = A (fp32 [N,Mp]), 4 = phase timestamps of the M x M kernels (uint64 ns [32]),
 *        5 = W (fp32 [N,Mp], after a backward), 6 = folded upstream gradients g_mu, g_var (fp32 [2,N], after a backward).
 *        Returns the padded inducing count Mp via *mp. */
int gpblur_debug_fetch(int which, long long N, int D, int M, const void* ws, void* out,
                       size_t out_bytes, int* mp, void* stream);

/* ---- the steps on either side of the GP blur in one training step (SURVEY section 8 (f), ranks 1 and 2) ----------
 * blur application (replaces denoise_model_2.add_gp_noise's `x + self.proj_up(eps_gp.permute(1, 2, 0))`,
 * /root/reference/denoising_model/denoise_model_2.py:36-38; proj_up = nn.Linear(1, d)):
 *   out[n, :] = x[n, :] + mean[n] * w_up + b_up          x, out [N, D] row-major, mean [N], w_up, b_up [D]
 * backward: g_out [N, D] -> g_mean [N], g_w [D], g_b [D] (the gradient of x is g_out itself).
 * loss assembly (replaces /root/reference/forecast_denoising.py:84, 87-89, 102-104):
 *   final[n] = h[n, :] . w_f + b_f                        h = rows (b, p) of a [B', P, D] view: h + b * h_bstride + p * D
 *   scalars  = [loss, mse, mll_error]:  mse = mean_n (y[n] - final[n])^2,  mll_error = -mean_b elbo[b] (elbo [B]),
 *              loss = mse + clip(lam, 0, 0.005) * mll_error            (y, elbo, lam nullable: their terms are 0)
 * backward: g_final [N] (nullable), g_loss, g_mse (device scalars, nullable) -> g_h [N, D] (contiguous), g_w [D],
 *   g_b [1], g_elbo [B], g_lam [1]; torch.clip passes the gradient of lam where 0 <= lam <= 0.005.
 * `scratch`: gpblur_step_scratch_floats(D) floats; `ticket`: a zeroed device word the kernel leaves at 0. */
size_t gpblur_step_scratch_floats(int D);
int gpblur_blur_apply_forward(const float* x, const float* mean, const float* w_up, const float* b_up, long long N,
                              int D, float* out, void* stream);
int gpblur_blur_apply_backward(const float* g_out, const float* mean, const float* w_up, long long N, int D,
                               float* g_mean, float* g_w, float* g_b, float* scratch, unsigned* ticket,
                               void* stream);
int gpblur_loss_forward(const float* h, long long h_bstride, int P, const float* w_f, const float* b_f, const float* y,
                        const float* elbo, long long B, const float* lam, long long N, int D, float* final_out,
                        float* scalars, float* scratch, unsigned* ticket, void* stream);
int gpblur_loss_backward(const float* h, long long h_bstride, int P, const float* w_f, const float* y,
                         const float* final_in, const float* scalars, const float* lam, const float* g_final,
                         const float* g_loss, const float* g_mse, long long B, long long N, int D, float* g_h,
                         float* g_w, float* g_b, float* g_elbo, float* g_lam, float* scratch, unsigned* ticket,
                         void* stream);

/* ---- window sampler on the device (SURVEY section 8 (f), rank 4) -------------------------------------------------
 * Replaces the per-window host materialisation of /root/reference/Utils/base_train.py:67-97 (sample_train_val_test:
 * one .iloc slice per sampled window) and the per-batch .to(device) of /root/reference/train.py:160-161.
 * table [rows, F] fp32 row-major: the encoder-input columns of the (id, time)-ordered series, entities back to back;
 * target [rows]: the target column; starts [B] int64: first table row of each window of T = time_steps rows
 * (< 0: the window stays zero-filled, as the reference's pre-zeroed arrays do when max_samples exceeds the number of
 * valid sampling locations).  Outputs: enc [B, n_enc, F] (`enc_inputs`), dec [B, T - n_enc - pred_len, F]
 * (`dec_inputs`, may be NULL when empty), y [B, pred_len] (`outputs[:, -pred_len:, :]`).  Bit-exact copies. */
int gpblur_window_gather(const float* table, const float* target, long long rows, int F, const long long* starts,
                         long long B, int T, int n_enc, int pred_len, float* enc, float* dec, float* y, void* stream);

/* ---- core of the ATA attention head (SURVEY section 8 (f), rank 3) ------------------------------------------------
 * Replaces /root/reference/forecasting_models/ATA.py:53-65 (two topk(k = 1) poolings, einsum / sqrt(d_k), softmax,
 * einsum) as called from /root/reference/modules/multi_head_attention.py:49-51.  The score matrix is rank one after
 * the pooling; scores / attn [B, H, Lq, Lk] are never materialised.
 *   qp [B, H, Lq, G], kp [B, H, Lk, G]  the multi-scale conv outputs as the reference reshapes them (G = 4 d_k),
 *   v  element (b, h, j, e) at v + b v_sb + h v_sh + j v_sl + e (the [B, Lk, H, DV] memory of `v_s`), DV <= 64,
 *   scale = 1 / sqrt(d_k);   ctx [B, Lq, H, DV] (= context.transpose(1, 2): what multi_head_attention.py:95 makes
 *   contiguous);  saved for the backward: q_pool / q_arg / lse [B, H, Lq], k_pool / k_arg [B, H, Lk].
 * backward: g_ctx [B, Lq, H, DV] -> g_qp, g_kp (pooled gradient at the arg-max element of each group, zeros
 * elsewhere: topk's backward), g_v [B, Lk, H, DV].  16-byte aligned qp / kp / g_qp / g_kp when G % 4 == 0. */
int gpblur_ata_forward(const float* qp, const float* kp, const float* v, long long v_sb, long long v_sh, long long v_sl,
                       int B, int H, int Lq, int Lk, int G, int DV, float scale, float* ctx, float* q_pool,
                       float* k_pool, int* q_arg, int* k_arg, float* lse, void* stream);
int gpblur_ata_backward(const float* g_ctx, const float* ctx, const float* v, long long v_sb, long long v_sh,
                        long long v_sl, const float* q_pool, const float* k_pool, const int* q_arg, const int* k_arg,
                        const float* lse, int B, int H, int Lq, int Lk, int G, int DV, float scale, float* g_qp,
                        float* g_kp, float* g_v, void* stream);
/* The same core for the head's conv stacks evaluated as ONE convolution (nf filter stacks as channel groups of a
 * [B, nf * C, L] output, C = H * d_k) instead of nf convolutions + torch.cat(dim = 0) (ATA.py:50-54): qp / kp / g_qp /
 * g_kp are [B, nf * C, Lq | Lk] buffers and every group is read / written at the place the cat would have put it, so
 * the results equal the plain entry points on the concatenated tensor.  Needs (C * Lq) % G == 0 and (C * Lk) % G == 0. */
int gpblur_ata_forward_fused_stacks(const float* qp, const float* kp, const float* v, long long v_sb, long long v_sh,
                                    long long v_sl, int B, int H, int Lq, int Lk, int G, int DV, int nf, float scale,
                                    float* ctx, float* q_pool, float* k_pool, int* q_arg, int* k_arg, float* lse,
                                    void* stream);
int gpblur_ata_backward_fused_stacks(const float* g_ctx, const float* ctx, const float* v, long long v_sb,
                                     long long v_sh, long long v_sl, const float* q_pool, const float* k_pool,
                                     const int* q_arg, const int* k_arg, const float* lse, int B, int H, int Lq, int Lk,
                                     int G, int DV, int nf, float scale, float* g_qp, float* g_kp, float* g_v,
                                     void* stream);


/* ---- data-parallel exchange: one-shot all-reduce of the flat gradient bucket over NVLink peer memory -------------
 * (one node, one process per GPU; replaces the all-reduce a torch DistributedDataParallel wrapper would issue for the
 * GP parameters - the reference itself trains on one device.)  Every rank allocates one communication buffer of
 * gpblur_peer_comm_bytes(n) with gpblur_peer_alloc, publishes the 64-byte IPC handle to its peers (any side channel:
 * torch.distributed all_gather_object, MPI, ...), maps theirs with gpblur_peer_open, and calls gpblur_peer_allreduce
 * once per step with the `world` pointers in RANK order (comm[rank] = its own buffer): bucket <- scale * sum over ranks,
 * summed in rank order (bit-identical on every rank).  The kernel is self-synchronising (flags in peer memory, a
 * device-resident step counter): it can be captured in a CUDA graph, and it traps instead of hanging if a peer never
 * arrives.  `bucket` must be 16-byte aligned; world <= 16.  These two functions allocate / free device memory. */
size_t gpblur_peer_comm_bytes(long long n);
int gpblur_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int gpblur_peer_open(const unsigned char* handle64, void** ptr);
int gpblur_peer_close(void* ptr);
int gpblur_peer_free(void* ptr);
int gpblur_peer_allreduce(float* bucket, long long n, int world, int rank, void* const* comm, float scale,
                          void* stream);

/* Developer probe: register a device buffer (>= 32 KB, zero-filled by the caller) that CTA 0 of the tensor-core
 * point kernels fills with clock64 event stamps (scripts/tc2_trace.py); NULL switches tracing off (default). */
int gpblur_debug_set_trace(void* device_buffer);

/* Optional per-stage timing for bench.py's roofline: while enabled, every launch is bracketed with CUDA
 * events on its own stream.  gpblur_profile_collect synchronises on the recorded events, writes the
 * accumulated milliseconds / launch counts per stage (order: mm_fwd, point_fwd, point_bwd, gram, wx,
 * mm_bwd, elbo_fwd, elbo_bwd, dx, sg_reduce; n >= 10) and clears the records. */
int gpblur_profile_enable(int on);
int gpblur_profile_collect(double* ms, unsigned long long* counts, int n);

/* Count of kernel launches issued by this library in this process (for bench.py's gpu_launches). */
unsigned long long gpblur_launch_count(void);
const char* gpblur_last_cuda_error(void);
const char* gpblur_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GPBLUR_H_ */
