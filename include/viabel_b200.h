/* libviabel_b200 -- C ABI of the B200-native hot path for jhuggins/viabel.
 *
 * The reference (pure Python, /root/reference/viabel) has no FFI of its own; its seams
 * are Python call signatures.  Each entry point below names the reference call it sits
 * under (file:line relative to the reference tree).  INTEGRATION.md shows the ctypes
 * binding a viabel maintainer would add.
 *
 * Conventions
 *  - every function returns 0 on success or a negative VB_ERR_* code; vb_last_error()
 *    returns a thread-local message for the last failure;
 *  - all array arguments are DEVICE pointers unless the name ends in `_host`;
 *  - matrices are row-major; `ld*` is the row pitch in elements;
 *  - no hidden allocation: scratch memory comes from the caller, sized by the matching
 *    *_workspace_bytes() query (256-byte aligned);
 *  - work is enqueued on `stream` and is asynchronous with respect to the host.
 */
#ifndef VIABEL_B200_H_
#define VIABEL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define VB_OK 0
#define VB_ERR_INVALID_ARG (-1)   /* -> ValueError   */
#define VB_ERR_UNSUPPORTED (-2)   /* -> NotImplementedError */
#define VB_ERR_CUDA (-3)          /* -> RuntimeError */
#define VB_ERR_WORKSPACE (-4)     /* -> RuntimeError (workspace too small) */
#define VB_ERR_NUMERIC (-5)       /* -> ValueError (e.g. all weights zero) */

/* variational families (viabel/approximations.py) */
#define VB_FAMILY_MF_GAUSSIAN 0   /* MFGaussian :192-251 */
#define VB_FAMILY_MF_STUDENT 1    /* MFStudentT :254-312 */

/* link functions of the built-in GLM model plugins (the reference evaluates user Python
 * code at models.py:27-39; these are the GPU-resident replacements) */
#define VB_LINK_LOGISTIC 0        /* log sigmoid(y * x.theta),  y in {-1,+1} */
#define VB_LINK_PROBIT 1          /* log Phi(y * x.theta),      y in {-1,+1} */
#define VB_LINK_GAUSSIAN 2        /* -0.5*((y - x.theta)*aux_s)^2 + log(aux_s), aux_s = 1/sigma_s */

/* objectives (viabel/objectives.py) */
#define VB_OBJ_EXCLUSIVE_KL 0       /* ExclusiveKL :154-168, entropy branch */
#define VB_OBJ_EXCLUSIVE_KL_PATH 1  /* ExclusiveKL use_path_deriv=True :156-159 */
#define VB_OBJ_ALPHA 2              /* AlphaDivergence :440-463 */

const char* vb_last_error(void);
int vb_version(void);
int vb_device_sm_count(void);

/* ---------------------------------------------------------------------------------------
 * Base draws.  Replaces numpy RandomState.randn / standard_t / chisquare at
 * approximations.py:216, :274, :345-347.  Philox4x32-10, counter = element index + offset,
 * so any sub-range can be regenerated and every rank draws identical values.
 * quantize: 0 = full precision; 1 = round each draw to bfloat16 (8-bit mantissa); 2 = round to
 * float16 (11-bit mantissa).  Quantised draws are exact operands of the tensor-core fast path.
 * ------------------------------------------------------------------------------------- */
int vb_philox_normal_f64(double* out, int64_t n, uint64_t seed, uint64_t offset, int quantize,
                         cudaStream_t stream);
int vb_philox_normal_f32(float* out, int64_t n, uint64_t seed, uint64_t offset, int quantize,
                         cudaStream_t stream);
int vb_philox_chisquare_f64(double* out, int64_t n, double df, uint64_t seed, uint64_t offset,
                            cudaStream_t stream);
int vb_philox_student_t_f64(double* out, int64_t n, double df, uint64_t seed, uint64_t offset,
                            int quantize, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Mean-field families: var_param = [mu(d), log_sigma(d)] (approximations.py:185-189).
 * ------------------------------------------------------------------------------------- */
/* theta[s,:] = mu + exp(log_sigma) * base[s,:]        (MFGaussian.sample :212-216,
 *                                                      MFStudentT.sample :270-274) */
int vb_mf_sample_f64(const double* var_param, const double* base, double* theta, int64_t S, int d,
                     cudaStream_t stream);
/* out[i] = log q(x[i,:]; var_param)                   (log_density :231-236, :281-286) */
int vb_mf_log_density_f64(const double* var_param, const double* x, int64_t n, int d, int family,
                          double df, double* out, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * GLM model plugin, float64 exact path.  One sweep over this rank's N observations:
 *   z[n,s]   = sum_j X[n,j] theta[s,j]
 *   out_ll[s]  = sum_n loglik(y_n, z[n,s])                             (always)
 *   out_gmu[j] = sum_n X[n,j] sum_s w[s] dloglik/dz[n,s]               (want_grad)
 *   out_ge[j]  = sum_n X[n,j] sum_s w[s] dloglik/dz[n,s] base[s,j]     (want_grad)
 * i.e. the S x N contraction X.Theta^T of the user's log_density (models.py:27-39) fused
 * with the link function and the back-projection that autograd's reverse sweep performs
 * (objectives.py:167, :448).  w == NULL means all ones; aux == NULL unless the link needs it.
 * Outputs are per-rank partial sums (the caller all-reduces them when N is sharded).
 * ------------------------------------------------------------------------------------- */
size_t vb_glm_sweep_workspace_bytes(int64_t N, int d, int64_t S);
int vb_glm_sweep_f64(const double* X, int64_t ldx, const double* y, int64_t N, int d, int link,
                     const double* theta, const double* base, const double* w, const double* aux,
                     int64_t S, int want_grad, double* out_ll, double* out_gmu, double* out_ge,
                     void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * GLM model plugin, tensor-core fast path (logistic link; tolerance 1e-4 relative).
 * Same contract and outputs (float64 sums) as vb_glm_sweep_f64, but the two contractions run
 * as tcgen05.mma on fp16 hi+lo operand splits fed by TMA (the two correction products of the first contraction on
 * e5m2 copies, kind::f8f6f4), with fp32 accumulators in TMEM.
 *
 * vb_glm_fast_create: one-off preprocessing of the model data into `model_mem` (1024-byte
 *   aligned device memory of vb_glm_fast_model_bytes(N,d) bytes, owned by the caller and kept
 *   alive for the lifetime of the handle): y*X split into fp16 hi and lo, zero padded.
 *   absmax_host (optional, HOST pointer) receives max|y*X|; values above 3e4 do not fit the
 *   fp16 operand range and are rejected with VB_ERR_UNSUPPORTED (use the float64 path), as is
 *   a NaN or infinite entry.
 * vb_glm_fast_sweep: S <= 256 samples per call.  want_grad bit 0: gradients wanted; bit 1: only
 *   sum_s ll[s] is needed (every out_ll[s] then receives the mean, plain ExclusiveKL).  `debug`
 *   (optional, device, 49152 floats per CTA + 128 int64) receives per-phase clock64 timestamps of
 *   CTA 0 in its 128 int64 after the floats.
 *   The kernel runs CTA pairs (tcgen05 cta_group::2, clusters of 2); a device that cannot
 *   schedule them gets VB_ERR_UNSUPPORTED (use the float64 path).
 * Workspace and model_mem must be 1024-byte aligned.
 * ------------------------------------------------------------------------------------- */
size_t vb_glm_fast_model_bytes(int64_t N, int d);
size_t vb_glm_fast_workspace_bytes(int64_t N, int d, int64_t S);
int vb_glm_fast_create(void** handle, const double* X, int64_t ldx, const double* y, int64_t N, int d,
                       int link, void* model_mem, size_t model_bytes, float* absmax_host,
                       cudaStream_t stream);
int vb_glm_fast_destroy(void* handle);
int vb_glm_fast_sweep(void* handle, const double* theta, const double* base, const double* w,
                      int64_t S, int want_grad, double* out_ll, double* out_gmu, double* out_ge,
                      void* workspace, size_t workspace_bytes, float* debug, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Objective assembly for mean-field families on "GLM likelihood + iid Gaussian prior"
 * models (objectives.py:154-168 and :440-463; gradients per SURVEY.md App. A.1).
 *
 * vb_mf_alpha_weights_f64: lw[s] = ll[s] + logprior(theta_s) - log q(theta_s); m = max lw;
 *   w[s] = exp(alpha*(lw[s]-m)); value = log(mean w)/alpha + m          (:456-459)
 * vb_mf_objective_finish_f64: value[0] and grad[2d] from the (all-reduced) sweep sums.
 *   For VB_OBJ_ALPHA pass the weights used in the sweep; otherwise w = NULL.
 *   The ExclusiveKL value is summed over blocks of 8 samples in a fixed order through
 *   vb_mf_objective_finish_workspace_bytes(S) bytes of workspace (VB_ERR_WORKSPACE below;
 *   not used, and may be NULL, for VB_OBJ_ALPHA or without value and logp).
 * ------------------------------------------------------------------------------------- */
int vb_mf_alpha_weights_f64(const double* var_param, const double* theta, const double* base,
                            const double* ll, int64_t S, int d, int family, double df,
                            double prior_sd, double alpha, double* lw, double* w, double* value,
                            cudaStream_t stream);
int vb_mf_objective_finish_f64(const double* var_param, const double* theta, const double* base,
                               const double* ll, const double* gmu, const double* ge,
                               const double* w, int64_t S, int d, int family, double df,
                               double prior_sd, int objective, double alpha, double* value,
                               double* grad, double* logp, void* workspace, size_t workspace_bytes,
                               cudaStream_t stream);
size_t vb_mf_objective_finish_workspace_bytes(int64_t S);

/* ---------------------------------------------------------------------------------------
 * Optimiser steps fused with the parameter update (optimization.py:188-197 RMSProp,
 * :308-326 Adam incl. the first-step aliasing quirk, objectives.py:57-59 update).
 * `first` != 0 on the first call after reset_state().  direction may be NULL.
 * ------------------------------------------------------------------------------------- */
int vb_rmsprop_step_f64(double* var_param, const double* grad, double* nu, double* direction,
                        int64_t P, double lr, double beta, double jitter, int first,
                        cudaStream_t stream);
int vb_adam_step_f64(double* var_param, const double* grad, double* m, double* nu,
                     double* direction, int64_t P, double lr, double beta1, double beta2,
                     double jitter, int first, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Peer-memory communicator (one process per GPU, NVLink / NVSwitch peer stores).  Replaces nothing in the
 * reference (single process); it is the exchange step of the data-sharded path (SURVEY.md 8(e)): the per-rank
 * sweep sums [ll(S), gmu(d), ge(d)] are summed with a one-shot all-reduce INSIDE the step's last kernel.
 *   vb_comm_create : allocates this rank's exchange buffer (cudaMalloc, 2 parities x world slots of slot_bytes)
 *                    and writes its 64-byte CUDA IPC handle to handle_out (HOST pointer);
 *   vb_comm_connect: all_handles = world x 64 bytes (HOST), rank order -- the caller all-gathers them with
 *                    whatever transport it has (torch.distributed in viabel_b200/parallel.py);
 *   vb_comm_connect_ptrs / vb_comm_buffer: the same for several ranks driven by one process;
 *   vb_comm_allreduce_sum_f64: in-place sum of n <= slot_bytes/8 doubles, summed in rank order on every
 *                    rank (bit-identical results everywhere); stream-ordered, no host synchronisation;
 *   vb_comm_error  : 1 if a collective gave up waiting for a peer (4 s), else 0 (synchronises the device).
 * ------------------------------------------------------------------------------------- */
#define VB_COMM_HANDLE_BYTES 64
int vb_comm_create(void** comm, int rank, int world, size_t slot_bytes, unsigned char* handle_out);
int vb_comm_connect(void* comm, const unsigned char* all_handles);
int vb_comm_connect_ptrs(void* comm, void* const* peer_ptrs);
void* vb_comm_buffer(void* comm);
int vb_comm_allreduce_sum_f64(void* comm, double* buf, int64_t n, cudaStream_t stream);
int vb_comm_error(void* comm);
int vb_comm_destroy(void* comm);

/* ---------------------------------------------------------------------------------------
 * Fused ELBO-gradient step: the three calls of the reference loop (optimization.py:95-98)
 *     value, grad = objective(var_param)              objectives.py:154-168, :440-463
 *     direction   = sgo.descent_direction(grad)       optimization.py:188-197 (RMSProp), :308-326 (Adam)
 *     var_param   = objective.update(var_param, lr * direction)        objectives.py:57-59
 * for ExclusiveKL (entropy or path-derivative form) or AlphaDivergence with a mean-field family on a GLM plugin,
 * enqueued with no host round trip.  ExclusiveKL is three kernels: [draw + reparameterise + operand pack] ->
 * [sweep] -> [partial reduction + cross-rank all-reduce through `comm` + value + gradient + optimiser +
 * histories].  AlphaDivergence is five: [draw + pack] -> [forward-only sweep] -> [ll reduction + all-reduce of
 * the S log-likelihoods + log weights + alpha weights + value] -> [weighted sweep] -> [the last kernel above,
 * with the alpha gradient].  Everything that changes from step to step (the draw-stream position, "first step"
 * of the optimiser, history slot) lives in `counters` on the device, so a captured CUDA graph of one call can
 * be replayed.
 *
 * Draws: ExclusiveKL: element i of step t is element counters[2] + t * (S*d rounded up to even) + i of the
 * family's Philox stream (vb_philox_normal_f64 / vb_philox_student_t_f64), t = counters[0].  AlphaDivergence:
 * the draws of step t are elements 0 .. S*d-1 of the stream of key seeds[t % seed_len] (a fresh seed per
 * iteration, objectives.py:455); the config's seed and counters[2] are not used.  With inject_base != 0 the
 * caller's `base` is used instead (parity by draw injection).
 * Errors: VB_ERR_INVALID_ARG for a non-finite or zero alpha, or AlphaDivergence without injection and without
 * seeds (seeds == NULL or seed_len <= 0); VB_ERR_WORKSPACE for a workspace below vb_mf_step_workspace_bytes.
 * ------------------------------------------------------------------------------------- */
typedef struct {
  int32_t family;        /* VB_FAMILY_MF_*                                             */
  int32_t objective;     /* VB_OBJ_EXCLUSIVE_KL, VB_OBJ_EXCLUSIVE_KL_PATH or VB_OBJ_ALPHA */
  int32_t S, d;          /* Monte Carlo samples, model dimension                        */
  int32_t optimizer;     /* 0: none (value + gradient only), 1: RMSProp, 2: Adam        */
  int32_t quantize;      /* draw quantisation, as vb_philox_normal_f64                  */
  int32_t inject_base;   /* != 0: `base` is an input                                    */
  int32_t reserved;
  double df;             /* MFStudentT degrees of freedom                               */
  double prior_sd;       /* iid N(0, prior_sd^2) prior of the GLM plugin (inf: flat)    */
  double lr;             /* learning rate                                               */
  double beta1;          /* RMSProp beta / Adam beta1                                   */
  double beta2;          /* Adam beta2                                                  */
  double jitter;
  uint64_t seed;         /* Philox key of the family's draw stream (ExclusiveKL)        */
  double alpha;          /* VB_OBJ_ALPHA: the divergence's alpha (finite, != 0)         */
} vb_step_config;

typedef struct {
  double* var_param;     /* [2d]  in/out (updated when optimizer != 0)                  */
  double* opt_m;         /* [2d]  Adam momentum (NULL otherwise)                        */
  double* opt_nu;        /* [2d]  RMSProp / Adam second-moment state                    */
  uint64_t* counters;    /* [4]   [0] steps taken (history index), [1] optimiser steps taken,
                          *       [2] stream offset of step 0 (caller-set), [3] reserved  */
  double* base;          /* [S,d] base draws of the step (out; in when inject_base)     */
  double* theta;         /* [S,d] out                                                   */
  double* value;         /* [1]   out                                                   */
  double* grad;          /* [2d]  out                                                   */
  double* logp;          /* [S]   out, optional: model log density per sample           */
  double* direction;     /* [2d]  out, optional: descent direction                      */
  double* value_hist;    /* [hist_len] optional: value_hist[step]                       */
  double* param_hist;    /* [ring, 2d] optional ring of the iterates after the update: row step % ring */
  double* grad_hist;     /* [ring, 2d] optional ring of the gradients                   */
  double* dir_hist;      /* [ring, 2d] optional ring of the descent directions          */
  int64_t hist_len, ring;
  const uint64_t* seeds; /* [seed_len] VB_OBJ_ALPHA without injection: Philox key of step t is
                          *       seeds[t % seed_len], read on the device when the step runs */
  int64_t seed_len;
} vb_step_buffers;

typedef struct {
  /* tensor-core path: handle of vb_glm_fast_create and its workspace; or NULL for the float64 path */
  void* fast_handle;
  void* fast_workspace;
  size_t fast_workspace_bytes;
  /* float64 path: the arguments of vb_glm_sweep_f64; sweep_workspace holds vb_glm_sweep_workspace_bytes
   * (rounded up to 256) + (S + 2d) * 8 bytes */
  const double* X;
  int64_t ldx;
  const double* y;
  int64_t N;
  int32_t link;
  int32_t reserved;
  void* sweep_workspace;
  size_t sweep_workspace_bytes;
} vb_step_model;

/* The workspace carries state between calls (the block tickets of the reducing kernels): zero it once before the
 * first call and hand the same buffer to every later call of the same engine.  Its size covers every objective. */
size_t vb_mf_step_workspace_bytes(int S, int d);
int vb_mf_step_glm(const vb_step_config* cfg, const vb_step_buffers* buf, const vb_step_model* model,
                   void* comm, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * GLM plugin: derivatives of the log-LIKELIHOOD at one point theta[d] (the caller adds the prior's part), for
 * the control-variate ExclusiveKL estimators (objectives.py:170-273), which take them from autograd:
 *   out_grad[d]      = grad f(theta)            `grad_f(m_mean)`             :203, :221
 *   out_hvp[K,d]     = H v_k for V[K,d]         `make_hvp(f_model)(m_mean)`  :220, :238, :256   (K in 0..4 or 8)
 *   out_hessian[d,d] = H (optional)             `hessian(f_model)(m_mean)`   :200-204
 *   out_ll[1]        = f(theta) (optional)
 * Gradient and HVPs are ONE pass over X; the Hessian is a weighted SYRK on the FP64 tensor pipe.
 * Logistic and probit links.
 * ------------------------------------------------------------------------------------- */
size_t vb_glm_point_workspace_bytes(int64_t N, int d, int K, int want_hessian);
int vb_glm_point_f64(const double* X, int64_t ldx, const double* y, int64_t N, int d, int link,
                     const double* theta, const double* V, int K, double* out_ll, double* out_grad,
                     double* out_hvp, double* out_hessian, void* workspace, size_t workspace_bytes,
                     cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Sample moments of x[n,d] (row-major, pitch ldx): the sample branch of wasserstein_bounds
 * (diagnostics.py:137-141) and the covariance all_diagnostics takes from np.cov (diagnostics.py:58-59).
 *   mean[d]; m2[d], m4[d] = sum_n (x_nj - mean_j)^2, ^4 (both or neither); cov[d,d] = np.cov(x.T) (optional,
 *   1/(n-1) normalisation, FP64 tensor-pipe SYRK).  Deterministic (fixed summation order).
 * ------------------------------------------------------------------------------------- */
size_t vb_sample_moments_workspace_bytes(int64_t n, int d, int want_cov);
int vb_sample_moments_f64(const double* x, int64_t n, int d, int64_t ldx, double* mean, double* m2, double* m4,
                          double* cov, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Device-side convergence statistics of FASO / RAABBVI on the iterate ring written by the fused step
 * (vb_step_buffers.param_hist: row t % ring holds the iterate after step t).  `end` is the physical row one past
 * the newest iterate; a window of W rows is rows end-W .. end-1 (mod ring), oldest first.
 *   vb_faso_rhat_f64  : max over parameters of the split-R-hat of the last W iterates, for nwin <= 16 window sizes
 *                       at once (windows_host: HOST array) -- _mc_diagnostics.py:124-184, optimization.py:551-563;
 *   vb_ring_mean_f64  : column means (and optionally sum (x-mean)^2) of a window -- the iterate average
 *                       (optimization.py:563, :568) and np.var(ddof=1) of MCSE (:119);
 *   vb_faso_center_f64: the window minus `mean`, zero padded to m rows, layout [m, P] -- the input of the
 *                       FFT autocovariance (_mc_diagnostics.py:21-37; the FFT is a cuFFT call made by the host side);
 *   vb_faso_ess_f64   : Geyer's initial positive / monotone sequence ESS of every parameter from the autocovariances
 *                       acov[t][p] = scale * acov_raw[t * ld + p] (_mc_diagnostics.py:56-99).  acov_raw is overwritten.
 * ------------------------------------------------------------------------------------- */
size_t vb_faso_rhat_workspace_bytes(int P, int nwin);
int vb_faso_rhat_f64(const double* hist, int64_t ring, int P, int64_t end, const int64_t* windows_host, int nwin,
                     double jitter, double* rhat_max, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int vb_ring_mean_f64(const double* hist, int64_t ring, int P, int64_t end, int64_t W, double* mean, double* css,
                     cudaStream_t stream);
int vb_faso_center_f64(const double* hist, int64_t ring, int P, int64_t end, int64_t W, int64_t m, const double* mean,
                       double* centered, cudaStream_t stream);
int vb_faso_ess_f64(double* acov_raw, int64_t ld, double scale, int64_t n_draw, int P, double* ess, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * DISInclusiveKL (objectives.py:283-416), forward-only in the model.
 *   vb_dis_bisection_f64: the ESS bisection on the tempering epsilon (:338-366) in one launch.  log_prior / log_p /
 *     log_q: [S]; w[S] receives exp(eps log_prior + (1 - eps) log_p - log_q) at the final midpoint (not max-shifted,
 *     as the reference); out4 = [eps (snapped to 0 / max_eps when that end point never moved), ESS, 1 if all weights
 *     are zero (the reference raises ValueError), sum w].
 *   vb_mf_score_f64: value[1] = -sum_r c_r log q(x_{i_r}; var_param), grad[2d] = its gradient wrt [mu, log sigma]
 *     (:405-416 differentiates approx.log_density at FIXED samples), c_r = scale * w[r] (w NULL: 1), i_r = idx[r]
 *     (idx NULL: r), x: [*, d].  Workspace: vb_mf_score_workspace_bytes(d).
 *   vb_mvt_score_f64: the same score for the full-rank MultivariateT (either reparameterisation: the score depends on
 *     var_param and the fixed rows only), grad[d + d(d+1)/2].  L^-1 on the device, then Y = (x - mu) L^-T, V = Y L^-1
 *     and the packed-triangle cotangent on the FP64 tensor pipe (about 3 n d^2 flops plus the d^3 / 3 of the
 *     inverse).  Workspace: vb_mvt_score_workspace_bytes(n, d), O(d^2 + n d).
 *   vb_lr_score_f64: the same score for LRGaussian, grad[2d + d k]; P = [C^-1 | -C^-1 B^T D^-1] (k x (k + d)), C C^T =
 *     I + B^T D^-2 B, may be NULL when k = 0.  About 8 n d k flops, nothing of size d x d.  Workspace:
 *     vb_lr_score_workspace_bytes(n, d, k), O(n (d + k)).
 *   All three: deterministic (fixed summation orders, no atomics), no host synchronisation; idx entries must lie in
 *   the rows of x (not checked on the device).
 * ------------------------------------------------------------------------------------- */
int vb_dis_bisection_f64(const double* log_prior, const double* log_p, const double* log_q, int64_t S,
                         double eps_guess, double max_eps, double ess_target, int max_its, double* w,
                         double* out4, cudaStream_t stream);
size_t vb_mf_score_workspace_bytes(int d);
int vb_mf_score_f64(const double* var_param, const double* x, const int64_t* idx, const double* w, double scale,
                    int64_t n, int d, int family, double df, double* value, double* grad, void* workspace,
                    size_t workspace_bytes, cudaStream_t stream);
size_t vb_mvt_score_workspace_bytes(int64_t n, int d);
int vb_mvt_score_f64(const double* var_param, const double* x, const int64_t* idx, const double* w, double scale,
                     int64_t n, int d, double df, double* value, double* grad, void* workspace, size_t workspace_bytes,
                     cudaStream_t stream);
size_t vb_lr_score_workspace_bytes(int64_t n, int d, int k);
int vb_lr_score_f64(const double* var_param, const double* P, const double* x, const int64_t* idx, const double* w,
                    double scale, int64_t n, int d, int k, double* value, double* grad, void* workspace,
                    size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Mean-field families on a plugin WITHOUT a fused sweep (targets, hierarchical regression, user models): reduce the
 * per-sample model gradients G[S,d] to gmu[j] = sum_s w_s G[s,j] and ge[j] = sum_s w_s G[s,j] base[s,j] (w NULL: 1) --
 * the inputs of vb_mf_objective_finish_f64; in the reference this is autograd's reverse sweep through
 * mu + sigma * eps (approximations.py:212-216 under objectives.py:161-167).
 * ------------------------------------------------------------------------------------- */
int vb_mf_reduce_grads_f64(const double* G, const double* w, const double* base, int64_t S, int d, double* gmu, double* ge,
                           cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * GLM plugin, PER-SAMPLE gradients (full-rank / low-rank / flow families: models.py:27-39 under autograd in the
 * reference).  The two GEMMs are vb_gemm_f64; this is the link step between them on a row chunk A[Nc,S] = y.(X_c
 * Theta^T): ll_accum[s] += sum_n loglik(A[n,s]) (deterministic), A[n,s] <- y_n dloglik/da in place.
 * ------------------------------------------------------------------------------------- */
size_t vb_glm_link_workspace_bytes(int64_t Nc, int S);
int vb_glm_link_f64(double* A, const double* y, int64_t Nc, int S, int link, double* ll_accum, void* workspace,
                    size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Product-target model plugins (north_star: "Gaussian/Student-t targets"): log density and per-sample gradient of
 * kind 0: sum_j N(theta_j; loc_j, scale_j), kind 1: sum_j t_df(theta_j; loc_j, scale_j) at theta[S,d].  In the
 * reference these are user Python log densities under autograd (models.py:27-39; tests/test_objectives.py:18-19).
 * log_norm_const is the theta-independent part (the caller's closed form); grad may be NULL (forward only, as
 * DISInclusiveKL needs).  logp[S], grad[S,d].
 * ------------------------------------------------------------------------------------- */
int vb_target_logp_grad_f64(const double* theta, int64_t S, int d, int kind, const double* loc, const double* scale,
                            double df, double log_norm_const, double* logp, double* grad, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Streaming log-weights for vi_diagnostics (convenience.py:136-179 samples_and_log_weights): for a mean-field
 * family and a product target (target_kind 0: sum_j N(theta_j; loc_j, scale_j), 1: sum_j t_{target_df}(theta_j;
 * loc_j, scale_j)) one kernel regenerates draw i = elements offset + i*d .. + d-1 of the family's Philox stream,
 * reparameterises and writes lw[i] = log p(theta_i) - log q(theta_i).  theta_out (optional, [n,d]) also stores the
 * samples; leave it NULL at scale (n = 1e8, d = 256 would be 204.8 GB).
 * ------------------------------------------------------------------------------------- */
int vb_mf_target_log_weights_f64(const double* var_param, int64_t n, int d, int family, double df, uint64_t seed,
                                 uint64_t offset, int quantize, int target_kind, const double* target_loc,
                                 const double* target_scale, double target_df, double* lw, double* theta_out,
                                 cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Float64 GEMM on the FP64 tensor pipe with fused scalings (the building block of the full-rank path):
 *   C[m,n] = ( alpha * sum_k A'(m,k) kscale[k] B'(k,n) ) * rowscale[m] / (divm[m] + divn[n]) + bias[n]
 *   A'(m,k) = trans_a ? A[k*lda + m] : A[m*lda + k];  B'(k,n) = trans_b ? B[n*ldb + k] : B[k*ldb + n];
 *   kscale / rowscale / bias / (divm, divn) are optional (NULL).
 * ------------------------------------------------------------------------------------- */
int vb_gemm_f64(int trans_a, int trans_b, int M, int N, int K, double alpha, const double* A, int64_t lda,
                const double* B, int64_t ldb, double* C, int64_t ldc, const double* kscale, const double* rowscale,
                const double* bias, const double* divm, const double* divn, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Full-rank MultivariateT (approximations.py:322-382, _distributions.py:7-38) and its objectives
 * (objectives.py:154-164, :443-460).  var_param = [mu(d), row-major lower triangle of F], L = tril(F,-1) +
 * diag(exp(diag F)), Sigma = L L^T.  The caller eigen-decomposes Sigma = V diag(w) V^T (cuSOLVER) between
 * vb_mvt_sigma_f64 and the rest; V is row-major with eigenvectors in its COLUMNS.
 *   vb_mvt_unpack_f64     L[d,d], half_logdet[1] = sum_i F_ii (= the entropy up to df-only constants, :351-354)
 *   vb_mvt_sigma_f64      Sigma = scale * L L^T                                   (mean_and_cov :359-362 uses df/(df-2))
 *   vb_mvt_transform_f64  P = (z / u) V, theta = mu + (P . sqrt(w)) V^T = mu + (z / u) sqrtm(Sigma), zu2[s] = |z_s/u_s|^2,
 *                         u_s = sqrt(chi2_s / df)                                 (sample :342-349)
 *   vb_mvt_objective_f64  value[1], grad[d + d(d+1)/2] of ExclusiveKL (entropy form) / AlphaDivergence from the
 *                         model's f[S], G[S,d] at theta: the sqrtm / Cholesky-parameter VJPs as five GEMMs.
 *                         VB_OBJ_EXCLUSIVE_KL_PATH (use_path_deriv=True, objectives.py:156-159): value = -mean(f - log q)
 *                         at var_param held fixed, gradient = the same VJPs of G + diag(kappa) Y without the entropy
 *                         term, Y = (theta - mu) Sigma^+ with the 1e-10 eigenvalue floor of log_density (:26-28),
 *                         kappa_s = (df + d) / (df + delta_s), delta_s = sum of P[s,k]^2 over w_k > 1e-10.  Needs
 *                         vb_mvt_path_workspace_bytes(S, d) of workspace (2 S + 3 d doubles more); VB_ERR_WORKSPACE below.
 *   vb_mvt_log_density_f64  multivariate_t_logpdf with the 1e-10 eigenvalue floor of the pseudo-inverse (:26-30)
 * ------------------------------------------------------------------------------------- */
int vb_mvt_unpack_f64(const double* var_param, int d, double* L, double* half_logdet, cudaStream_t stream);
int vb_mvt_sigma_f64(const double* L, int d, double scale, double* Sigma, cudaStream_t stream);
size_t vb_mvt_transform_workspace_bytes(int S, int d);
int vb_mvt_transform_f64(const double* var_param, const double* z, const double* chi2, double df, int S, int d,
                         const double* w, const double* V, double* P, double* theta, double* zu2, void* workspace,
                         size_t workspace_bytes, cudaStream_t stream);
size_t vb_mvt_objective_workspace_bytes(int S, int d);
size_t vb_mvt_path_workspace_bytes(int S, int d);
int vb_mvt_objective_f64(const double* L, const double* half_logdet, const double* w, const double* V,
                         const double* P, const double* zu2, const double* f, const double* G, int S, int d,
                         double df, int objective, double alpha, double* value, double* grad, void* workspace,
                         size_t workspace_bytes, cudaStream_t stream);
size_t vb_mvt_log_density_workspace_bytes(int64_t n, int d);
int vb_mvt_log_density_f64(const double* var_param, const double* w, const double* V, const double* x, int64_t n, int d,
                           double df, double* out, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Full-rank MultivariateT in the Cholesky reparameterisation (MultivariateT(..., reparam='cholesky')): theta_s =
 * mu + L z_s / u_s instead of the reference's mu + (z_s / u_s) sqrtm(Sigma) (approximations.py:342-349).  Same
 * distribution, same objectives as functions of var_param, a different per-draw map; no eigensolver, no d x d
 * temporaries, O(S d^2) float64 tensor-core work.  Deterministic (fixed summation order, no atomics).
 *   vb_mvt_chol_transform_f64  theta[S,d] = mu + diag(1/u) z L^T, inv_u[S] = 1/u_s, zu2[S] = |z_s/u_s|^2,
 *                              u_s = sqrt(chi2_s / df)                             (sample :342-349)
 *   vb_mvt_chol_objective_f64  value[1], grad[d + d(d+1)/2] of ExclusiveKL (entropy form, objectives.py:154-164) /
 *                              AlphaDivergence (:443-460) from the model's f[S], G[S,d] at theta:
 *                              grad_mu = c sum_s sv_s G_s,  Fbar[i,j] = c sum_s sv_s G[s,i] z[s,j]/u_s (j < i),
 *                              Fbar[i,i] = (c sum_s sv_s G[s,i] z[s,i]/u_s) L_ii + diag_add;
 *                              c = -1/S, sv = 1, diag_add = -1 (ExclusiveKL) or c = alpha/S, sv_s = exp(lw_s - max lw)^alpha,
 *                              diag_add = c sum_s sv_s (AlphaDivergence).
 *                              VB_OBJ_EXCLUSIVE_KL_PATH (use_path_deriv=True, objectives.py:156-159): value =
 *                              -mean(f - log q) at var_param held fixed; the formulas above with c = -1/S, sv = 1,
 *                              diag_add = 0 and G replaced by G + diag(kappa) Y, Y = diag(1/u) z L^-1, kappa_s =
 *                              (df + d) / (df + zu2_s).  L^-1 is formed on the device (64 x 64 diagonal blocks by
 *                              substitution, then log2 doubling levels), so this form needs
 *                              vb_mvt_chol_path_workspace_bytes(S, d) of workspace (O(d^2 + S d)); VB_ERR_WORKSPACE below.
 * ------------------------------------------------------------------------------------- */
int vb_mvt_chol_transform_f64(const double* var_param, const double* z, const double* chi2, double df, int S, int d,
                              double* theta, double* inv_u, double* zu2, cudaStream_t stream);
size_t vb_mvt_chol_objective_workspace_bytes(int S, int d);
size_t vb_mvt_chol_path_workspace_bytes(int S, int d);
int vb_mvt_chol_objective_f64(const double* var_param, const double* z, const double* inv_u, const double* zu2,
                              const double* f, const double* G, int S, int d, double df, int objective, double alpha,
                              double* value, double* grad, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Streaming log-weights of the full-rank MultivariateT for vi_diagnostics (convenience.py:136-179), never storing
 * samples[n, d].  For global draw i in [first, first + count) of an n_total-draw call: chi2_i = element offset + i of
 * the chi-square stream, z_i[j] = element offset + n_total + (n_total & 1) + i*d + j of the normal stream (what
 * MultivariateT.base_draws(n_total) draws), theta_i = mu + M z_i / u_i, u_i = sqrt(chi2_i / df), with M = L from the
 * packed triangle of var_param when A == NULL (Cholesky mode) or M = A (d x d row-major, sqrtm mode: A = V diag(sqrt w)
 * V^T formed by the caller).  log q_i is the closed form in |z_i / u_i|^2; lw[i - first] = log p(theta_i) - log q_i for
 * target_kind 0 (sum_j N(theta_j; loc_j, scale_j)) or 1 (sum_j t_{target_df}(theta_j; loc_j, scale_j)), -log q_i for
 * target_kind -1.  theta_out[count, d] (optional) receives theta, so that the caller can add any model's log p.
 * Deterministic: a slice equals the same draws of a longer call bit for bit.  Workspace does not depend on n.
 * ------------------------------------------------------------------------------------- */
size_t vb_mvt_target_log_weights_workspace_bytes(int d);
int vb_mvt_target_log_weights_f64(const double* var_param, const double* A, int64_t n_total, int64_t first,
                                  int64_t count, int d, double df, uint64_t seed, uint64_t offset, int target_kind,
                                  const double* target_loc, const double* target_scale, double target_df, double* lw,
                                  double* theta_out, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Streaming log-weights of the low-rank LRGaussian (Sigma = B B^T + D^2, D = diag(exp(log_sigma)), var_param =
 * [mu(d), log_sigma(d), B(d,k) row-major]) for vi_diagnostics, never storing samples[n, d].  For global draw i in
 * [first, first + count) of an n_total-draw call: z_i[l] = element offset + i*k + l and eps_i[j] = element
 * offset + n_total*k + ((n_total*k) & 1) + i*d + j of the normal stream (what LRGaussian.base_draws(n_total) draws),
 * theta_i = mu + B z_i + sigma * eps_i.  With u_i = [z_i, eps_i], log q_i = -1/2 (d log 2 pi + |u_i|^2 - |P u_i|^2)
 * - sum_j log sigma_j + sum_l log P_ll, where P (k x (k+d) row-major, formed by the caller) = [C^-1 | -C^-1 B^T D^-1]
 * and C C^T = I + B^T D^-2 B.  P's left k x k block must be the lower-triangular C^-1 with a positive diagonal: half
 * the log-determinant is read from that diagonal.  P may be NULL when k = 0.  lw and theta_out as in
 * vb_mvt_target_log_weights_f64.  Deterministic: a slice equals the same draws of a longer call bit for bit.
 * Workspace does not depend on n.
 * ------------------------------------------------------------------------------------- */
size_t vb_lr_target_log_weights_workspace_bytes(int d, int k);
int vb_lr_target_log_weights_f64(const double* var_param, const double* P, int64_t n_total, int64_t first,
                                 int64_t count, int d, int k, uint64_t seed, uint64_t offset, int target_kind,
                                 const double* target_loc, const double* target_scale, double target_df, double* lw,
                                 double* theta_out, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Hierarchical linear regression plugin (BASELINE configs[3]) with per-sample gradients: a grouped contraction
 * (no block-expanded design matrix).  X[N,p], y[N] sorted by group; goff[G+1] device int64 row offsets;
 * theta[S,D], D = G p + p + 2 = [beta (group-major), m, log tau, log sigma]; p <= 32.
 * ------------------------------------------------------------------------------------- */
size_t vb_hier_workspace_bytes(int G, int S);
int vb_hier_logp_grad_f64(const double* X, const double* y, const int64_t* goff, int64_t N, int p, int G,
                          const double* theta, int S, double* out_lp, double* out_grad, void* workspace,
                          size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------
 * Pareto-smoothed importance sampling and divergence-bound moments
 * (viabel/_psis.py:113-209 psislw, :212-332 gpdfitnew, :335-377 gpinv, :380-396 sumlogs;
 *  viabel/diagnostics.py:148-186 divergence_bound).
 *
 * vb_psislw_f64: one column of log-weights lw[n] -> smoothed, normalised log-weights out[n]
 * (out may alias lw = the reference's overwrite_lw; out == NULL computes k-hat and the bound moments [7], [8]
 * only, in ONE pass over lw: 8 bytes of traffic per draw instead of 24).
 * result[16] (device doubles): [0] k-hat (inf when the tail has <= 4 entries), [1] GPD sigma,
 * [2] n2 = tail length, [3] shifted cutoff, [4] log-sum-exp, [5] max(lw), [6] status
 * (0 ok; 1 = the sampled threshold missed, call again with exact=1; 2 = internal overflow),
 * [7] sum(out+lse), [8] sum exp(2(out+lse)) (moments for the CUBO/ELBO bounds), [9] M,
 * [10] candidates examined, [11] 1 if the tail was smoothed (k-hat >= 1/3).
 * tail_idx (optional, [tail capacity]) receives the tail indices in ascending index order
 * and tail_rank their rank (0 = smallest) among the tail values -- ties ranked by index.
 * ------------------------------------------------------------------------------------- */
size_t vb_psis_workspace_bytes(int64_t n, double reff);
int64_t vb_psis_tail_capacity(int64_t n, double reff);
int vb_psislw_f64(const double* lw, double* out, int64_t n, double reff, int exact, double* result,
                  int64_t* tail_idx, int32_t* tail_rank, void* workspace, size_t workspace_bytes,
                  cudaStream_t stream);

/* vb_psislw_batch_f64: every column of an n x m matrix of log-weights smoothed separately, in one launch
 * (viabel/_psis.py:113-209 for 2-D lw, and psisloo :69-110).  Column j starts at lw + j*ld (column-major, ld >= n);
 * one CTA holds one column in shared memory, so n may not exceed vb_psis_batch_max_n(reff) (VB_ERR_UNSUPPORTED
 * above it; the limit falls as reff falls, because the tail length M can reach 0.2 n).  Same results as
 * vb_psislw_f64 on each column: maximum and cutoff bit-equal, the same tail set, ties ranked by index.
 *   out    [n x m, leading dimension ldo >= n] smoothed, normalised log-weights; may be lw itself (with ldo == ld)
 *          or NULL (no write).
 *   khat   [m] k-hat per column (+inf when the tail has <= 4 entries or the column holds a NaN).
 *   result [m][16] or NULL: per-column rows in the layout of vb_psislw_f64's result[] -- [0] k-hat, [1] sigma,
 *          [2] n2, [3] shifted cutoff, [4] log-sum-exp, [5] max, [9] M, [10] n, [11] smoothed; the other slots are 0.
 *   loo    [m] or NULL: log-sum-exp over i of (out_i + (-lw_i)), psisloo's sumlogs(lw_smoothed + log_lik) for
 *          lw = -log_lik.  With out == NULL this makes psisloo one read of the matrix.
 * m == 0 is a no-op.  VB_ERR_INVALID_ARG for n <= 1, m < 0, ld < n, ldo < n (with out), reff <= 0 or a NULL lw /
 * khat; nothing is written then.  No host synchronisation; repeated calls are bitwise equal. */
int64_t vb_psis_batch_max_n(double reff);
int vb_psislw_batch_f64(const double* lw, int64_t ld, int64_t n, int64_t m, double reff, double* out, int64_t ldo,
                        double* khat, double* result, double* loo, cudaStream_t stream);

/* Draw-sharded PSIS (SURVEY.md 8(e)): the n_global log-weights of ONE column are split over `world`
 * ranks, rank r holding n_local consecutive draws starting at global index idx_off.  Same
 * algorithm and results as vb_psislw_f64 (= viabel/_psis.py:113-209), in three stream-ordered
 * stages with ONE fixed-size exchange between the first two (host side: NCCL all-gather); no
 * host synchronisation is needed until result[] is read.
 *   vb_psis_dist_local : threshold + pass A over the local draws, local cutoff, then the rank's
 *                        RECORD (device, vb_psis_dist_record_doubles doubles): [local max, c_r =
 *                        local (M+1)-th largest, log-sum-exp of the draws not in the record,
 *                        count], the rank's top M+1 values (local tail padded with copies of c_r)
 *                        and their GLOBAL indices (int64 bit patterns; -1 for the padding).
 *   vb_psis_dist_global: replicated on every rank, on the `world` records concatenated in rank
 *                        order: global cutoff = (M+1)-th largest of the union, tail ranking, GPD
 *                        fit, smoothed tail, log-sum-exp.  result[] as for vb_psislw_f64
 *                        (status 1 if ANY rank's sampled threshold missed: rerun with exact=1).
 *   vb_psis_dist_apply : pass B over the local draws + scatter of the smoothed tail entries this
 *                        rank owns; result[7], result[8] are this rank's SHARE of the moments
 *                        (sum over ranks = the global moments; rank 0 carries the tail's part).
 * All three take the same workspace (vb_psis_dist_workspace_bytes), which carries the state. */
size_t vb_psis_dist_workspace_bytes(int64_t n_local, int64_t n_global, double reff, int world);
int64_t vb_psis_dist_record_doubles(int64_t n_global, double reff);
int vb_psis_dist_local(const double* lw, int64_t n_local, int64_t idx_off, int64_t n_global, double reff,
                       int world, int exact, double* record, void* workspace, size_t workspace_bytes,
                       cudaStream_t stream);
int vb_psis_dist_global(const double* records, int64_t n_local, int64_t n_global, double reff, int world,
                        double* result, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int vb_psis_dist_apply(const double* lw, double* out, int64_t n_local, int64_t idx_off, int64_t n_global,
                       double reff, int world, int rank, double* result, void* workspace,
                       size_t workspace_bytes, cudaStream_t stream);

/* divergence_bound moments in ONE read of lw after the max (diagnostics.py:148-198), out8 = 8 device doubles:
 * [0] max(lw), [1] sum r, [2] sum lw, [3] scratch, [4] sum (lw - max)^2, [5] sum r^2, with r = exp(lw - max)^alpha.
 * [4] and [5] give the Monte Carlo standard errors mean_and_check_mc_error warns about. */
int vb_divergence_moments_f64(const double* lw, int64_t n, double alpha, double* out8,
                              cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VIABEL_B200_H_ */
