/* libblr_cuda -- C ABI of the B200-native FiniteBLR inference path.
 *
 * This is the drop-in boundary for BayesianLinearRegressors.jl's hot path.  The reference has
 * no FFI of its own (its boundary is Julia method dispatch, SURVEY.md section 8b); each entry
 * point below names the reference method body (file:line under the reference repo) whose work
 * it replaces.  The Julia glue (`julia/src/`) and the Python host mirror
 * (`bayesianlinearregressors.jl_b200/`) bind exactly these symbols; see INTEGRATION.md.
 *
 * Conventions
 *   - plain C types only; every matrix is Float64, column-major (Julia / LAPACK order);
 *   - status return: 0 ok; >0 = LAPACK-style `info` of a failed Cholesky (leading minor of
 *     that order is not positive definite -> LinearAlgebra.PosDefException(info));
 *     <0 = BLR_E_* argument / CUDA / NCCL error, text via blr_last_error(ctx);
 *   - one context drives one GPU (one process per GPU under torchrun, or several contexts in
 *     one Julia process); a context is not re-entrant; every call sets its own device;
 *   - host pointers are borrowed for the duration of the call only (`GC.@preserve`);
 *   - "dev" pointers are device addresses on the context's GPU, borrowed while the handle lives;
 *   - there is NO CPU fallback: without a usable sm_100 device blr_ctx_create fails.
 */
#ifndef BLR_CUDA_H
#define BLR_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BLR_VERSION 100 /* 0.1.0 */

/* error codes (negative) */
#define BLR_E_INVALID (-1)   /* bad argument (shape, null pointer, unknown kind) */
#define BLR_E_CUDA (-2)      /* CUDA runtime error */
#define BLR_E_NCCL (-3)      /* NCCL error / NCCL not loadable */
#define BLR_E_DIM (-4)       /* length(y) != size(X, 2)  (src/bayesian_linear_regression.jl:74) */
#define BLR_E_NODEVICE (-5)  /* no sm_100 device: the product path refuses to run */
#define BLR_E_NOMEM (-6)

/* input layouts: x_as_colvecs, src/bayesian_linear_regression.jl:20-31 */
#define BLR_COLVECS 0 /* D x N column-major: observation contiguous, element (d,n) at n*ld + d */
#define BLR_ROWVECS 1 /* N x D column-major: feature contiguous,     element (n,d) at d*ld + n */

/* precision-matrix kinds of BayesianLinearRegressor.Λw (src/bayesian_linear_regression.jl:11-14) */
#define BLR_LAMBDA_DIAGONAL 0 /* `lambda` = D diagonal entries (LinearAlgebra.Diagonal) */
#define BLR_LAMBDA_DENSE 1    /* `lambda` = D x D symmetric, column-major, leading dim ld (Matrix / Symmetric / PDMat.mat) */

/* observation-noise kinds of FiniteGP.Σy */
#define BLR_NOISE_SCALAR 0 /* Diagonal(Fill(σ², N)) : f(X, 0.1) */
#define BLR_NOISE_VECTOR 1 /* Diagonal(v)           : f(X, Diagonal(v)) */
/* Observation-noise variances must be positive wherever the reference factorises Σy (posterior / logpdf :79, rand :52):
 * a non-positive entry returns info > 0 (-> PosDefException(info), info = its 1-based index when known to this rank,
 * else 1).  mean / var / cov only add diag(Σy) (:37,:42) and accept anything, as the reference does. */
#define BLR_NOISE_DENSE 2  /* dense N x N Σy (the reference's test fixtures, test/test_utils.jl:7-8): small-N side path --
                              Σy is factorised on the device and X, y are whitened before the same Gram kernel runs */

typedef struct blr_ctx blr_ctx;
typedef struct blr_x blr_x;         /* device design matrix (this rank's N-shard) */
typedef struct blr_vec blr_vec;     /* device N-vector (targets y, noise variances σ²) */
typedef struct blr_stats blr_stats; /* packed sufficient statistics [G(DxD) | r(D) | q | ℓ | n] on device */
typedef struct blr_post blr_post;   /* device-resident regressor: mw, chol(Λw) (+ inverse factor), cached for predict */

typedef struct blr_prior {
    const double* mw;     /* host, D */
    int lambda_kind;      /* BLR_LAMBDA_* */
    const double* lambda; /* host */
    int64_t ld;           /* leading dimension for DENSE (>= D); ignored for DIAGONAL */
    int64_t D;            /* length(mw) = size(Λw, 1).  Checked against size(X, 1) / the statistics' dimension by every
                             entry point that takes a prior (BLR_E_DIM on mismatch -- the reference throws
                             DimensionMismatch from `X' * mw`, src/bayesian_linear_regression.jl:33); 0 = unchecked */
} blr_prior;

typedef struct blr_noise {
    int kind;           /* BLR_NOISE_* */
    double scalar;      /* σ² when kind == SCALAR */
    const blr_vec* vec; /* σ²_n when kind == VECTOR (same N partition as X) */
    const double* dense; /* host, N x N symmetric column-major when kind == DENSE (single GPU: couples observations) */
    int64_t dense_ld;    /* leading dimension of `dense` (>= N) */
} blr_noise;

/* ------------------------------------------------------------------ context */
int blr_version(void);
int blr_ctx_create(blr_ctx** out, int device);
int blr_ctx_destroy(blr_ctx* ctx);
const char* blr_last_error(const blr_ctx* ctx);
int blr_ctx_sync(blr_ctx* ctx);
/* cudaStream_t all kernels of this context are launched on (for CUDA-event timing by the host). */
int blr_ctx_stream(blr_ctx* ctx, void** stream_out);
/* Numerical form of the D x D phase and of the factor applications (per context; default BLR_FORM_DIRECT, or the
 * environment variable BLR_FORM=whitened at blr_ctx_create).
 *   BLR_FORM_DIRECT   : L' = chol(Λw + G); `var` / `rand` apply an explicit inverse factor (tensor-core GEMMs).
 *   BLR_FORM_WHITENED : the reference's own evaluation order -- Λεy = chol(Uw⁻ᵀ G Uw⁻¹ + I)
 *                       (src/bayesian_linear_regression.jl:81,86), mεy = Λεy \ (Bt'δy) (:64), T = Λεy.U * Uw (:67),
 *                       m' = mw + Uw \ mεy (:68), and triangular SOLVES `Uw' \ X` in var / cov (:36,:41) and `Uw \ randn`
 *                       in rand (:51); no inverse is formed anywhere.  About 8x the D x D flops and plain-DFMA solves in
 *                       `var`; results agree with the direct form to rounding (DESIGN.md section 2). */
#define BLR_FORM_DIRECT 0
#define BLR_FORM_WHITENED 1
int blr_ctx_set_form(blr_ctx* ctx, int form);
int blr_ctx_get_form(const blr_ctx* ctx, int* form_out);
/* Stream ordering for BORROWED device buffers (blr_x_wrap_device / blr_vec_wrap_device, the *_dev outputs): the context
 * launches on its own non-blocking stream, which does not synchronise with the caller's streams implicitly.
 *   blr_ctx_wait_stream: everything already enqueued on `producer` (cudaStream_t, NULL = legacy default stream) happens
 *                        before any later work of this context  (inputs produced by the caller's kernels);
 *   blr_stream_wait_ctx: everything this context has enqueued happens before later work on `consumer`  (outputs). */
int blr_ctx_wait_stream(blr_ctx* ctx, void* producer);
int blr_stream_wait_ctx(blr_ctx* ctx, void* consumer);
/* number of libblr_cuda kernels launched by this context so far. */
int64_t blr_launch_count(const blr_ctx* ctx);
/* Device-event timings (ms) of the last blr_stats_accumulate / blr_infer* call:
 * out[0]=prep (δ, 1/σ²), out[1]=Gram kernel, out[2]=split reduce, out[3]=factorise+solve, out[4..7]=0. */
int blr_last_timings(blr_ctx* ctx, double* out8);

/* Page-locked host memory for result buffers (D2H at PCIe speed instead of through the driver's pageable staging). */
int blr_host_alloc(blr_ctx* ctx, int64_t bytes, void** out);
int blr_host_free(blr_ctx* ctx, void* p);

/* ------------------------------------------------------------------ multi-GPU (N-sharded observations)
 * One rank per GPU; the only exchange of the path is one sum-allreduce of the packed statistics
 * (SURVEY.md section 8e).  NCCL is dlopen'ed on first use. */
int blr_nccl_unique_id(void* out128);
int blr_comm_init_rank(blr_ctx* ctx, const void* id128, int nranks, int rank);
/* One process driving n GPUs (one context per device, e.g. a Julia session): rank i = ctxs[i]; the communicators are
 * created inside one NCCL group.  blr_stats_allreduce_all is the matching grouped in-place sum of stats[i] on ctxs[i]. */
int blr_comm_init_all(blr_ctx** ctxs, int n);
int blr_comm_destroy(blr_ctx* ctx);

/* ------------------------------------------------------------------ data handles */
int blr_x_upload(blr_ctx* ctx, const double* host, int64_t D, int64_t N, int64_t ld, int layout, blr_x** out);
int blr_x_wrap_device(blr_ctx* ctx, const double* dev, int64_t D, int64_t N, int64_t ld, int layout, blr_x** out);
int blr_x_alloc(blr_ctx* ctx, int64_t D, int64_t N, int layout, blr_x** out);
int blr_x_device_ptr(blr_ctx* ctx, const blr_x* x, double** dev_out, int64_t* ld_out);
int blr_x_free(blr_ctx* ctx, blr_x* x);
int blr_vec_upload(blr_ctx* ctx, const double* host, int64_t n, blr_vec** out);
int blr_vec_wrap_device(blr_ctx* ctx, const double* dev, int64_t n, blr_vec** out);
int blr_vec_alloc(blr_ctx* ctx, int64_t n, blr_vec** out);
int blr_vec_device_ptr(blr_ctx* ctx, const blr_vec* v, double** dev_out);
int blr_vec_download(blr_ctx* ctx, const blr_vec* v, double* host);
int blr_vec_free(blr_ctx* ctx, blr_vec* v);

/* bench-only synthetic generators (counter-based Philox4x32-10; SURVEY.md section 8d):
 *   X ~ N(0,1) iid;  σ²_n = exp(z_n);  y = X' w* + σ_n ε_n  with w* ~ N(0, I_D). */
int blr_x_synth(blr_ctx* ctx, blr_x* x, uint64_t seed, int64_t n_offset);
int blr_vec_synth_noise(blr_ctx* ctx, blr_vec* sigma2, uint64_t seed, int64_t n_offset);
int blr_vec_synth_targets(blr_ctx* ctx, const blr_x* x, const blr_vec* sigma2, uint64_t seed, int64_t n_offset,
                          blr_vec* y);

/* device-resident random Fourier features for BasisFunctionRegressor
 * (replaces ϕ(x) of src/basis_function_regression.jl:41 for ϕ(x) = sqrt(2/D) cos(W x + b)):
 * xin: d_in x N ColVecs; W host D x d_in column-major; b host D; out: new D x N ColVecs handle. */
int blr_x_rff(blr_ctx* ctx, const blr_x* xin, const double* W, const double* b, int64_t D, blr_x** out);
/* the general one-layer device feature map  out = scale * act(W x + b)  (blr_x_rff is act = COS, scale = sqrt(2/D)); any
 * other ϕ (src/basis_function_regression.jl:34-37: an arbitrary callable) stays on the device by producing its output in
 * device memory and handing it over with blr_x_wrap_device + blr_ctx_wait_stream (INTEGRATION.md, "device feature maps"). */
#define BLR_ACT_COS 0
#define BLR_ACT_TANH 1
#define BLR_ACT_RELU 2
#define BLR_ACT_IDENTITY 3
#define BLR_ACT_SIN 4
int blr_x_features(blr_ctx* ctx, const blr_x* xin, const double* W, const double* b, int64_t D, int act, double scale,
                   blr_x** out);
/* Vector-Jacobian product of blr_x_features for a cotangent dΦ (what blr_logpdf_grads.dX_dev holds), so gradients reach the
 * feature map's parameters and inputs (the reference differentiates ϕ with Zygote).  With z_n = W x_n + b and
 * g_dn = dΦ_dn * scale * act'(z_dn)  (act' = -sin, 1 - tanh², 1[z > 0] (0 at z = 0), 1, cos for COS, TANH, RELU, IDENTITY, SIN):
 *   dW = Σ_n g_n x_n'  (host, D x d_in column-major, W's layout)    db = Σ_n g_n  (host, D)    dx_n = W' g_n  (device, d_in x N)
 * W, b, act and scale mean what they mean for blr_x_features (blr_x_rff: act = COS, scale = sqrt(2/D)).
 *   dphi_dev : device, D x N ColVecs, leading dimension ld_dphi >= D;   dxin_dev : device, d_in x N ColVecs, ld_dxin >= d_in.
 * Any output may be NULL (not computed); a call that requests nothing launches nothing.  N == 0 writes zeros to dW and db.
 * BLR_E_INVALID for RowVecs xin, d_in outside 1 .. 384, an unknown act, NULL W / b / dphi_dev, D < 1, or a leading dimension
 * too small.  z is recomputed (the forward saves nothing) and no N x D workspace is used.  With a communicator dW and db are
 * summed over ranks (one all-reduce of D (d_in + 1) doubles, D when only db is requested) and replicated; dxin covers this
 * rank's shard.  Fixed-order sums: repeated
 * calls are bit-identical. */
int blr_x_features_vjp(blr_ctx* ctx, const blr_x* xin, const double* W, const double* b, int64_t D, int act, double scale,
                       const double* dphi_dev, int64_t ld_dphi, double* dW_host, double* db_host, double* dxin_dev, int64_t ld_dxin);

/* ------------------------------------------------------------------ inference
 * replaces __compute_inference_quantities / logpdf / posterior,
 * src/bayesian_linear_regression.jl:55-89, and the reverse-mode derivative of logpdf (blr_logpdf_grad) */
int blr_stats_create(blr_ctx* ctx, int64_t D, blr_stats** out);
int blr_stats_free(blr_ctx* ctx, blr_stats* s);
int blr_stats_zero(blr_ctx* ctx, blr_stats* s);
/* stats += [X S X', X S δ, δ'Sδ, Σ log σ², N] of this shard, δ = y - X'mw, S = diag(1/σ²)
 * (the O(N D²) part of :81-:86 in closed form).  May be called repeatedly (chunked / streamed data). */
int blr_stats_accumulate(blr_ctx* ctx, blr_stats* s, const double* mw_host, const blr_x* x, const blr_vec* y,
                         const blr_noise* noise);
/* Same, from HOST arrays (what a Julia caller holds): the observations are streamed to the device in chunks of
 * `chunk` observations through two staging buffers, copies on a second stream overlapped with the Gram kernel
 * of the previous chunk.  X: D x N (COLVECS) or N x D (ROWVECS) column-major with leading dimension ld;
 * sigma2_host: N noise variances when noise_kind == BLR_NOISE_VECTOR, else ignored.  Pinned host memory
 * gives full PCIe overlap; pageable memory works (staged by the driver). */
int blr_stats_accumulate_host(blr_ctx* ctx, blr_stats* s, const double* mw_host, const double* X, int64_t D, int64_t N,
                              int64_t ld, int layout, const double* y, int noise_kind, double noise_scalar,
                              const double* sigma2_host, int64_t chunk);
/* in-place NCCL sum over ranks; no-op without a communicator. */
int blr_stats_allreduce(blr_ctx* ctx, blr_stats* s);
int blr_stats_allreduce_all(blr_ctx** ctxs, blr_stats** stats, int n);
int blr_stats_device_ptr(blr_ctx* ctx, const blr_stats* s, double** dev_out, int64_t* len_out);
int blr_stats_download(blr_ctx* ctx, const blr_stats* s, double* host);
int blr_stats_upload(blr_ctx* ctx, blr_stats* s, const double* host);
/* posterior + logpdf from reduced statistics (replicated on every rank).  Any output may be NULL.
 *   logpdf_out : 1      log marginal likelihood                                     (:57)
 *   m_post     : D      posterior mean                                              (:68)
 *   T_post     : D x D  upper-triangular factor, T'T = posterior precision, ld = D  (:67)
 *   L_post     : D x D  posterior precision Λw + X S X' (symmetric), ld = D         (:92)
 *   post_out   : device-resident posterior regressor for mean/var/rand              */
int blr_infer_from_stats(blr_ctx* ctx, const blr_prior* prior, const blr_stats* s, double* logpdf_out, double* m_post,
                         double* T_post, double* L_post, blr_post** post_out);
/* zero + accumulate + allreduce + infer_from_stats in one call. */
int blr_infer(blr_ctx* ctx, const blr_prior* prior, const blr_x* x, const blr_vec* y, const blr_noise* noise,
              double* logpdf_out, double* m_post, double* T_post, double* L_post, blr_post** post_out);
/* log marginal likelihood of k observation vectors under one regressor and one set of inputs -- AbstractGPs'
 * `logpdf(fx, Y::AbstractMatrix)`, the form the reference's conformance test calls (test/bayesian_linear_regression.jl:7-9),
 * which with the reference's `logpdf` (:55-58) re-runs __compute_inference_quantities (:72-89) once per column.  Only δy (:84)
 * depends on y: here the Gram pass, the factorisation and the log-determinants run ONCE; every further column costs a share of
 * one skinny pass R = X Σy⁻¹ (Y - X'mw) over X and one forward solve.
 *   Y_dev : device, N x k column-major, leading dimension ldy >= N;   logpdf_out : host, k.
 * Scalar / vector Σy only (dense Σy: BLR_E_INVALID -- loop blr_infer).  Statistics are all-reduced when a communicator is set. */
int blr_logpdf_multi(blr_ctx* ctx, const blr_prior* prior, const blr_x* x, const double* Y_dev, int64_t ldy, int64_t k,
                     const blr_noise* noise, double* logpdf_out);
/* Gradients of the log marginal likelihood (:55-58) with respect to every input, in closed form from the posterior of the same
 * call (type-II maximum likelihood of mw, Λw, Σy, and backpropagation into whatever produced X or y).  With s_n = 1/σ²_n,
 * Q = inverse posterior precision, m' the posterior mean, u = m' - mw and e_n = y_n - x_n'm':
 *   ∂/∂x_n = s_n (e_n m' - Q x_n)    ∂/∂y_n = -s_n e_n    ∂/∂σ²_n = (s_n² (x_n'Q x_n + e_n²) - s_n) / 2
 *   ∂/∂mw  = Λw u                    ∂/∂Λw  = -(Q - Λw⁻¹ + u u') / 2  (the symmetric G with dℓ = <G, dΛw>; its diagonal for
 *                                                                      a Diagonal prior)
 * Any field may be NULL (not computed); a pass over the observations runs only when a per-observation output or the scalar
 * dsigma2 is requested.  logpdf_out (may be NULL) is bit-identical to blr_infer's.  Scalar / vector Σy only (dense Σy:
 * BLR_E_INVALID).  Per-observation outputs cover this rank's shard; the others are replicated on every rank. */
typedef struct blr_logpdf_grads {
    double* dmw;         /* host, D */
    double* dlambda;     /* host: D (BLR_LAMBDA_DIAGONAL) or D x D column-major, ld = D (BLR_LAMBDA_DENSE) */
    double* dsigma2;     /* host, 1 value: BLR_NOISE_SCALAR (summed over all ranks) */
    double* dsigma2_dev; /* device, N: BLR_NOISE_VECTOR (this rank's shard) */
    double* dy_dev;      /* device, N (this rank's shard) */
    double* dX_dev;      /* device, same layout as x (this rank's shard) */
    int64_t ld_dX;       /* >= D (COLVECS) or >= N (ROWVECS) */
} blr_logpdf_grads;
int blr_logpdf_grad(blr_ctx* ctx, const blr_prior* prior, const blr_x* x, const blr_vec* y, const blr_noise* noise,
                    double* logpdf_out, const blr_logpdf_grads* g);
/* Gradients of L = Σ_j c_j ℓ_j, ℓ_j the log marginal likelihood of column j of Y (blr_logpdf_multi), c = weights (host, k;
 * NULL = all ones: a reverse-mode rule passes its cotangent here).  With c̄ = Σ_j c_j, m'_j the posterior mean of column j,
 * M' = [m'_1 .. m'_k], u_j = m'_j - mw, U = [u_1 .. u_k] and e_jn = y_jn - x_n'm'_j (each line the single-column formula summed):
 *   ∂/∂x_n = s_n (Σ_j c_j e_jn m'_j - c̄ Q x_n)    ∂/∂Y[n, j] = -c_j s_n e_jn
 *   ∂/∂σ²_n = (s_n² (c̄ x_n'Q x_n + Σ_j c_j e_jn²) - c̄ s_n) / 2
 *   ∂/∂mw  = Λw U c                                ∂/∂Λw = -(c̄ (Q - Λw⁻¹) + U diag(c) U') / 2  (its diagonal for a Diagonal prior)
 * g is a blr_logpdf_grads whose dy_dev is N x k column-major with leading dimension ldy, like Y_dev; every other field as for
 * blr_logpdf_grad.  logpdf_out (host, k; may be NULL) is bit-identical to blr_logpdf_multi's.  k == 0 writes zeros to every
 * requested output.  The O(N D²) work is one GEMM over [X ; E'] with K = D + k rounded up to 16, so k columns cost about one
 * blr_logpdf_grad call, not k.  Scalar / vector Σy only; per-observation outputs cover this rank's shard, the others are
 * replicated on every rank. */
int blr_logpdf_multi_grad(blr_ctx* ctx, const blr_prior* prior, const blr_x* x, const double* Y_dev, int64_t ldy, int64_t k,
                          const blr_noise* noise, const double* weights, double* logpdf_out, const blr_logpdf_grads* g);

/* ------------------------------------------------------------------ prediction / sampling
 * replaces mean / var / mean_and_var / rand, src/bayesian_linear_regression.jl:33-53,
 * and the weight draw of src/sampling_functions.jl:29,35,44 */
int blr_post_create(blr_ctx* ctx, const blr_prior* prior, int64_t D, blr_post** out); /* factorises Λw once */
int blr_post_free(blr_ctx* ctx, blr_post* p);
int blr_post_dim(const blr_post* p, int64_t* D_out);
/* mean_n = x_n'mw,  var_n = |Uw^-T x_n|² + σ²_n; outputs are host (or device if *_dev) N-vectors; either may be NULL. */
int blr_mean_var(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, double* mean_host,
                 double* var_host);
int blr_mean_var_dev(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, double* mean_dev,
                     double* var_dev);
/* N x N covariance α'α + Σy (cov, :35-38); C host column-major ld = N. */
int blr_cov(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, double* C_host);
/* Y (N x S, column-major) = X'(mw + Uw^-1 Zw) + sqrt(σ²) .* Zy  (:51-52).
 * Zw (D x S) / Zy (N x S) host standard-normal draws in the reference's order, or NULL to draw on
 * device (Philox, `seed`). */
int blr_rand_finite(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, int64_t S, const double* Zw,
                    const double* Zy, uint64_t seed, double* Y_host);
int blr_rand_finite_dev(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, int64_t S,
                        const double* Zw_host, const double* Zy_dev, uint64_t seed, double* Y_dev);
/* W (D x S) = mw .+ Uw \ Z */
int blr_rand_weights(blr_ctx* ctx, blr_post* p, int64_t S, const double* Z, uint64_t seed, double* W_host);
/* out_n = x_n'w for one weight sample (BLRFunctionSample call, src/sampling_functions.jl:17-19) */
int blr_apply_weights(blr_ctx* ctx, const blr_x* x, const double* w_host, double* out_host);

/* ------------------------------------------------------------------ on-box calibration of the fp64 roofline
 * (BASELINE.md: "fp64 peak must be calibrated on-box").  Pure DMMA.8x8x4 issue loop over all SMs and a
 * device-to-device copy; results in TFLOP/s (2 flop per FMA) and GB/s (read + write bytes). */
int blr_calibrate_dmma(blr_ctx* ctx, double* tflops_out);
/* issue-rate probe: `warps_per_sm` warps on every SM, each with `n_acc` (1..32, power of two) independent DMMA chains */
int blr_calibrate_dmma_cfg(blr_ctx* ctx, int warps_per_sm, int n_acc, double* tflops_out);
/* the Gram kernel's consumer instruction mix on a resident shared-memory stage (no TMA, no barriers): hardware TFLOP/s */
int blr_calibrate_gram_inner(blr_ctx* ctx, double* tflops_out);
/* DMMA and DFMA loops side by side on every SM: out[0] = DMMA TFLOP/s, out[1] = DFMA TFLOP/s achieved concurrently */
int blr_calibrate_mixed(blr_ctx* ctx, double* tflops2_out);
int blr_calibrate_dfma(blr_ctx* ctx, double* tflops_out);
int blr_calibrate_hbm(blr_ctx* ctx, double* gbs_out);

#ifdef __cplusplus
}
#endif
#endif /* BLR_CUDA_H */
