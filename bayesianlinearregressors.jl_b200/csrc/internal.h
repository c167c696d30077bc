// Internal declarations shared by the translation units of libblr_cuda.
#pragma once
#include <cuda.h>  // CUtensorMap (type only)
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/blr_cuda.h"

struct blr_x {
    double* p = nullptr;
    int64_t D = 0, N = 0, ld = 0;
    int layout = BLR_COLVECS;
    bool owned = false;
};
struct blr_vec {
    double* p = nullptr;
    int64_t n = 0;
    bool owned = false;
};
// packed statistics: G (D*D, column-major, full symmetric) | r (D) | q | ℓ | n   -> D*D + D + 3 doubles
struct blr_stats {
    double* p = nullptr;
    int64_t D = 0;
    int64_t len() const { return D * D + D + 3; }
    double* G() const { return p; }
    double* r() const { return p + D * D; }
    double* scal() const { return p + D * D + D; }  // q, ℓ, n
};
// device-resident regressor (prior or posterior)
struct blr_post {
    int64_t D = 0;
    double* mw = nullptr;    // D
    double* L = nullptr;     // D x D lower Cholesky factor of Λw (Λw = L L'), column-major; upper part zero
    double* W = nullptr;     // D x D lower, W = inv(L); built lazily for var / rand
    double* Lam = nullptr;   // D x D precision (kept for download)
    double* Wp = nullptr;    // zero-padded copy of W (+ padded mw) in the layout of the TMA predict kernels
    bool has_W = false;
    cudaStream_t stream = nullptr;  // stream the buffers were allocated on (stream-ordered pool)
};

struct blr_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    int64_t launches = 0;
    // scratch
    double* ws = nullptr;  // gram partial workspace
    size_t ws_bytes = 0;
    double* nbuf = nullptr;  // per-observation scratch (s, t = sδ), 2 * npad doubles
    size_t nbuf_bytes = 0;
    double* dinv = nullptr;  // packed inverse diagonal blocks for the wavefront solves
    size_t dinv_bytes = 0;
    double* small = nullptr;  // small device scratch (scalars, block partial sums)
    size_t small_bytes = 0;
    int* d_info = nullptr;
    double* h_in = nullptr;   // page-locked input staging of infer_solve: [mw | diag(Λw) | logdet Λw] in ONE H2D copy
    double* h_res = nullptr;  // page-locked result staging: [info | logpdf | m_post (SMALL_VEC)] -> one sync per inference
    int* d_flags = nullptr;  // wavefront-solve ready flags (one per 64-row block), compared against flag_epoch
    int flag_epoch = 0;
    int* tflags = nullptr;   // ready flags of the fused tiled D x D kernel (one per tile + 2 per block row + abort)
    size_t tflags_n = 0;
    int dxd_occ = 0;         // resident CTAs per SM of dxd_fused_kernel (occupancy query, cached)
    int dxd_legacy = 0;      // BLR_DXD=legacy: round-1 multi-launch D x D phase (A/B and fallback for debugging)
    int form = 0;            // BLR_FORM_DIRECT / BLR_FORM_WHITENED (blr_ctx_set_form, BLR_FORM=whitened): whitened.cu
    cudaEvent_t ev[8] = {};
    bool ev_valid[4] = {};
    // stream-K schedule of the Gram fast path (cached by shape)
    int* sched = nullptr;
    size_t sched_bytes = 0;
    int64_t sched_key[4] = {-1, -1, -1, -1};
    int sched_T = 0, sched_nseg = 0;
    int64_t gram_period_obs = 0;  // observations per L2 period of the Gram kernel (0 = single period; BLR_GRAM_PERIOD_OBS)
    int gram_stages = 0;   // ring depth override for gram_kt == 16 (BLR_GRAM_STAGES = 6)
    int var_small_max = 128;  // marginals: largest D served by the streaming small-D kernel (W in shared memory: 136 KB at D = 128); BLR_VAR_SMALL_MAX in [64, 128]
    int mid_ring = 1;      // K1m: team-of-two-warps ring kernel for 64 < D <= 96 (BLR_MID_RING=0: one padded 128-row tile of K1)
    int small_ring = 1;    // K1s: per-warp TMA ring for 16 < D <= 64, D % 8 == 0, aligned ColVecs (BLR_SMALL_RING=0: register-fed kernel)
    int rand_pp = 1;       // K7: 1 = two consumer groups on alternating point tiles when the draws are SUPPLIED (8.2 ms against 9.6 ms at
                           // D = 512, N* = 2^22, S = 64), single-group kernel for device draws (9.79 ms; two-group 9.97); 0 = always
                           // single-group, 2 = always two-group (BLR_RAND_PP)
    int rand_unfused = 0;  // K7 two-group with device draws: 1 = draw a chunk's normals in a pass of their own (9.83 ms: no gain, the
                           // generator costs the same 1.5 ms on its own) (BLR_RAND_UNFUSED)
    int var_cfg = 1;       // marginals fast path: 1 = <4 x 64 rows, 64 points> (default), 0 = <8 x 64 rows, 32 points> (BLR_VAR_CFG=0)
    int gram_unit = 1;     // homoscedastic noise: run the Gram kernel unscaled and apply 1/σ² in the reduction (BLR_GRAM_UNIT=0: off)
    int gram_cs = 1;       // Gram consumer tiling: 1 = hybrid (column strips, 1 x 8 warps, on off-diagonal tiles), 0 = 2 x 4 (BLR_GRAM_CS)
    int gram_kt = 32;      // observations per pipeline stage of the Gram kernel: 16 or 32 (BLR_GRAM_KT)
    int diag_weight = 0;   // cost of a diagonal-tile stage relative to W_OFF = 64; 0 = auto: 38 for the hybrid tiling, 40 for
                           // 2 x 4 (both measured best; BLR_DIAG_WEIGHT overrides)
    // host-streaming path (blr_stats_accumulate_host): copy stream, two staging slots
    cudaStream_t copy_stream = nullptr;
    double* stage[2] = {nullptr, nullptr};
    size_t stage_bytes = 0;
    cudaEvent_t ev_copied[2] = {}, ev_consumed[2] = {};
    bool stage_used[2] = {false, false};  // ev_consumed[b] has been recorded since the slot was (re)allocated
    cudaEvent_t ev_xstream = nullptr;     // blr_ctx_wait_stream / blr_stream_wait_ctx
    // NCCL (dlopen'ed)
    void* nccl_comm = nullptr;
    int nranks = 1, rank = 0;
};

namespace blr {

// internal status of infer_solve: Σ log σ² is not finite, i.e. some observation-noise variance is <= 0 (or NaN)
constexpr int BLR_INFO_NOISE = 0x7ffffff0;

// layout of blr_ctx::small (doubles)
constexpr int PERIOD_COUNTER_SLOT = 448;  // index into blr_ctx::d_flags (wavefront flags use < 256)
constexpr int SMALL_PREP = 0;        // prep-kernel block partials (2 per block, <= 4096)
constexpr int SMALL_SC = 4096;       // scalars
constexpr int SMALL_VEC = 16384;     // capacity of each D-vector slot (max supported D)
constexpr int SMALL_RHS = 8192;
constexpr int SMALL_MW = SMALL_RHS + SMALL_VEC;
constexpr int SMALL_DTMP = SMALL_MW + SMALL_VEC;
constexpr int SMALL_U = SMALL_DTMP + SMALL_VEC + 8;  // backward-solve output of the fused D x D kernel (8 spare doubles: the
                                                     // staged host inputs [mw | diag Λw | logdet Λw] span SMALL_MW .. +2D+1)
constexpr int SMALL_TOTAL = SMALL_U + SMALL_VEC;

int set_err(blr_ctx* ctx, int code, const std::string& msg);
int cuda_fail(blr_ctx* ctx, cudaError_t e, const char* what);
// stream-ordered allocations for per-call objects (no device-wide synchronisation, memory retained by the pool)
cudaError_t dev_alloc(blr_ctx* ctx, double** p, size_t bytes);
void dev_free(cudaStream_t stream, void* p);
int ensure_ws(blr_ctx* ctx, size_t bytes);
int ensure_nbuf(blr_ctx* ctx, size_t bytes);
int ensure_dinv(blr_ctx* ctx, size_t bytes);
// 0, or the 1-based index of the first non-positive variance (PosDefException info of Diagonal(v)); synchronises
int check_noise_vector(blr_ctx* ctx, const double* v, int64_t N);

#define BLR_CUDA_OK(ctx, call)                                           \
    do {                                                                 \
        cudaError_t _e = (call);                                         \
        if (_e != cudaSuccess) return ::blr::cuda_fail(ctx, _e, #call);  \
    } while (0)
#define BLR_CHECK_LAUNCH(ctx, name)                                             \
    do {                                                                        \
        (ctx)->launches++;                                                      \
        cudaError_t _e = cudaGetLastError();                                    \
        if (_e != cudaSuccess) return ::blr::cuda_fail(ctx, _e, "launch " name); \
    } while (0)
#define BLR_TRY(call)          \
    do {                       \
        int _r = (call);       \
        if (_r != 0) return _r; \
    } while (0)

// ---- gram.cu
// stats += local shard statistics.  s_noise: scalar σ² when sigma2 == nullptr.
int gram_accumulate(blr_ctx* ctx, blr_stats* st, const double* mw_dev, bool mw_is_zero, const blr_x* x,
                    const double* y, const double* sigma2, double sigma2_scalar, bool padded_odd = false);

// ---- gram_small.cu: D <= 64, any layout / alignment; adds this shard's statistics into st.  D <= 16: K0 fused (reads
// y, σ² itself, s / t unused, `partial` is scratch for 2 doubles per CTA); otherwise s, t, partial come from prep_kernel.
bool gram_small_fused(const blr_ctx* ctx, const blr_x* x);
int gram_small(blr_ctx* ctx, blr_stats* st, const blr_x* x, const double* y, const double* sigma2, double sigma2_scalar,
               const double* mw_dev, bool mw_is_zero, const double* s, const double* t, double* partial, int partial_blocks);

// ---- chol_tiled.cu
// inputs / outputs of the finalize step of the fused D x D kernel (all device pointers)
struct DxdFinalize {
    const double* stat_scal;  // q, ℓ, n of the reduced statistics
    const double* mw;         // prior mean
    double* m_post;           // out: mw + u
    const double* logdet_w;   // logdet Λw
    double* sc;               // out: [1] logdet Λ', [2] z'z, [3] logpdf
};
// One cooperative launch: A (lower triangle in) -> Cholesky factor (lower, strict upper zeroed); optionally z = L^-1 z in
// place, u = L^-T z, and the finalize step.  info_dev: 4 device ints, [0] = LAPACK-style info, [1] = noise flag, [3] = abort.
int dxd_fused(blr_ctx* ctx, double* A, int64_t D, int* info_dev, double* z, double* u, const DxdFinalize* fin);

int gram_small_reduce(blr_ctx* ctx, blr_stats* st, const double* P, const double* Pr, int DP, int nblocks, int D, const double* partial,
                      int partial_blocks, double n_obs);  // gram_small.cu
// ---- gram_mid.cu: 64 < D <= 96 (even, aligned ColVecs): two warps own the matrix together, preparation fused in
bool gram_mid_eligible(const blr_ctx* ctx, const blr_x* x, bool padded_odd);
int gram_mid(blr_ctx* ctx, blr_stats* st, const blr_x* x, const double* y, const double* sigma2, double sigma2_scalar,
             const double* mw_dev, bool mw_is_zero, double* partial, bool padded_odd);
int repack_colvecs(blr_ctx* ctx, const double* X, int64_t ld, int64_t D, int64_t n, double* out, int64_t ldo);  // gram.cu

// ---- whitened.cu (the reference's literal numerical form, opt-in: blr_ctx::form == BLR_FORM_WHITENED)
int trsm_lower(blr_ctx* ctx, const double* L, int64_t ldl, int64_t D, double* B, int64_t ldb, int64_t K, bool trans);
int dxd_whitened(blr_ctx* ctx, blr_post* p, const double* Lw, const blr_stats* st, double* rhs, double* usol, const double* mwd,
                 double* sc, int* info_post);
int diag_factor_dense(blr_ctx* ctx, const double* diag_dev, int64_t D, double* Lw);
int solve_alpha(blr_ctx* ctx, const blr_post* p, const blr_x* x, int64_t n0, int64_t n, double* alpha);
int predict_mean_var_literal(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* sigma2, double sigma2_scalar,
                             double* mean_dev, double* var_dev);

// ---- chol.cu
// In-place lower Cholesky of the column-major D x D matrix A (only the lower triangle is read);
// strictly-upper part is zeroed.  *info_dev (device int) receives 0 or the 1-based failing order.
int potrf_lower(blr_ctx* ctx, double* A, int64_t D, int* info_dev);
// synchronising read of ctx->d_info after potrf_lower(..., ctx->d_info): *info_host = LAPACK-style info; error if the
// fused kernel's watchdog fired
int read_info(blr_ctx* ctx, int* info_host);
// W = inv(L) (lower triangular, column-major), strictly-upper part zeroed.
int trtri_lower(blr_ctx* ctx, const double* L, double* W, int64_t D);
// Solve L z = b (forward) then optionally L' u = z (backward); b overwritten.  zz_out (device) = z'z.
int trtri_diag_packed(blr_ctx* ctx, const double* L, int64_t D, double* Dinv);
int trsv_lower_forward(blr_ctx* ctx, const double* L, int64_t D, const double* Dinv, double* b);
int trsv_lower_backward(blr_ctx* ctx, const double* L, int64_t D, const double* Dinv, double* b);
// out[0] = 2 * sum log diag(L)
int logdet_from_chol(blr_ctx* ctx, const double* L, int64_t D, double* out_dev);
int infer_solve(blr_ctx* ctx, const blr_prior* prior, const blr_stats* st, double* logpdf_out, double* m_post,
                double* T_post, double* L_post, blr_post** post_out);
int post_from_prior(blr_ctx* ctx, const blr_prior* prior, int64_t D, blr_post** out);
// Z_j = L^-1 R_j in place (K columns of D contiguous doubles), zz_dev[j] = Z_j'Z_j
int forward_solve_multi(blr_ctx* ctx, const blr_post* p, double* R, int64_t K, double* zz_dev);
int post_ensure_W(blr_ctx* ctx, blr_post* p);
void post_release(blr_post* p);

// ---- predict.cu
int predict_mean_var(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* sigma2, double sigma2_scalar,
                     double* mean_dev, double* var_dev);
int predict_cov(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* sigma2, double sigma2_scalar, double* C_dev);
int sample_weights(blr_ctx* ctx, blr_post* p, int64_t S, const double* Z_dev, double* W_dev);
// noiseless: Y = X'Wsamp alone (no draws made, sigma2 / Zy not read)
int sample_finite(blr_ctx* ctx, const blr_x* x, const double* Wsamp_dev, int64_t S, const double* sigma2,
                  double sigma2_scalar, const double* Zy_dev, uint64_t seed, double* Y_dev, bool noiseless = false);
int apply_weights(blr_ctx* ctx, const blr_x* x, const double* w_dev, double* out_dev);
// C[m, n] = beta * C + Σ_k A[m, k] B[k, n] with arbitrary element strides (small / odd shapes; plain DFMA)
int gemm_generic(blr_ctx* ctx, int64_t M, int64_t Nn, int64_t K, const double* A, int64_t as_m, int64_t as_k,
                 const double* B, int64_t bs_k, int64_t bs_n, double* C, int64_t cs_m, int64_t cs_n, double beta);

// ---- rhs_multi.cu: R_out[j] = X Σy⁻¹ (Y_j - pm) (K x D, column j contiguous), q_out[j] = (Y_j - pm)' Σy⁻¹ (Y_j - pm); pm = X'mw or nullptr
int rhs_multi(blr_ctx* ctx, const blr_x* x, const double* Y, int64_t ldy, int64_t K, const double* sigma2,
              double sigma2_scalar, const double* pm, double* R_out, double* q_out);

// ---- predict_tma.cu
bool predict_fast_eligible(const blr_post* p, const blr_x* x);
bool sample_fast_eligible(const blr_x* x);
struct RandChunk {
    int64_t ldy, ldz, n_global, N_global;
};
int sample_finite_fast(blr_ctx* ctx, const blr_x* x, const double* Wsamp_dev, int64_t S, const double* sigma2,
                       double sigma2_scalar, const double* Zy_dev, uint64_t seed, double* Y_dev, const RandChunk* chunk = nullptr,
                       bool noiseless = false);
int predict_mean_var_fast(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* sigma2, double sigma2_scalar,
                          double* mean_dev, double* var_dev);
// 2-D tiled TMA map of a column-major fp64 matrix (inner x outer, leading dimension ld), 128-byte swizzled boxes
int make_tmap_2d_f64(blr_ctx* ctx, CUtensorMap* out, const double* base, uint64_t inner, uint64_t outer, uint64_t ld,
                     uint32_t box_inner, uint32_t box_outer);

// ---- grad.cu: gradients of the log marginal likelihood from the posterior p of the same call
// e, h by the predict path with zero noise; on exit se = s ⊙ e; dy, dsig (N) and dsig_sum (device scalar) may be null
int grad_obs(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* y, const double* sigma2, double sigma2_scalar,
             double* se, double* var, double* dy, double* dsig, double* dsig_sum);
// u (D scratch) = m' - mw; dmw = Λw u; dlam = -1/2 (Q - Λw⁻¹ + u u') (dense, ld = D; Q read with leading dimension ldq) or its
// diagonal (Q not read).  mw_dev, lam_dev (Diagonal prior only): the prior on the device; dmw / dlam may be null
int grad_prior(blr_ctx* ctx, const blr_prior* prior, blr_post* p, const double* mw_dev, const double* lam_dev, const double* Q,
               int64_t ldq, double* u, double* dmw, double* dlam);
bool grad_x_fast_eligible(const blr_post* p, const blr_x* x, const double* dX, int64_t ld_dX);
// shape of the Q buffer grad_x reads: zero-padded to the pass height and the stage depth of the fast kernel, else D x D
void grad_q_shape(const blr_post* p, bool fast, int64_t* ldq, int64_t* dk);
int grad_q(blr_ctx* ctx, blr_post* p, double* Qp, int64_t ldq, int64_t dk);
// dX = -Q X S + m' se'  in x's layout
int grad_x(blr_ctx* ctx, const blr_post* p, const blr_x* x, const double* Qp, int64_t ldq, int64_t dk, bool fast,
           const double* se, const double* sigma2, double sigma2_scalar, double* dX, int64_t ld_dX);
// rank k (blr_logpdf_multi_grad), L = Σ_j c_j ℓ_j with c = c_dev (device, k), c̄ = cbar; kp = k rounded up to 16.
// U (D x k): column 0 is overwritten with m'_0 - mw, columns 1 .. k-1 = W'Z_j (Z = L⁻¹R of the forward pass); M = mw + U
int grad_means_multi(blr_ctx* ctx, blr_post* p, const double* mw_dev, const double* Z, int64_t k, double* U, double* M);
// XM (N x k scratch) = X'M; mean, var (N scratch) = x_n'm'_0, h_n (only when dsig / dsig_sum); E (kp x N, point-major; may be
// null) = residuals; dY (ld ldy), dsig (N) and dsig_sum (device scalar) may be null
int grad_obs_multi(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* M, int64_t k, int64_t kp, const double* Y, int64_t ldy,
                   const double* sigma2, double sigma2_scalar, const double* c_dev, double cbar, double* XM, double* mean,
                   double* var, double* E, double* dY, double* dsig, double* dsig_sum);
// uc (D scratch) = U c; dmw = Λw U c; dlam = -1/2 (c̄ (Q - Λw⁻¹) + U diag(c) U') or its diagonal; dmw / dlam may be null
int grad_prior_multi(blr_ctx* ctx, const blr_prior* prior, blr_post* p, const double* lam_dev, const double* Q, int64_t ldq,
                     const double* U, int64_t k, const double* c_dev, double cbar, double* uc, double* dmw, double* dlam);
// A (ldq x (dk + kp), Q in its first dk columns) = [-c̄ Q | M diag(c)] in place
int grad_a_multi(blr_ctx* ctx, double* A, int64_t ldq, int64_t dk, int64_t kp, int64_t D, int64_t k, const double* M,
                 const double* c_dev, double cbar);
// dX = S A [X ; E'] in x's layout
int grad_x_multi(blr_ctx* ctx, const blr_post* p, const blr_x* x, const double* A, int64_t ldq, int64_t dk, int64_t k, int64_t kp,
                 bool fast, const double* E, const double* sigma2, double sigma2_scalar, double* dX, int64_t ld_dX);

// ---- synth.cu
int synth_normal(blr_ctx* ctx, double* out, int64_t rows, int64_t cols, int64_t ld, uint64_t seed, uint64_t stream_id,
                 int64_t col_offset);
int synth_noise(blr_ctx* ctx, double* sigma2, int64_t n, uint64_t seed, int64_t n_offset);
int synth_targets(blr_ctx* ctx, const blr_x* x, const double* sigma2, uint64_t seed, int64_t n_offset, double* y);
int affine_features(blr_ctx* ctx, const blr_x* xin, const double* W_dev, const double* b_dev, int64_t D, int act, double scale,
                    double* out, int64_t ldo);
int rff_features(blr_ctx* ctx, const blr_x* xin, const double* W_dev, const double* b_dev, int64_t D, double* out,
                 int64_t ldo);
int transpose_to_colvecs(blr_ctx* ctx, const blr_x* x, double* out, int64_t ldo);

// ---- features_grad.cu: VJP of affine_features for the cotangent dphi (D x N, leading dimension ldp).  dWb (may be null) =
// [dW (D x d_in) | db (D)], column-major, from S point ranges through ws (S x D x (d_in + 1)); with_w = false computes and writes
// only the db part.
// dx (may be null) = W'g, d_in x N with leading dimension lddx.  S from features_vjp_splits.
int features_vjp_splits(const blr_ctx* ctx, int64_t N, int64_t D, int64_t din);
int features_vjp(blr_ctx* ctx, const blr_x* xin, const double* W_dev, const double* b_dev, int64_t D, int act, double scale,
                 const double* dphi, int64_t ldp, double* dWb, double* ws, int S, bool with_w, double* dx, int64_t lddx);

// ---- calib.cu
int calib_dmma(blr_ctx* ctx, double* tflops);
int calib_dfma(blr_ctx* ctx, double* tflops);
int calib_mixed(blr_ctx* ctx, double* tflops2);
int calib_gram_inner(blr_ctx* ctx, double* tflops);  // gram.cu
int calib_dmma_cfg(blr_ctx* ctx, int warps, int nacc, double* tflops);
int calib_hbm(blr_ctx* ctx, double* gbs);

}  // namespace blr
