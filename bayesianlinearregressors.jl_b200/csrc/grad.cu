// Gradients of the log marginal likelihood (reference src/bayesian_linear_regression.jl:55-58) with respect to every input,
// in closed form from the posterior of the same call.  With S = diag(s), s_n = 1/σ²_n, P = Λw + X S X' the posterior precision,
// Q = P⁻¹ = W'W (W = inv(L), P = L L'), m' the posterior mean, u = m' - mw, e_n = y_n - x_n'm' and h_n = x_n'Q x_n:
//
//     ∂ℓ/∂x_n  = s_n (e_n m' - Q x_n)          ∂ℓ/∂y_n = -s_n e_n          ∂ℓ/∂σ²_n = ½ (s_n² (h_n + e_n²) - s_n)
//     ∂ℓ/∂mw   = Λw u                          ∂ℓ/∂Λw  = -½ (Q - Λw⁻¹ + u u')   (symmetric; its diagonal for a Diagonal prior)
//
// (the X and σ² terms by the envelope theorem: the quadratic term of ℓ is the minimum over w of the penalised residual).
// e is computed exactly, from a pass over X with m' -- not expanded from the statistics as q - 2u'r + u'Gu, which cancels at
// high signal-to-noise.  e and h come from the predict path with zero noise (K6 where eligible).
//
// grad_x, the hot path: dX = -Q X S + m' (s ⊙ e)' is a dense GEMM with M = D rows, K = D, N points and a fused epilogue.  It is
// K6 (predict_tma.cu) without the triangle: one persistent CTA per SM on tiles of 64 points, 256-row passes, X fed by 2-D tiled
// TMA boxes with the 128-byte swizzle, columns of the zero-padded Q by 1-D bulk copies, a 4-stage mbarrier ring, DMMA.8x8x4.
// The epilogue scales in registers and stages each 32-row x 8-point block of a warp through shared memory, so that one store
// instruction writes two whole 256-byte column segments of dX (ColVecs: a point's features are contiguous).
//
// Rank k (blr_logpdf_multi_grad): the gradient of L = Σ_j c_j ℓ_j with respect to x_n is s_n [-c̄ Q | M' diag(c)] [x_n ; e_n]
// (c̄ = Σ_j c_j, M' = [m'_1 .. m'_k], e_jn = y_jn - x_n'm'_j): the same GEMM with K = D + kp, the A buffer Q extended by kp =
// k rounded up to 16 columns and, for the stages beyond the padded D, B read by a second tensor map over E (kp x N, point-major)
// with the same box and swizzle.  The epilogue is s_n acc.  e comes exactly from X'M', the noiseless product of the rand path.
#include <cuda.h>
#include <math.h>

#include <algorithm>

#include "common.cuh"
#include "internal.h"

namespace blr {
namespace gk {
constexpr int KT = 16;            // features per stage (one 128-byte swizzle span per point)
constexpr int STAGES = 4;
constexpr int MI = 4;             // 8-row blocks per warp: a warp owns 32 consecutive rows of the pass
constexpr int NP = 64;            // points per tile
constexpr int NI = NP / 8;
constexpr int CONSUMER_WARPS = 8;
constexpr int R = CONSUMER_WARPS * MI * 8;  // 256 rows per pass
constexpr int LDA = R + 4;        // A row stride (doubles): == 4 mod 16, conflict-free fragment loads
constexpr int LDE = MI * 8 + 4;   // epilogue staging stride per point (doubles): 2 * LDE == 8 mod 16, conflict-free fragment stores
constexpr int PRODUCER_WARPS = 4;  // A columns 0-7 | A columns 8-15 | first half of the points | second half
constexpr int THREADS = (CONSUMER_WARPS + PRODUCER_WARPS) * 32;
struct __align__(1024) Stage {
    double b[NP * KT];  // [point][k], 128-byte TMA swizzle (swz128); 1024-byte aligned
    double a[KT * LDA]; // [k][row - r_base]
};
struct Smem {
    Stage st[STAGES];
    double ep[CONSUMER_WARPS][8 * LDE];  // per-warp epilogue staging: 8 points x 32 rows
    unsigned long long full[STAGES];
    unsigned long long empty[STAGES];
};
}  // namespace gk

struct GradXParams {
    const double* Qp;  // ldq x dk, zero outside D x D (rank k: ldq x (dk + kp), A = [-c̄ Q | M' diag(c)])
    int64_t ldq;       // multiple of gk::R
    int dk;            // multiple of gk::KT
    int kp;            // rank k: rows of E, a multiple of gk::KT; 0 for a single column
    int D;
    int64_t N;
    const double* m;       // posterior mean, D
    const double* se;      // s_n e_n, N
    const double* sigma2;  // N, or null: s = s_scalar
    double s_scalar;
    double* dX;
    int64_t ld;
};

// tme: the tensor map over E (rank k); the single-column instantiation does not read it
template <bool MULTI>
__global__ void __launch_bounds__(gk::THREADS, 1) grad_x_tma_kernel(const GradXParams p, const __grid_constant__ CUtensorMap tmx,
                                                                    const __grid_constant__ CUtensorMap tme) {
    using namespace gk;
    extern __shared__ unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(smem_u32(&sm.full[i]), PRODUCER_WARPS * RING_LANES);
            mbar_init(smem_u32(&sm.empty[i]), CONSUMER_WARPS * RING_LANES);
        }
        mbar_fence_init();
    }
    fence_proxy_async();
    __syncthreads();

    const int64_t ntiles = (p.N + NP - 1) / NP;
    const int npass = (int)(p.ldq / R);
    const int nst = p.dk / KT + (MULTI ? p.kp / KT : 0);

    if (warp >= CONSUMER_WARPS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        const int pw = warp - CONSUMER_WARPS;
        int it = 0;
        for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int64_t p0 = tile * NP;
            for (int ps = 0; ps < npass; ++ps) {
                const int r_base = ps * R;
                for (int si = 0; si < nst; ++si, ++it) {
                    const int k0 = si * KT;
                    const int stg = it % STAGES;
                    const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
                    mbar_wait(smem_u32(&sm.empty[stg]), ph ^ 1u);
                    Stage& S = sm.st[stg];
                    const uint32_t bar = smem_u32(&sm.full[stg]);
                    if (pw < 2) {  // 8 columns of Q each, rows r_base .. r_base + R
                        ring_expect(bar, (uint32_t)(KT / 2) * R * 8u, lane);
                        if (lane < KT / 2) {
                            const int kr = pw * (KT / 2) + lane;
                            bulk_g2s(smem_u32(&S.a[kr * LDA]), p.Qp + (int64_t)(k0 + kr) * p.ldq + r_base, (uint32_t)R * 8u, bar);
                        }
                    } else {  // one box {KT features, NP / 2 points}; beyond D or N zero-filled and still counted
                        const int pbase = (pw - 2) * (NP / 2);
                        ring_expect(bar, (uint32_t)(NP / 2) * KT * 8u, lane);
                        if (lane == 0) {
                            if (MULTI && k0 >= p.dk)
                                tma_load_2d(smem_u32(&S.b[pbase * KT]), &tme, k0 - p.dk, (int)(p0 + pbase), bar);
                            else
                                tma_load_2d(smem_u32(&S.b[pbase * KT]), &tmx, k0, (int)(p0 + pbase), bar);
                        }
                    }
                }
            }
        }
        return;
    }

    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    const int g = lane >> 2, kq = lane & 3;
    int boff[4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) boff[kk] = swz128(g, kk * 4 + kq);
    double* ep = sm.ep[warp];
    const int rl = 2 * (lane & 15), pl = lane >> 4;  // epilogue: row pair within the warp's 32 rows, point within a pair
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t p0 = tile * NP;
        for (int ps = 0; ps < npass; ++ps) {
            const int r_base = ps * R;
            double acc[MI][NI][2];
#pragma unroll
            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                for (int ni = 0; ni < NI; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
            for (int si = 0; si < nst; ++si, ++it) {
                const int stg = it % STAGES;
                const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
                mbar_wait(smem_u32(&sm.full[stg]), ph);
                const Stage& S = sm.st[stg];
                const double* Ap = S.a + warp * (MI * 8) + g;
#pragma unroll
                for (int kk = 0; kk < KT / 4; ++kk) {
                    const int kl = kk * 4 + kq;
                    double a[MI], b[NI];
#pragma unroll
                    for (int mi = 0; mi < MI; ++mi) a[mi] = Ap[kl * LDA + mi * 8];
#pragma unroll
                    for (int ni = 0; ni < NI; ++ni) b[ni] = S.b[ni * 8 * KT + boff[kk]];
#pragma unroll
                    for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                        for (int ni = 0; ni < NI; ++ni) dmma884(acc[mi][ni], a[mi], b[ni]);
                }
                ring_release(smem_u32(&sm.empty[stg]), lane);
            }
            // epilogue: dX[row, n] = se_n m'[row] - s_n (Q X)[row, n]; rank k: s_n (A [X ; E'])[row, n]
            const int row = r_base + warp * (MI * 8) + rl;
            const double m0 = !MULTI && row < p.D ? p.m[row] : 0.0, m1 = !MULTI && row + 1 < p.D ? p.m[row + 1] : 0.0;
#pragma unroll
            for (int ni = 0; ni < NI; ++ni) {
#pragma unroll
                for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                    for (int c = 0; c < 2; ++c) ep[(2 * kq + c) * LDE + mi * 8 + g] = acc[mi][ni][c];
                __syncwarp();
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int pt = 2 * q + pl;
                    const int64_t n = p0 + ni * 8 + pt;
                    if (n < p.N && row < p.D) {
                        const double2 v = *reinterpret_cast<const double2*>(&ep[pt * LDE + rl]);
                        const double s = p.sigma2 ? 1.0 / p.sigma2[n] : p.s_scalar;
                        double* dst = p.dX + n * p.ld + row;
                        double o0, o1;
                        if constexpr (MULTI) {
                            o0 = s * v.x;
                            o1 = s * v.y;
                        } else {
                            const double se = p.se[n];
                            o0 = fma(se, m0, -s * v.x);
                            o1 = fma(se, m1, -s * v.y);
                        }
                        if (row + 1 < p.D)
                            *reinterpret_cast<double2*>(dst) = make_double2(o0, o1);
                        else
                            dst[0] = o0;
                    }
                }
                __syncwarp();
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// The per-observation pass: on entry mean = x_n'm', var = h_n; on exit mean = s_n e_n (what grad_x needs).
// dsig_part: one partial sum of ∂ℓ/∂σ²_n per block (scalar noise), reduced in a fixed order by grad_sum_kernel.
__global__ void __launch_bounds__(256) grad_obs_kernel(int64_t N, const double* __restrict__ y, const double* __restrict__ sigma2,
                                                       double sigma2_scalar, double* __restrict__ mean, const double* __restrict__ var,
                                                       double* __restrict__ dy, double* __restrict__ dsig, double* __restrict__ dsig_part) {
    __shared__ double red[32];
    double part = 0.0;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        const double s = 1.0 / (sigma2 ? sigma2[n] : sigma2_scalar);
        const double e = y[n] - mean[n];
        const double d = 0.5 * (s * s * (var[n] + e * e) - s);
        mean[n] = s * e;
        if (dy) dy[n] = -s * e;
        if (dsig) dsig[n] = d;
        part += d;
    }
    if (dsig_part) {
        part = block_sum(part, red);
        if (threadIdx.x == 0) dsig_part[blockIdx.x] = part;
    }
}
__global__ void __launch_bounds__(1024) grad_sum_kernel(const double* __restrict__ part, int n, double* __restrict__ out) {
    __shared__ double red[32];
    double v = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) v += part[i];
    v = block_sum(v, red);
    if (threadIdx.x == 0) *out = v;
}

// dX[d, n] = se_n m'[d] - s_n dX[d, n] in either layout (the generic path's epilogue after gemm_generic wrote Q X)
template <int LAYOUT>
__global__ void __launch_bounds__(256) grad_x_epilogue_kernel(double* __restrict__ dX, int64_t ld, int64_t D, int64_t N,
                                                              const double* __restrict__ m, const double* __restrict__ se,
                                                              const double* __restrict__ sigma2, double s_scalar) {
    const int64_t total = D * N;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        // ColVecs: d fastest (contiguous); RowVecs: n fastest (contiguous)
        const int64_t d = LAYOUT == BLR_COLVECS ? e % D : e / N, n = LAYOUT == BLR_COLVECS ? e / D : e % N;
        double* v = dX + (LAYOUT == BLR_COLVECS ? n * ld + d : d * ld + n);
        const double s = sigma2 ? 1.0 / sigma2[n] : s_scalar;
        *v = fma(se[n], m[d], -s * *v);
    }
}

// u = m' - mw;  Diagonal prior (lam != null): dmw = λ ⊙ u, dlam_i = -½ (Q_ii - 1/λ_i + u_i²) with Q_ii = Σ_k W[k, i]² (W lower);
// a warp per feature, fixed-order sums
__global__ void __launch_bounds__(256) grad_prior_diag_kernel(int D, const double* __restrict__ mpost, const double* __restrict__ mw,
                                                              const double* __restrict__ lam, const double* __restrict__ W,
                                                              double* __restrict__ u, double* __restrict__ dmw, double* __restrict__ dlam) {
    const int lane = threadIdx.x & 31;
    for (int i = blockIdx.x * 8 + (threadIdx.x >> 5); i < D; i += gridDim.x * 8) {
        const double ui = mpost[i] - mw[i];
        double q = 0.0;
        if (dlam)
            for (int k = i + lane; k < D; k += 32) q = fma(W[(int64_t)i * D + k], W[(int64_t)i * D + k], q);
        q = warp_sum(q);
        if (lane == 0) {
            u[i] = ui;
            if (dmw && lam) dmw[i] = lam[i] * ui;
            if (dlam) dlam[i] = -0.5 * (q - 1.0 / lam[i] + ui * ui);
        }
    }
}
// Dense prior: dlam = -½ (Q - Λw⁻¹ + u u')
__global__ void __launch_bounds__(256) grad_prior_dense_kernel(int64_t D, const double* __restrict__ Q, int64_t ldq,
                                                               const double* __restrict__ Li, const double* __restrict__ u,
                                                               double* __restrict__ dlam) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < D * D; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e % D, c = e / D;
        dlam[e] = -0.5 * (Q[c * ldq + r] - Li[e] + u[r] * u[c]);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
bool grad_x_fast_eligible(const blr_post* p, const blr_x* x, const double* dX, int64_t ld_dX) {
    return predict_fast_eligible(p, x) && (ld_dX % 2) == 0 && (reinterpret_cast<uintptr_t>(dX) & 15) == 0;
}

int grad_obs(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* y, const double* sigma2, double sigma2_scalar,
             double* se, double* var, double* dy, double* dsig, double* dsig_sum) {
    const int64_t N = x->N;
    if (N == 0) {
        if (dsig_sum) BLR_CUDA_OK(ctx, cudaMemsetAsync(dsig_sum, 0, sizeof(double), ctx->stream));
        return 0;
    }
    BLR_TRY(predict_mean_var(ctx, p, x, nullptr, 0.0, se, var));
    // the grid depends on N alone: the partial sums, hence the scalar, are the same on every call
    const int grid = (int)std::min<int64_t>((N + 255) / 256, 1024);
    double* part = dsig_sum ? ctx->small + SMALL_PREP : nullptr;
    grad_obs_kernel<<<grid, 256, 0, ctx->stream>>>(N, y, sigma2, sigma2_scalar, se, var, dy, dsig, part);
    BLR_CHECK_LAUNCH(ctx, "grad_obs_kernel");
    if (dsig_sum) {
        grad_sum_kernel<<<1, 1024, 0, ctx->stream>>>(part, grid, dsig_sum);
        BLR_CHECK_LAUNCH(ctx, "grad_sum_kernel");
    }
    return 0;
}

int grad_prior(blr_ctx* ctx, const blr_prior* prior, blr_post* p, const double* mw_dev, const double* lam_dev, const double* Q,
               int64_t ldq, double* u, double* dmw, double* dlam) {
    const int64_t D = p->D;
    cudaStream_t sm = ctx->stream;
    if (prior->lambda_kind == BLR_LAMBDA_DIAGONAL) {
        if (dlam) BLR_TRY(post_ensure_W(ctx, p));
        grad_prior_diag_kernel<<<(int)std::min<int64_t>((D + 7) / 8, ctx->sm_count * 4), 256, 0, sm>>>(
            (int)D, p->mw, mw_dev, lam_dev, dlam ? p->W : nullptr, u, dmw, dlam);
        BLR_CHECK_LAUNCH(ctx, "grad_prior_diag_kernel");
        return 0;
    }
    grad_prior_diag_kernel<<<(int)std::min<int64_t>((D + 7) / 8, ctx->sm_count * 4), 256, 0, sm>>>((int)D, p->mw, mw_dev, nullptr,
                                                                                                    nullptr, u, nullptr, nullptr);
    BLR_CHECK_LAUNCH(ctx, "grad_prior_diag_kernel");
    // Λw (dense upload) and, for dlam, Λw⁻¹ = Ww'Ww from the prior's own factor
    blr_post* pw = nullptr;
    BLR_TRY(post_from_prior(ctx, prior, D, &pw));
    double* Li = nullptr;
    int rc = 0;
    if (dmw) rc = gemm_generic(ctx, D, 1, D, pw->Lam, 1, D, u, 1, D, dmw, 1, D, 0.0);
    if (rc == 0 && dlam) {
        cudaError_t e = dev_alloc(ctx, &Li, (size_t)D * D * sizeof(double));
        if (e != cudaSuccess) rc = cuda_fail(ctx, e, "cudaMallocAsync(Λw⁻¹)");
        if (rc == 0) rc = post_ensure_W(ctx, pw);
        if (rc == 0) rc = gemm_generic(ctx, D, D, D, pw->W, D, 1, pw->W, 1, D, Li, 1, D, 0.0);
        if (rc == 0) {
            grad_prior_dense_kernel<<<(int)std::min<int64_t>((D * D + 255) / 256, ctx->sm_count * 8), 256, 0, sm>>>(D, Q, ldq, Li, u,
                                                                                                                    dlam);
            BLR_CHECK_LAUNCH(ctx, "grad_prior_dense_kernel");
        }
    }
    dev_free(sm, Li);
    post_release(pw);
    return rc;
}

// Q = W'W into the zero-padded ldq x dk buffer (rows >= D and columns >= D are zero)
int grad_q(blr_ctx* ctx, blr_post* p, double* Qp, int64_t ldq, int64_t dk) {
    const int64_t D = p->D;
    BLR_TRY(post_ensure_W(ctx, p));
    if (ldq != D || dk != D) BLR_CUDA_OK(ctx, cudaMemsetAsync(Qp, 0, (size_t)ldq * dk * sizeof(double), ctx->stream));
    return gemm_generic(ctx, D, D, D, p->W, D, 1, p->W, 1, D, Qp, 1, ldq, 0.0);
}

void grad_q_shape(const blr_post* p, bool fast, int64_t* ldq, int64_t* dk) {
    const int64_t D = p->D;
    *ldq = fast ? (D + gk::R - 1) / gk::R * gk::R : D;
    *dk = fast ? (D + gk::KT - 1) / gk::KT * gk::KT : D;
}

int grad_x(blr_ctx* ctx, const blr_post* p, const blr_x* x, const double* Qp, int64_t ldq, int64_t dk, bool fast,
           const double* se, const double* sigma2, double sigma2_scalar, double* dX, int64_t ld_dX) {
    const int64_t D = p->D, N = x->N;
    if (N == 0) return 0;
    const double s_scalar = sigma2 ? 0.0 : 1.0 / sigma2_scalar;
    if (fast) {
        GradXParams gp;
        gp.Qp = Qp;
        gp.ldq = ldq;
        gp.dk = (int)dk;
        gp.D = (int)D;
        gp.N = N;
        gp.m = p->mw;
        gp.se = se;
        gp.sigma2 = sigma2;
        gp.s_scalar = s_scalar;
        gp.dX = dX;
        gp.ld = ld_dX;
        gp.kp = 0;
        const int smem = (int)sizeof(gk::Smem) + 1024;
        BLR_CUDA_OK(ctx, cudaFuncSetAttribute(grad_x_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        CUtensorMap tmx;
        BLR_TRY(make_tmap_2d_f64(ctx, &tmx, x->p, (uint64_t)D, (uint64_t)N, (uint64_t)x->ld, gk::KT, gk::NP / 2));
        const int grid = (int)std::min<int64_t>((N + gk::NP - 1) / gk::NP, ctx->sm_count);
        grad_x_tma_kernel<false><<<grid, gk::THREADS, smem, ctx->stream>>>(gp, tmx, tmx);
        BLR_CHECK_LAUNCH(ctx, "grad_x_tma_kernel");
        return 0;
    }
    // generic path (any layout / alignment): Q X by gemm_generic in column blocks it can address, then the epilogue
    const bool colv = x->layout == BLR_COLVECS;
    const int64_t block = (int64_t)1 << 20;
    for (int64_t a = 0; a < N; a += block) {
        const int64_t nb = std::min(block, N - a);
        const double* Xa = x->p + (colv ? a * x->ld : a);
        double* Ca = dX + (colv ? a * ld_dX : a);
        BLR_TRY(gemm_generic(ctx, D, nb, D, Qp, 1, ldq, Xa, colv ? 1 : x->ld, colv ? x->ld : 1, Ca, colv ? 1 : ld_dX,
                             colv ? ld_dX : 1, 0.0));
    }
    const int grid = (int)std::min<int64_t>((D * N + 255) / 256, (int64_t)ctx->sm_count * 16);
    if (colv)
        grad_x_epilogue_kernel<BLR_COLVECS><<<grid, 256, 0, ctx->stream>>>(dX, ld_dX, D, N, p->mw, se, sigma2, s_scalar);
    else
        grad_x_epilogue_kernel<BLR_ROWVECS><<<grid, 256, 0, ctx->stream>>>(dX, ld_dX, D, N, p->mw, se, sigma2, s_scalar);
    BLR_CHECK_LAUNCH(ctx, "grad_x_epilogue_kernel");
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// Rank k (blr_logpdf_multi_grad): gradients of L = Σ_j c_j ℓ_j, c̄ = Σ_j c_j; U = [u_1 .. u_k] (D x k), M' = mw + U.

// U[:, 0] = m'_0 - mw (columns >= 1 already hold W'Z_j); M'[:, j] = m'_0 for j = 0, else mw + u_j
__global__ void __launch_bounds__(256) grad_means_kernel(int64_t D, int64_t k, const double* __restrict__ mpost,
                                                         const double* __restrict__ mw, double* __restrict__ U, double* __restrict__ M) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < D * k; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e % D;
        if (e < D) {
            U[e] = mpost[r] - mw[r];
            M[e] = mpost[r];
        } else {
            M[e] = mw[r] + U[e];
        }
    }
}

// the per-observation pass: on entry XM[n + j N] = x_n'm'_j; writes e_jn into E (point-major, kp rows, rows >= k zero) when
// E is given, dY[n + j ldy] = -c_j s_n e_jn, and ∂L/∂σ²_n = ½ (s_n² (c̄ h_n + Σ_j c_j e_jn²) - c̄ s_n) (h = var) into dsig and /
// or the per-block partial sums reduced by grad_sum_kernel in a fixed order
__global__ void __launch_bounds__(256) grad_obs_multi_kernel(int64_t N, int k, int kp, const double* __restrict__ XM,
                                                             const double* __restrict__ Y, int64_t ldy, const double* __restrict__ sigma2,
                                                             double sigma2_scalar, const double* __restrict__ c, double cbar,
                                                             const double* __restrict__ var, double* __restrict__ E,
                                                             double* __restrict__ dY, double* __restrict__ dsig,
                                                             double* __restrict__ dsig_part) {
    __shared__ double red[32];
    double part = 0.0;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        const double s = 1.0 / (sigma2 ? sigma2[n] : sigma2_scalar);
        double t = 0.0;
        for (int j = 0; j < k; ++j) {
            const double e = Y[j * ldy + n] - XM[j * N + n];
            t = fma(c[j] * e, e, t);
            if (E) E[n * kp + j] = e;
            if (dY) dY[j * ldy + n] = -c[j] * s * e;
        }
        if (E)
            for (int j = k; j < kp; ++j) E[n * kp + j] = 0.0;
        if (var) {
            const double d = 0.5 * (s * s * fma(cbar, var[n], t) - cbar * s);
            if (dsig) dsig[n] = d;
            part += d;
        }
    }
    if (dsig_part) {
        part = block_sum(part, red);
        if (threadIdx.x == 0) dsig_part[blockIdx.x] = part;
    }
}

// A = [-c̄ Q | M' diag(c)]: Q (the first dk columns, ld ldq) scaled in place, then kp columns c_j m'_j (zero beyond D and k)
__global__ void __launch_bounds__(256) grad_a_multi_kernel(double* __restrict__ A, int64_t ldq, int64_t dk, int64_t kp, int64_t D,
                                                           int64_t k, const double* __restrict__ M, const double* __restrict__ c,
                                                           double cbar) {
    const int64_t total = ldq * (dk + kp);
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e % ldq, col = e / ldq;
        if (col < dk) {
            A[e] = -cbar * A[e];
        } else {
            const int64_t j = col - dk;
            A[e] = (j < k && r < D) ? c[j] * M[j * D + r] : 0.0;
        }
    }
}

// dX[d, n] *= s_n in either layout (the generic rank-k path's epilogue after gemm_generic wrote A [X ; E'])
template <int LAYOUT>
__global__ void __launch_bounds__(256) grad_x_scale_kernel(double* __restrict__ dX, int64_t ld, int64_t D, int64_t N,
                                                           const double* __restrict__ sigma2, double s_scalar) {
    const int64_t total = D * N;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t d = LAYOUT == BLR_COLVECS ? e % D : e / N, n = LAYOUT == BLR_COLVECS ? e / D : e % N;
        double* v = dX + (LAYOUT == BLR_COLVECS ? n * ld + d : d * ld + n);
        *v *= sigma2 ? 1.0 / sigma2[n] : s_scalar;
    }
}

// Diagonal prior (lam != null): dmw_i = λ_i (U c)_i, dlam_i = -½ (c̄ (Q_ii - 1/λ_i) + Σ_j c_j U_ij²); dense prior (lam == null):
// uc = U c only.  A warp per feature, fixed-order sums.
__global__ void __launch_bounds__(256) grad_prior_multi_diag_kernel(int D, int k, const double* __restrict__ U,
                                                                    const double* __restrict__ c, double cbar,
                                                                    const double* __restrict__ lam, const double* __restrict__ W,
                                                                    double* __restrict__ uc, double* __restrict__ dmw,
                                                                    double* __restrict__ dlam) {
    const int lane = threadIdx.x & 31;
    for (int i = blockIdx.x * 8 + (threadIdx.x >> 5); i < D; i += gridDim.x * 8) {
        double q = 0.0;
        if (dlam)
            for (int kk = i + lane; kk < D; kk += 32) q = fma(W[(int64_t)i * D + kk], W[(int64_t)i * D + kk], q);
        q = warp_sum(q);
        if (lane == 0) {
            double a = 0.0, t = 0.0;
            for (int j = 0; j < k; ++j) {
                const double v = U[(int64_t)j * D + i];
                a = fma(c[j], v, a);
                t = fma(c[j] * v, v, t);
            }
            uc[i] = a;
            if (dmw && lam) dmw[i] = lam[i] * a;
            if (dlam) dlam[i] = -0.5 * fma(cbar, q - 1.0 / lam[i], t);
        }
    }
}
// Dense prior: dlam = -½ (c̄ (Q - Λw⁻¹) + U diag(c) U')
__global__ void __launch_bounds__(256) grad_prior_multi_dense_kernel(int64_t D, int64_t k, const double* __restrict__ Q, int64_t ldq,
                                                                     const double* __restrict__ Li, const double* __restrict__ U,
                                                                     const double* __restrict__ c, double cbar,
                                                                     double* __restrict__ dlam) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < D * D; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e % D, cc = e / D;
        double t = 0.0;
        for (int64_t j = 0; j < k; ++j) t = fma(c[j] * U[j * D + r], U[j * D + cc], t);
        dlam[e] = -0.5 * fma(cbar, Q[cc * ldq + r] - Li[e], t);
    }
}

int grad_means_multi(blr_ctx* ctx, blr_post* p, const double* mw_dev, const double* Z, int64_t k, double* U, double* M) {
    const int64_t D = p->D;
    if (k > 1) {
        BLR_TRY(post_ensure_W(ctx, p));
        // u_j = W'Z_j = Q R_j:  (W'Z)[d, j] = Σ_i W[i, d] Z[i, j]
        BLR_TRY(gemm_generic(ctx, D, k - 1, D, p->W, D, 1, Z, 1, D, U + D, 1, D, 0.0));
    }
    grad_means_kernel<<<(int)std::min<int64_t>((D * k + 255) / 256, (int64_t)ctx->sm_count * 8), 256, 0, ctx->stream>>>(
        D, k, p->mw, mw_dev, U, M);
    BLR_CHECK_LAUNCH(ctx, "grad_means_kernel");
    return 0;
}

int grad_obs_multi(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* M, int64_t k, int64_t kp, const double* Y, int64_t ldy,
                   const double* sigma2, double sigma2_scalar, const double* c_dev, double cbar, double* XM, double* mean,
                   double* var, double* E, double* dY, double* dsig, double* dsig_sum) {
    const int64_t N = x->N;
    const bool wsig = dsig || dsig_sum;
    if (N == 0) {
        if (dsig_sum) BLR_CUDA_OK(ctx, cudaMemsetAsync(dsig_sum, 0, sizeof(double), ctx->stream));
        return 0;
    }
    BLR_TRY(sample_finite(ctx, x, M, k, nullptr, 0.0, nullptr, 0, XM, true));
    if (wsig) BLR_TRY(predict_mean_var(ctx, p, x, nullptr, 0.0, mean, var));
    // the grid depends on N alone: the partial sums, hence the scalar, are the same on every call
    const int grid = (int)std::min<int64_t>((N + 255) / 256, 1024);
    double* part = dsig_sum ? ctx->small + SMALL_PREP : nullptr;
    grad_obs_multi_kernel<<<grid, 256, 0, ctx->stream>>>(N, (int)k, (int)kp, XM, Y, ldy, sigma2, sigma2_scalar, c_dev, cbar,
                                                         wsig ? var : nullptr, E, dY, dsig, part);
    BLR_CHECK_LAUNCH(ctx, "grad_obs_multi_kernel");
    if (dsig_sum) {
        grad_sum_kernel<<<1, 1024, 0, ctx->stream>>>(part, grid, dsig_sum);
        BLR_CHECK_LAUNCH(ctx, "grad_sum_kernel");
    }
    return 0;
}

int grad_prior_multi(blr_ctx* ctx, const blr_prior* prior, blr_post* p, const double* lam_dev, const double* Q, int64_t ldq,
                     const double* U, int64_t k, const double* c_dev, double cbar, double* uc, double* dmw, double* dlam) {
    const int64_t D = p->D;
    cudaStream_t sm = ctx->stream;
    const bool diagonal = prior->lambda_kind == BLR_LAMBDA_DIAGONAL;
    if (diagonal && dlam) BLR_TRY(post_ensure_W(ctx, p));
    grad_prior_multi_diag_kernel<<<(int)std::min<int64_t>((D + 7) / 8, ctx->sm_count * 4), 256, 0, sm>>>(
        (int)D, (int)k, U, c_dev, cbar, diagonal ? lam_dev : nullptr, diagonal && dlam ? p->W : nullptr, uc, diagonal ? dmw : nullptr,
        diagonal ? dlam : nullptr);
    BLR_CHECK_LAUNCH(ctx, "grad_prior_multi_diag_kernel");
    if (diagonal) return 0;
    // Λw (dense upload) and, for dlam, Λw⁻¹ = Ww'Ww from the prior's own factor
    blr_post* pw = nullptr;
    BLR_TRY(post_from_prior(ctx, prior, D, &pw));
    double* Li = nullptr;
    int rc = 0;
    if (dmw) rc = gemm_generic(ctx, D, 1, D, pw->Lam, 1, D, uc, 1, D, dmw, 1, D, 0.0);
    if (rc == 0 && dlam) {
        cudaError_t e = dev_alloc(ctx, &Li, (size_t)D * D * sizeof(double));
        if (e != cudaSuccess) rc = cuda_fail(ctx, e, "cudaMallocAsync(Λw⁻¹)");
        if (rc == 0) rc = post_ensure_W(ctx, pw);
        if (rc == 0) rc = gemm_generic(ctx, D, D, D, pw->W, D, 1, pw->W, 1, D, Li, 1, D, 0.0);
        if (rc == 0) {
            grad_prior_multi_dense_kernel<<<(int)std::min<int64_t>((D * D + 255) / 256, ctx->sm_count * 8), 256, 0, sm>>>(
                D, k, Q, ldq, Li, U, c_dev, cbar, dlam);
            BLR_CHECK_LAUNCH(ctx, "grad_prior_multi_dense_kernel");
        }
    }
    dev_free(sm, Li);
    post_release(pw);
    return rc;
}

int grad_a_multi(blr_ctx* ctx, double* A, int64_t ldq, int64_t dk, int64_t kp, int64_t D, int64_t k, const double* M,
                 const double* c_dev, double cbar) {
    const int64_t total = ldq * (dk + kp);
    grad_a_multi_kernel<<<(int)std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 8), 256, 0, ctx->stream>>>(
        A, ldq, dk, kp, D, k, M, c_dev, cbar);
    BLR_CHECK_LAUNCH(ctx, "grad_a_multi_kernel");
    return 0;
}

int grad_x_multi(blr_ctx* ctx, const blr_post* p, const blr_x* x, const double* A, int64_t ldq, int64_t dk, int64_t k, int64_t kp,
                 bool fast, const double* E, const double* sigma2, double sigma2_scalar, double* dX, int64_t ld_dX) {
    const int64_t D = p->D, N = x->N;
    if (N == 0) return 0;
    const double s_scalar = sigma2 ? 0.0 : 1.0 / sigma2_scalar;
    if (fast) {
        GradXParams gp;
        gp.Qp = A;
        gp.ldq = ldq;
        gp.dk = (int)dk;
        gp.kp = (int)kp;
        gp.D = (int)D;
        gp.N = N;
        gp.m = nullptr;
        gp.se = nullptr;
        gp.sigma2 = sigma2;
        gp.s_scalar = s_scalar;
        gp.dX = dX;
        gp.ld = ld_dX;
        const int smem = (int)sizeof(gk::Smem) + 1024;
        BLR_CUDA_OK(ctx, cudaFuncSetAttribute(grad_x_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        CUtensorMap tmx, tme;
        BLR_TRY(make_tmap_2d_f64(ctx, &tmx, x->p, (uint64_t)D, (uint64_t)N, (uint64_t)x->ld, gk::KT, gk::NP / 2));
        BLR_TRY(make_tmap_2d_f64(ctx, &tme, E, (uint64_t)kp, (uint64_t)N, (uint64_t)kp, gk::KT, gk::NP / 2));
        const int grid = (int)std::min<int64_t>((N + gk::NP - 1) / gk::NP, ctx->sm_count);
        grad_x_tma_kernel<true><<<grid, gk::THREADS, smem, ctx->stream>>>(gp, tmx, tme);
        BLR_CHECK_LAUNCH(ctx, "grad_x_tma_kernel<rank k>");
        return 0;
    }
    // generic path: -c̄ Q X, then + M' diag(c) E' (β = 1), by gemm_generic in column blocks it can address; then dX *= s_n
    const bool colv = x->layout == BLR_COLVECS;
    const int64_t block = (int64_t)1 << 20;
    for (int64_t a = 0; a < N; a += block) {
        const int64_t nb = std::min(block, N - a);
        const double* Xa = x->p + (colv ? a * x->ld : a);
        double* Ca = dX + (colv ? a * ld_dX : a);
        const int64_t cs_m = colv ? 1 : ld_dX, cs_n = colv ? ld_dX : 1;
        BLR_TRY(gemm_generic(ctx, D, nb, D, A, 1, ldq, Xa, colv ? 1 : x->ld, colv ? x->ld : 1, Ca, cs_m, cs_n, 0.0));
        BLR_TRY(gemm_generic(ctx, D, nb, k, A + dk * ldq, 1, ldq, E + a * kp, 1, kp, Ca, cs_m, cs_n, 1.0));
    }
    const int grid = (int)std::min<int64_t>((D * N + 255) / 256, (int64_t)ctx->sm_count * 16);
    if (colv)
        grad_x_scale_kernel<BLR_COLVECS><<<grid, 256, 0, ctx->stream>>>(dX, ld_dX, D, N, sigma2, s_scalar);
    else
        grad_x_scale_kernel<BLR_ROWVECS><<<grid, 256, 0, ctx->stream>>>(dX, ld_dX, D, N, sigma2, s_scalar);
    BLR_CHECK_LAUNCH(ctx, "grad_x_scale_kernel");
    return 0;
}

}  // namespace blr
