// K6/K7: prediction-side kernels -- mean, marginal variances, covariance, sampling.
//
// Reference work replaced (src/bayesian_linear_regression.jl):
//   mean  :33      X' mw
//   var   :40-43   α = Uw' \ X ; sum(abs2, α; dims=1) .+ diag(Σy)      (Uw' = L, lower factor of Λw)
//   cov   :35-38   α'α + Σy
//   rand  :49-53   X'(mw .+ Uw \ Zw) .+ Uy' Zy
// and src/sampling_functions.jl:29,35,44 (weight draws), :17-19 (BLRFunctionSample call).
//
// The triangular solve against N columns is recast as a triangular GEMM with the explicit inverse factor
// W = inv(L) (built once per regressor, cached on the device): α = W X, var_n = |W x_n|² + σ²_n.  α is never
// written to HBM: each CTA owns a tile of test points, sweeps the row blocks of W and folds the squares into
// per-point sums held in registers (shuffle reduction across the fragment rows).
#include <math.h>

#include <algorithm>

#include "blockgemm.cuh"
#include "common.cuh"
#include "internal.h"
#include "philox.cuh"

namespace blr {

// ---------------------------------------------------------------------------------------------
// out_n = x_n' w   (mean :33, BLRFunctionSample call)
template <int LAYOUT>
__global__ void __launch_bounds__(256) apply_weights_kernel(const double* __restrict__ X, int64_t ld, int D, int64_t N,
                                                            const double* __restrict__ w, double* __restrict__ out) {
    if (LAYOUT == BLR_COLVECS) {
        const int lane = threadIdx.x & 31;
        const int64_t warps = (int64_t)gridDim.x * 8;
        for (int64_t n = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); n < N; n += warps) {
            const double* col = X + n * ld;
            double dot = 0.0;
            for (int d = lane; d < D; d += 32) dot = fma(col[d], __ldg(w + d), dot);
            dot = warp_sum(dot);
            if (lane == 0) out[n] = dot;
        }
    } else {
        const int64_t stride = (int64_t)gridDim.x * 256;
        for (int64_t n = (int64_t)blockIdx.x * 256 + threadIdx.x; n < N; n += stride) {
            double dot = 0.0;
            for (int d = 0; d < D; ++d) dot = fma(X[(int64_t)d * ld + n], __ldg(w + d), dot);
            out[n] = dot;
        }
    }
}

int apply_weights(blr_ctx* ctx, const blr_x* x, const double* w_dev, double* out_dev) {
    if (x->N == 0) return 0;
    const int D = (int)x->D;
    if (x->layout == BLR_COLVECS) {
        const int grid = (int)std::min<int64_t>((x->N + 7) / 8, (int64_t)ctx->sm_count * 16);
        apply_weights_kernel<BLR_COLVECS><<<grid, 256, 0, ctx->stream>>>(x->p, x->ld, D, x->N, w_dev, out_dev);
    } else {
        const int grid = (int)std::min<int64_t>((x->N + 255) / 256, (int64_t)ctx->sm_count * 16);
        apply_weights_kernel<BLR_ROWVECS><<<grid, 256, 0, ctx->stream>>>(x->p, x->ld, D, x->N, w_dev, out_dev);
    }
    BLR_CHECK_LAUNCH(ctx, "apply_weights_kernel");
    return 0;
}

// ---------------------------------------------------------------------------------------------
// var_n = |W x_n|² + σ²_n for a tile of 64 test points per CTA (DMMA block GEMMs, α stays on chip).
template <int LAYOUT>
__global__ void __launch_bounds__(bg::THREADS) var_kernel(const double* __restrict__ W, int D,
                                                          const double* __restrict__ X, int64_t ld, int64_t N,
                                                          const double* __restrict__ sigma2, double sigma2_scalar,
                                                          double* __restrict__ var) {
    __shared__ double smA[bg::SMEM_A], smB[bg::SMEM_B];
    __shared__ double colsum[2][bg::BS];
    const int64_t p0 = (int64_t)blockIdx.x * bg::BS;
    const int pvalid = (int)min((int64_t)bg::BS, N - p0);
    const int nblk = (D + bg::BS - 1) / bg::BS;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wm = warp >> 1, wn = warp & 1;
    double csum[4][2];
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) csum[ni][0] = csum[ni][1] = 0.0;

    for (int ib = 0; ib < nblk; ++ib) {
        double acc[4][4][2];
        acc_zero(acc);
        const int r0 = ib * bg::BS;
        for (int kb = 0; kb <= ib; ++kb) {
            const int k0 = kb * bg::BS;
            const int kc = min(bg::BS, D - k0);
            // A (m, k) = W[r0 + m, k0 + k] ; B (k, n) = X[k0 + k, p0 + n]
            if (LAYOUT == BLR_COLVECS)
                cta_gemm64<true>(acc, W + (int64_t)k0 * D + r0, D, D - r0, X + p0 * ld + k0, ld, pvalid, kc, smA, smB);
            else
                cta_gemm64<false>(acc, W + (int64_t)k0 * D + r0, D, D - r0, X + (int64_t)k0 * ld + p0, ld, pvalid, kc, smA,
                                  smB);
        }
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) {
                csum[ni][0] = fma(acc[mi][ni][0], acc[mi][ni][0], csum[ni][0]);
                csum[ni][1] = fma(acc[mi][ni][1], acc[mi][ni][1], csum[ni][1]);
            }
    }
    // fold the 8 fragment rows (lane >> 2) of each column, then the two row-warps
#pragma unroll
    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            double v = csum[ni][c];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            if ((lane >> 2) == 0) colsum[wm][wn * 32 + ni * 8 + (lane & 3) * 2 + c] = v;
        }
    __syncthreads();
    if (threadIdx.x < pvalid) {
        const int64_t n = p0 + threadIdx.x;
        var[n] = (colsum[0][threadIdx.x] + colsum[1][threadIdx.x]) + (sigma2 ? sigma2[n] : sigma2_scalar);
    }
}

// ---------------------------------------------------------------------------------------------
#ifndef BLR_VAR_SMALL_GB34
#define BLR_VAR_SMALL_GB34 2  // groups of 8 points in flight per warp trip for 16 < D <= 24 (MI = 4 would spill at two)
#endif
// Small-D marginals (D <= 64): W lives in shared memory, every warp streams groups of 8 test points straight from HBM
// into m8n8k4 B fragments (lane (k, g) reads feature 4*kk + k of point p + g: whole 32-byte sectors in both layouts),
// α = W x stays in 2 accumulators per 8-row block, squares are folded by shuffles; the mean rides on the same fragments.
template <int MI>
__global__ void __launch_bounds__(256, MI <= 8 ? 2 : 1) var_small_kernel(const double* __restrict__ W, const double* __restrict__ mw, int D,
                                                        const double* __restrict__ X, int64_t sd, int64_t sn, int64_t N,
                                                        const double* __restrict__ sigma2, double sigma2_scalar,
                                                        double* __restrict__ mean, double* __restrict__ var) {
    constexpr int DP = MI * 8, KK = DP / 4, LDW = DP + 4;
    extern __shared__ __align__(16) double var_small_smem[];  // (D <= 128: up to 136 KB, hence dynamic)
    double* Ws = var_small_smem;       // Ws[k * LDW + m] = W[m, k]
    double* mws = Ws + DP * LDW;       // [DP]
    for (int e = threadIdx.x; e < DP * DP; e += 256) {
        const int m = e % DP, k = e / DP;
        Ws[k * LDW + m] = (m < D && k < D && m >= k) ? W[(int64_t)k * D + m] : 0.0;
    }
    if (threadIdx.x < DP) mws[threadIdx.x] = threadIdx.x < D ? mw[threadIdx.x] : 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31, g = lane >> 2, kq = lane & 3;
    const int64_t nwarps = (int64_t)gridDim.x * 8;
    const int64_t ngroups = (N + 7) / 8;
    double a_mw[KK];
#pragma unroll
    for (int kk = 0; kk < KK; ++kk) a_mw[kk] = mws[kk * 4 + kq];
    // GB groups of 8 points per trip, loads first: like the small-D Gram kernel this is bound by bytes in flight
    constexpr int GB = (MI == 1 ? 8 : (MI == 2 ? 4 : (MI == 3 ? BLR_VAR_SMALL_GB34 : 1)));
    for (int64_t grp0 = ((int64_t)blockIdx.x * 8 + (threadIdx.x >> 5)) * GB; grp0 < ngroups; grp0 += nwarps * GB) {
        double b[GB][KK];
#pragma unroll
        for (int gb = 0; gb < GB; ++gb) {
            const int64_t pt = (grp0 + gb) * 8 + g;
            const bool pok = pt < N;
#pragma unroll
            for (int kk = 0; kk < KK; ++kk) {
                const int k = kk * 4 + kq;
                b[gb][kk] = (pok && k < D) ? X[(int64_t)k * sd + pt * sn] : 0.0;
            }
        }
#pragma unroll
        for (int gb = 0; gb < GB; ++gb) {
            const int64_t p0 = (grp0 + gb) * 8, pt = p0 + g;
            if (p0 >= N) break;
            const bool pok = pt < N;
            double acc[MI][2];
#pragma unroll
            for (int mi = 0; mi < MI; ++mi) acc[mi][0] = acc[mi][1] = 0.0;
            double macc = 0.0;
#pragma unroll
            for (int kk = 0; kk < KK; ++kk) {
                macc = fma(a_mw[kk], b[gb][kk], macc);
#pragma unroll
                for (int mi = 0; mi < MI; ++mi) {
                    if (mi * 8 + 7 >= kk * 4) {  // W[m, k] = 0 for k > m: static triangular skip
                        const double a = Ws[(kk * 4 + kq) * LDW + mi * 8 + g];
                        dmma884(acc[mi], a, b[gb][kk]);
                    }
                }
            }
            double v0 = 0.0, v1 = 0.0;
#pragma unroll
            for (int mi = 0; mi < MI; ++mi) {
                v0 = fma(acc[mi][0], acc[mi][0], v0);
                v1 = fma(acc[mi][1], acc[mi][1], v1);
            }
#pragma unroll
            for (int o = 4; o <= 16; o <<= 1) {
                v0 += __shfl_xor_sync(0xffffffffu, v0, o);
                v1 += __shfl_xor_sync(0xffffffffu, v1, o);
            }
            macc += __shfl_xor_sync(0xffffffffu, macc, 1);
            macc += __shfl_xor_sync(0xffffffffu, macc, 2);
            if (var && g == 0) {  // lane kq owns points p0 + 2 kq, p0 + 2 kq + 1
                const int64_t q0 = p0 + kq * 2;
                if (q0 < N) var[q0] = v0 + (sigma2 ? sigma2[q0] : sigma2_scalar);
                if (q0 + 1 < N) var[q0 + 1] = v1 + (sigma2 ? sigma2[q0 + 1] : sigma2_scalar);
            }
            if (mean && kq == 0 && pok) mean[pt] = macc;
        }
    }
}

// D <= 8: one thread per test point (an m8n8k4 tile would be mostly padding and the warp-per-8-points schedule above is
// bound by instruction issue): W (lower triangle) and mw live in registers, X is read once with coalesced loads
// (16-byte vector loads for ColVecs with ld == D), D (D + 1) / 2 + 2 D DFMAs per point.
template <int DT, bool VEC>
__global__ void __launch_bounds__(DT == 8 ? 128 : 256, DT == 2 ? 4 : 3)
    var_tiny_kernel(const double* __restrict__ W, const double* __restrict__ mw, int D, const double* __restrict__ X,
                    int64_t sd, int64_t sn, int64_t N, const double* __restrict__ sigma2, double sigma2_scalar,
                    double* __restrict__ mean, double* __restrict__ var) {
    double w[DT * (DT + 1) / 2], m[DT];
#pragma unroll
    for (int i = 0; i < DT; ++i) {
        m[i] = i < D ? mw[i] : 0.0;
#pragma unroll
        for (int k = 0; k <= i; ++k) w[i * (i + 1) / 2 + k] = (i < D) ? W[(int64_t)k * D + i] : 0.0;
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
#pragma unroll(DT == 8 ? 1 : 2)
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += stride) {
        double x[DT];
        if (VEC) {
            const double2* col = reinterpret_cast<const double2*>(X + n * DT);
#pragma unroll
            for (int h = 0; h < DT / 2; ++h) {
                const double2 v2 = col[h];
                x[2 * h] = v2.x;
                x[2 * h + 1] = v2.y;
            }
        } else {
#pragma unroll
            for (int d = 0; d < DT; ++d) x[d] = (d < D) ? X[(int64_t)d * sd + n * sn] : 0.0;
        }
        double v = 0.0, mu = 0.0;
#pragma unroll
        for (int i = 0; i < DT; ++i) {
            mu = fma(x[i], m[i], mu);
            double al = 0.0;
#pragma unroll
            for (int k = 0; k <= i; ++k) al = fma(w[i * (i + 1) / 2 + k], x[k], al);
            v = fma(al, al, v);
        }
        if (var) var[n] = v + (sigma2 ? sigma2[n] : sigma2_scalar);
        if (mean) mean[n] = mu;
    }
}

template <int DT>
static int launch_var_tiny(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* sigma2, double sigma2_scalar,
                           double* mean_dev, double* var_dev) {
    constexpr int THREADS = DT == 8 ? 128 : 256;
    const bool colv = x->layout == BLR_COLVECS;
    const int64_t sd = colv ? 1 : x->ld, sn = colv ? x->ld : 1;
    const int grid = (int)std::max<int64_t>(
        1, std::min<int64_t>((x->N + THREADS - 1) / THREADS, (int64_t)ctx->sm_count * (DT == 2 ? 4 : 3)));
    const bool vec = colv && p->D == DT && x->ld == DT && (reinterpret_cast<uintptr_t>(x->p) & 15) == 0;
    if (vec)
        var_tiny_kernel<DT, true><<<grid, THREADS, 0, ctx->stream>>>(p->W, p->mw, (int)p->D, x->p, sd, sn, x->N, sigma2,
                                                                    sigma2_scalar, mean_dev, var_dev);
    else
        var_tiny_kernel<DT, false><<<grid, THREADS, 0, ctx->stream>>>(p->W, p->mw, (int)p->D, x->p, sd, sn, x->N, sigma2,
                                                                     sigma2_scalar, mean_dev, var_dev);
    BLR_CHECK_LAUNCH(ctx, "var_tiny_kernel");
    return 0;
}

template <int MI>
static int launch_var_small(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* sigma2, double sigma2_scalar,
                            double* mean_dev, double* var_dev) {
    const bool colv = x->layout == BLR_COLVECS;
    const int64_t sd = colv ? 1 : x->ld, sn = colv ? x->ld : 1;
    constexpr int DP = MI * 8;
    const int smem = (DP * (DP + 4) + DP) * (int)sizeof(double);
    if (smem > 48 * 1024) BLR_CUDA_OK(ctx, cudaFuncSetAttribute(var_small_kernel<MI>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int grid = (int)std::min<int64_t>(((x->N + 7) / 8 + 7) / 8, (int64_t)ctx->sm_count * (MI <= 8 ? 4 : 1));
    var_small_kernel<MI><<<std::max(grid, 1), 256, smem, ctx->stream>>>(p->W, p->mw, (int)p->D, x->p, sd, sn, x->N, sigma2,
                                                                      sigma2_scalar, mean_dev, var_dev);
    BLR_CHECK_LAUNCH(ctx, "var_small_kernel");
    return 0;
}

int predict_mean_var(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* sigma2, double sigma2_scalar,
                     double* mean_dev, double* var_dev) {
    if (x->N == 0) return 0;
    if (ctx->form == BLR_FORM_WHITENED) return predict_mean_var_literal(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
    if (var_dev && p->D > 64 && p->D <= ctx->var_small_max) {
        // 64 < D <= 128 (BLR_VAR_SMALL_MAX): W still fits shared memory and the streaming kernel of the small-D regime beats the
        // tiled one, whose 128-row pass and short per-tile pipeline leave it at 6 .. 19 TF here (measured per 2^20 .. 2^21 points:
        // D = 66 1.47 -> 0.56 ms, D = 96 1.07 -> 0.60 ms, D = 128 0.89 -> 0.72 ms); any layout, any alignment, no staging
        BLR_TRY(post_ensure_W(ctx, p));
        switch ((p->D + 7) / 8) {
            case 9: return launch_var_small<9>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 10: return launch_var_small<10>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 11: return launch_var_small<11>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 12: return launch_var_small<12>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 13: return launch_var_small<13>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 14: return launch_var_small<14>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 15: return launch_var_small<15>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            default: return launch_var_small<16>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
        }
    }
    if (var_dev && predict_fast_eligible(p, x))
        return predict_mean_var_fast(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
    if (var_dev && p->D > 64 && x->N >= 32) {
        // Inputs the TMA kernel cannot address -- RowVecs, or ColVecs with an odd leading dimension (dense odd D) or a misaligned
        // base -- are staged block by block into an aligned ColVecs buffer (one extra read + write of X: 32 / D of the pass)
        // instead of running the DFMA-fed generic kernel.
        const int64_t D = p->D, N = x->N, ldt = D + (D % 2);
        const int64_t block = std::min<int64_t>(N, std::max<int64_t>((int64_t)1 << 16, ((int64_t)1 << 27) / ldt));
        double* stage = nullptr;
        BLR_CUDA_OK(ctx, cudaMallocAsync(&stage, (size_t)ldt * block * sizeof(double), ctx->stream));
        int rc = 0;
        for (int64_t a = 0; a < N && rc == 0; a += block) {
            blr_x sub;
            sub.p = stage;
            sub.D = D;
            sub.N = std::min(block, N - a);
            sub.ld = ldt;
            sub.layout = BLR_COLVECS;
            if (x->layout == BLR_COLVECS) {
                rc = repack_colvecs(ctx, x->p + a * x->ld, x->ld, D, sub.N, stage, ldt);
            } else {
                blr_x view = *x;
                view.p = x->p + a;
                view.N = sub.N;
                view.owned = false;
                rc = transpose_to_colvecs(ctx, &view, stage, ldt);  // the pad row (odd D) is never read: the tensor map has D rows
            }
            if (rc != 0) break;
            if (sub.N >= 32) {
                rc = predict_mean_var_fast(ctx, p, &sub, sigma2 ? sigma2 + a : nullptr, sigma2_scalar,
                                           mean_dev ? mean_dev + a : nullptr, var_dev + a);
            } else {  // a tail shorter than a point tile
                rc = predict_mean_var(ctx, p, &sub, sigma2 ? sigma2 + a : nullptr, sigma2_scalar,
                                      mean_dev ? mean_dev + a : nullptr, var_dev + a);
            }
        }
        cudaFreeAsync(stage, ctx->stream);
        return rc;
    }
    if (var_dev && p->D <= 64) {
        BLR_TRY(post_ensure_W(ctx, p));
        if (p->D <= 2) return launch_var_tiny<2>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
        if (p->D <= 4) return launch_var_tiny<4>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
        if (p->D <= 8) return launch_var_tiny<8>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
        // one instantiation per multiple of 8 features: padding D = 24 to 32 or D = 40 to 64 costs 1.8x / 2.6x the tensor work
        switch ((p->D + 7) / 8) {
            case 2: return launch_var_small<2>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 3: return launch_var_small<3>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 4: return launch_var_small<4>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 5: return launch_var_small<5>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 6: return launch_var_small<6>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            case 7: return launch_var_small<7>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
            default: return launch_var_small<8>(ctx, p, x, sigma2, sigma2_scalar, mean_dev, var_dev);
        }
    }
    if (mean_dev) BLR_TRY(apply_weights(ctx, x, p->mw, mean_dev));
    if (var_dev) {
        BLR_TRY(post_ensure_W(ctx, p));
        const int64_t grid = (x->N + bg::BS - 1) / bg::BS;
        if (grid > 0x7fffffff) return set_err(ctx, BLR_E_INVALID, "too many test points for one launch");
        if (x->layout == BLR_COLVECS)
            var_kernel<BLR_COLVECS><<<(int)grid, bg::THREADS, 0, ctx->stream>>>(p->W, (int)p->D, x->p, x->ld, x->N, sigma2,
                                                                              sigma2_scalar, var_dev);
        else
            var_kernel<BLR_ROWVECS><<<(int)grid, bg::THREADS, 0, ctx->stream>>>(p->W, (int)p->D, x->p, x->ld, x->N, sigma2,
                                                                              sigma2_scalar, var_dev);
        BLR_CHECK_LAUNCH(ctx, "var_kernel");
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Generic strided GEMM (plain DFMA, 32 x 32 tiles): C[m, n] = beta * C + Σ_k A[m, k] B[k, n].
// Used for the small-N "next" rows (cov) and the first version of rand; not a throughput path.
__global__ void __launch_bounds__(256) gemm_generic_kernel(int64_t M, int64_t Nn, int64_t K, const double* __restrict__ A,
                                                           int64_t as_m, int64_t as_k, const double* __restrict__ B,
                                                           int64_t bs_k, int64_t bs_n, double* __restrict__ C,
                                                           int64_t cs_m, int64_t cs_n, double beta) {
    __shared__ double As[32][33], Bs[32][33];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t m0 = (int64_t)blockIdx.x * 32, n0 = (int64_t)blockIdx.y * 32;
    double c00 = 0, c01 = 0, c10 = 0, c11 = 0;
    for (int64_t k0 = 0; k0 < K; k0 += 32) {
        __syncthreads();
        for (int e = threadIdx.x; e < 1024; e += 256) {
            // pick the thread -> element map that walks the unit-stride direction of each operand
            const int a_m = (as_m <= as_k) ? e % 32 : e / 32, a_k = (as_m <= as_k) ? e / 32 : e % 32;
            As[a_k][a_m] = (m0 + a_m < M && k0 + a_k < K) ? A[(m0 + a_m) * as_m + (k0 + a_k) * as_k] : 0.0;
            const int b_n = (bs_n <= bs_k) ? e % 32 : e / 32, b_k = (bs_n <= bs_k) ? e / 32 : e % 32;
            Bs[b_k][b_n] = (n0 + b_n < Nn && k0 + b_k < K) ? B[(k0 + b_k) * bs_k + (n0 + b_n) * bs_n] : 0.0;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < 32; ++k) {
            const double a0 = As[k][ty * 2], a1 = As[k][ty * 2 + 1], b0 = Bs[k][tx * 2], b1 = Bs[k][tx * 2 + 1];
            c00 = fma(a0, b0, c00);
            c01 = fma(a0, b1, c01);
            c10 = fma(a1, b0, c10);
            c11 = fma(a1, b1, c11);
        }
    }
    const double cc[2][2] = {{c00, c01}, {c10, c11}};
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j) {
            const int64_t m = m0 + ty * 2 + i, n = n0 + tx * 2 + j;
            if (m < M && n < Nn) {
                double* dst = C + m * cs_m + n * cs_n;
                *dst = (beta == 0.0) ? cc[i][j] : beta * (*dst) + cc[i][j];
            }
        }
}

int gemm_generic(blr_ctx* ctx, int64_t M, int64_t Nn, int64_t K, const double* A, int64_t as_m, int64_t as_k,
                        const double* B, int64_t bs_k, int64_t bs_n, double* C, int64_t cs_m, int64_t cs_n, double beta) {
    if (M == 0 || Nn == 0) return 0;
    const int64_t gx = (M + 31) / 32, gy = (Nn + 31) / 32;
    if (gy > 65535) return set_err(ctx, BLR_E_INVALID, "gemm_generic: too many column tiles");
    gemm_generic_kernel<<<dim3((unsigned)gx, (unsigned)gy), 256, 0, ctx->stream>>>(M, Nn, K, A, as_m, as_k, B, bs_k, bs_n, C,
                                                                                  cs_m, cs_n, beta);
    BLR_CHECK_LAUNCH(ctx, "gemm_generic_kernel");
    return 0;
}

__global__ void add_diag_noise_kernel(double* __restrict__ C, int64_t N, const double* __restrict__ sigma2,
                                      double sigma2_scalar) {
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x)
        C[n * N + n] += sigma2 ? sigma2[n] : sigma2_scalar;
}

// cov = α'α + Σy, α = W X  (N x N output: small-N path, "next" row of SURVEY.md section 8f)
int predict_cov(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* sigma2, double sigma2_scalar, double* C_dev) {
    const int64_t D = p->D, N = x->N;
    if (N == 0) return 0;
    const bool literal = ctx->form == BLR_FORM_WHITENED;
    if (!literal) BLR_TRY(post_ensure_W(ctx, p));
    double* alpha = nullptr;
    BLR_CUDA_OK(ctx, cudaMallocAsync(&alpha, (size_t)D * N * sizeof(double), ctx->stream));
    const bool colv = x->layout == BLR_COLVECS;
    // α (D x N, column-major) = W (D x D, column-major) * X;  literal form: α = Uw' \ X by triangular solve (:36)
    int rc = literal ? solve_alpha(ctx, p, x, 0, N, alpha)
                     : gemm_generic(ctx, D, N, D, p->W, 1, D, x->p, colv ? 1 : x->ld, colv ? x->ld : 1, alpha, 1, D, 0.0);
    // C = α'α
    if (rc == 0) rc = gemm_generic(ctx, N, N, D, alpha, D, 1, alpha, 1, D, C_dev, 1, N, 0.0);
    if (rc == 0) {
        add_diag_noise_kernel<<<(int)std::min<int64_t>((N + 255) / 256, 1024), 256, 0, ctx->stream>>>(C_dev, N, sigma2,
                                                                                                   sigma2_scalar);
        ctx->launches++;
    }
    cudaFreeAsync(alpha, ctx->stream);
    return rc;
}

// ---------------------------------------------------------------------------------------------
// Weight draws: Wsamp (D x S) = mw .+ Uw \ Z = mw .+ L^-T Z = mw .+ W' Z
__global__ void add_col_vector_kernel(double* __restrict__ A, int64_t D, int64_t S, const double* __restrict__ v) {
    const int64_t total = D * S;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x)
        A[e] += v[e % D];
}

int sample_weights(blr_ctx* ctx, blr_post* p, int64_t S, const double* Z_dev, double* W_dev) {
    const int64_t D = p->D;
    if (S == 0) return 0;
    if (ctx->form == BLR_FORM_WHITENED) {
        // literal form: Uw \ Z by back substitution against the factor (:51)
        BLR_CUDA_OK(ctx, cudaMemcpyAsync(W_dev, Z_dev, (size_t)D * S * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        BLR_TRY(trsm_lower(ctx, p->L, D, D, W_dev, D, S, true));
    } else {
        BLR_TRY(post_ensure_W(ctx, p));
        // (W' Z)[d, s] = Σ_k W[k, d] Z[k, s]
        BLR_TRY(gemm_generic(ctx, D, S, D, p->W, D, 1, Z_dev, 1, D, W_dev, 1, D, 0.0));
    }
    add_col_vector_kernel<<<(int)std::min<int64_t>((D * S + 255) / 256, (int64_t)ctx->sm_count * 8), 256, 0, ctx->stream>>>(
        W_dev, D, S, p->mw);
    BLR_CHECK_LAUNCH(ctx, "add_col_vector_kernel");
    return 0;
}

// Y[n, s] += sqrt(σ²_n) * z,  z = Zy[n, s] when supplied, else Philox normal: stream 7, pair index n + (s / 2) * N,
// first / second member of the pair for even / odd s (same indexing as the fused epilogue of rand_tma_kernel)
__global__ void add_obs_noise_kernel(double* __restrict__ Y, int64_t N, int64_t S, const double* __restrict__ sigma2,
                                     double sigma2_scalar, const double* __restrict__ Zy, uint64_t seed) {
    const int64_t total = N * S;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t n = e % N;
        const double sd = sqrt(sigma2 ? sigma2[n] : sigma2_scalar);
        double z;
        if (Zy) {
            z = Zy[e];
        } else {
            const int64_t sidx = e / N;
            double z0, z1;
            philox_normal_pair(seed, 7, (uint64_t)n + (uint64_t)(sidx >> 1) * (uint64_t)N, z0, z1);
            z = (sidx & 1) ? z1 : z0;
        }
        Y[e] = fma(sd, z, Y[e]);
    }
}

int sample_finite(blr_ctx* ctx, const blr_x* x, const double* Wsamp_dev, int64_t S, const double* sigma2,
                  double sigma2_scalar, const double* Zy_dev, uint64_t seed, double* Y_dev, bool noiseless) {
    const int64_t N = x->N, D = x->D;
    if (N == 0 || S == 0) return 0;
    if (sample_fast_eligible(x))
        return sample_finite_fast(ctx, x, Wsamp_dev, S, sigma2, sigma2_scalar, Zy_dev, seed, Y_dev, nullptr, noiseless);
    const bool colv = x->layout == BLR_COLVECS;
    if (D >= 64 && N >= 128) {
        // RowVecs, or ColVecs with an odd leading dimension / misaligned base: blocks of points staged into an aligned ColVecs
        // buffer and run by the single-group TMA kernel (outputs, draws and Philox counters addressed in the whole problem)
        const int64_t ldt = D + (D % 2);
        const int64_t block = std::min<int64_t>(N, std::max<int64_t>((int64_t)1 << 16, ((int64_t)1 << 27) / ldt));
        double* stage = nullptr;
        BLR_CUDA_OK(ctx, cudaMallocAsync(&stage, (size_t)ldt * block * sizeof(double), ctx->stream));
        int rc = 0;
        for (int64_t a = 0; a < N && rc == 0; a += block) {
            blr_x sub;
            sub.p = stage;
            sub.D = D;
            sub.N = std::min(block, N - a);
            sub.ld = ldt;
            sub.layout = BLR_COLVECS;
            if (colv) {
                rc = repack_colvecs(ctx, x->p + a * x->ld, x->ld, D, sub.N, stage, ldt);
            } else {
                blr_x view = *x;
                view.p = x->p + a;
                view.N = sub.N;
                view.owned = false;
                rc = transpose_to_colvecs(ctx, &view, stage, ldt);
            }
            const RandChunk ck = {N, N, a, N};
            if (rc == 0)
                rc = sample_finite_fast(ctx, &sub, Wsamp_dev, S, sigma2 ? sigma2 + a : nullptr, sigma2_scalar,
                                        Zy_dev ? Zy_dev + a : nullptr, seed, Y_dev + a, &ck, noiseless);
        }
        cudaFreeAsync(stage, ctx->stream);
        return rc;
    }
    // Y (N x S) = X' Wsamp : A[m = n, k = d] = X[d, n]
    BLR_TRY(gemm_generic(ctx, N, S, D, x->p, colv ? x->ld : 1, colv ? 1 : x->ld, Wsamp_dev, 1, D, Y_dev, 1, N, 0.0));
    if (noiseless) return 0;
    add_obs_noise_kernel<<<(int)std::min<int64_t>((N * S + 255) / 256, (int64_t)ctx->sm_count * 16), 256, 0, ctx->stream>>>(
        Y_dev, N, S, sigma2, sigma2_scalar, Zy_dev, seed);
    BLR_CHECK_LAUNCH(ctx, "add_obs_noise_kernel");
    return 0;
}

}  // namespace blr
