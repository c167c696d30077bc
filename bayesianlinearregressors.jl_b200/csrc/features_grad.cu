// Vector-Jacobian product of the device feature map ϕ(x) = scale * act(W x + b) (blr_x_features, synth.cu): for a cotangent
// dΦ (D x N ColVecs), with z_n = W x_n + b and g_dn = dΦ_dn * scale * act'(z_dn),
//   dW = Σ_n g_n x_n'      db = Σ_n g_n      dx_n = W' g_n.
// The forward saves nothing, so both kernels recompute z on the tensor cores and form g in registers; no N x D array is ever
// written.  The dW and dx contractions want opposite loop orders (dW: feature blocks outer, the partial held in registers;
// dx: point tiles outer, the sum over all features held in registers), so each output has its own kernel, and each reads dΦ
// once (DESIGN.md, K10):
//   features_vjp_w_kernel : grid (D / 64, d_in / BN, S).  CTA = one 64-feature block x a contiguous range of 64-point tiles;
//                           per tile z (64 x 64, K = d_in), g -> shared memory, dW block += G X' (K = 64 points); db as row sums of
//                           the g tile.  Partials go to a CTA-private slice of an S x D x (d_in + 1) workspace, summed over S in a
//                           fixed order by features_vjp_reduce_kernel.
//   features_vjp_x_kernel : grid (N / 64, d_in / BN).  CTA = one 64-point tile; loops over all feature blocks: z, g, then
//                           dXᵀ (64 points x BN) += Gᵀ W_blk (K = 64 features).
// Every contraction is a 64 x BN CTA tile on DMMA.8x8x4 (BN = 32 for d_in <= 32, else 64), operands staged through padded
// shared memory by element loaders that zero everything out of range, so any 1 <= d_in, D >= 1, N and leading dimension take
// the same path.  No atomics: repeated calls are bit-identical.
#include <math.h>

#include <algorithm>

#include "common.cuh"
#include "internal.h"

namespace blr {
namespace fg {
constexpr int BM = 64;        // tile rows (features for z and dW, points for dXᵀ)
constexpr int BP = 64;        // points per tile
constexpr int KH = 32;        // k extent staged per pass
constexpr int LDP = BM + 4;   // [k][m] rows: 68 == 4 (mod 16) doubles, conflict-free fragment loads
constexpr int LDQ = KH + 4;   // [n][k] rows
constexpr int LDG = 68;       // g tile in shared memory
constexpr int THREADS = 128;  // 2 x 2 warps, each a 32 x (BN / 2) register tile
constexpr int SMEM_A = KH * LDP;
constexpr int SMEM_B = 64 * LDQ;
constexpr int SMEM_G = 64 * LDG;
constexpr size_t SMEM_BYTES = (size_t)(SMEM_A + SMEM_B + SMEM_G) * sizeof(double);
}  // namespace fg

// C(64 x 16 NI) += A(64 x kc) B(kc x 16 NI) with A(m, k) = la(m, k), B(k, n) = lb(k, n); the loaders return 0 out of range.
// B_KFAST: B is contiguous along k in memory, so the staging loop walks k fastest.
template <int NI, bool B_KFAST, typename LA, typename LB>
__device__ __forceinline__ void tile_mma(double (&acc)[4][NI][2], int kc, LA la, LB lb, double* smA, double* smB) {
    using namespace fg;
    constexpr int BN = 16 * NI;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wm = warp >> 1, wn = warp & 1;
    for (int kh = 0; kh < kc; kh += KH) {
        const int kr = kc - kh, k4r = min(KH, (kr + 3) & ~3);  // stage only the k4 steps the MMA loop reads
        __syncthreads();
        for (int e = tid; e < k4r * BM; e += THREADS) {
            const int m = e % BM, k = e / BM;
            smA[k * LDP + m] = (k < kr) ? la(m, kh + k) : 0.0;
        }
        for (int e = tid; e < k4r * BN; e += THREADS) {
            const int k = B_KFAST ? e % k4r : e / BN, n = B_KFAST ? e / k4r : e % BN;
            smB[n * LDQ + k] = (k < kr) ? lb(kh + k, n) : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int k4 = 0; k4 < KH; k4 += 4)
            if (k4 < kr) warp_mma_k4<4, NI>(acc, smA + k4 * LDP + wm * 32, 1, LDP, smB + (wn * 8 * NI) * LDQ + k4, LDQ, 1, lane);
    }
}

template <int NI>
__device__ __forceinline__ void tile_zero(double (&acc)[4][NI][2]) {
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < NI; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
}

// f(mi, row, col, value&) for every accumulator element of this thread, row in [0, 64), col in [0, 16 NI)
template <int NI, typename F>
__device__ __forceinline__ void tile_foreach(double (&acc)[4][NI][2], F f) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wm = warp >> 1, wn = warp & 1, g = lane >> 2, kq = lane & 3;
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < NI; ++ni)
#pragma unroll
            for (int c = 0; c < 2; ++c) f(mi, wm * 32 + mi * 8 + g, wn * 8 * NI + ni * 8 + kq * 2 + c, acc[mi][ni][c]);
}

// act'(z); relu' is 0 at z = 0 (torch, Flux).  tanh' = sech² z = 4e / (1 + e)², e = exp(-2|z|): 1 - tanh² z cancels once
// |z| grows (relative error 1e-8 at |z| = 10, exactly 0 from |z| ≈ 19.1), this form keeps full relative accuracy, cannot
// overflow, and is 0 only where sech² z itself underflows.
template <int ACT>
__device__ __forceinline__ double feature_act_grad(double z) {
    if (ACT == BLR_ACT_COS) return -sin(z);
    if (ACT == BLR_ACT_SIN) return cos(z);
    if (ACT == BLR_ACT_TANH) {
        const double e = exp(-2.0 * fabs(z)), r = __drcp_rn(1.0 + e);  // a reciprocal, not a division: no fix-up path
        return 4.0 * e * r * r;
    }
    if (ACT == BLR_ACT_RELU) return z > 0.0 ? 1.0 : 0.0;
    return 1.0;
}

struct VjpArgs {
    const double* X;  // d_in x N ColVecs
    int64_t ldx;
    int din;
    int64_t N;
    const double* W;  // D x d_in column-major (device)
    const double* b;  // D
    int D;
    double scale;
    const double* dphi;  // D x N
    int64_t ldp;
};

// z tile (features d0.. x points n0..) on DMMA, then g = dΦ * scale * act'(z + b) into acc (0 outside D x N)
template <int ACT>
__device__ __forceinline__ void g_tile(const VjpArgs& a, int d0, int64_t n0, double (&acc)[4][4][2], double* smA, double* smB) {
    tile_zero<4>(acc);
    const double* W = a.W;
    const double* X = a.X;
    const int D = a.D;
    const int64_t N = a.N, ldx = a.ldx;
    tile_mma<4, true>(
        acc, a.din, [=](int m, int k) { return d0 + m < D ? W[(d0 + m) + (int64_t)k * D] : 0.0; },
        [=](int k, int n) { return n0 + n < N ? X[k + (n0 + n) * ldx] : 0.0; }, smA, smB);
    tile_foreach<4>(acc, [&](int, int r, int c, double& v) {
        const int d = d0 + r;
        const int64_t n = n0 + c;
        v = (d < D && n < N) ? a.dphi[d + n * a.ldp] * a.scale * feature_act_grad<ACT>(v + a.b[d]) : 0.0;
    });
}

template <int ACT, int NI>
__global__ void __launch_bounds__(fg::THREADS, 2) features_vjp_w_kernel(VjpArgs a, int64_t tiles_per_split, bool with_w,
                                                                     double* __restrict__ ws) {
    using namespace fg;
    extern __shared__ __align__(16) double sm[];
    double *smA = sm, *smB = smA + SMEM_A, *Gs = smB + SMEM_B;
    constexpr int BN = 16 * NI;
    const int d0 = blockIdx.x * BM, i0 = blockIdx.y * BN;
    const int64_t ntiles = (a.N + BP - 1) / BP;
    const int64_t t0 = (int64_t)blockIdx.z * tiles_per_split, t1 = min(ntiles, t0 + tiles_per_split);
    const bool with_b = blockIdx.y == 0;
    double accw[4][NI][2];
    tile_zero<NI>(accw);
    double dbr = 0.0;  // thread r < 64: db of feature d0 + r over this CTA's points
    const double* X = a.X;
    const int64_t ldx = a.ldx, N = a.N;
    const int din = a.din;
    for (int64_t t = t0; t < t1; ++t) {
        const int64_t n0 = t * BP;
        double accz[4][4][2];
        g_tile<ACT>(a, d0, n0, accz, smA, smB);
        tile_foreach<4>(accz, [&](int, int r, int c, double& v) { Gs[r + c * LDG] = v; });  // [point][feature]
        __syncthreads();
        if (with_b && threadIdx.x < BM)
            for (int c = 0; c < BP; ++c) dbr += Gs[threadIdx.x + c * LDG];
        if (with_w)
            tile_mma<NI, false>(
                accw, (int)min((int64_t)BP, N - n0), [=](int m, int k) { return Gs[m + k * LDG]; },
                [=](int k, int n) { return i0 + n < din ? X[(i0 + n) + (n0 + k) * ldx] : 0.0; }, smA, smB);
    }
    const int64_t len = (int64_t)a.D * (din + 1);
    double* out = ws + (int64_t)blockIdx.z * len;
    if (with_w)
        tile_foreach<NI>(accw, [&](int, int r, int c, double& v) {
            if (d0 + r < a.D && i0 + c < din) out[(d0 + r) + (int64_t)(i0 + c) * a.D] = v;
        });
    if (with_b && threadIdx.x < BM && d0 + (int)threadIdx.x < a.D) out[(int64_t)din * a.D + d0 + threadIdx.x] = dbr;
}

// out[off + j] = Σ_s ws[s * len + off + j], j < cnt, s = 0 .. S-1 in order (off = D d_in, cnt = D: the db column alone)
__global__ void __launch_bounds__(256) features_vjp_reduce_kernel(const double* __restrict__ ws, int64_t len, int64_t off,
                                                                  int64_t cnt, int S, double* __restrict__ out) {
    for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < cnt; j += (int64_t)gridDim.x * 256) {
        double s = 0.0;
        for (int k = 0; k < S; ++k) s += ws[(int64_t)k * len + off + j];
        out[off + j] = s;
    }
}

template <int ACT, int NI>
__global__ void __launch_bounds__(fg::THREADS) features_vjp_x_kernel(VjpArgs a, double* __restrict__ dx, int64_t lddx) {
    using namespace fg;
    extern __shared__ __align__(16) double sm[];
    double *smA = sm, *smB = smA + SMEM_A, *Gs = smB + SMEM_B;
    constexpr int BN = 16 * NI;
    const int64_t n0 = (int64_t)blockIdx.x * BP;
    const int i0 = blockIdx.y * BN;
    const double* W = a.W;
    const int D = a.D, din = a.din;
    double accx[4][NI][2];
    tile_zero<NI>(accx);
    for (int d0 = 0; d0 < D; d0 += BM) {
        double accz[4][4][2];
        g_tile<ACT>(a, d0, n0, accz, smA, smB);
        tile_foreach<4>(accz, [&](int, int r, int c, double& v) { Gs[c + r * LDG] = v; });  // [feature][point]
        tile_mma<NI, true>(
            accx, min(BM, D - d0), [=](int m, int k) { return Gs[m + k * LDG]; },
            [=](int k, int n) { return i0 + n < din ? W[(d0 + k) + (int64_t)(i0 + n) * D] : 0.0; }, smA, smB);
    }
    tile_foreach<NI>(accx, [&](int, int r, int c, double& v) {
        if (n0 + r < a.N && i0 + c < din) dx[(i0 + c) + (n0 + r) * lddx] = v;
    });
}

template <int ACT>
static int features_vjp_launch(blr_ctx* ctx, const VjpArgs& a, double* dWb, double* ws, int S, int64_t tiles_per_split,
                               bool with_w, double* dx, int64_t lddx) {
    using namespace fg;
    const bool narrow = a.din <= 32;
    if (dWb) {
        const unsigned gy = with_w ? (unsigned)((a.din + (narrow ? 31 : 63)) / (narrow ? 32 : 64)) : 1u;
        const dim3 grid((unsigned)((a.D + BM - 1) / BM), gy, (unsigned)S);
        auto k = narrow ? features_vjp_w_kernel<ACT, 2> : features_vjp_w_kernel<ACT, 4>;
        BLR_CUDA_OK(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        k<<<grid, THREADS, SMEM_BYTES, ctx->stream>>>(a, tiles_per_split, with_w, ws);
        BLR_CHECK_LAUNCH(ctx, "features_vjp_w_kernel");
        // without dW the workspace holds only the db column: reduce that alone
        const int64_t len = (int64_t)a.D * (a.din + 1), off = with_w ? 0 : (int64_t)a.D * a.din, cnt = len - off;
        const int rgrid = (int)std::min<int64_t>((cnt + 255) / 256, (int64_t)ctx->sm_count * 8);
        features_vjp_reduce_kernel<<<rgrid, 256, 0, ctx->stream>>>(ws, len, off, cnt, S, dWb);
        BLR_CHECK_LAUNCH(ctx, "features_vjp_reduce_kernel");
    }
    if (dx) {
        const dim3 grid((unsigned)((a.N + BP - 1) / BP), (unsigned)((a.din + (narrow ? 31 : 63)) / (narrow ? 32 : 64)));
        auto k = narrow ? features_vjp_x_kernel<ACT, 2> : features_vjp_x_kernel<ACT, 4>;
        BLR_CUDA_OK(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        k<<<grid, THREADS, SMEM_BYTES, ctx->stream>>>(a, dx, lddx);
        BLR_CHECK_LAUNCH(ctx, "features_vjp_x_kernel");
    }
    return 0;
}

int features_vjp_splits(const blr_ctx* ctx, int64_t N, int64_t D, int64_t din) {
    // about eight CTAs per SM over (feature block, d_in block, point range), so the last wave is a small share; never more
    // ranges than point tiles
    const int64_t blocks = ((D + fg::BM - 1) / fg::BM) * (din <= 32 ? 1 : (din + 63) / 64), ntiles = (N + fg::BP - 1) / fg::BP;
    return (int)std::max<int64_t>(1, std::min<int64_t>(ntiles, (8 * (int64_t)ctx->sm_count + blocks - 1) / blocks));
}

int features_vjp(blr_ctx* ctx, const blr_x* xin, const double* W_dev, const double* b_dev, int64_t D, int act, double scale,
                 const double* dphi, int64_t ldp, double* dWb, double* ws, int S, bool with_w, double* dx, int64_t lddx) {
    const VjpArgs a{xin->p, xin->ld, (int)xin->D, xin->N, W_dev, b_dev, (int)D, scale, dphi, ldp};
    const int64_t ntiles = (xin->N + fg::BP - 1) / fg::BP;
    const int64_t tps = S > 0 ? (ntiles + S - 1) / S : 0;  // S = 0: no dW / db requested
    switch (act) {
        case BLR_ACT_COS: return features_vjp_launch<BLR_ACT_COS>(ctx, a, dWb, ws, S, tps, with_w, dx, lddx);
        case BLR_ACT_TANH: return features_vjp_launch<BLR_ACT_TANH>(ctx, a, dWb, ws, S, tps, with_w, dx, lddx);
        case BLR_ACT_RELU: return features_vjp_launch<BLR_ACT_RELU>(ctx, a, dWb, ws, S, tps, with_w, dx, lddx);
        case BLR_ACT_IDENTITY: return features_vjp_launch<BLR_ACT_IDENTITY>(ctx, a, dWb, ws, S, tps, with_w, dx, lddx);
        case BLR_ACT_SIN: return features_vjp_launch<BLR_ACT_SIN>(ctx, a, dWb, ws, S, tps, with_w, dx, lddx);
        default: return set_err(ctx, BLR_E_INVALID, "unknown activation");
    }
}

}  // namespace blr
