// K6 fast path: marginal means and variances for ColVecs test points at throughput scale
//
//     mean_n = x_n' mw            var_n = |W x_n|² + σ²_n ,   W = inv(L),  Λw = L L'
//
// (reference src/bayesian_linear_regression.jl:33 and :40-43: `α = Uw' \ X; sum(abs2, α; dims=1) .+ diag(Σy)`;
// the reference materialises the D x N matrix α, here α never leaves the SM).
//
// Shape of the computation: α = W X is a triangular GEMM with M = D rows, N = points, K = D.  One persistent CTA
// per SM owns tiles of 32 points and keeps α (up to 512 rows x 32 points = 128 KB) in registers as DMMA.8x8x4
// accumulators: 8 consumer warps, warp tile 64 rows x 32 points.  The K dimension is streamed in stages of 16:
//   A operand = 16 columns of W (rows >= the stage's first non-zero row), [k][row] in shared memory, 1-D bulk copies (2 KB each),
//   B operand = 16 features of the tile's points, [point][k] in shared memory: ONE 2-D tiled TMA load per producer warp and
//               stage (cp.async.bulk.tensor.2d, tensor map over X, 128-byte swizzle instead of row padding, ragged edges
//               zero-filled by the hardware) -- round 1 issued one 128-byte bulk copy per point, 64 per stage, and the
//               serial issue of those copies (~100 cycles apiece) was as long as a stage takes to consume,
// through a 3-stage mbarrier ring.  X is read from HBM exactly
// once; W (2 MB at D = 512) streams from L2.
// Triangular balance: warp w owns the 8-row blocks {w, 15 - w, 16 + w, 31 - w, ...}, so every warp loses sub-tiles
// at the same rate as k advances; which sub-tile rows are live is a compile-time template parameter (run-time predication
// of mma.sync serialises the tensor pipe, see gram.cu).
// D > 512 is handled in row passes of 512 rows (the point tile is re-streamed per pass).
#include <cuda.h>  // CUtensorMap types only: the encoder is fetched through cudaGetDriverEntryPoint, libcuda is not linked
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <string>

#include "common.cuh"
#include "internal.h"
#include "philox.cuh"

namespace blr {
namespace vk {
constexpr int KT = 16;          // features per stage
constexpr int STAGES = 3;
static_assert(KT == 16, "the point tile is one 128-byte swizzle span (16 doubles) per point");
constexpr int CONSUMER_WARPS = 8;
// cp.async.bulk is a uniform-datapath instruction: the per-lane copies of a warp are issued one after another.
// Four producer warps (A columns 0-7 | A columns 8-15 | first half of the points | second half) keep the issue rate ahead of
// the consumers; 12 warps x 168 registers is exactly the register file.
constexpr int PRODUCER_WARPS = 4;
constexpr int THREADS = (CONSUMER_WARPS + PRODUCER_WARPS) * 32;
// MI: 64-row blocks of α per pass; NP: points per tile (32, 64 or 128).  MI * NP / 8 = 32 accumulator tiles per warp either way:
// <8, 32> keeps all 512 rows of a D <= 512 problem in one pass; <4, 64> runs 256-row passes on twice the points (half the W
// traffic per point, 25 % fewer pipeline stages per point and no 16-DMMA stages; the point tile is re-streamed per pass).
template <int MI, int NP>
struct Cfg {
    static constexpr int R = MI * 64;      // rows of α per pass
    static constexpr int LDA = R + 4;      // A row stride (doubles): == 4 mod 16
    static constexpr int NI = NP / 8;      // 8-point blocks per tile
    struct __align__(1024) Stage {
        double b[NP * KT];    // [point][k], 128 bytes per point, 128-byte TMA swizzle (swz128); 1024-byte aligned
        double a[KT * LDA];   // [k][row - r_base]
        double mw[KT];
    };
    struct Smem {
        Stage st[STAGES];
        double red[CONSUMER_WARPS][NP];
        double mred[NP];
        unsigned long long full[STAGES];
        unsigned long long empty[STAGES];
    };
};
}  // namespace vk

struct VarParams {
    const double* Wp;   // padded inverse factor: ldw x dk, column-major, zeros outside the lower triangle / beyond D
    int64_t ldw;        // multiple of R
    int D;
    int64_t N;          // test points (ColVecs, reached through the tensor map)
    const double* mwp;  // prior mean padded with zeros to a multiple of KT
    const double* sigma2;
    double sigma2_scalar;
    double* mean;       // may be null
    double* var;        // may be null
};

// one stage for one consumer warp; sub-tile rows mi >= M0 are live
template <int MI, int NI, int M0>
__device__ __forceinline__ void var_consume(double (&acc)[MI][NI][2], const double* __restrict__ As,
                                            const double* __restrict__ Bs, int warp, int g, int kq, const int (&boff)[4]) {
    using C = vk::Cfg<MI, NI * 8>;
    // row block of (warp, mi): 8 mi + warp for even mi, 8 mi + 7 - warp for odd mi (see var_tma_kernel)
    const double* Ap0 = As + warp * 8 + g;
    const double* Ap1 = As + (7 - warp) * 8 + g;
#pragma unroll
    for (int kk = 0; kk < vk::KT / 4; ++kk) {
        const int kl = kk * 4 + kq;
        double a[MI], b[NI];
#pragma unroll
        for (int mi = M0; mi < MI; ++mi) a[mi] = ((mi & 1) ? Ap1 : Ap0)[kl * C::LDA + mi * 64];
#pragma unroll
        for (int ni = 0; ni < NI; ++ni) b[ni] = Bs[ni * 8 * vk::KT + boff[kk]];  // point 8 ni + g, feature 4 kk + kq
#pragma unroll
        for (int mi = M0; mi < MI; ++mi)
#pragma unroll
            for (int ni = 0; ni < NI; ++ni) dmma884(acc[mi][ni], a[mi], b[ni]);
    }
}

template <int MI, int NI>
__device__ __forceinline__ void var_consume_dispatch(double (&acc)[MI][NI][2], const double* As, const double* Bs,
                                                     int warp, int g, int kq, int m0, const int (&boff)[4]) {
    // warp-uniform compare chain (a switch compiles to an indirect branch, measured 2.6 % slower)
    if (m0 <= 0) var_consume<MI, NI, 0>(acc, As, Bs, warp, g, kq, boff);
    else if (m0 == 1) var_consume<MI, NI, (1 < MI ? 1 : MI)>(acc, As, Bs, warp, g, kq, boff);
    else if (m0 == 2) var_consume<MI, NI, (2 < MI ? 2 : MI)>(acc, As, Bs, warp, g, kq, boff);
    else if (m0 == 3) var_consume<MI, NI, (3 < MI ? 3 : MI)>(acc, As, Bs, warp, g, kq, boff);
    else if (m0 == 4) var_consume<MI, NI, (4 < MI ? 4 : MI)>(acc, As, Bs, warp, g, kq, boff);
    else if (m0 == 5) var_consume<MI, NI, (5 < MI ? 5 : MI)>(acc, As, Bs, warp, g, kq, boff);
    else if (m0 == 6) var_consume<MI, NI, (6 < MI ? 6 : MI)>(acc, As, Bs, warp, g, kq, boff);
    else if (m0 == 7) var_consume<MI, NI, (7 < MI ? 7 : MI)>(acc, As, Bs, warp, g, kq, boff);
    // m0 >= MI: nothing live for this warp in this stage
}

// Stage order within a row pass: heavy (small k: many live rows) and light (large k) stages alternate, so the time a
// (STAGES - 1)-deep prefetch covers stays ~constant instead of collapsing at the light end of the triangle.
__device__ __forceinline__ int var_stage_k0(int s, int nst) {
    return ((s & 1) ? (nst - 1 - (s >> 1)) : (s >> 1)) * vk::KT;
}

template <int MI, int NP>
__global__ void __launch_bounds__(vk::THREADS, 1) var_tma_kernel(const VarParams p, const __grid_constant__ CUtensorMap tmx) {
    using namespace vk;
    using C = Cfg<MI, NP>;
    constexpr int NI = C::NI;
    extern __shared__ unsigned char smem_raw[];
    // the swizzled point tiles need 1024-byte alignment: align by hand (the launcher asks for 1 KB more than sizeof(Smem))
    typename C::Smem& sm = *reinterpret_cast<typename C::Smem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    {
        double* z = reinterpret_cast<double*>(sm.st);
        const int nz = (int)(sizeof(typename C::Stage) * STAGES / sizeof(double));
        for (int i = tid; i < nz; i += THREADS) z[i] = 0.0;
    }
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
    const int npass = (int)(p.ldw / C::R);

    if (warp >= CONSUMER_WARPS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");  // producers hand their registers to the consumer warpgroups
        // ------------------------------------------------------------ producer warps (TMA)
        const int pw = warp - CONSUMER_WARPS;
        int it = 0;
        for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int64_t p0 = tile * NP;
            for (int ps = 0; ps < npass; ++ps) {
                const int r_base = ps * C::R;
                const int kmax = min(p.D, r_base + C::R);  // W[row][k] = 0 for k > row
                const int nst = (kmax + KT - 1) / KT;
                for (int si = 0; si < nst; ++si, ++it) {
                    const int k0 = var_stage_k0(si, nst);
                    const int stg = it % STAGES;
                    const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
                    mbar_wait(smem_u32(&sm.empty[stg]), ph ^ 1u);
                    typename C::Stage& S = sm.st[stg];
                    const uint32_t bar = smem_u32(&sm.full[stg]);
                    const int r_lo = max(r_base, (k0 / 64) * 64);     // first row that can be non-zero in this stage
                    const int rows = r_base + C::R - r_lo;
                    const bool with_mw = (ps == npass - 1);
                    if (pw < 2) {  // 8 columns of W each
                        ring_expect(bar, (uint32_t)(KT / 2) * rows * 8u + ((pw == 0 && with_mw) ? KT * 8u : 0u), lane);
                        if (lane < KT / 2) {
                            const int kr = pw * (KT / 2) + lane;
                            bulk_g2s(smem_u32(&S.a[kr * C::LDA + (r_lo - r_base)]), p.Wp + (int64_t)(k0 + kr) * p.ldw + r_lo,
                                     (uint32_t)rows * 8u, bar);
                        }
                        if (lane == 0 && pw == 0 && with_mw) bulk_g2s(smem_u32(S.mw), p.mwp + k0, KT * 8u, bar);
                    } else {       // half of the tile's points each: one 2-D box {KT features, NP / 2 points}; whatever lies
                                   // beyond D or N is zero-filled by the TMA unit and still counted, so the byte count is fixed
                        const int pbase = (pw - 2) * (NP / 2);
                        ring_expect(bar, (uint32_t)(NP / 2) * KT * 8u, lane);
                        if (lane == 0) tma_load_2d(smem_u32(&S.b[pbase * KT]), &tmx, k0, (int)(p0 + pbase), bar);
                    }
                }
            }
        }
        return;
    }

    // ---------------------------------------------------------------- consumer warps (DMMA)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");  // 128 x 40 + 256 x 232 = 384 x 168
    const int g = lane >> 2, kq = lane & 3;
    int boff[4];  // swizzled offset of (point g, feature 4 kk + kq) within an 8-point block of the point tile
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) boff[kk] = swz128(g, kk * 4 + kq);
    constexpr int PP = NP / 16;               // mean: points per thread
    const int mk = tid & 15, mpg = tid >> 4;  // mean: feature within the stage, point group
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t p0 = tile * NP;
        double macc[PP];
#pragma unroll
        for (int j = 0; j < PP; ++j) macc[j] = 0.0;
        for (int ps = 0; ps < npass; ++ps) {
            const int r_base = ps * C::R;
            const int kmax = min(p.D, r_base + C::R);
            double acc[MI][NI][2];
#pragma unroll
            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                for (int ni = 0; ni < NI; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
            const int nst = (kmax + KT - 1) / KT;
            for (int si = 0; si < nst; ++si, ++it) {
                const int k0 = var_stage_k0(si, nst);
                const int stg = it % STAGES;
                const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
                mbar_wait(smem_u32(&sm.full[stg]), ph);
                const typename C::Stage& S = sm.st[stg];
                // Warp w owns the 8-row blocks b(mi) = 8 mi + (mi odd ? 7 - w : w) of this pass (boustrophedon, so that
                // every warp -- and every SM sub-partition -- loses sub-tiles at the same rate as k advances: with the
                // plain 8 mi + w map warps 6, 7 carry 20 % more DMMAs than warps 0, 1).  Block b holds rows
                // r_base + 8 b .. + 7 and is live iff its last row >= k0; b grows with mi, so the live set is mi >= m0.
                // Closed form of  #{mi : 64 mi + 8 wp(mi) < q},  q = k0 - r_base - 7,  wp = warp (mi even) or 7 - warp (odd):
                // every mi < q / 64 qualifies, mi = q / 64 qualifies iff 8 wp(mi) < q mod 64, larger mi never do.
                const int q = k0 - r_base - 7;
                int m0 = 0;
                if (q > 0) {
                    const int ms = q >> 6, rem = q & 63;
                    m0 = min(ms, MI);
                    if (ms < MI && 8 * ((ms & 1) ? 7 - warp : warp) < rem) ++m0;
                }
                var_consume_dispatch<MI, NI>(acc, S.a, S.b, warp, g, kq, m0, boff);
                if (ps == npass - 1) {  // the last row pass streams every feature k < D
                    const double mwk = S.mw[mk];
#pragma unroll
                    for (int j = 0; j < PP; ++j) macc[j] = fma(mwk, S.b[swz128(PP * mpg + j, mk)], macc[j]);
                }
                ring_release(smem_u32(&sm.empty[stg]), lane);
            }
            // fold this pass: squares over the warp's rows (registers, then the 8 fragment rows by shuffle) into the
            // warp's per-point slots in shared memory (each slot has a single owner lane: no synchronisation needed)
#pragma unroll
            for (int ni = 0; ni < NI; ++ni)
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    double v = 0.0;
#pragma unroll
                    for (int mi = 0; mi < MI; ++mi) v = fma(acc[mi][ni][c], acc[mi][ni][c], v);
                    v += __shfl_xor_sync(0xffffffffu, v, 4);
                    v += __shfl_xor_sync(0xffffffffu, v, 8);
                    v += __shfl_xor_sync(0xffffffffu, v, 16);
                    if (g == 0) {
                        double* slot = &sm.red[warp][ni * 8 + kq * 2 + c];
                        *slot = (ps == 0) ? v : *slot + v;
                    }
                }
        }
#pragma unroll
        for (int j = 0; j < PP; ++j) {  // fold the 16 features held by 16 consecutive lanes
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) macc[j] += __shfl_xor_sync(0xffffffffu, macc[j], o);
            if (mk == 0) sm.mred[PP * mpg + j] = macc[j];
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (tid < NP && p0 + tid < p.N) {
            const int64_t n = p0 + tid;
            if (p.var) {
                double v = 0.0;
#pragma unroll
                for (int w = 0; w < CONSUMER_WARPS; ++w) v += sm.red[w][tid];
                p.var[n] = v + (p.sigma2 ? p.sigma2[n] : p.sigma2_scalar);
            }
            if (p.mean) p.mean[n] = sm.mred[tid];
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");  // slots are rewritten by the next tile
    }
}

// Wp (ldw x dk) = zero-padded copy of the lower-triangular W (D x D, ld = D); mwp = zero-padded mw
__global__ void pad_inverse_factor_kernel(const double* __restrict__ W, int D, double* __restrict__ Wp, int64_t ldw, int dk,
                                          const double* __restrict__ mw, double* __restrict__ mwp) {
    const int64_t total = ldw * dk;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(e % ldw), c = (int)(e / ldw);
        Wp[e] = (r < D && c < D && r >= c) ? W[(int64_t)c * D + r] : 0.0;
    }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < dk; i += gridDim.x * blockDim.x) mwp[i] = (i < D) ? mw[i] : 0.0;
}

// Tensor map of a column-major fp64 matrix for 2-D tiled TMA loads: `inner` contiguous elements per column, `outer` columns
// `ld` elements apart, boxes of box_inner x box_outer elements stored with the 128-byte swizzle (box_inner * 8 <= 128 bytes),
// out-of-range elements read as zero.  cuTensorMapEncodeTiled is a host-side encoder; it is looked up through the runtime
// (cudaGetDriverEntryPoint) so the library keeps linking against nothing but cudart.
int make_tmap_2d_f64(blr_ctx* ctx, CUtensorMap* out, const double* base, uint64_t inner, uint64_t outer, uint64_t ld,
                     uint32_t box_inner, uint32_t box_outer) {
    typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static encode_fn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        BLR_CUDA_OK(ctx, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !fn) return set_err(ctx, BLR_E_CUDA, "cuTensorMapEncodeTiled is not available");
        encode = (encode_fn)fn;
    }
    if (box_inner * 8u > 128u || box_inner > 256u || box_outer > 256u || (ld & 1) || (reinterpret_cast<uintptr_t>(base) & 15) ||
        outer >= (1ull << 31) || inner >= (1ull << 31))
        return set_err(ctx, BLR_E_INVALID, "matrix not addressable by a 2-D tensor map");
    const cuuint64_t dims[2] = {inner, outer};
    const cuuint64_t strides[1] = {ld * sizeof(double)};  // bytes between columns (a multiple of 16: ld is even)
    const cuuint32_t box[2] = {box_inner, box_outer};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_err(ctx, BLR_E_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return 0;
}

template <int MI, int NP>
static int launch_var_tma(blr_ctx* ctx, const VarParams& vp, const blr_x* x) {
    using C = vk::Cfg<MI, NP>;
    const int smem = (int)sizeof(typename C::Smem) + 1024;  // + slack for the in-kernel 1024-byte alignment
    BLR_CUDA_OK(ctx, cudaFuncSetAttribute(var_tma_kernel<MI, NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CUtensorMap tmx;  // test points: D features (contiguous) x N points; one box = 16 features of half a point tile
    BLR_TRY(make_tmap_2d_f64(ctx, &tmx, x->p, (uint64_t)x->D, (uint64_t)x->N, (uint64_t)x->ld, vk::KT, NP / 2));
    const int64_t ntiles = (vp.N + NP - 1) / NP;
    const int grid = (int)std::min<int64_t>(ntiles, ctx->sm_count);
    var_tma_kernel<MI, NP><<<grid, vk::THREADS, smem, ctx->stream>>>(vp, tmx);
    BLR_CHECK_LAUNCH(ctx, "var_tma_kernel");
    return 0;
}

bool predict_fast_eligible(const blr_post* p, const blr_x* x) {
    // (odd D is fine: the 2-D tensor map zero-fills beyond D and the inverse factor is zero-padded; only the row pitch and the
    // base of X are bound by TMA's 16-byte rule)
    return x->layout == BLR_COLVECS && p->D > 64 && (x->ld % 2) == 0 &&
           (reinterpret_cast<uintptr_t>(x->p) & 15) == 0 && x->N >= 32 && x->N < (1ll << 31);
}

int predict_mean_var_fast(blr_ctx* ctx, blr_post* p, const blr_x* x, const double* sigma2, double sigma2_scalar,
                          double* mean_dev, double* var_dev) {
    const int D = (int)p->D;
    const bool wide = ctx->var_cfg == 1 && x->N >= 64;  // 256-row passes on 64-point tiles
    // D <= 128: one 128-row pass on 128-point tiles (a 256-row pass would spend half its DMMAs on zero rows); the choice depends
    // on D alone because the padded factor Wp is cached with the posterior in the layout of the chosen pass height
    const int MI = D <= 128 ? 2 : ((D <= 256 || ctx->var_cfg == 1) ? 4 : 8);
    const int R = MI * 64;
    const int64_t ldw = ((D + R - 1) / R) * (int64_t)R;
    const int dk = ((D + vk::KT - 1) / vk::KT) * vk::KT;
    if (!p->Wp) {
        BLR_TRY(post_ensure_W(ctx, p));
        BLR_CUDA_OK(ctx, dev_alloc(ctx, &p->Wp, (size_t)(ldw * dk + dk) * sizeof(double)));
        pad_inverse_factor_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(p->W, D, p->Wp, ldw, dk, p->mw, p->Wp + ldw * dk);
        BLR_CHECK_LAUNCH(ctx, "pad_inverse_factor_kernel");
    }
    VarParams vp;
    vp.Wp = p->Wp;
    vp.ldw = ldw;
    vp.D = D;
    vp.N = x->N;
    vp.mwp = p->Wp + ldw * dk;
    vp.sigma2 = sigma2;
    vp.sigma2_scalar = sigma2_scalar;
    vp.mean = mean_dev;
    vp.var = var_dev;
    if (MI == 2) return launch_var_tma<2, 128>(ctx, vp, x);
    if (MI == 8) return launch_var_tma<8, 32>(ctx, vp, x);
    return wide ? launch_var_tma<4, 64>(ctx, vp, x) : launch_var_tma<4, 32>(ctx, vp, x);
}


// ====================================================================================================
// K7 fast path: Y (N x S) = X' Wsamp + sqrt(σ²) .* Z      (reference src/bayesian_linear_regression.jl:52)
//
// GEMM with M = points, N = samples, K = D.  One persistent CTA per SM owns tiles of 128 points x 64 samples
// (8 warps as 4 x 2, warp tile 32 x 32 on DMMA.8x8x4); X is streamed once per 64-sample block through a TMA
// bulk-copy ring ([point][k] rows of 32 features), the sample weights come pre-transposed ([k][sample], 512-byte
// rows) from L2.  The noise term is fused into the epilogue: Z supplied (parity mode) or Philox on the fly.
namespace rk {
constexpr int TP = 128;         // points per tile
constexpr int TS = 64;          // samples per block
constexpr int KT = 32;          // features per stage
constexpr int STAGES = 4;
constexpr int LDB = TS + 4;     // [k][sample]
constexpr int CONSUMER_WARPS = 8;
constexpr int PRODUCER_WARPS = 4;  // each: ONE 2-D TMA box (16 features x 64 points) + 8 bulk copies of sample-weight rows
static_assert(KT == 32 && TP == 128, "producer warp pw loads feature half (pw & 1) of point half (pw >> 1)");
constexpr int THREADS = (CONSUMER_WARPS + PRODUCER_WARPS) * 32;
struct __align__(1024) Stage {
    double a[KT / 16][TP * 16];  // points: two sub-tiles of 16 features, [point][k] with the 128-byte TMA swizzle (swz128)
    double b[KT * LDB];          // sample weights [k][sample]
};
struct Smem {
    Stage st[STAGES];
    unsigned long long full[STAGES];
    unsigned long long empty[STAGES];
};
}  // namespace rk

struct RandParams {
    int D;
    int64_t N;
    const double* Wt;   // [nsb][dk][64]: transposed, zero-padded sample weights
    int dk;             // D rounded up to KT
    int S;
    const double* sigma2;
    double sigma2_scalar;
    const double* Zy;   // N x S column-major, or null
    uint64_t seed;
    bool noise;         // false: Y = X'W alone (no draws, sigma2 / Zy not read)
    double* Y;          // N x S column-major
    int64_t ldy, ldz;   // leading dimensions of Y and Zy (two-group kernel; the single-group kernel uses N for both)
    int64_t n_global;   // index of this launch's first point in the whole problem and the whole problem's N: the Philox counter
    int64_t N_global;   // of pair (n, s) is n + (s >> 1) N over the WHOLE problem, whatever the chunking
};

__global__ void __launch_bounds__(rk::THREADS, 1) rand_tma_kernel(const RandParams p, const __grid_constant__ CUtensorMap tmx) {
    using namespace rk;
    extern __shared__ unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));  // swizzle: 1 KB aligned
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    {
        double* z = reinterpret_cast<double*>(sm.st);
        const int nz = (int)(sizeof(Stage) * STAGES / sizeof(double));
        for (int i = tid; i < nz; i += THREADS) z[i] = 0.0;
    }
    if (tid == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(smem_u32(&sm.full[i]), PRODUCER_WARPS * RING_LANES);
            mbar_init(smem_u32(&sm.empty[i]), CONSUMER_WARPS * RING_LANES);
        }
        mbar_fence_init();
    }
    fence_proxy_async();
    __syncthreads();

    const int64_t ntiles = (p.N + TP - 1) / TP;
    const int nsb = (p.S + TS - 1) / TS;

    if (warp >= CONSUMER_WARPS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        const int pw = warp - CONSUMER_WARPS;  // producer pw: points 32 pw .. 32 pw + 31 and W rows 8 pw .. 8 pw + 7
        int it = 0;
        for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int64_t p0 = tile * TP;
            for (int sb = 0; sb < nsb; ++sb) {
                const double* Wsb = p.Wt + (int64_t)sb * p.dk * TS;
                for (int k0 = 0; k0 < p.D; k0 += KT, ++it) {
                    const int stg = it % STAGES;
                    const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
                    mbar_wait(smem_u32(&sm.empty[stg]), ph ^ 1u);
                    Stage& S = sm.st[stg];
                    const uint32_t bar = smem_u32(&sm.full[stg]);
                    // one box {16 features, 64 points} per warp; beyond D or N the TMA unit writes zeros and still counts the bytes
                    ring_expect(bar, (uint32_t)(TP / 2) * 16u * 8u + (uint32_t)(KT / 4) * TS * 8u, lane);
                    if (lane == 0)
                        tma_load_2d(smem_u32(&S.a[pw & 1][(pw >> 1) * (TP / 2) * 16]), &tmx, k0 + 16 * (pw & 1),
                                    (int)(p0 + (pw >> 1) * (TP / 2)), bar);
                    if (lane < KT / 4) {
                        const int kr = pw * (KT / 4) + lane;
                        bulk_g2s(smem_u32(&S.b[kr * LDB]), Wsb + (int64_t)(k0 + kr) * TS, TS * 8u, bar);
                    }
                }
            }
        }
        return;
    }

    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");
    const int wm = warp >> 1, wn = warp & 1, g = lane >> 2, kq = lane & 3;
    int aoff[4];  // swizzled offset of (point wm * 32 + g, feature 4 j + kq) within a 16-feature sub-tile
#pragma unroll
    for (int j = 0; j < 4; ++j) aoff[j] = wm * 32 * 16 + swz128(g, j * 4 + kq);
    int it = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t p0 = tile * TP;
        for (int sb = 0; sb < nsb; ++sb) {
            double acc[4][4][2];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
            for (int k0 = 0; k0 < p.D; k0 += KT, ++it) {
                const int stg = it % STAGES;
                const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
                mbar_wait(smem_u32(&sm.full[stg]), ph);
                const Stage& S = sm.st[stg];
                const double* Bp = S.b + wn * 32 + g;
#pragma unroll
                for (int kk = 0; kk < KT / 4; ++kk) {
                    const int kl = kk * 4 + kq;
                    double a[4], b[4];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi) a[mi] = S.a[kk >> 2][mi * 8 * 16 + aoff[kk & 3]];
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) b[ni] = Bp[kl * LDB + ni * 8];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                        for (int ni = 0; ni < 4; ++ni) dmma884(acc[mi][ni], a[mi], b[ni]);
                }
                ring_release(smem_u32(&sm.empty[stg]), lane);
            }
            // epilogue: add the observation noise and store (column-major N x S)
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int64_t n = p0 + wm * 32 + mi * 8 + g;
                if (n < p.N) {
                    const double sd = p.noise ? sqrt(p.sigma2 ? p.sigma2[n] : p.sigma2_scalar) : 0.0;
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) {
                        const int s0 = sb * TS + wn * 32 + ni * 8 + kq * 2;  // even
                        if (s0 < p.S) {
                            double z0 = 0.0, z1 = 0.0;
                            if (p.noise) {
                                if (p.Zy) {
                                    z0 = p.Zy[(int64_t)s0 * p.ldz + n];
                                    z1 = (s0 + 1 < p.S) ? p.Zy[(int64_t)(s0 + 1) * p.ldz + n] : 0.0;
                                } else {
                                    philox_normal_pair(p.seed, 7, (uint64_t)(p.n_global + n) + (uint64_t)(s0 >> 1) * (uint64_t)p.N_global,
                                                       z0, z1);
                                }
                            }
                            p.Y[(int64_t)s0 * p.ldy + n] = fma(sd, z0, acc[mi][ni][0]);
                            if (s0 + 1 < p.S) p.Y[(int64_t)(s0 + 1) * p.ldy + n] = fma(sd, z1, acc[mi][ni][1]);
                        }
                    }
                }
            }
        }
    }
}

// Wt[sb][k][j] = Wsamp[k, sb*64 + j]  (zero beyond D / S)
__global__ void transpose_samples_kernel(const double* __restrict__ Wsamp, int D, int S, double* __restrict__ Wt, int dk,
                                         int nsb) {
    const int64_t total = (int64_t)nsb * dk * rk::TS;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int j = (int)(e % rk::TS);
        const int k = (int)((e / rk::TS) % dk);
        const int sb = (int)(e / ((int64_t)rk::TS * dk));
        const int s = sb * rk::TS + j;
        Wt[e] = (k < D && s < S) ? Wsamp[(int64_t)s * D + k] : 0.0;
    }
}

int sample_finite_pp(blr_ctx* ctx, const blr_x* x, const double* Wsamp_dev, int64_t S, const double* sigma2,
                     double sigma2_scalar, const double* Zy_dev, uint64_t seed, double* Y_dev);

bool sample_fast_eligible(const blr_x* x) {
    // (odd D is fine for the single-group kernel: the tensor map over X zero-fills beyond D, the sample weights are re-packed)
    return x->layout == BLR_COLVECS && x->D >= 64 && (x->ld % 2) == 0 &&
           (reinterpret_cast<uintptr_t>(x->p) & 15) == 0 && x->N >= 128 && x->N < (1ll << 31);
}

// chunk != nullptr: x holds points [n_global, n_global + x->N) of a problem of N_global points (a staged block of an input the
// tensor map cannot address); sigma2 / Zy_dev / Y_dev already point at the block's first point, ldy / ldz span the whole problem.
int sample_finite_fast(blr_ctx* ctx, const blr_x* x, const double* Wsamp_dev, int64_t S, const double* sigma2,
                       double sigma2_scalar, const double* Zy_dev, uint64_t seed, double* Y_dev, const RandChunk* chunk,
                       bool noiseless) {
    const int D = (int)x->D;
    // the two-group kernel reads the sample weights through a tensor map over the D x S matrix itself: D must be even
    if (!noiseless && !chunk && (D % 2) == 0 && (ctx->rand_pp == 2 || (ctx->rand_pp == 1 && Zy_dev != nullptr))) {
        const int r = sample_finite_pp(ctx, x, Wsamp_dev, S, sigma2, sigma2_scalar, Zy_dev, seed, Y_dev);
        if (r <= 0) return r;  // 1: weights not 16-byte aligned -> the default kernel
    }
    const int dk = ((D + rk::KT - 1) / rk::KT) * rk::KT;
    const int nsb = (int)((S + rk::TS - 1) / rk::TS);
    double* Wt = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &Wt, (size_t)nsb * dk * rk::TS * sizeof(double)));
    transpose_samples_kernel<<<std::min(ctx->sm_count * 4, nsb * dk), 256, 0, ctx->stream>>>(Wsamp_dev, D, (int)S, Wt, dk, nsb);
    BLR_CHECK_LAUNCH(ctx, "transpose_samples_kernel");
    RandParams rp;
    rp.D = D;
    rp.N = x->N;
    rp.Wt = Wt;
    rp.dk = dk;
    rp.S = (int)S;
    rp.sigma2 = sigma2;
    rp.sigma2_scalar = sigma2_scalar;
    rp.Zy = Zy_dev;
    rp.seed = seed;
    rp.noise = !noiseless;
    rp.Y = Y_dev;
    rp.ldy = chunk ? chunk->ldy : x->N;
    rp.ldz = chunk ? chunk->ldz : x->N;
    rp.n_global = chunk ? chunk->n_global : 0;
    rp.N_global = chunk ? chunk->N_global : x->N;
    const int smem = (int)sizeof(rk::Smem) + 1024;  // + slack for the in-kernel 1024-byte alignment
    CUtensorMap tmx;  // points: D features (contiguous) x N points; one box = 16 features of 64 points
    int rc = make_tmap_2d_f64(ctx, &tmx, x->p, (uint64_t)x->D, (uint64_t)x->N, (uint64_t)x->ld, 16, rk::TP / 2);
    cudaError_t e = (rc == 0) ? cudaFuncSetAttribute(rand_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) : cudaSuccess;
    if (rc == 0 && e == cudaSuccess) {
        const int64_t ntiles = (x->N + rk::TP - 1) / rk::TP;
        rand_tma_kernel<<<(int)std::min<int64_t>(ntiles, ctx->sm_count), rk::THREADS, smem, ctx->stream>>>(rp, tmx);
        ctx->launches++;
        e = cudaGetLastError();
    }
    dev_free(ctx->stream, Wt);
    if (rc != 0) return rc;
    if (e != cudaSuccess) return cuda_fail(ctx, e, "launch rand_tma_kernel");
    return 0;
}

// ====================================================================================================
// K7, two-group kernel (default when the draws are supplied; BLR_RAND_PP): TWO consumer groups of four warps, each with its own tiles of 128 points x 64 samples
// (warp tile 32 x 64), its own 4-stage ring of 16-feature stages and its own producer warp; warps w and w + 4 share an SM
// sub-partition, so while one group is in its epilogue the other group's warp has the DMMA pipe to itself.  Both operands by
// 2-D tiled TMA (tensor maps over X and over the D x S sample-weight matrix itself; one swizzled offset table serves both
// fragments).  Measurements and the dead ends on the way: DESIGN.md, section 4 (K7).
// The per-pair epilogue (draw or load z, add the noise, store) as a real call instead of 32 inlined copies: with two groups executing DIFFERENT code at the same time
// (one in its main loop, one in its epilogue) the unrolled epilogue (~64 KB of SASS) evicted the main loop from the instruction
// cache -- ncu: no_instruction was the top stall (5.3 per issue), 64.9 ms at cfg4 against 38.8 ms for the single-group kernel.
// Four pairs per call (one point, samples s0 + 8 j + {0, 1}, j = 0..3): the four Philox -> log / sincospi -> sqrt chains are
// independent and interleave; 32 strictly serial single-pair calls made a group's epilogue nearly as long as the other
// group's main loop (two-group kernel with device draws 9.94 ms against 8.57 ms with supplied draws, D = 512, N* = 2^22).
__device__ __noinline__ void rand_emit4(double* __restrict__ Y, const double* __restrict__ Zy, int64_t ldy, int64_t ldz, int S,
                                        uint64_t seed, uint64_t ctr0, uint64_t Ng, int64_t n, int s0, double sd, double a00,
                                        double a01, double a10, double a11, double a20, double a21, double a30, double a31) {
    const double a[4][2] = {{a00, a01}, {a10, a11}, {a20, a21}, {a30, a31}};
    double z[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int s = s0 + 8 * j;
        z[j][0] = z[j][1] = 0.0;
        if (s < S) {
            if (Zy) {
                z[j][0] = Zy[(int64_t)s * ldz + n];
                if (s + 1 < S) z[j][1] = Zy[(int64_t)(s + 1) * ldz + n];
            } else {
                philox_normal_pair(seed, 7, ctr0 + (uint64_t)n + (uint64_t)(s >> 1) * Ng, z[j][0], z[j][1]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int s = s0 + 8 * j;
        if (s < S) Y[(int64_t)s * ldy + n] = fma(sd, z[j][0], a[j][0]);
        if (s + 1 < S) Y[(int64_t)(s + 1) * ldy + n] = fma(sd, z[j][1], a[j][1]);
    }
}

// The draws of points [0, cnt) of a chunk (global indices n_global + n) for all S samples, with exactly the counters of the fused
// epilogue: pair (n, s even) = Philox(seed, stream 7, n + (s / 2) N_global) -> (z_s, z_{s+1}).  Z is cnt x S, ld = ldz.
__global__ void __launch_bounds__(256) rand_draws_kernel(double* __restrict__ Z, int64_t ldz, int64_t cnt, int S, uint64_t seed,
                                                         uint64_t n_global, uint64_t N_global) {
    const int64_t npair_cols = (S + 1) / 2, total = npair_cols * cnt;
    for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (int64_t)gridDim.x * 256) {
        const int64_t sp = e / cnt, n = e % cnt;
        double z0, z1;
        philox_normal_pair(seed, 7, n_global + (uint64_t)n + (uint64_t)sp * N_global, z0, z1);
        Z[2 * sp * ldz + n] = z0;
        if (2 * sp + 1 < S) Z[(2 * sp + 1) * ldz + n] = z1;
    }
}

namespace rp {
constexpr int TP = 128, TS = 64, KT = 16, STAGES = 4, GROUPS = 2, GROUP_WARPS = 4;
constexpr int CONSUMER_WARPS = GROUPS * GROUP_WARPS;
// setmaxnreg.sync.aligned is a WARPGROUP operation (four contiguous warps): the producer side is a full warpgroup, warps 8 and
// 9 produce, warps 10 and 11 only hand their registers over and exit (a two-warp producer side hangs the kernel)
constexpr int THREADS = (CONSUMER_WARPS + 4) * 32;
struct __align__(1024) Stage {
    double a[TP * 16];  // points:         [point][16 features], swz128
    double b[TS * 16];  // sample weights: [sample][16 features], swz128
};
constexpr uint32_t STAGE_BYTES = (uint32_t)((TP + TS) * 16 * sizeof(double));
struct Smem {
    // barriers first; the stages follow at the next 1 KB boundary
    unsigned long long full[GROUPS][STAGES];
    unsigned long long empty[GROUPS][STAGES];
    unsigned long long go;  // mbarrier, one arrival: group 0 is half way through its first tile, group 1 may start
    Stage st[GROUPS][STAGES];
};
}  // namespace rp

__global__ void __launch_bounds__(rp::THREADS, 1) rand_pp_kernel(const RandParams p, const __grid_constant__ CUtensorMap tmx,
                                                                 const __grid_constant__ CUtensorMap tmw) {
    using namespace rp;
    extern __shared__ unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int gi = 0; gi < GROUPS; ++gi)
            for (int i = 0; i < STAGES; ++i) {
                mbar_init(smem_u32(&sm.full[gi][i]), RING_LANES);
                mbar_init(smem_u32(&sm.empty[gi][i]), GROUP_WARPS * RING_LANES);
            }
        mbar_init(smem_u32(&sm.go), 1);
        mbar_fence_init();
    }
    fence_proxy_async();
    __syncthreads();  // no zero fill: every byte of a stage is written by the TMA boxes of the phase that is read
    const int64_t ntiles = (p.N + TP - 1) / TP;
    const int nsb = (p.S + TS - 1) / TS;
    const int nst = (p.D + KT - 1) / KT;

    if (warp >= CONSUMER_WARPS) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
        const int grp = warp - CONSUMER_WARPS;
        if (grp >= GROUPS) return;
        // Barrier addresses as plain registers, opaque to the optimiser: ptxas otherwise addresses both barriers with NEGATIVE
        // immediates off one shared base register ([R + -0x100]), which compute-sanitizer synccheck mis-resolves -- it reported
        // every first wait as "Missing init" and faulted the kernel (tool-only; same SASS otherwise).
        uint32_t ebase = smem_u32(&sm.empty[grp][0]), fbase = smem_u32(&sm.full[grp][0]);
        asm volatile("" : "+r"(ebase), "+r"(fbase));
        int it = 0;
        // the CTA's j-th tile is blockIdx.x + j gridDim.x; group grp takes j = grp, grp + 2, ...
        for (int64_t tile = blockIdx.x + (int64_t)grp * gridDim.x; tile < ntiles; tile += (int64_t)GROUPS * gridDim.x) {
            const int p0 = (int)(tile * TP);
            for (int sb = 0; sb < nsb; ++sb)
                for (int si = 0; si < nst; ++si, ++it) {
                    const int stg = it % STAGES;
                    mbar_wait(ebase + 8u * (uint32_t)stg, ((uint32_t)(it / STAGES) & 1u) ^ 1u);
                    Stage& S = sm.st[grp][stg];
                    const uint32_t bar = fbase + 8u * (uint32_t)stg;
                    ring_expect(bar, STAGE_BYTES, lane);  // out-of-range features / points / samples are zero-filled and counted
                    if (lane == 0) {
                        tma_load_2d(smem_u32(S.a), &tmx, si * KT, p0, bar);
                        tma_load_2d(smem_u32(S.b), &tmw, si * KT, sb * TS, bar);
                    }
                }
        }
        return;
    }

    asm volatile("setmaxnreg.inc.sync.aligned.u32 232;");  // 128 x 40 + 256 x 232 = 384 x 168
    const int grp = warp / GROUP_WARPS, wq = warp % GROUP_WARPS, g = lane >> 2, kq = lane & 3;
    int off[4];  // swizzled offset of (row g, feature 4 j + kq) within an 8-row block
#pragma unroll
    for (int j = 0; j < 4; ++j) off[j] = swz128(g, j * 4 + kq);
    if (grp == 1) mbar_wait(smem_u32(&sm.go), 0u);  // start half a tile behind group 0
    int it = 0;
    bool first = true;
    for (int64_t tile = blockIdx.x + (int64_t)grp * gridDim.x; tile < ntiles; tile += (int64_t)GROUPS * gridDim.x) {
        const int64_t p0 = tile * TP;
        for (int sb = 0; sb < nsb; ++sb) {
            double acc[4][8][2];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 8; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
            for (int si = 0; si < nst; ++si, ++it) {
                const int stg = it % STAGES;
                mbar_wait(smem_u32(&sm.full[grp][stg]), (uint32_t)(it / STAGES) & 1u);
                const Stage& S = sm.st[grp][stg];
#pragma unroll
                for (int kk = 0; kk < KT / 4; ++kk) {
                    const double* Ah = S.a + wq * 32 * 16 + off[kk];
                    const double* Bh = S.b + off[kk];
                    double a[4], b[8];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi) a[mi] = Ah[mi * 8 * 16];
#pragma unroll
                    for (int ni = 0; ni < 8; ++ni) b[ni] = Bh[ni * 8 * 16];
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                        for (int ni = 0; ni < 8; ++ni) dmma884(acc[mi][ni], a[mi], b[ni]);
                }
                ring_release(smem_u32(&sm.empty[grp][stg]), lane);
                if (first && grp == 0 && warp == 0 && lane == 0 && sb == 0 && si == nst / 2) mbar_arrive(smem_u32(&sm.go));
            }
            first = false;
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int64_t n = p0 + wq * 32 + mi * 8 + g;
                if (n < p.N) {
                    const double sd = sqrt(p.sigma2 ? p.sigma2[n] : p.sigma2_scalar);
#pragma unroll
                    for (int nh = 0; nh < 2; ++nh) {
                        const int s0 = sb * TS + nh * 32 + kq * 2;  // even; samples s0 + 8 j + {0, 1}
                        if (s0 < p.S)
                            rand_emit4(p.Y, p.Zy, p.ldy, p.ldz, p.S, p.seed, (uint64_t)p.n_global, (uint64_t)p.N_global, n, s0, sd, acc[mi][4 * nh][0], acc[mi][4 * nh][1], acc[mi][4 * nh + 1][0],
                                       acc[mi][4 * nh + 1][1], acc[mi][4 * nh + 2][0], acc[mi][4 * nh + 2][1], acc[mi][4 * nh + 3][0],
                                       acc[mi][4 * nh + 3][1]);
                    }
                }
            }
        }
    }
}

// One launch of the two-group kernel on points [n0, n0 + cnt) of x
static int launch_rand_pp(blr_ctx* ctx, const blr_x* x, int64_t n0, int64_t cnt, const double* Wsamp_dev, int64_t S,
                          const double* sigma2, double sigma2_scalar, const double* Zy, int64_t ldz, uint64_t seed, double* Y_dev) {
    RandParams rp_;
    rp_.D = (int)x->D;
    rp_.N = cnt;
    rp_.Wt = nullptr;
    rp_.dk = 0;
    rp_.S = (int)S;
    rp_.sigma2 = sigma2 ? sigma2 + n0 : nullptr;
    rp_.sigma2_scalar = sigma2_scalar;
    rp_.Zy = Zy;
    rp_.seed = seed;
    rp_.noise = true;
    rp_.Y = Y_dev + n0;
    rp_.ldy = x->N;
    rp_.ldz = ldz;
    rp_.n_global = n0;
    rp_.N_global = x->N;
    const int smem = (int)sizeof(rp::Smem) + 1024;
    CUtensorMap tmx, tmw;
    BLR_TRY(make_tmap_2d_f64(ctx, &tmx, x->p + n0 * x->ld, (uint64_t)x->D, (uint64_t)cnt, (uint64_t)x->ld, 16, rp::TP));
    BLR_TRY(make_tmap_2d_f64(ctx, &tmw, Wsamp_dev, (uint64_t)x->D, (uint64_t)S, (uint64_t)x->D, 16, rp::TS));
    BLR_CUDA_OK(ctx, cudaFuncSetAttribute(rand_pp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int64_t ntiles = (cnt + rp::TP - 1) / rp::TP;
    const int grid = (int)std::min<int64_t>((ntiles + rp::GROUPS - 1) / rp::GROUPS, ctx->sm_count);
    rand_pp_kernel<<<grid, rp::THREADS, smem, ctx->stream>>>(rp_, tmx, tmw);
    BLR_CHECK_LAUNCH(ctx, "rand_pp_kernel");
    return 0;
}

// Wsamp_dev must be 16-byte aligned (it is a TMA source); returns 1 if the variant does not apply.
// Device draws (Zy_dev == nullptr) are UN-FUSED by default: the ~68 scalar fp64 instructions per pair of draws run on the pipe
// DMMA runs on, and inside the GEMM's epilogue they cost 1.8 ms per 2^22 x 64 outputs against ~0.5 ms as a pass of their own
// (rand_draws_kernel, same Philox counters) followed by the supplied-draws epilogue (two loads, two FMAs, two stores).  The
// draws of a chunk of points live in a bounded scratch buffer.
int sample_finite_pp(blr_ctx* ctx, const blr_x* x, const double* Wsamp_dev, int64_t S, const double* sigma2,
                     double sigma2_scalar, const double* Zy_dev, uint64_t seed, double* Y_dev) {
    if ((reinterpret_cast<uintptr_t>(Wsamp_dev) & 15) != 0) return 1;
    const int64_t N = x->N;
    if (Zy_dev || !ctx->rand_unfused) return launch_rand_pp(ctx, x, 0, N, Wsamp_dev, S, sigma2, sigma2_scalar, Zy_dev, N, seed, Y_dev);
    // chunk: <= 64 Mi draws (512 MiB), a multiple of 2 x 128 points x #SMs so that every CTA gets whole tile pairs
    const int64_t unit = (int64_t)rp::TP * rp::GROUPS * ctx->sm_count;
    int64_t chunk = std::max<int64_t>(unit, ((int64_t)1 << 26) / std::max<int64_t>(S, 1) / unit * unit);
    chunk = std::min(chunk, (N + 1) / 2 * 2);
    double* Z = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &Z, (size_t)(chunk * S) * sizeof(double)));
    int rc = 0;
    for (int64_t n0 = 0; n0 < N && rc == 0; n0 += chunk) {
        const int64_t cnt = std::min(chunk, N - n0);
        const int64_t work = (S + 1) / 2 * cnt;
        rand_draws_kernel<<<(int)std::min<int64_t>((work + 255) / 256, (int64_t)ctx->sm_count * 16), 256, 0, ctx->stream>>>(
            Z, chunk, cnt, (int)S, seed, (uint64_t)n0, (uint64_t)N);
        ctx->launches++;
        if (cudaGetLastError() != cudaSuccess) rc = set_err(ctx, BLR_E_CUDA, "launch rand_draws_kernel");
        if (rc == 0) rc = launch_rand_pp(ctx, x, n0, cnt, Wsamp_dev, S, sigma2, sigma2_scalar, Z, chunk, seed, Y_dev);
    }
    dev_free(ctx->stream, Z);
    return rc;
}

}  // namespace blr
