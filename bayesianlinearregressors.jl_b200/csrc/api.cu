// C ABI of libblr_cuda (declared in include/blr_cuda.h): contexts, handles, and the entry points the Julia
// glue / Python host mirror bind.  No torch types, no exceptions across the boundary, no CPU fallback.
#include <dlfcn.h>
#include <math.h>
#include <nccl.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "internal.h"

namespace blr {

int set_err(blr_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    return code;
}
int cuda_fail(blr_ctx* ctx, cudaError_t e, const char* what) {
    if (ctx) ctx->err = std::string(what) + ": " + cudaGetErrorString(e);
    cudaGetLastError();  // clear the sticky-less error state
    return (e == cudaErrorMemoryAllocation) ? BLR_E_NOMEM : BLR_E_CUDA;
}
static int grow(blr_ctx* ctx, double** buf, size_t* cap, size_t bytes) {
    if (*cap >= bytes) return 0;
    if (*buf) {
        BLR_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
        BLR_CUDA_OK(ctx, cudaFree(*buf));
        *buf = nullptr;
        *cap = 0;
    }
    BLR_CUDA_OK(ctx, cudaMalloc(buf, bytes));
    *cap = bytes;
    return 0;
}
cudaError_t dev_alloc(blr_ctx* ctx, double** p, size_t bytes) {
    return cudaMallocAsync(reinterpret_cast<void**>(p), std::max<size_t>(bytes, 16), ctx->stream);
}
void dev_free(cudaStream_t stream, void* p) {
    if (p) cudaFreeAsync(p, stream);
}
int ensure_ws(blr_ctx* ctx, size_t bytes) { return grow(ctx, &ctx->ws, &ctx->ws_bytes, bytes); }
int ensure_nbuf(blr_ctx* ctx, size_t bytes) { return grow(ctx, &ctx->nbuf, &ctx->nbuf_bytes, bytes); }
int ensure_dinv(blr_ctx* ctx, size_t bytes) { return grow(ctx, &ctx->dinv, &ctx->dinv_bytes, bytes); }

// ---------------------------------------------------------------------------------------------- NCCL via dlopen
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*CommGetAsyncError)(ncclComm_t, ncclResult_t*) = nullptr;  // optional
    std::string why;
};
static NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return &api;
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (api.handle) break;
    }
    if (!api.handle) {
        api.why = std::string("dlopen(libnccl.so.2) failed: ") + dlerror();
        return &api;
    }
    api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.handle, "ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.handle, "ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.handle, "ncclCommDestroy");
    api.GroupStart = (decltype(api.GroupStart))dlsym(api.handle, "ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))dlsym(api.handle, "ncclGroupEnd");
    api.AllReduce = (decltype(api.AllReduce))dlsym(api.handle, "ncclAllReduce");
    api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.handle, "ncclGetErrorString");
    api.CommGetAsyncError = (decltype(api.CommGetAsyncError))dlsym(api.handle, "ncclCommGetAsyncError");
    if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllReduce || !api.GetErrorString) {
        api.why = "libnccl is missing required symbols";
        api.handle = nullptr;
    }
    return &api;
}
static int nccl_fail(blr_ctx* ctx, ncclResult_t r, const char* what) {
    NcclApi* a = nccl_api();
    return set_err(ctx, BLR_E_NCCL, std::string(what) + ": " + (a->GetErrorString ? a->GetErrorString(r) : "?"));
}

// require_pd: the caller factorises Σy (`_cholesky(fx.Σy)`, src/bayesian_linear_regression.jl:52,:79), so a non-positive
// variance is a PosDefException.  Scalar noise is checked here (info = 1: Diagonal(Fill(σ², N)) fails at its first entry);
// a vector is checked on the device (Σ log σ² is not finite / check_noise_vector).  mean / var / cov only add diag(Σy) (:37,:42).
// a communicator that hit an asynchronous error (peer died, NVLink fault) reports it here, not through the enqueue call
int nccl_async_check(blr_ctx* ctx) {
    NcclApi* a = nccl_api();
    if (!ctx->nccl_comm || !a->CommGetAsyncError) return 0;
    ncclResult_t st = ncclSuccess;
    const ncclResult_t r = a->CommGetAsyncError((ncclComm_t)ctx->nccl_comm, &st);
    if (r != ncclSuccess) return nccl_fail(ctx, r, "ncclCommGetAsyncError");
    if (st != ncclSuccess && st != ncclInProgress) return nccl_fail(ctx, st, "NCCL asynchronous error");
    return 0;
}

static int noise_args(blr_ctx* ctx, const blr_noise* noise, int64_t N, const double** vec, double* scalar, bool require_pd = false) {
    if (!noise) return set_err(ctx, BLR_E_INVALID, "noise is NULL");
    *vec = nullptr;
    *scalar = 0.0;
    if (noise->kind == BLR_NOISE_SCALAR) {
        *scalar = noise->scalar;
        if (require_pd && N > 0 && !(noise->scalar > 0.0)) {
            set_err(ctx, 1, "observation noise variance is not positive");
            return 1;
        }
        return 0;
    }
    if (noise->kind == BLR_NOISE_VECTOR) {
        if (!noise->vec) return set_err(ctx, BLR_E_INVALID, "noise.vec is NULL");
        if (noise->vec->n != N) return set_err(ctx, BLR_E_DIM, "length(diag(Σy)) != number of inputs");
        *vec = noise->vec->p;
        return 0;
    }
    return set_err(ctx, BLR_E_INVALID, "unknown noise kind");
}

// first index (1-based) with a non-positive (or NaN) variance, or INT_MAX-ish if none: *info = min(*info, n + 1)
__global__ void check_noise_kernel(const double* __restrict__ v, int64_t N, int* __restrict__ info) {
    int bad = 0x7fffffff;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x)
        if (!(v[n] > 0.0)) bad = min(bad, (int)(n + 1 < 0x7ffffffe ? n + 1 : 0x7ffffffe));
    if (bad != 0x7fffffff) atomicMin(info, bad);
}
// Synchronising check (error paths and rand): returns 0 or the PosDefException info of Diagonal(v).
int check_noise_vector(blr_ctx* ctx, const double* v, int64_t N) {
    if (!v || N == 0) return 0;
    int* slot = ctx->d_info + 1;
    const int big = 0x7fffffff;
    BLR_CUDA_OK(ctx, cudaMemcpyAsync(slot, &big, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    check_noise_kernel<<<(int)std::min<int64_t>((N + 255) / 256, ctx->sm_count * 8), 256, 0, ctx->stream>>>(v, N, slot);
    ctx->launches++;
    int info = 0;
    BLR_CUDA_OK(ctx, cudaMemcpyAsync(&info, slot, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    BLR_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    if (info == big) return 0;
    set_err(ctx, info, "observation noise variance is not positive");
    return info;
}

// ---------------------------------------------------------------------------------------------- dense Σy side path
// (SURVEY.md section 8f item 2; reference src/bayesian_linear_regression.jl:79,:81-82 with a dense `_cholesky(fx.Σy)`.)
struct DenseNoise {
    int64_t N = 0;
    double* S = nullptr;     // Σy (N x N, column-major)
    double* L = nullptr;     // lower Cholesky factor, Σy = L L'  (Σy.U' of the reference)
    double* diag = nullptr;  // diag(Σy)
    double* scal = nullptr;  // [0] = logdet Σy
};
__global__ void dense_diag_kernel(const double* __restrict__ S, int64_t N, double* __restrict__ diag) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x)
        diag[i] = S[i * N + i];
}
__global__ void add_to_scalar_kernel(double* __restrict__ dst, const double* __restrict__ src) {
    if (blockIdx.x == 0 && threadIdx.x == 0) dst[0] += src[0];
}
__global__ void add_matrix_kernel(double* __restrict__ C, const double* __restrict__ A, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) C[e] += A[e];
}
static void dense_noise_release(blr_ctx* ctx, DenseNoise* dn) {
    dev_free(ctx->stream, dn->S);
    dn->S = dn->L = dn->diag = dn->scal = nullptr;
}
// uploads Σy, factorises it (PosDefException info > 0 on failure), extracts diag and logdet
static int dense_noise_prepare(blr_ctx* ctx, const blr_noise* noise, int64_t N, DenseNoise* dn) {
    if (!noise->dense) return set_err(ctx, BLR_E_INVALID, "noise.dense is NULL");
    const int64_t ld = noise->dense_ld > 0 ? noise->dense_ld : N;
    if (ld < N) return set_err(ctx, BLR_E_DIM, "size(Σy) does not match the number of inputs");
    if (ctx->nranks > 1) return set_err(ctx, BLR_E_INVALID, "dense observation noise couples observations: single GPU only");
    dn->N = N;
    double* buf = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &buf, (size_t)(2 * N * N + N + 2) * sizeof(double)));
    dn->S = buf;
    dn->L = buf + N * N;
    dn->diag = dn->L + N * N;
    dn->scal = dn->diag + N;
    cudaStream_t sm = ctx->stream;
    cudaError_t e = cudaMemcpy2DAsync(dn->S, (size_t)N * sizeof(double), noise->dense, (size_t)ld * sizeof(double),
                                      (size_t)N * sizeof(double), (size_t)N, cudaMemcpyHostToDevice, sm);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dn->L, dn->S, (size_t)N * N * sizeof(double), cudaMemcpyDeviceToDevice, sm);
    if (e != cudaSuccess) {
        dense_noise_release(ctx, dn);
        return cuda_fail(ctx, e, "upload Σy");
    }
    dense_diag_kernel<<<(int)std::min<int64_t>((N + 255) / 256, 1024), 256, 0, sm>>>(dn->S, N, dn->diag);
    ctx->launches++;
    int rc = potrf_lower(ctx, dn->L, N, ctx->d_info);
    if (rc == 0) rc = logdet_from_chol(ctx, dn->L, N, dn->scal);
    int info = 0;
    if (rc == 0) rc = read_info(ctx, &info);
    if (rc == 0 && info != 0) rc = info;
    if (rc != 0) dense_noise_release(ctx, dn);
    return rc;
}

}  // namespace blr

using namespace blr;

#define CTX_ENTER(ctx)                                                   \
    do {                                                                 \
        if (!(ctx)) return BLR_E_INVALID;                                \
        cudaError_t _e = cudaSetDevice((ctx)->device);                   \
        if (_e != cudaSuccess) return cuda_fail(ctx, _e, "cudaSetDevice"); \
    } while (0)

extern "C" {

int blr_version(void) { return BLR_VERSION; }

int blr_ctx_create(blr_ctx** out, int device) {
    if (!out) return BLR_E_INVALID;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) {
        cudaGetLastError();
        return BLR_E_NODEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return BLR_E_NODEVICE;
    if (prop.major != 10) return BLR_E_NODEVICE;  // sm_100a cubin only: no other architecture, no fallback
    if (cudaSetDevice(device) != cudaSuccess) return BLR_E_CUDA;
    blr_ctx* ctx = new (std::nothrow) blr_ctx();
    if (!ctx) return BLR_E_NOMEM;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    cudaError_t e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    {   // keep freed blocks in the device's default pool: steady-state calls never hit cudaMalloc / cudaFree
        cudaMemPool_t pool;
        if (e == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    for (int i = 0; i < 8 && e == cudaSuccess; ++i) e = cudaEventCreate(&ctx->ev[i]);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->small, (size_t)SMALL_TOTAL * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_info, 8 * sizeof(int));  // [0] Cholesky info, [1] noise flag, [3] watchdog; [4..7] same for the prior's factor
    if (e == cudaSuccess) e = cudaMallocHost(&ctx->h_in, (size_t)(2 * SMALL_VEC + 8) * sizeof(double));
    if (e == cudaSuccess) e = cudaMallocHost(&ctx->h_res, (size_t)(SMALL_VEC + 8) * sizeof(double));
    // copy stream + hand-over events: host-streaming accumulation and the overlapped precision download
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_consumed[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_xstream, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->d_flags, 512 * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(ctx->d_flags, 0, 512 * sizeof(int));
    if (e != cudaSuccess || ctx->sm_count * 16 > SMALL_SC) {
        blr_ctx_destroy(ctx);
        return BLR_E_CUDA;
    }
    ctx->small_bytes = (size_t)SMALL_TOTAL * sizeof(double);
    if (const char* po = getenv("BLR_GRAM_PERIOD_OBS")) {
        const long long v = atoll(po);
        if (v >= 32) ctx->gram_period_obs = v;
    }
    if (const char* st = getenv("BLR_GRAM_STAGES")) ctx->gram_stages = atoi(st);
    if (const char* k = getenv("BLR_GRAM_KT")) {
        if (atoi(k) == 16) ctx->gram_kt = 16;
        if (atoi(k) == 32) ctx->gram_kt = 32;
    }
    if (const char* v = getenv("BLR_DXD")) ctx->dxd_legacy = (strcmp(v, "legacy") == 0) ? 1 : 0;
    if (const char* v = getenv("BLR_FORM")) ctx->form = (strcmp(v, "whitened") == 0) ? BLR_FORM_WHITENED : BLR_FORM_DIRECT;
    if (const char* v = getenv("BLR_GRAM_UNIT")) ctx->gram_unit = atoi(v) != 0 ? 1 : 0;
    if (const char* v = getenv("BLR_GRAM_CS")) ctx->gram_cs = atoi(v) != 0 ? 1 : 0;
    if (const char* v = getenv("BLR_VAR_CFG")) ctx->var_cfg = atoi(v) == 0 ? 0 : 1;
    if (const char* v = getenv("BLR_RAND_PP")) ctx->rand_pp = std::max(0, std::min(2, atoi(v)));
    if (const char* v = getenv("BLR_RAND_UNFUSED")) ctx->rand_unfused = atoi(v) != 0 ? 1 : 0;
    if (const char* v = getenv("BLR_SMALL_RING")) ctx->small_ring = atoi(v) != 0 ? 1 : 0;
    if (const char* v = getenv("BLR_MID_RING")) ctx->mid_ring = atoi(v) != 0 ? 1 : 0;
    if (const char* v = getenv("BLR_VAR_SMALL_MAX")) ctx->var_small_max = std::max(64, std::min(128, atoi(v)));
    if (const char* w = getenv("BLR_DIAG_WEIGHT")) {
        const int v = atoi(w);
        if (v >= 8 && v <= 128) ctx->diag_weight = v;
    }
    *out = ctx;
    return 0;
}

int blr_ctx_destroy(blr_ctx* ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    blr_comm_destroy(ctx);
    cudaFree(ctx->ws);
    cudaFree(ctx->nbuf);
    cudaFree(ctx->dinv);
    cudaFree(ctx->small);
    cudaFree(ctx->d_info);
    if (ctx->h_res) cudaFreeHost(ctx->h_res);
    if (ctx->h_in) cudaFreeHost(ctx->h_in);
    cudaFree(ctx->d_flags);
    cudaFree(ctx->tflags);
    cudaFree(ctx->sched);
    cudaFree(ctx->stage[0]);
    cudaFree(ctx->stage[1]);
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
        if (ctx->ev_consumed[i]) cudaEventDestroy(ctx->ev_consumed[i]);
    }
    if (ctx->ev_xstream) cudaEventDestroy(ctx->ev_xstream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    for (int i = 0; i < 8; ++i)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return 0;
}

const char* blr_last_error(const blr_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int blr_ctx_sync(blr_ctx* ctx) {
    CTX_ENTER(ctx);
    BLR_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
int blr_ctx_set_form(blr_ctx* ctx, int form) {
    if (!ctx) return BLR_E_INVALID;
    if (form != BLR_FORM_DIRECT && form != BLR_FORM_WHITENED) return set_err(ctx, BLR_E_INVALID, "unknown numerical form");
    ctx->form = form;
    return 0;
}

int blr_ctx_get_form(const blr_ctx* ctx, int* form_out) {
    if (!ctx || !form_out) return BLR_E_INVALID;
    *form_out = ctx->form;
    return 0;
}

int blr_ctx_stream(blr_ctx* ctx, void** stream_out) {
    if (!ctx || !stream_out) return BLR_E_INVALID;
    *stream_out = (void*)ctx->stream;
    return 0;
}
// Order this context's stream after everything already enqueued on `producer` (a cudaStream_t of the same device; NULL = the
// legacy default stream): borrowed device buffers (blr_x_wrap_device / blr_vec_wrap_device) written by another stream.
int blr_ctx_wait_stream(blr_ctx* ctx, void* producer) {
    CTX_ENTER(ctx);
    BLR_CUDA_OK(ctx, cudaEventRecord(ctx->ev_xstream, (cudaStream_t)producer));
    BLR_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_xstream, 0));
    return 0;
}
// The other direction: make `consumer` wait for everything enqueued on this context's stream (results written into borrowed
// device buffers by the *_dev entry points).
int blr_stream_wait_ctx(blr_ctx* ctx, void* consumer) {
    CTX_ENTER(ctx);
    BLR_CUDA_OK(ctx, cudaEventRecord(ctx->ev_xstream, ctx->stream));
    BLR_CUDA_OK(ctx, cudaStreamWaitEvent((cudaStream_t)consumer, ctx->ev_xstream, 0));
    return 0;
}
int64_t blr_launch_count(const blr_ctx* ctx) { return ctx ? ctx->launches : 0; }

int blr_last_timings(blr_ctx* ctx, double* out8) {
    CTX_ENTER(ctx);
    if (!out8) return BLR_E_INVALID;
    for (int i = 0; i < 8; ++i) out8[i] = 0.0;
    BLR_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    float ms;
    if (ctx->ev_valid[0]) {
        for (int i = 0; i < 3; ++i) {
            BLR_CUDA_OK(ctx, cudaEventElapsedTime(&ms, ctx->ev[i], ctx->ev[i + 1]));
            out8[i] = ms;
        }
    }
    if (ctx->ev_valid[3]) {
        BLR_CUDA_OK(ctx, cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]));
        out8[3] = ms;
    }
    return 0;
}

int blr_host_alloc(blr_ctx* ctx, int64_t bytes, void** out) {
    CTX_ENTER(ctx);
    if (!out || bytes < 0) return BLR_E_INVALID;
    *out = nullptr;
    BLR_CUDA_OK(ctx, cudaHostAlloc(out, (size_t)std::max<int64_t>(bytes, 8), cudaHostAllocDefault));
    return 0;
}
int blr_host_free(blr_ctx* ctx, void* p) {
    if (!p) return 0;
    if (ctx) cudaSetDevice(ctx->device);
    cudaFreeHost(p);
    return 0;
}

// ---------------------------------------------------------------------------------------------- NCCL
int blr_nccl_unique_id(void* out128) {
    NcclApi* a = nccl_api();
    if (!a->handle || !out128) return BLR_E_NCCL;
    ncclUniqueId id;
    if (a->GetUniqueId(&id) != ncclSuccess) return BLR_E_NCCL;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(out128, &id, 128);
    return 0;
}
int blr_comm_init_rank(blr_ctx* ctx, const void* id128, int nranks, int rank) {
    CTX_ENTER(ctx);
    NcclApi* a = nccl_api();
    if (!a->handle) return set_err(ctx, BLR_E_NCCL, a->why);
    if (!id128 || nranks < 1 || rank < 0 || rank >= nranks) return set_err(ctx, BLR_E_INVALID, "bad communicator args");
    blr_comm_destroy(ctx);
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclComm_t comm;
    ncclResult_t r = a->CommInitRank(&comm, nranks, id, rank);
    if (r != ncclSuccess) return nccl_fail(ctx, r, "ncclCommInitRank");
    ctx->nccl_comm = (void*)comm;
    ctx->nranks = nranks;
    ctx->rank = rank;
    return 0;
}
// One process driving several GPUs (one context per device -- a Julia session): rank i = ctxs[i].  The n
// ncclCommInitRank calls must be in flight together, hence the group.
int blr_comm_init_all(blr_ctx** ctxs, int n) {
    if (!ctxs || n < 1) return BLR_E_INVALID;
    for (int i = 0; i < n; ++i)
        if (!ctxs[i]) return BLR_E_INVALID;
    NcclApi* a = nccl_api();
    if (!a->handle || !a->GroupStart || !a->GroupEnd) return set_err(ctxs[0], BLR_E_NCCL, a->handle ? "libnccl lacks group calls" : a->why);
    for (int i = 0; i < n; ++i) blr_comm_destroy(ctxs[i]);
    if (n == 1) return 0;
    ncclUniqueId id;
    ncclResult_t r = a->GetUniqueId(&id);
    if (r != ncclSuccess) return nccl_fail(ctxs[0], r, "ncclGetUniqueId");
    std::vector<ncclComm_t> comms((size_t)n, nullptr);
    r = a->GroupStart();
    for (int i = 0; i < n && r == ncclSuccess; ++i) {
        cudaSetDevice(ctxs[i]->device);
        r = a->CommInitRank(&comms[(size_t)i], n, id, i);
    }
    const ncclResult_t re = a->GroupEnd();
    if (r == ncclSuccess) r = re;
    if (r != ncclSuccess) return nccl_fail(ctxs[0], r, "ncclCommInitRank (group)");
    for (int i = 0; i < n; ++i) {
        ctxs[i]->nccl_comm = (void*)comms[(size_t)i];
        ctxs[i]->nranks = n;
        ctxs[i]->rank = i;
    }
    return 0;
}
// Grouped in-place sum of stats[i] (resident on ctxs[i]'s device) over the contexts of a blr_comm_init_all communicator.
int blr_stats_allreduce_all(blr_ctx** ctxs, blr_stats** stats, int n) {
    if (!ctxs || !stats || n < 1) return BLR_E_INVALID;
    if (n == 1) return 0;
    NcclApi* a = nccl_api();
    if (!a->handle || !a->GroupStart || !a->GroupEnd) return set_err(ctxs[0], BLR_E_NCCL, a->handle ? "libnccl lacks group calls" : a->why);
    for (int i = 0; i < n; ++i) {
        if (!ctxs[i] || !stats[i] || !ctxs[i]->nccl_comm || ctxs[i]->nranks != n)
            return set_err(ctxs[0], BLR_E_INVALID, "contexts are not the n ranks of one communicator");
        if (stats[i]->len() != stats[0]->len()) return set_err(ctxs[0], BLR_E_DIM, "statistics of different dimension");
    }
    ncclResult_t r = a->GroupStart();
    for (int i = 0; i < n && r == ncclSuccess; ++i) {
        cudaSetDevice(ctxs[i]->device);
        r = a->AllReduce(stats[i]->p, stats[i]->p, (size_t)stats[i]->len(), ncclFloat64, ncclSum, (ncclComm_t)ctxs[i]->nccl_comm,
                         ctxs[i]->stream);
    }
    const ncclResult_t re = a->GroupEnd();
    if (r == ncclSuccess) r = re;
    if (r != ncclSuccess) return nccl_fail(ctxs[0], r, "ncclAllReduce (group)");
    for (int i = 0; i < n; ++i) BLR_TRY(nccl_async_check(ctxs[i]));
    return 0;
}
int blr_comm_destroy(blr_ctx* ctx) {
    if (!ctx || !ctx->nccl_comm) return 0;
    NcclApi* a = nccl_api();
    if (a->handle) a->CommDestroy((ncclComm_t)ctx->nccl_comm);
    ctx->nccl_comm = nullptr;
    ctx->nranks = 1;
    ctx->rank = 0;
    return 0;
}

// ---------------------------------------------------------------------------------------------- handles
static int check_x_shape(blr_ctx* ctx, int64_t D, int64_t N, int64_t ld, int layout) {
    if (D < 1 || N < 0) return set_err(ctx, BLR_E_INVALID, "bad design-matrix shape");
    if (layout != BLR_COLVECS && layout != BLR_ROWVECS) return set_err(ctx, BLR_E_INVALID, "unknown layout");
    const int64_t rows = (layout == BLR_COLVECS) ? D : N;
    if (ld < std::max<int64_t>(rows, 1)) return set_err(ctx, BLR_E_INVALID, "leading dimension too small");
    return 0;
}

int blr_x_alloc(blr_ctx* ctx, int64_t D, int64_t N, int layout, blr_x** out) {
    CTX_ENTER(ctx);
    if (!out) return BLR_E_INVALID;
    const int64_t rows = (layout == BLR_COLVECS) ? D : N, cols = (layout == BLR_COLVECS) ? N : D;
    const int64_t ld = std::max<int64_t>(rows + (rows & 1), 2);  // even leading dimension: 16-byte aligned columns
    BLR_TRY(check_x_shape(ctx, D, N, ld, layout));
    blr_x* x = new blr_x();
    x->D = D;
    x->N = N;
    x->ld = ld;
    x->layout = layout;
    x->owned = true;
    // stream-ordered pool: a feature map re-evaluated per call (blr_x_rff) must not pay cudaMalloc / cudaFree each time
    cudaError_t e = dev_alloc(ctx, &x->p, (size_t)ld * cols * sizeof(double));
    if (e != cudaSuccess) {
        delete x;
        return cuda_fail(ctx, e, "cudaMallocAsync(X)");
    }
    *out = x;
    return 0;
}

int blr_x_upload(blr_ctx* ctx, const double* host, int64_t D, int64_t N, int64_t ld, int layout, blr_x** out) {
    CTX_ENTER(ctx);
    if (!out || (!host && N > 0)) return set_err(ctx, BLR_E_INVALID, "null pointer");
    BLR_TRY(check_x_shape(ctx, D, N, ld, layout));
    blr_x* x = nullptr;
    BLR_TRY(blr_x_alloc(ctx, D, N, layout, &x));
    const int64_t rows = (layout == BLR_COLVECS) ? D : N, cols = (layout == BLR_COLVECS) ? N : D;
    if (rows > 0 && cols > 0) {
        cudaError_t e = cudaMemcpy2DAsync(x->p, (size_t)x->ld * sizeof(double), host, (size_t)ld * sizeof(double),
                                          (size_t)rows * sizeof(double), (size_t)cols, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            blr_x_free(ctx, x);
            return cuda_fail(ctx, e, "upload X");
        }
    }
    *out = x;
    return 0;
}

int blr_x_wrap_device(blr_ctx* ctx, const double* dev, int64_t D, int64_t N, int64_t ld, int layout, blr_x** out) {
    if (!ctx || !out || !dev) return BLR_E_INVALID;
    BLR_TRY(check_x_shape(ctx, D, N, ld, layout));
    blr_x* x = new blr_x();
    x->p = const_cast<double*>(dev);
    x->D = D;
    x->N = N;
    x->ld = ld;
    x->layout = layout;
    x->owned = false;
    *out = x;
    return 0;
}

int blr_x_device_ptr(blr_ctx* ctx, const blr_x* x, double** dev_out, int64_t* ld_out) {
    if (!ctx || !x) return BLR_E_INVALID;
    if (dev_out) *dev_out = x->p;
    if (ld_out) *ld_out = x->ld;
    return 0;
}

int blr_x_free(blr_ctx* ctx, blr_x* x) {
    if (!x) return 0;
    if (ctx) cudaSetDevice(ctx->device);
    if (x->owned && x->p) {
        if (ctx && ctx->stream)
            dev_free(ctx->stream, x->p);
        else
            cudaFree(x->p);
    }
    delete x;
    return 0;
}

int blr_vec_alloc(blr_ctx* ctx, int64_t n, blr_vec** out) {
    CTX_ENTER(ctx);
    if (!out || n < 0) return BLR_E_INVALID;
    blr_vec* v = new blr_vec();
    v->n = n;
    v->owned = true;
    cudaError_t e = dev_alloc(ctx, &v->p, (size_t)n * sizeof(double));
    if (e != cudaSuccess) {
        delete v;
        return cuda_fail(ctx, e, "cudaMallocAsync(vec)");
    }
    *out = v;
    return 0;
}
int blr_vec_upload(blr_ctx* ctx, const double* host, int64_t n, blr_vec** out) {
    CTX_ENTER(ctx);
    if (!out || (!host && n > 0)) return set_err(ctx, BLR_E_INVALID, "null pointer");
    blr_vec* v = nullptr;
    BLR_TRY(blr_vec_alloc(ctx, n, &v));
    if (n > 0) {
        cudaError_t e = cudaMemcpyAsync(v->p, host, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) {
            blr_vec_free(ctx, v);
            return cuda_fail(ctx, e, "upload vec");
        }
    }
    *out = v;
    return 0;
}
int blr_vec_wrap_device(blr_ctx* ctx, const double* dev, int64_t n, blr_vec** out) {
    if (!ctx || !out || !dev || n < 0) return BLR_E_INVALID;
    blr_vec* v = new blr_vec();
    v->p = const_cast<double*>(dev);
    v->n = n;
    v->owned = false;
    *out = v;
    return 0;
}
int blr_vec_device_ptr(blr_ctx* ctx, const blr_vec* v, double** dev_out) {
    if (!ctx || !v || !dev_out) return BLR_E_INVALID;
    *dev_out = v->p;
    return 0;
}
int blr_vec_download(blr_ctx* ctx, const blr_vec* v, double* host) {
    CTX_ENTER(ctx);
    if (!v || !host) return BLR_E_INVALID;
    if (v->n == 0) return 0;
    BLR_CUDA_OK(ctx, cudaMemcpyAsync(host, v->p, (size_t)v->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    BLR_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
int blr_vec_free(blr_ctx* ctx, blr_vec* v) {
    if (!v) return 0;
    if (ctx) cudaSetDevice(ctx->device);
    if (v->owned && v->p) {
        if (ctx && ctx->stream)
            dev_free(ctx->stream, v->p);
        else
            cudaFree(v->p);
    }
    delete v;
    return 0;
}

// ---------------------------------------------------------------------------------------------- synthetic data
int blr_x_synth(blr_ctx* ctx, blr_x* x, uint64_t seed, int64_t n_offset) {
    CTX_ENTER(ctx);
    if (!x) return BLR_E_INVALID;
    if (x->layout != BLR_COLVECS) return set_err(ctx, BLR_E_INVALID, "blr_x_synth generates ColVecs data");
    return synth_normal(ctx, x->p, x->D, x->N, x->ld, seed, 0, n_offset);
}
int blr_vec_synth_noise(blr_ctx* ctx, blr_vec* sigma2, uint64_t seed, int64_t n_offset) {
    CTX_ENTER(ctx);
    if (!sigma2) return BLR_E_INVALID;
    return synth_noise(ctx, sigma2->p, sigma2->n, seed, n_offset);
}
int blr_vec_synth_targets(blr_ctx* ctx, const blr_x* x, const blr_vec* sigma2, uint64_t seed, int64_t n_offset,
                          blr_vec* y) {
    CTX_ENTER(ctx);
    if (!x || !sigma2 || !y) return BLR_E_INVALID;
    if (sigma2->n != x->N || y->n != x->N) return set_err(ctx, BLR_E_DIM, "vector lengths do not match X");
    return synth_targets(ctx, x, sigma2->p, seed, n_offset, y->p);
}

int blr_x_features(blr_ctx* ctx, const blr_x* xin, const double* W, const double* b, int64_t D, int act, double scale,
                   blr_x** out) {
    CTX_ENTER(ctx);
    if (!xin || !W || !b || !out || D < 1) return set_err(ctx, BLR_E_INVALID, "bad feature-map arguments");
    const int64_t din = xin->D;
    double *Wd = nullptr, *bd = nullptr;
    blr_x* phi = nullptr;
    BLR_TRY(blr_x_alloc(ctx, D, xin->N, BLR_COLVECS, &phi));
    cudaError_t e = dev_alloc(ctx, &Wd, (size_t)D * din * sizeof(double));
    if (e == cudaSuccess) e = dev_alloc(ctx, &bd, (size_t)D * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpyAsync(Wd, W, (size_t)D * din * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(bd, b, (size_t)D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    int rc = (e == cudaSuccess) ? affine_features(ctx, xin, Wd, bd, D, act, scale, phi->p, phi->ld) : cuda_fail(ctx, e, "feature-map upload");
    dev_free(ctx->stream, Wd);
    dev_free(ctx->stream, bd);
    if (rc != 0) {
        blr_x_free(ctx, phi);
        return rc;
    }
    *out = phi;
    return 0;
}
int blr_x_rff(blr_ctx* ctx, const blr_x* xin, const double* W, const double* b, int64_t D, blr_x** out) {
    return blr_x_features(ctx, xin, W, b, D, BLR_ACT_COS, sqrt(2.0 / (double)(D > 0 ? D : 1)), out);
}

int blr_x_features_vjp(blr_ctx* ctx, const blr_x* xin, const double* W, const double* b, int64_t D, int act, double scale,
                       const double* dphi_dev, int64_t ld_dphi, double* dW_host, double* db_host, double* dxin_dev, int64_t ld_dxin) {
    CTX_ENTER(ctx);
    if (!xin || !W || !b || !dphi_dev || D < 1) return set_err(ctx, BLR_E_INVALID, "bad feature-map VJP arguments");
    if (xin->layout != BLR_COLVECS) return set_err(ctx, BLR_E_INVALID, "device feature maps expect ColVecs inputs");
    const int64_t din = xin->D, N = xin->N;
    if (din < 1 || din > 384) return set_err(ctx, BLR_E_INVALID, "device feature map: d_in must be 1 .. 384");
    if (act < BLR_ACT_COS || act > BLR_ACT_SIN) return set_err(ctx, BLR_E_INVALID, "unknown activation");
    if (ld_dphi < D) return set_err(ctx, BLR_E_INVALID, "ld_dphi too small");
    if (dxin_dev && ld_dxin < din) return set_err(ctx, BLR_E_INVALID, "ld_dxin too small");
    const bool want_wb = dW_host || db_host;
    if (!want_wb && !dxin_dev) return 0;

    // device scratch: [W (D x d_in) | b (D) | dW, db (D x (d_in + 1)) | per-range partials (S x D x (d_in + 1))]
    const int64_t len = D * (din + 1);
    const int S = (want_wb && N > 0) ? features_vjp_splits(ctx, N, D, din) : 0;
    double* buf = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &buf, (size_t)(D * din + D + (want_wb ? len * (1 + S) : 0)) * sizeof(double)));
    double *Wd = buf, *bd = Wd + D * din, *dWb = bd + D, *ws = dWb + len;
    auto done = [&](int rc) {
        dev_free(ctx->stream, buf);
        return rc;
    };
    cudaError_t e = cudaMemcpyAsync(Wd, W, (size_t)D * din * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(bd, b, (size_t)D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && want_wb && N == 0) e = cudaMemsetAsync(dWb, 0, (size_t)len * sizeof(double), ctx->stream);
    if (e != cudaSuccess) return done(cuda_fail(ctx, e, "feature-map VJP upload"));
    if (N > 0) {
        const int rc = features_vjp(ctx, xin, Wd, bd, D, act, scale, dphi_dev, ld_dphi, want_wb ? dWb : nullptr, ws, S, dW_host != nullptr,
                                    dxin_dev, ld_dxin);
        if (rc != 0) return done(rc);
    }
    if (want_wb && ctx->nccl_comm && ctx->nranks > 1) {
        // [dW | db] in one all-reduce, or the db column alone when dW is not requested
        const int64_t off = dW_host ? 0 : D * din;
        NcclApi* a = nccl_api();
        ncclResult_t r = a->AllReduce(dWb + off, dWb + off, (size_t)(len - off), ncclFloat64, ncclSum, (ncclComm_t)ctx->nccl_comm,
                                      ctx->stream);
        const int rc = (r != ncclSuccess) ? nccl_fail(ctx, r, "ncclAllReduce") : nccl_async_check(ctx);
        if (rc != 0) return done(rc);
    }
    if (dW_host) e = cudaMemcpyAsync(dW_host, dWb, (size_t)D * din * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && db_host) e = cudaMemcpyAsync(db_host, dWb + D * din, (size_t)D * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return done(cuda_fail(ctx, e, "download feature-map gradients"));
    return done(0);
}

// ---------------------------------------------------------------------------------------------- inference
int blr_stats_create(blr_ctx* ctx, int64_t D, blr_stats** out) {
    CTX_ENTER(ctx);
    if (!out || D < 1 || D > SMALL_VEC) return set_err(ctx, BLR_E_INVALID, "bad D (1 <= D <= 16384)");
    blr_stats* s = new blr_stats();
    s->D = D;
    cudaError_t e = dev_alloc(ctx, &s->p, (size_t)s->len() * sizeof(double));
    if (e != cudaSuccess) {
        delete s;
        return cuda_fail(ctx, e, "cudaMallocAsync(stats)");
    }
    *out = s;
    return blr_stats_zero(ctx, s);
}
int blr_stats_free(blr_ctx* ctx, blr_stats* s) {
    if (!s) return 0;
    if (ctx) {
        cudaSetDevice(ctx->device);
        dev_free(ctx->stream, s->p);
    } else {
        cudaFree(s->p);
    }
    delete s;
    return 0;
}
int blr_stats_zero(blr_ctx* ctx, blr_stats* s) {
    CTX_ENTER(ctx);
    if (!s) return BLR_E_INVALID;
    BLR_CUDA_OK(ctx, cudaMemsetAsync(s->p, 0, (size_t)s->len() * sizeof(double), ctx->stream));
    return 0;
}

int blr_stats_accumulate(blr_ctx* ctx, blr_stats* s, const double* mw_host, const blr_x* x, const blr_vec* y,
                         const blr_noise* noise) {
    CTX_ENTER(ctx);
    if (!s || !x || !y || !mw_host) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (x->D != s->D) return set_err(ctx, BLR_E_INVALID, "size(X, 1) != length(mw)");
    if (y->n != x->N) return set_err(ctx, BLR_E_DIM, "length(y) != size(fx.x.X, 2)");
    if (noise && noise->kind == BLR_NOISE_DENSE) {
        // whiten with the factor of Σy and reuse the diagonal-noise path:  à = L^-1 X' (N x D, a RowVecs matrix),
        // ỹ = L^-1 y, unit noise;  logdet Σy is added to ℓ afterwards.
        const int64_t N = x->N, D = x->D;
        if (N == 0) return 0;
        DenseNoise dn;
        BLR_TRY(dense_noise_prepare(ctx, noise, N, &dn));
        double* buf = nullptr;
        cudaError_t e = dev_alloc(ctx, &buf, (size_t)(N * N + N * D + N) * sizeof(double));
        if (e != cudaSuccess) {
            dense_noise_release(ctx, &dn);
            return cuda_fail(ctx, e, "cudaMallocAsync(whiten)");
        }
        double *Wy = buf, *At = buf + N * N, *yt = At + N * D;
        const bool colv = x->layout == BLR_COLVECS;
        int rc = trtri_lower(ctx, dn.L, Wy, N);
        // Ã[n, d] = Σ_m Wy[n, m] X[d, m]
        if (rc == 0) rc = gemm_generic(ctx, N, D, N, Wy, 1, N, x->p, colv ? x->ld : 1, colv ? 1 : x->ld, At, 1, N, 0.0);
        if (rc == 0) rc = gemm_generic(ctx, N, 1, N, Wy, 1, N, y->p, 1, N, yt, 1, N, 0.0);
        if (rc == 0) {
            bool zero = true;
            for (int64_t i = 0; i < D; ++i)
                if (mw_host[i] != 0.0) zero = false;
            double* mwd = ctx->small + SMALL_MW;
            if (!zero) {
                e = cudaMemcpyAsync(mwd, mw_host, (size_t)D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
                if (e != cudaSuccess) rc = cuda_fail(ctx, e, "upload mw");
            }
            blr_x xw;
            xw.p = At;
            xw.D = D;
            xw.N = N;
            xw.ld = N;
            xw.layout = BLR_ROWVECS;
            if (rc == 0) rc = gram_accumulate(ctx, s, mwd, zero, &xw, yt, nullptr, 1.0);
        }
        if (rc == 0) {
            add_to_scalar_kernel<<<1, 32, 0, ctx->stream>>>(s->scal() + 1, dn.scal);
            ctx->launches++;
        }
        dev_free(ctx->stream, buf);
        dense_noise_release(ctx, &dn);
        return rc;
    }
    const double* sig = nullptr;
    double sig_scalar = 0.0;
    BLR_TRY(noise_args(ctx, noise, x->N, &sig, &sig_scalar, true));
    bool zero = true;
    for (int64_t i = 0; i < s->D; ++i)
        if (mw_host[i] != 0.0) {
            zero = false;
            break;
        }
    double* mwd = ctx->small + SMALL_MW;
    if (!zero)
        BLR_CUDA_OK(ctx, cudaMemcpyAsync(mwd, mw_host, (size_t)s->D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    return gram_accumulate(ctx, s, mwd, zero, x, y->p, sig, sig_scalar);
}

int blr_stats_accumulate_host(blr_ctx* ctx, blr_stats* s, const double* mw_host, const double* X, int64_t D, int64_t N,
                              int64_t ld, int layout, const double* y, int noise_kind, double noise_scalar,
                              const double* sigma2_host, int64_t chunk) {
    CTX_ENTER(ctx);
    if (!s || !mw_host || (N > 0 && (!X || !y))) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (D != s->D) return set_err(ctx, BLR_E_INVALID, "size(X, 1) != length(mw)");
    BLR_TRY(check_x_shape(ctx, D, N, ld, layout));
    if (noise_kind != BLR_NOISE_SCALAR && noise_kind != BLR_NOISE_VECTOR) return set_err(ctx, BLR_E_INVALID, "unknown noise kind");
    if (noise_kind == BLR_NOISE_VECTOR && N > 0 && !sigma2_host) return set_err(ctx, BLR_E_INVALID, "sigma2_host is NULL");
    if (N == 0) return 0;
    if (noise_kind == BLR_NOISE_SCALAR && !(noise_scalar > 0.0)) {  // cholesky(Diagonal(Fill(σ², N))) fails at entry 1
        set_err(ctx, 1, "observation noise variance is not positive");
        return 1;
    }
    if (chunk <= 0) chunk = 1 << 16;
    chunk = std::min<int64_t>((chunk + 15) / 16 * 16, (N + 15) / 16 * 16);
    // staging slot: X chunk (D x chunk, ld = D rounded to even; or chunk x D) | y chunk | σ² chunk
    const int64_t ldx = (layout == BLR_COLVECS) ? D + (D & 1) : chunk;
    const size_t x_elems = (size_t)((layout == BLR_COLVECS) ? ldx * chunk : chunk * D);
    const size_t slot_bytes = (x_elems + 2 * (size_t)chunk) * sizeof(double);
    if (ctx->stage_bytes < slot_bytes) {
        BLR_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
        BLR_CUDA_OK(ctx, cudaStreamSynchronize(ctx->copy_stream));
        for (int i = 0; i < 2; ++i) {
            if (ctx->stage[i]) BLR_CUDA_OK(ctx, cudaFree(ctx->stage[i]));
            ctx->stage[i] = nullptr;
        }
        ctx->stage_bytes = 0;
        for (int i = 0; i < 2; ++i) BLR_CUDA_OK(ctx, cudaMalloc(&ctx->stage[i], slot_bytes));
        ctx->stage_bytes = slot_bytes;
        ctx->stage_used[0] = ctx->stage_used[1] = false;
    }
    bool zero = true;
    for (int64_t i = 0; i < D; ++i)
        if (mw_host[i] != 0.0) {
            zero = false;
            break;
        }
    double* mwd = ctx->small + SMALL_MW;
    if (!zero)
        BLR_CUDA_OK(ctx, cudaMemcpyAsync(mwd, mw_host, (size_t)D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    int it = 0;
    for (int64_t a = 0; a < N; a += chunk, ++it) {
        const int64_t nb = std::min(chunk, N - a);
        const int b = it & 1;
        double* xs = ctx->stage[b];
        double* ys = xs + x_elems;
        double* ss = ys + chunk;
        // the slot may still be read by a Gram kernel of THIS call (it >= 2) or of a previous call on this context (the
        // function returns without synchronising): always order the copy after the slot's last consumer
        if (ctx->stage_used[b]) BLR_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_consumed[b], 0));
        if (layout == BLR_COLVECS && ld == D && ldx == D)  // contiguous block of columns: one linear copy
            BLR_CUDA_OK(ctx, cudaMemcpyAsync(xs, X + a * ld, (size_t)D * nb * sizeof(double), cudaMemcpyHostToDevice,
                                             ctx->copy_stream));
        else if (layout == BLR_COLVECS)
            BLR_CUDA_OK(ctx, cudaMemcpy2DAsync(xs, (size_t)ldx * sizeof(double), X + a * ld, (size_t)ld * sizeof(double),
                                               (size_t)D * sizeof(double), (size_t)nb, cudaMemcpyHostToDevice,
                                               ctx->copy_stream));
        else
            BLR_CUDA_OK(ctx, cudaMemcpy2DAsync(xs, (size_t)ldx * sizeof(double), X + a, (size_t)ld * sizeof(double),
                                               (size_t)nb * sizeof(double), (size_t)D, cudaMemcpyHostToDevice,
                                               ctx->copy_stream));
        BLR_CUDA_OK(ctx, cudaMemcpyAsync(ys, y + a, (size_t)nb * sizeof(double), cudaMemcpyHostToDevice, ctx->copy_stream));
        if (noise_kind == BLR_NOISE_VECTOR)
            BLR_CUDA_OK(ctx, cudaMemcpyAsync(ss, sigma2_host + a, (size_t)nb * sizeof(double), cudaMemcpyHostToDevice,
                                             ctx->copy_stream));
        BLR_CUDA_OK(ctx, cudaEventRecord(ctx->ev_copied[b], ctx->copy_stream));
        BLR_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_copied[b], 0));
        blr_x xv;
        xv.p = xs;
        xv.D = D;
        xv.N = nb;
        xv.ld = ldx;
        xv.layout = layout;
        BLR_TRY(gram_accumulate(ctx, s, mwd, zero, &xv, ys, noise_kind == BLR_NOISE_VECTOR ? ss : nullptr, noise_scalar));
        BLR_CUDA_OK(ctx, cudaEventRecord(ctx->ev_consumed[b], ctx->stream));
        ctx->stage_used[b] = true;
    }
    return 0;
}

int blr_stats_allreduce(blr_ctx* ctx, blr_stats* s) {
    CTX_ENTER(ctx);
    if (!s) return BLR_E_INVALID;
    if (!ctx->nccl_comm || ctx->nranks == 1) return 0;
    NcclApi* a = nccl_api();
    ncclResult_t r =
        a->AllReduce(s->p, s->p, (size_t)s->len(), ncclFloat64, ncclSum, (ncclComm_t)ctx->nccl_comm, ctx->stream);
    if (r != ncclSuccess) return nccl_fail(ctx, r, "ncclAllReduce");
    return nccl_async_check(ctx);
}
int blr_stats_device_ptr(blr_ctx* ctx, const blr_stats* s, double** dev_out, int64_t* len_out) {
    if (!ctx || !s) return BLR_E_INVALID;
    if (dev_out) *dev_out = s->p;
    if (len_out) *len_out = s->len();
    return 0;
}
int blr_stats_download(blr_ctx* ctx, const blr_stats* s, double* host) {
    CTX_ENTER(ctx);
    if (!s || !host) return BLR_E_INVALID;
    BLR_CUDA_OK(ctx, cudaMemcpyAsync(host, s->p, (size_t)s->len() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    BLR_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
int blr_stats_upload(blr_ctx* ctx, blr_stats* s, const double* host) {
    CTX_ENTER(ctx);
    if (!s || !host) return BLR_E_INVALID;
    BLR_CUDA_OK(ctx, cudaMemcpyAsync(s->p, host, (size_t)s->len() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    BLR_CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int blr_infer_from_stats(blr_ctx* ctx, const blr_prior* prior, const blr_stats* s, double* logpdf_out, double* m_post,
                         double* T_post, double* L_post, blr_post** post_out) {
    CTX_ENTER(ctx);
    if (!prior || !s || !prior->mw || !prior->lambda) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (prior->D > 0 && prior->D != s->D) return set_err(ctx, BLR_E_DIM, "length(mw) != dimension of the statistics");
    const int rc = infer_solve(ctx, prior, s, logpdf_out, m_post, T_post, L_post, post_out);
    if (rc == BLR_INFO_NOISE) {  // which entry is not known from the statistics alone: report the first
        set_err(ctx, 1, "observation noise variance is not positive");
        return 1;
    }
    return rc;
}

int blr_infer(blr_ctx* ctx, const blr_prior* prior, const blr_x* x, const blr_vec* y, const blr_noise* noise,
              double* logpdf_out, double* m_post, double* T_post, double* L_post, blr_post** post_out) {
    CTX_ENTER(ctx);
    if (!prior || !x) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (prior->D > 0 && prior->D != x->D) return set_err(ctx, BLR_E_DIM, "size(X, 1) != length(mw)");
    blr_stats* s = nullptr;
    BLR_TRY(blr_stats_create(ctx, x->D, &s));
    int rc = blr_stats_accumulate(ctx, s, prior->mw, x, y, noise);
    if (rc == 0) rc = blr_stats_allreduce(ctx, s);
    if (rc == 0 && (!prior->mw || !prior->lambda)) rc = set_err(ctx, BLR_E_INVALID, "null argument");
    if (rc == 0) rc = infer_solve(ctx, prior, s, logpdf_out, m_post, T_post, L_post, post_out);
    blr_stats_free(ctx, s);
    if (rc == BLR_INFO_NOISE) {
        // Σ log σ² was not finite: some variance is <= 0 (or NaN).  Report Diagonal(σ²)'s PosDefException index when this
        // rank holds the offending entry (another rank's shard may hold it: then the index is not known here).
        int info = 1;
        if (noise && noise->kind == BLR_NOISE_VECTOR && noise->vec) {
            const int loc = check_noise_vector(ctx, noise->vec->p, noise->vec->n);
            if (loc != 0) info = loc;
        }
        set_err(ctx, info, "observation noise variance is not positive");
        return info;
    }
    return rc;
}

// The body of logpdf(fx, Y::AbstractMatrix) shared by blr_logpdf_multi and blr_logpdf_multi_grad (arguments validated, k >= 1):
// accumulate column 0, R = X Σy⁻¹ (Y_j - X'mw) of columns 1 .. k-1, all-reduce, infer_solve, Z_j = L⁻¹ R_j in place.  On
// return the caller owns *s (the reduced statistics), *post (the posterior of column 0) and *extra = [Z (K x D) | q (K) | zz (K) |
// q_0 | z_0'z_0] (K = k - 1; null when K = 0), whatever the status; logpdf_out (host, k) is filled on success.
static int logpdf_multi_forward(blr_ctx* ctx, const blr_prior* prior, const blr_x* x, const double* Y_dev, int64_t ldy, int64_t k,
                                const blr_noise* noise, double* logpdf_out, blr_stats** s_out, blr_post** post_out,
                                double** extra_out) {
    const int64_t D = x->D, N = x->N, K = k - 1;
    blr_vec y0;  // column 0 goes down the ordinary path: Gram statistics, factorisation, logpdf_0
    y0.p = const_cast<double*>(Y_dev);
    y0.n = N;
    BLR_TRY(blr_stats_create(ctx, D, s_out));
    blr_stats* s = *s_out;
    int rc = blr_stats_accumulate(ctx, s, prior->mw, x, &y0, noise);
    if (rc != 0) return rc;
    if (K > 0) {
        cudaError_t e = dev_alloc(ctx, extra_out, (size_t)(K * D + 2 * K + 2) * sizeof(double));
        if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaMallocAsync(logpdf_multi)");
        const double* sig = nullptr;
        double sig_scalar = 0.0;
        rc = noise_args(ctx, noise, N, &sig, &sig_scalar, true);
        if (rc != 0) return rc;
        bool zero = true;
        for (int64_t i = 0; i < D; ++i)
            if (prior->mw[i] != 0.0) zero = false;
        double* pm = nullptr;  // X'mw, shared by every column
        if (!zero && N > 0) {
            e = dev_alloc(ctx, &pm, (size_t)N * sizeof(double));
            if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaMallocAsync(pm)");
            // blr_stats_accumulate left mw in ctx->small + SMALL_MW (stream-ordered)
            rc = apply_weights(ctx, x, ctx->small + SMALL_MW, pm);
        }
        if (rc == 0) rc = rhs_multi(ctx, x, Y_dev + ldy, ldy, K, sig, sig_scalar, pm, *extra_out, *extra_out + K * D);
        dev_free(ctx->stream, pm);
        if (rc != 0) return rc;
    }
    double* extra = *extra_out;
    rc = blr_stats_allreduce(ctx, s);
    if (rc == 0 && K > 0 && ctx->nccl_comm && ctx->nranks > 1) {
        NcclApi* a = nccl_api();
        ncclResult_t r = a->AllReduce(extra, extra, (size_t)(K * D + K), ncclFloat64, ncclSum, (ncclComm_t)ctx->nccl_comm, ctx->stream);
        rc = (r != ncclSuccess) ? nccl_fail(ctx, r, "ncclAllReduce") : nccl_async_check(ctx);
    }
    if (rc != 0) return rc;
    rc = infer_solve(ctx, prior, s, logpdf_out, nullptr, nullptr, nullptr, post_out);
    if (rc == BLR_INFO_NOISE) {
        int info = 1;
        if (noise && noise->kind == BLR_NOISE_VECTOR && noise->vec) {
            const int loc = check_noise_vector(ctx, noise->vec->p, noise->vec->n);
            if (loc != 0) info = loc;
        }
        set_err(ctx, info, "observation noise variance is not positive");
        return info;
    }
    if (rc != 0 || K == 0) return rc;
    // logpdf_j - logpdf_0 = -1/2 [(q_j - q_0) - (z_j'z_j - z_0'z_0)]: every other term of (:57) is common to the columns
    double* tail = extra + K * D;
    BLR_TRY(forward_solve_multi(ctx, *post_out, extra, K, tail + K));
    std::vector<double> h((size_t)(2 * K + 2));
    cudaError_t e = cudaMemcpyAsync(tail + 2 * K, s->scal(), sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(tail + 2 * K + 1, ctx->small + SMALL_SC + 2, sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(h.data(), tail, h.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "download logpdf_multi");
    const double q0 = h[2 * K], zz0 = h[2 * K + 1];
    for (int64_t j = 0; j < K; ++j) logpdf_out[j + 1] = logpdf_out[0] - 0.5 * ((h[j] - q0) - (h[K + j] - zz0));
    return 0;
}

int blr_logpdf_multi(blr_ctx* ctx, const blr_prior* prior, const blr_x* x, const double* Y_dev, int64_t ldy, int64_t k,
                     const blr_noise* noise, double* logpdf_out) {
    CTX_ENTER(ctx);
    if (!prior || !x || !prior->mw || !prior->lambda || (k > 0 && (!Y_dev || !logpdf_out)) || k < 0)
        return set_err(ctx, BLR_E_INVALID, "null argument");
    if (prior->D > 0 && prior->D != x->D) return set_err(ctx, BLR_E_DIM, "size(X, 1) != length(mw)");
    if (k == 0) return 0;
    if (ldy < x->N) return set_err(ctx, BLR_E_DIM, "size(Y, 1) != size(fx.x.X, 2)");
    if (noise && noise->kind == BLR_NOISE_DENSE)
        return set_err(ctx, BLR_E_INVALID, "blr_logpdf_multi: dense Σy is not supported (loop blr_infer over the columns)");
    blr_stats* s = nullptr;
    blr_post* post = nullptr;
    double* extra = nullptr;
    const int rc = logpdf_multi_forward(ctx, prior, x, Y_dev, ldy, k, noise, logpdf_out, &s, &post, &extra);
    dev_free(ctx->stream, extra);
    if (s) blr_stats_free(ctx, s);
    if (post) post_release(post);
    return rc;
}

int blr_logpdf_grad(blr_ctx* ctx, const blr_prior* prior, const blr_x* x, const blr_vec* y, const blr_noise* noise,
                    double* logpdf_out, const blr_logpdf_grads* g) {
    CTX_ENTER(ctx);
    if (!prior || !x || !y || !noise || !prior->mw || !prior->lambda) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (prior->D > 0 && prior->D != x->D) return set_err(ctx, BLR_E_DIM, "size(X, 1) != length(mw)");
    if (y->n != x->N) return set_err(ctx, BLR_E_DIM, "length(y) != size(fx.x.X, 2)");
    if (noise->kind == BLR_NOISE_DENSE) return set_err(ctx, BLR_E_INVALID, "blr_logpdf_grad: dense Σy is not supported");
    const blr_logpdf_grads none = {};
    const blr_logpdf_grads& G = g ? *g : none;
    const bool vector_noise = noise->kind == BLR_NOISE_VECTOR;
    if ((G.dsigma2 && vector_noise) || (G.dsigma2_dev && !vector_noise))
        return set_err(ctx, BLR_E_INVALID, "dsigma2 (scalar noise) / dsigma2_dev (vector noise) does not match the noise kind");
    const int64_t D = x->D, N = x->N;
    if (G.dX_dev && G.ld_dX < std::max<int64_t>(x->layout == BLR_COLVECS ? D : N, 1))
        return set_err(ctx, BLR_E_INVALID, "ld_dX too small");
    const double* sig = nullptr;
    double sig_scalar = 0.0;
    BLR_TRY(noise_args(ctx, noise, N, &sig, &sig_scalar, true));

    // the value: exactly blr_infer's path (accumulate, all-reduce, infer_solve), keeping the posterior
    blr_stats* s = nullptr;
    blr_post* post = nullptr;
    double* buf = nullptr;
    BLR_TRY(blr_stats_create(ctx, D, &s));
    auto done = [&](int rc) {
        dev_free(ctx->stream, buf);
        blr_stats_free(ctx, s);
        if (post) post_release(post);
        return rc;
    };
    int rc = blr_stats_accumulate(ctx, s, prior->mw, x, y, noise);
    if (rc == 0) rc = blr_stats_allreduce(ctx, s);
    if (rc == 0) rc = infer_solve(ctx, prior, s, logpdf_out, nullptr, nullptr, nullptr, &post);
    if (rc == BLR_INFO_NOISE) {
        int info = 1;
        if (vector_noise && noise->vec) {
            const int loc = check_noise_vector(ctx, noise->vec->p, noise->vec->n);
            if (loc != 0) info = loc;
        }
        set_err(ctx, info, "observation noise variance is not positive");
        return done(info);
    }
    if (rc != 0) return done(rc);

    // device scratch: [se (N) | var (N) | Q (ldq x dk) | u (D) | mw (D) | λ (D) | dmw (D) | dλ (D or D x D) | Σ ∂/∂σ² (1)]
    const bool obs = G.dX_dev || G.dy_dev || G.dsigma2_dev || G.dsigma2;
    const bool diagonal = prior->lambda_kind == BLR_LAMBDA_DIAGONAL;
    const bool needQ = G.dX_dev || (G.dlambda && !diagonal);
    const bool fast = G.dX_dev && grad_x_fast_eligible(post, x, G.dX_dev, G.ld_dX);
    int64_t ldq = 0, dk = 0;
    if (needQ) grad_q_shape(post, fast, &ldq, &dk);
    const int64_t nse = obs ? 2 * N : 0, nq = ldq * dk, ndl = diagonal ? D : D * D;
    cudaError_t e = dev_alloc(ctx, &buf, (size_t)(nse + nq + 4 * D + ndl + 1) * sizeof(double));
    if (e != cudaSuccess) return done(cuda_fail(ctx, e, "cudaMallocAsync(logpdf_grad)"));
    double *se = buf, *var = se + N, *Q = buf + nse, *u = Q + nq, *mwd = u + D, *lamd = mwd + D, *dmw = lamd + D, *dlam = dmw + D,
           *dsum = dlam + ndl;
    if (obs) {
        rc = grad_obs(ctx, post, x, y->p, sig, sig_scalar, se, var, G.dy_dev, G.dsigma2_dev, G.dsigma2 ? dsum : nullptr);
        if (rc == 0 && G.dsigma2 && ctx->nccl_comm && ctx->nranks > 1) {
            NcclApi* a = nccl_api();
            ncclResult_t r = a->AllReduce(dsum, dsum, 1, ncclFloat64, ncclSum, (ncclComm_t)ctx->nccl_comm, ctx->stream);
            rc = (r != ncclSuccess) ? nccl_fail(ctx, r, "ncclAllReduce") : nccl_async_check(ctx);
        }
        if (rc != 0) return done(rc);
    }
    if (needQ) {
        rc = grad_q(ctx, post, Q, ldq, dk);
        if (rc != 0) return done(rc);
    }
    if (G.dmw || G.dlambda) {
        e = cudaMemcpyAsync(mwd, prior->mw, (size_t)D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess && diagonal)
            e = cudaMemcpyAsync(lamd, prior->lambda, (size_t)D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) return done(cuda_fail(ctx, e, "upload prior"));
        rc = grad_prior(ctx, prior, post, mwd, diagonal ? lamd : nullptr, Q, ldq, u, G.dmw ? dmw : nullptr, G.dlambda ? dlam : nullptr);
        if (rc != 0) return done(rc);
    }
    if (G.dX_dev) {
        rc = grad_x(ctx, post, x, Q, ldq, dk, fast, se, sig, sig_scalar, G.dX_dev, G.ld_dX);
        if (rc != 0) return done(rc);
    }
    if (G.dmw) e = cudaMemcpyAsync(G.dmw, dmw, (size_t)D * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && G.dlambda)
        e = cudaMemcpyAsync(G.dlambda, dlam, (size_t)ndl * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && G.dsigma2) e = cudaMemcpyAsync(G.dsigma2, dsum, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return done(cuda_fail(ctx, e, "download logpdf gradients"));
    return done(0);
}

int blr_logpdf_multi_grad(blr_ctx* ctx, const blr_prior* prior, const blr_x* x, const double* Y_dev, int64_t ldy, int64_t k,
                          const blr_noise* noise, const double* weights, double* logpdf_out, const blr_logpdf_grads* g) {
    CTX_ENTER(ctx);
    if (!prior || !x || !noise || !prior->mw || !prior->lambda || k < 0 || (k > 0 && !Y_dev))
        return set_err(ctx, BLR_E_INVALID, "null argument");
    if (prior->D > 0 && prior->D != x->D) return set_err(ctx, BLR_E_DIM, "size(X, 1) != length(mw)");
    if (k > 0 && ldy < x->N) return set_err(ctx, BLR_E_DIM, "size(Y, 1) != size(fx.x.X, 2)");
    if (noise->kind == BLR_NOISE_DENSE) return set_err(ctx, BLR_E_INVALID, "blr_logpdf_multi_grad: dense Σy is not supported");
    const blr_logpdf_grads none = {};
    const blr_logpdf_grads& G = g ? *g : none;
    const bool vector_noise = noise->kind == BLR_NOISE_VECTOR;
    if ((G.dsigma2 && vector_noise) || (G.dsigma2_dev && !vector_noise))
        return set_err(ctx, BLR_E_INVALID, "dsigma2 (scalar noise) / dsigma2_dev (vector noise) does not match the noise kind");
    const int64_t D = x->D, N = x->N;
    const bool colv = x->layout == BLR_COLVECS;
    if (G.dX_dev && G.ld_dX < std::max<int64_t>(colv ? D : N, 1)) return set_err(ctx, BLR_E_INVALID, "ld_dX too small");
    const bool diagonal = prior->lambda_kind == BLR_LAMBDA_DIAGONAL;
    const int64_t ndl = diagonal ? D : D * D;
    if (k == 0) {  // L is an empty sum: every requested gradient is zero
        cudaStream_t sm = ctx->stream;
        if (G.dmw) std::fill(G.dmw, G.dmw + D, 0.0);
        if (G.dlambda) std::fill(G.dlambda, G.dlambda + ndl, 0.0);
        if (G.dsigma2) *G.dsigma2 = 0.0;
        if (G.dsigma2_dev && N > 0) BLR_CUDA_OK(ctx, cudaMemsetAsync(G.dsigma2_dev, 0, (size_t)N * sizeof(double), sm));
        if (G.dX_dev && N > 0 && D > 0) {
            const int64_t rows = colv ? D : N, cols = colv ? N : D;
            BLR_CUDA_OK(ctx, cudaMemset2DAsync(G.dX_dev, (size_t)G.ld_dX * sizeof(double), 0, (size_t)rows * sizeof(double), (size_t)cols, sm));
        }
        BLR_CUDA_OK(ctx, cudaStreamSynchronize(sm));
        return 0;
    }
    const double* sig = nullptr;
    double sig_scalar = 0.0;
    BLR_TRY(noise_args(ctx, noise, N, &sig, &sig_scalar, true));
    std::vector<double> c_host(weights ? weights : nullptr, weights ? weights + k : nullptr), lp_host;
    if (!weights) c_host.assign((size_t)k, 1.0);
    double cbar = 0.0;
    for (int64_t j = 0; j < k; ++j) cbar += c_host[j];
    if (!logpdf_out) {
        lp_host.resize((size_t)k);
        logpdf_out = lp_host.data();
    }

    // the value: exactly blr_logpdf_multi's path, keeping the posterior of column 0 and Z = L⁻¹R of the others
    blr_stats* s = nullptr;
    blr_post* post = nullptr;
    double *extra = nullptr, *buf = nullptr;
    auto done = [&](int rc) {
        dev_free(ctx->stream, buf);
        dev_free(ctx->stream, extra);
        if (s) blr_stats_free(ctx, s);
        if (post) post_release(post);
        return rc;
    };
    int rc = logpdf_multi_forward(ctx, prior, x, Y_dev, ldy, k, noise, logpdf_out, &s, &post, &extra);
    if (rc != 0) return done(rc);

    // device scratch: [A (ldq x (dk + kp)) | E (kp x N) | c (k) | U (D x k) | M' (D x k) | uc (D) | mw (D) | λ (D) | dmw (D) |
    //                  dλ (D or D x D) | Σ ∂/∂σ² (1) | XM (N x k) | mean, h (2N)]: A and E first, where the tensor copies need
    //                  16-byte alignment (ldq and kp are multiples of 16 on the fast path)
    const bool obs = G.dX_dev || G.dy_dev || G.dsigma2_dev || G.dsigma2;
    const bool wsig = G.dsigma2_dev || G.dsigma2;
    const bool needQ = G.dX_dev || (G.dlambda && !diagonal);
    const bool fast = G.dX_dev && grad_x_fast_eligible(post, x, G.dX_dev, G.ld_dX);
    const int64_t kp = (k + 15) / 16 * 16;
    int64_t ldq = 0, dk = 0;
    if (needQ) grad_q_shape(post, fast, &ldq, &dk);
    const int64_t nsmall = k + 2 * D * k + 5 * D + ndl + 1, nxm = obs ? N * k : 0, nh = wsig ? 2 * N : 0,
                  ne = G.dX_dev ? kp * N : 0, na = needQ ? ldq * (dk + (G.dX_dev ? kp : 0)) : 0;
    cudaError_t e = dev_alloc(ctx, &buf, (size_t)(nsmall + nxm + nh + ne + na) * sizeof(double));
    if (e != cudaSuccess) return done(cuda_fail(ctx, e, "cudaMallocAsync(logpdf_multi_grad)"));
    double *A = buf, *E = A + na, *c = E + ne, *U = c + k, *M = U + D * k, *uc = M + D * k, *mwd = uc + D, *lamd = mwd + D,
           *dmw = lamd + D, *dlam = dmw + D, *dsum = dlam + ndl, *XM = dsum + 1, *hbuf = XM + nxm;
    e = cudaMemcpyAsync(c, c_host.data(), (size_t)k * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(mwd, prior->mw, (size_t)D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && diagonal)
        e = cudaMemcpyAsync(lamd, prior->lambda, (size_t)D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) return done(cuda_fail(ctx, e, "upload weights / prior"));
    // U and M' are replicated: R, hence Z, was all-reduced by the forward pass
    rc = grad_means_multi(ctx, post, mwd, extra, k, U, M);
    if (rc == 0 && obs) {
        rc = grad_obs_multi(ctx, post, x, M, k, kp, Y_dev, ldy, sig, sig_scalar, c, cbar, XM, hbuf, wsig ? hbuf + N : nullptr,
                            G.dX_dev ? E : nullptr, G.dy_dev, G.dsigma2_dev, G.dsigma2 ? dsum : nullptr);
        if (rc == 0 && G.dsigma2 && ctx->nccl_comm && ctx->nranks > 1) {
            NcclApi* a = nccl_api();
            ncclResult_t r = a->AllReduce(dsum, dsum, 1, ncclFloat64, ncclSum, (ncclComm_t)ctx->nccl_comm, ctx->stream);
            rc = (r != ncclSuccess) ? nccl_fail(ctx, r, "ncclAllReduce") : nccl_async_check(ctx);
        }
    }
    if (rc == 0 && needQ) rc = grad_q(ctx, post, A, ldq, dk);
    if (rc == 0 && (G.dmw || G.dlambda))
        rc = grad_prior_multi(ctx, prior, post, diagonal ? lamd : nullptr, A, ldq, U, k, c, cbar, uc, G.dmw ? dmw : nullptr,
                              G.dlambda ? dlam : nullptr);
    if (rc == 0 && G.dX_dev) {
        rc = grad_a_multi(ctx, A, ldq, dk, kp, D, k, M, c, cbar);
        if (rc == 0) rc = grad_x_multi(ctx, post, x, A, ldq, dk, k, kp, fast, E, sig, sig_scalar, G.dX_dev, G.ld_dX);
    }
    if (rc != 0) return done(rc);
    if (G.dmw) e = cudaMemcpyAsync(G.dmw, dmw, (size_t)D * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && G.dlambda)
        e = cudaMemcpyAsync(G.dlambda, dlam, (size_t)ndl * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && G.dsigma2) e = cudaMemcpyAsync(G.dsigma2, dsum, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return done(cuda_fail(ctx, e, "download logpdf gradients"));
    return done(0);
}

// ---------------------------------------------------------------------------------------------- prediction
int blr_post_create(blr_ctx* ctx, const blr_prior* prior, int64_t D, blr_post** out) {
    CTX_ENTER(ctx);
    if (!prior || !out || !prior->mw || !prior->lambda || D < 1 || D > SMALL_VEC)
        return set_err(ctx, BLR_E_INVALID, "bad prior");
    if (prior->D > 0 && prior->D != D) return set_err(ctx, BLR_E_DIM, "length(mw) != D");
    return post_from_prior(ctx, prior, D, out);
}
int blr_post_free(blr_ctx* ctx, blr_post* p) {
    if (!p) return 0;
    if (ctx) cudaSetDevice(ctx->device);
    post_release(p);
    return 0;
}
int blr_post_dim(const blr_post* p, int64_t* D_out) {
    if (!p || !D_out) return BLR_E_INVALID;
    *D_out = p->D;
    return 0;
}

int blr_mean_var_dev(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, double* mean_dev,
                     double* var_dev) {
    CTX_ENTER(ctx);
    if (!p || !x) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (x->D != p->D) return set_err(ctx, BLR_E_INVALID, "size(X, 1) != length(mw)");
    if (noise && noise->kind == BLR_NOISE_DENSE) {  // only diag(Σy) enters the marginal variances (:42)
        if (x->N == 0) return 0;
        DenseNoise dn;
        BLR_TRY(dense_noise_prepare(ctx, noise, x->N, &dn));
        const int rc = predict_mean_var(ctx, p, x, dn.diag, 0.0, mean_dev, var_dev);
        dense_noise_release(ctx, &dn);
        return rc;
    }
    const double* sig = nullptr;
    double sig_scalar = 0.0;
    BLR_TRY(noise_args(ctx, noise, x->N, &sig, &sig_scalar));
    return predict_mean_var(ctx, p, x, sig, sig_scalar, mean_dev, var_dev);
}

int blr_mean_var(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, double* mean_host,
                 double* var_host) {
    CTX_ENTER(ctx);
    if (!p || !x) return set_err(ctx, BLR_E_INVALID, "null argument");
    const int64_t N = x->N;
    if (N == 0) return 0;
    double* buf = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &buf, (size_t)2 * N * sizeof(double)));
    int rc = blr_mean_var_dev(ctx, p, x, noise, mean_host ? buf : nullptr, var_host ? buf + N : nullptr);
    cudaError_t e = cudaSuccess;
    if (rc == 0 && mean_host)
        e = cudaMemcpyAsync(mean_host, buf, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (rc == 0 && e == cudaSuccess && var_host)
        e = cudaMemcpyAsync(var_host, buf + N, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx->stream, buf);
    if (rc != 0) return rc;
    if (e != cudaSuccess) return cuda_fail(ctx, e, "download mean/var");
    if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "mean_var sync");
    return 0;
}

int blr_cov(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, double* C_host) {
    CTX_ENTER(ctx);
    if (!p || !x || !C_host) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (x->D != p->D) return set_err(ctx, BLR_E_INVALID, "size(X, 1) != length(mw)");
    const int64_t N = x->N;
    if (N == 0) return 0;
    const double* sig = nullptr;
    double sig_scalar = 0.0;
    DenseNoise dn;
    const bool dense = noise && noise->kind == BLR_NOISE_DENSE;
    if (dense)
        BLR_TRY(dense_noise_prepare(ctx, noise, N, &dn));
    else
        BLR_TRY(noise_args(ctx, noise, N, &sig, &sig_scalar));
    double* C = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &C, (size_t)N * N * sizeof(double)));
    int rc = predict_cov(ctx, p, x, sig, sig_scalar, C);
    if (dense) {
        if (rc == 0) {
            add_matrix_kernel<<<(int)std::min<int64_t>((N * N + 255) / 256, 2048), 256, 0, ctx->stream>>>(C, dn.S, N * N);
            ctx->launches++;
        }
        dense_noise_release(ctx, &dn);
    }
    cudaError_t e = cudaSuccess;
    if (rc == 0) e = cudaMemcpyAsync(C_host, C, (size_t)N * N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx->stream, C);
    if (rc != 0) return rc;
    if (e != cudaSuccess) return cuda_fail(ctx, e, "download cov");
    if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "cov sync");
    return 0;
}

int blr_rand_weights(blr_ctx* ctx, blr_post* p, int64_t S, const double* Z, uint64_t seed, double* W_host) {
    CTX_ENTER(ctx);
    if (!p || !W_host || S < 0) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (S == 0) return 0;
    const int64_t D = p->D;
    double* buf = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &buf, (size_t)2 * (D + 1) * S * sizeof(double)));
    double *Zd = buf, *Wd = buf + (D + 1) * S;
    int rc = 0;
    cudaError_t e = cudaSuccess;
    if (Z)
        e = cudaMemcpyAsync(Zd, Z, (size_t)D * S * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    else
        rc = synth_normal(ctx, Zd, D, S, D, seed, 5, 0);
    if (rc == 0 && e == cudaSuccess) rc = sample_weights(ctx, p, S, Zd, Wd);
    if (rc == 0 && e == cudaSuccess)
        e = cudaMemcpyAsync(W_host, Wd, (size_t)D * S * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx->stream, buf);
    if (rc != 0) return rc;
    if (e != cudaSuccess) return cuda_fail(ctx, e, "rand_weights copy");
    if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "rand_weights sync");
    return 0;
}

int blr_rand_finite_dev(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, int64_t S,
                        const double* Zw_host, const double* Zy_dev, uint64_t seed, double* Y_dev) {
    CTX_ENTER(ctx);
    if (!p || !x || !Y_dev || S < 0) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (x->D != p->D) return set_err(ctx, BLR_E_INVALID, "size(X, 1) != length(mw)");
    if (S == 0 || x->N == 0) return 0;
    const int64_t D = p->D;
    const double* sig = nullptr;
    double sig_scalar = 0.0;
    DenseNoise dn;
    const bool dense = noise && noise->kind == BLR_NOISE_DENSE;
    if (dense) {
        BLR_TRY(dense_noise_prepare(ctx, noise, x->N, &dn));
    } else {
        BLR_TRY(noise_args(ctx, noise, x->N, &sig, &sig_scalar, true));
        BLR_TRY(check_noise_vector(ctx, sig, x->N));  // `_cholesky(fx.Σy)` (:52): PosDefException for a non-positive variance
    }
    double* buf = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &buf, (size_t)(2 * (D + 1) * S + 2) * sizeof(double)));
    double *Zd = buf, *Wd = buf + (((D + 1) * S + 1) & ~(int64_t)1);  // even offset: 16-byte aligned (a TMA source in the two-group rand kernel)
    int rc = 0;
    cudaError_t e = cudaSuccess;
    if (Zw_host)
        e = cudaMemcpyAsync(Zd, Zw_host, (size_t)D * S * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    else
        rc = synth_normal(ctx, Zd, D, S, D, seed, 5, 0);
    if (rc == 0 && e == cudaSuccess) rc = sample_weights(ctx, p, S, Zd, Wd);
    if (dense) {
        // Y = X'w + Uy' Zy with Uy' = L (dense lower factor): noiseless product first, then Y += L Z  (:52)
        const int64_t N = x->N;
        if (rc == 0 && e == cudaSuccess) rc = sample_finite(ctx, x, Wd, S, nullptr, 0.0, nullptr, seed, Y_dev);
        double* Zgen = nullptr;
        if (rc == 0 && e == cudaSuccess && !Zy_dev) {
            e = dev_alloc(ctx, &Zgen, (size_t)(N + 1) * S * sizeof(double));
            if (e == cudaSuccess) rc = synth_normal(ctx, Zgen, N, S, N, seed, 7, 0);
        }
        if (rc == 0 && e == cudaSuccess)
            rc = gemm_generic(ctx, N, S, N, dn.L, 1, N, Zy_dev ? Zy_dev : Zgen, 1, N, Y_dev, 1, N, 1.0);
        dev_free(ctx->stream, Zgen);
        dense_noise_release(ctx, &dn);
    } else if (rc == 0 && e == cudaSuccess) {
        rc = sample_finite(ctx, x, Wd, S, sig, sig_scalar, Zy_dev, seed, Y_dev);
    }
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx->stream, buf);
    if (rc != 0) return rc;
    if (e != cudaSuccess) return cuda_fail(ctx, e, "rand_finite copy");
    if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "rand_finite sync");
    return 0;
}

int blr_rand_finite(blr_ctx* ctx, blr_post* p, const blr_x* x, const blr_noise* noise, int64_t S, const double* Zw,
                    const double* Zy, uint64_t seed, double* Y_host) {
    CTX_ENTER(ctx);
    if (!p || !x || !Y_host || S < 0) return set_err(ctx, BLR_E_INVALID, "null argument");
    const int64_t N = x->N;
    if (S == 0 || N == 0) return 0;
    double *Yd = nullptr, *Zyd = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &Yd, (size_t)N * S * sizeof(double)));
    cudaError_t e = cudaSuccess;
    if (Zy) {
        e = dev_alloc(ctx, &Zyd, (size_t)N * S * sizeof(double));
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(Zyd, Zy, (size_t)N * S * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    }
    int rc = (e == cudaSuccess) ? blr_rand_finite_dev(ctx, p, x, noise, S, Zw, Zyd, seed, Yd) : 0;
    if (rc == 0 && e == cudaSuccess)
        e = cudaMemcpyAsync(Y_host, Yd, (size_t)N * S * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx->stream, Yd);
    dev_free(ctx->stream, Zyd);
    if (rc != 0) return rc;
    if (e != cudaSuccess) return cuda_fail(ctx, e, "rand_finite copy");
    if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "rand_finite sync");
    return 0;
}

int blr_apply_weights(blr_ctx* ctx, const blr_x* x, const double* w_host, double* out_host) {
    CTX_ENTER(ctx);
    if (!x || !w_host || !out_host) return set_err(ctx, BLR_E_INVALID, "null argument");
    if (x->N == 0) return 0;
    double* buf = nullptr;
    BLR_CUDA_OK(ctx, dev_alloc(ctx, &buf, (size_t)(x->N + x->D) * sizeof(double)));
    cudaError_t e = cudaMemcpyAsync(buf + x->N, w_host, (size_t)x->D * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    int rc = (e == cudaSuccess) ? apply_weights(ctx, x, buf + x->N, buf) : 0;
    if (rc == 0 && e == cudaSuccess)
        e = cudaMemcpyAsync(out_host, buf, (size_t)x->N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e2 = cudaStreamSynchronize(ctx->stream);
    dev_free(ctx->stream, buf);
    if (rc != 0) return rc;
    if (e != cudaSuccess) return cuda_fail(ctx, e, "apply_weights copy");
    if (e2 != cudaSuccess) return cuda_fail(ctx, e2, "apply_weights sync");
    return 0;
}

// ---------------------------------------------------------------------------------------------- calibration
int blr_calibrate_dmma(blr_ctx* ctx, double* tflops_out) {
    CTX_ENTER(ctx);
    if (!tflops_out) return BLR_E_INVALID;
    return calib_dmma(ctx, tflops_out);
}
int blr_calibrate_dmma_cfg(blr_ctx* ctx, int warps_per_sm, int n_acc, double* tflops_out) {
    CTX_ENTER(ctx);
    if (!tflops_out) return BLR_E_INVALID;
    return calib_dmma_cfg(ctx, warps_per_sm, n_acc, tflops_out);
}
int blr_calibrate_gram_inner(blr_ctx* ctx, double* tflops_out) {
    CTX_ENTER(ctx);
    if (!tflops_out) return BLR_E_INVALID;
    return calib_gram_inner(ctx, tflops_out);
}
int blr_calibrate_mixed(blr_ctx* ctx, double* tflops2_out) {
    CTX_ENTER(ctx);
    if (!tflops2_out) return BLR_E_INVALID;
    return calib_mixed(ctx, tflops2_out);
}
int blr_calibrate_dfma(blr_ctx* ctx, double* tflops_out) {
    CTX_ENTER(ctx);
    if (!tflops_out) return BLR_E_INVALID;
    return calib_dfma(ctx, tflops_out);
}
int blr_calibrate_hbm(blr_ctx* ctx, double* gbs_out) {
    CTX_ENTER(ctx);
    if (!gbs_out) return BLR_E_INVALID;
    return calib_hbm(ctx, gbs_out);
}

}  // extern "C"
