// =====================================================================================
// kite_capi.cu -- extern "C" layer of libkite_b200.so (declared in include/kite_b200.h).
// Thin: argument checks, template dispatch, launches on the context's stream.  No CPU
// fallback anywhere: every entry point ends in a kernel launch or an error code.
// =====================================================================================
#include <dlfcn.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "kite_consts.h"
#include "kite_launch.h"

using namespace kite;

// ---- minimal NCCL surface, resolved at run time (no link-time dependency) -------------------------
typedef struct { char internal[128]; } nccl_unique_id_t;
typedef void* nccl_comm_t;
typedef int (*pfn_ncclGetUniqueId)(nccl_unique_id_t*);
typedef int (*pfn_ncclCommInitRank)(nccl_comm_t*, int, nccl_unique_id_t, int);
typedef int (*pfn_ncclAllGather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t);
typedef int (*pfn_ncclCommDestroy)(nccl_comm_t);
typedef const char* (*pfn_ncclGetErrorString)(int);
struct NcclApi {
    void* handle = nullptr;
    pfn_ncclGetUniqueId GetUniqueId = nullptr;
    pfn_ncclCommInitRank CommInitRank = nullptr;
    pfn_ncclAllGather AllGather = nullptr;
    pfn_ncclCommDestroy CommDestroy = nullptr;
    pfn_ncclGetErrorString GetErrorString = nullptr;
    bool ok() const { return handle && GetUniqueId && CommInitRank && AllGather && CommDestroy; }
};
static NcclApi& nccl_api() {
    static NcclApi api;
    if (api.handle) return api;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    for (const char* n : names) { h = dlopen(n, RTLD_NOW | RTLD_NOLOAD); if (h) break; }   // reuse torch's copy if loaded
    if (!h) for (const char* n : names) { h = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
    if (!h) return api;
    api.handle = h;
    api.GetUniqueId = (pfn_ncclGetUniqueId)dlsym(h, "ncclGetUniqueId");
    api.CommInitRank = (pfn_ncclCommInitRank)dlsym(h, "ncclCommInitRank");
    api.AllGather = (pfn_ncclAllGather)dlsym(h, "ncclAllGather");
    api.CommDestroy = (pfn_ncclCommDestroy)dlsym(h, "ncclCommDestroy");
    api.GetErrorString = (pfn_ncclGetErrorString)dlsym(h, "ncclGetErrorString");
    return api;
}

struct DevBuf {
    void* ptr = nullptr; size_t bytes = 0;
    int reserve(size_t n) {
        if (n <= bytes) return 0;
        if (ptr) cudaFree(ptr);
        ptr = nullptr; bytes = 0;
        cudaError_t e = cudaMalloc(&ptr, n);
        if (e != cudaSuccess) return (int)e;
        bytes = n; return 0;
    }
    void release() { if (ptr) cudaFree(ptr); ptr = nullptr; bytes = 0; }
};

struct kite_ctx {
    KiteConsts K;
    kite_params params;
    int device = 0;
    int model_kind = 0;
    cudaStream_t stream = nullptr;       // compute stream in use
    cudaStream_t own_stream = nullptr;
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_cmp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
    std::string err;
    long long launches = 0;
    DevBuf small;                        // W / V / compD staging
    DevBuf scratch;                      // output of the FP64 peak microbenchmark
    DevBuf ekf_lines;                    // ekf predict: pre-step state lines of the resident warps (TMA kernel)
    DevBuf pipe[2];                      // host-pipeline chunk buffers
    DevBuf shared_u, shared_y;
    DevBuf node_w;                       // collocated-cost node weights
    DevBuf counters;                     // dynamic work counters of the persistent kernels
    nccl_comm_t comm = nullptr;
    int nranks = 1, rank = 0;
    int32_t* status_out = nullptr;       // kite_set_status_buffer: per-unit flags of the sensitivity / EKF / collocation calls
};

static int fail(kite_ctx* c, int code, const std::string& msg) { if (c) c->err = msg; return code; }
static int cuda_fail(kite_ctx* c, cudaError_t e, const char* where) {
    return fail(c, KITE_ERR_CUDA, std::string(where) + ": " + cudaGetErrorString(e));
}
#define CK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call); } while (0)
#define LAUNCH_CHECK(name) do { ctx->launches++; cudaError_t e__ = cudaGetLastError(); if (e__ != cudaSuccess) return cuda_fail(ctx, e__, name); } while (0)


extern "C" {

const char* kite_version(void) { return "kite_b200 0.1 (sm_100a)"; }

int kite_create(kite_ctx** out, const kite_params* params, int model_kind, int device) {
    if (!out || !params) return KITE_ERR_ARG;
    if (model_kind < 0 || model_kind > 2) return KITE_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return KITE_ERR_CUDA;   // no CPU fallback
    kite_ctx* ctx = new kite_ctx();
    ctx->device = device; ctx->model_kind = model_kind; ctx->params = *params;
    ctx->K = make_consts(*params, model_kind);
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx; return KITE_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    *out = ctx;
    return KITE_OK;
}

int kite_destroy(kite_ctx* ctx) {
    if (!ctx) return KITE_ERR_ARG;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->comm && nccl_api().ok()) nccl_api().CommDestroy(ctx->comm);
    ctx->small.release(); ctx->scratch.release(); ctx->ekf_lines.release(); ctx->pipe[0].release(); ctx->pipe[1].release();
    ctx->shared_u.release(); ctx->shared_y.release(); ctx->node_w.release(); ctx->counters.release();
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_h2d[i]) cudaEventDestroy(ctx->ev_h2d[i]);
        if (ctx->ev_cmp[i]) cudaEventDestroy(ctx->ev_cmp[i]);
        if (ctx->ev_d2h[i]) cudaEventDestroy(ctx->ev_d2h[i]);
    }
    if (ctx->h2d_stream) cudaStreamDestroy(ctx->h2d_stream);
    if (ctx->d2h_stream) cudaStreamDestroy(ctx->d2h_stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return KITE_OK;
}

int kite_set_stream(kite_ctx* ctx, void* s) {
    if (!ctx) return KITE_ERR_ARG;
    ctx->stream = (cudaStream_t)s;      // NULL = the CUDA default stream
    return KITE_OK;
}
int kite_set_status_buffer(kite_ctx* ctx, int32_t* status_d) {
    if (!ctx) return KITE_ERR_ARG;
    ctx->status_out = status_d;
    return KITE_OK;
}
int kite_reset_stream(kite_ctx* ctx) {
    if (!ctx) return KITE_ERR_ARG;
    ctx->stream = ctx->own_stream;
    return KITE_OK;
}
int kite_device_malloc(void** ptr_out, size_t bytes) {
    if (!ptr_out) return KITE_ERR_ARG;
    return cudaMalloc(ptr_out, bytes) == cudaSuccess ? KITE_OK : KITE_ERR_CUDA;
}
int kite_device_free(void* ptr) { return cudaFree(ptr) == cudaSuccess ? KITE_OK : KITE_ERR_CUDA; }
int kite_ctx_malloc(kite_ctx* ctx, void** ptr_out, size_t bytes) {
    if (!ctx || !ptr_out) return fail(ctx, KITE_ERR_ARG, "kite_ctx_malloc: bad argument");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMalloc(ptr_out, bytes));
    return KITE_OK;
}
int kite_ctx_free(kite_ctx* ctx, void* ptr) {
    if (!ctx) return KITE_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaFree(ptr));
    return KITE_OK;
}
int kite_copy_h2d(kite_ctx* ctx, void* dst_d, const void* src_h, size_t bytes) {
    if (!ctx || !dst_d || !src_h) return fail(ctx, KITE_ERR_ARG, "kite_copy_h2d: bad argument");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(dst_d, src_h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KITE_OK;
}
int kite_copy_d2h(kite_ctx* ctx, void* dst_h, const void* src_d, size_t bytes) {
    if (!ctx || !dst_h || !src_d) return fail(ctx, KITE_ERR_ARG, "kite_copy_d2h: bad argument");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(dst_h, src_d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KITE_OK;
}
int kite_synchronize(kite_ctx* ctx) {
    if (!ctx) return KITE_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return KITE_OK;
}
const char* kite_last_error(const kite_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
long long kite_launch_count(const kite_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ---------------------------------------------------------------- pointwise ----------------------
static int point_eval(kite_ctx* ctx, long B, long ld, const double* x, const double* u, const double* p, double* f,
                      double* Jx, double* Ju, bool jac, double* fa = nullptr) {
    if (ctx && B == 0) return KITE_OK;
    if (!ctx || !x || B < 0 || ld < B) return fail(ctx, KITE_ERR_ARG, "point_eval: bad argument");
    const bool rigid = ctx->model_kind == KITE_MODEL_RIGID_BODY;
    if (!rigid && !u) return fail(ctx, KITE_ERR_ARG, "point_eval: u is required for the kite models");
    if (rigid && p) return fail(ctx, KITE_ERR_STATE, "point_eval: rigid body has no aero parameters");
    CK(cudaSetDevice(ctx->device));
    if (jac) {
        // zero only the B valid columns of every row: with ld > B the padding (a neighbouring sub-batch of a larger
        // [rows][ld] allocation) must stay untouched
        if (Jx) CK(cudaMemset2DAsync(Jx, sizeof(double) * (size_t)ld, 0, sizeof(double) * (size_t)B, 169, ctx->stream));
        if (Ju) CK(cudaMemset2DAsync(Ju, sizeof(double) * (size_t)ld, 0, sizeof(double) * (size_t)B, 39, ctx->stream));
    }
    PointArgs a{ctx->K, B, ld, x, u, p, f, Jx, Ju, fa};
    launch_point_eval(a, rigid, p != nullptr, jac, ctx->stream);
    LAUNCH_CHECK("k_point_eval");
    return KITE_OK;
}

int kite_rhs_batch(kite_ctx* ctx, long B, long ld, const double* x_d, const double* u_d, const double* p_d, double* f_d) {
    if (!f_d) return fail(ctx, KITE_ERR_ARG, "kite_rhs_batch: f_d is null");
    return point_eval(ctx, B, ld, x_d, u_d, p_d, f_d, nullptr, nullptr, false);
}
int kite_jac_sparsity(int model_kind, int has_arm, int wrt_u, int* row_out, int* col_out) {
    if (model_kind < 0 || model_kind > 2) return KITE_ERR_ARG;
    const bool rigid = model_kind == KITE_MODEL_RIGID_BODY;
    int n = 0;
    const int ncol = wrt_u ? 3 : 13;
    for (int j = 0; j < ncol; ++j)                   // CCS order: columns, rows ascending inside a column
        for (int i = 0; i < 13; ++i) {
            const bool nz = wrt_u ? (!rigid && ju_nz(i, j)) : (rigid ? jx_nz_rigid(i, j) : jx_nz(i, j, has_arm != 0));
            if (!nz) continue;
            if (row_out) row_out[n] = i;
            if (col_out) col_out[n] = j;
            ++n;
        }
    return n;
}
int kite_aero_batch(kite_ctx* ctx, long B, long ld, const double* x_d, const double* u_d, const double* p_d, double* F_d) {
    if (!F_d) return fail(ctx, KITE_ERR_ARG, "kite_aero_batch: F_d is null");
    if (ctx && ctx->model_kind == KITE_MODEL_RIGID_BODY) return fail(ctx, KITE_ERR_STATE, "kite_aero_batch: kite models only");
    return point_eval(ctx, B, ld, x_d, u_d, p_d, nullptr, nullptr, nullptr, false, F_d);
}
int kite_jac_batch(kite_ctx* ctx, long B, long ld, const double* x_d, const double* u_d, const double* p_d, double* Jx_d,
                   double* Ju_d) {
    if (!Jx_d && !Ju_d) return fail(ctx, KITE_ERR_ARG, "kite_jac_batch: both outputs null");
    return point_eval(ctx, B, ld, x_d, u_d, p_d, nullptr, Jx_d, Ju_d, true);
}

// ---------------------------------------------------------------- rollout ------------------------
int kite_rk4_rollout(kite_ctx* ctx, long B, long ld, long N, double h, const double* x0_d, const double* u_d, int u_mode,
                     const double* p_d, double* xf_d, double* traj_d, long save_every, const double* y_d, double* cost_d,
                     int32_t* status_d, long index0) {
    if (ctx && B == 0) return KITE_OK;      // empty batch: nothing to do, pointers may be null
    if (!ctx || B < 0 || N < 0 || ld < B || !xf_d) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout: bad argument");
    if (u_mode < 0 || u_mode > 3) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout: bad u_mode");
    const bool rigid = ctx->model_kind == KITE_MODEL_RIGID_BODY;
    if (u_mode != KITE_U_SYNTH && !x0_d) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout: x0_d is null");
    if (u_mode != KITE_U_SYNTH && !u_d && !rigid) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout: u_d is null");
    if (rigid && (p_d || u_mode == KITE_U_SYNTH)) return fail(ctx, KITE_ERR_STATE, "kite_rk4_rollout: not valid for rigid body");
    if ((y_d != nullptr) != (cost_d != nullptr)) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout: y_d and cost_d go together");
    if (y_d && N == 0) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout: the fitting cost averages over the steps and needs N > 0");
    if (traj_d && save_every <= 0) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout: save_every must be > 0");
    if (N >= (1L << 31) || save_every >= (1L << 31)) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout: N and save_every must be below 2^31");
    if (B == 0) return KITE_OK;
    CK(cudaSetDevice(ctx->device));
    RolloutArgs a{ctx->K, B, ld, N, h, make_rk_tab(h), x0_d, u_d, p_d, xf_d, traj_d, save_every > 0 ? save_every : 1, y_d, cost_d, status_d, index0};
    if (rigid && !u_d) { a.u = x0_d; u_mode = 0; }   // controls do not enter the rigid-body RHS; dummy readable pointer
    if (u_mode <= 1) launch_rollout_01(a, u_mode, rigid, p_d != nullptr, ctx->stream);
    else launch_rollout_23(a, u_mode, rigid, p_d != nullptr, ctx->stream);
    LAUNCH_CHECK("k_rk4_rollout");
    return KITE_OK;
}

int kite_synth_inputs(kite_ctx* ctx, long B, long ld, long N, long index0, double* x0_d, double* u_d) {
    if (!ctx || B < 0 || ld < B || N < 0) return fail(ctx, KITE_ERR_ARG, "kite_synth_inputs: bad argument");
    if (B == 0) return KITE_OK;
    CK(cudaSetDevice(ctx->device));
    SynthArgs a{B, ld, N, index0, x0_d, u_d};
    launch_synth_inputs(a, ctx->stream);
    LAUNCH_CHECK("k_synth_inputs");
    return KITE_OK;
}

int kite_synth_id_params(kite_ctx* ctx, long B, long ld, long index0, const double* pref_h, double* p_d) {
    if (!ctx || B < 0 || ld < B || !p_d) return fail(ctx, KITE_ERR_ARG, "kite_synth_id_params: bad argument");
    if (B == 0) return KITE_OK;
    CK(cudaSetDevice(ctx->device));
    const kite_params& P = ctx->params;
    const double nominal[21] = {P.CL0, P.CLa_total, P.CD0_total, P.CYb, P.Cm0, P.Cma, P.Cnb, P.Clb, P.CLq, P.Cmq, P.CYr,
                                P.Cnr, P.Clr, P.CYp, P.Clp, P.Cnp, P.CLde, P.CYdr, P.Cmde, P.Cndr, P.Cldr};
    SynthParamArgs a{};
    a.B = B; a.ld = ld; a.index0 = index0; a.p = p_d;
    for (int c = 0; c < 21; ++c) a.ref[c] = pref_h ? pref_h[c] : nominal[c];
    launch_synth_id_params(a, ctx->stream);
    LAUNCH_CHECK("k_synth_id_params");
    return KITE_OK;
}

// Host-pointer rollout: chunk over trajectories, double-buffered H2D / compute / D2H on three streams.
static int rollout_host_pipeline(kite_ctx* ctx, long B, long N, double h, const double* x0_h, const double* u_h, int u_mode,
                                 const double* p_h, double* xf_h, const double* y_h, double* cost_h, int32_t* status_h);
int kite_rk4_rollout_host(kite_ctx* ctx, long B, long N, double h, const double* x0_h, const double* u_h, int u_mode,
                          const double* p_h, double* xf_h, const double* y_h, double* cost_h, int32_t* status_h) {
    if (ctx && B == 0) return KITE_OK;
    if (!ctx || B < 0 || N < 0 || !xf_h) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout_host: bad argument");
    if (u_mode < 0 || u_mode > 2 || !x0_h) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout_host: bad u_mode / x0");
    const bool rigid = ctx->model_kind == KITE_MODEL_RIGID_BODY;
    if (!u_h && !rigid) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout_host: u_h is null");
    if ((y_h != nullptr) != (cost_h != nullptr)) return fail(ctx, KITE_ERR_ARG, "kite_rk4_rollout_host: y/cost go together");
    CK(cudaSetDevice(ctx->device));
    const int rc = rollout_host_pipeline(ctx, B, N, h, x0_h, u_h, u_mode, p_h, xf_h, y_h, cost_h, status_h);
    if (rc != KITE_OK) {
        // an error in the middle of the pipeline leaves copies on the caller's host buffers and kernels in flight on three
        // streams: drain them before handing the buffers back (the first error message is kept)
        const std::string first = ctx->err;
        if (ctx->h2d_stream) cudaStreamSynchronize(ctx->h2d_stream);
        cudaStreamSynchronize(ctx->stream);
        if (ctx->d2h_stream) cudaStreamSynchronize(ctx->d2h_stream);
        cudaGetLastError();
        ctx->err = first;
    }
    return rc;
}
static int rollout_host_pipeline(kite_ctx* ctx, long B, long N, double h, const double* x0_h, const double* u_h, int u_mode,
                                 const double* p_h, double* xf_h, const double* y_h, double* cost_h, int32_t* status_h) {
    const bool rigid = ctx->model_kind == KITE_MODEL_RIGID_BODY;
    if (!ctx->h2d_stream) {
        CK(cudaStreamCreateWithFlags(&ctx->h2d_stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CK(cudaEventCreateWithFlags(&ctx->ev_h2d[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->ev_cmp[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->ev_d2h[i], cudaEventDisableTiming));
        }
    }
    const bool per_step = (u_mode == KITE_U_PER_STEP);
    const long u_rows = rigid && !u_h ? 0 : (per_step ? 3 * N : (u_mode == KITE_U_CONST ? 3 : 0));
    // chunk size: ~512 MiB of per-trajectory input per buffer, multiple of 1024 trajectories
    const double bytes_per_traj = 8.0 * (13 + u_rows + (p_h ? 21 : 0) + 13 + 1) + 4.0;
    long Bc = (long)(512.0 * 1024 * 1024 / bytes_per_traj);
    Bc = std::max(1024L, (Bc / 1024) * 1024);
    if (Bc > B) Bc = B;
    const long rows_in = 13 + u_rows + (p_h ? 21 : 0);
    const size_t chunk_bytes = sizeof(double) * (size_t)Bc * (rows_in + 13 + 1) + sizeof(int32_t) * (size_t)Bc;
    for (int i = 0; i < 2; ++i)
        if (ctx->pipe[i].reserve(chunk_bytes)) return fail(ctx, KITE_ERR_CUDA, "kite_rk4_rollout_host: cudaMalloc failed");
    const double* u_shared_d = nullptr; const double* y_d = nullptr;
    if (u_mode == KITE_U_SHARED && u_h) {
        if (ctx->shared_u.reserve(sizeof(double) * 3 * (size_t)std::max(N, 1L))) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
        CK(cudaMemcpyAsync(ctx->shared_u.ptr, u_h, sizeof(double) * 3 * (size_t)N, cudaMemcpyHostToDevice, ctx->stream));
        u_shared_d = (const double*)ctx->shared_u.ptr;
    }
    if (y_h) {
        if (ctx->shared_y.reserve(sizeof(double) * 13 * (size_t)std::max(N, 1L))) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
        CK(cudaMemcpyAsync(ctx->shared_y.ptr, y_h, sizeof(double) * 13 * (size_t)N, cudaMemcpyHostToDevice, ctx->stream));
        y_d = (const double*)ctx->shared_y.ptr;
    }
    const long nchunks = (B + Bc - 1) / Bc;
    const size_t pitch_h = sizeof(double) * (size_t)B;
    for (long j = 0; j < nchunks; ++j) {
        const int b = (int)(j & 1);
        const long off = j * Bc, n = std::min(Bc, B - off);
        double* base = (double*)ctx->pipe[b].ptr;
        double* x0_d = base;
        double* u_d = x0_d + 13 * Bc;
        double* p_d = u_d + u_rows * Bc;
        double* xf_d = p_d + (p_h ? 21 : 0) * Bc;
        double* cost_d = xf_d + 13 * Bc;
        int32_t* st_d = (int32_t*)(cost_d + Bc);
        const size_t pitch_d = sizeof(double) * (size_t)Bc, width = sizeof(double) * (size_t)n;
        if (j >= 2) CK(cudaStreamWaitEvent(ctx->h2d_stream, ctx->ev_cmp[b], 0));     // inputs of chunk j-2 consumed
        CK(cudaMemcpy2DAsync(x0_d, pitch_d, x0_h + off, pitch_h, width, 13, cudaMemcpyHostToDevice, ctx->h2d_stream));
        if (u_rows) CK(cudaMemcpy2DAsync(u_d, pitch_d, u_h + off, pitch_h, width, (size_t)u_rows, cudaMemcpyHostToDevice, ctx->h2d_stream));
        if (p_h) CK(cudaMemcpy2DAsync(p_d, pitch_d, p_h + off, pitch_h, width, 21, cudaMemcpyHostToDevice, ctx->h2d_stream));
        CK(cudaEventRecord(ctx->ev_h2d[b], ctx->h2d_stream));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_h2d[b], 0));
        if (j >= 2) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_d2h[b], 0));         // outputs of chunk j-2 drained
        const double* uk = (u_mode == KITE_U_SHARED) ? u_shared_d : (u_rows ? u_d : nullptr);
        int rc = kite_rk4_rollout(ctx, n, Bc, N, h, x0_d, uk, u_mode, p_h ? p_d : nullptr, xf_d, nullptr, 0, y_d,
                                  y_h ? cost_d : nullptr, status_h ? st_d : nullptr, off);
        if (rc != KITE_OK) return rc;
        CK(cudaEventRecord(ctx->ev_cmp[b], ctx->stream));
        CK(cudaStreamWaitEvent(ctx->d2h_stream, ctx->ev_cmp[b], 0));
        CK(cudaMemcpy2DAsync(xf_h + off, pitch_h, xf_d, pitch_d, width, 13, cudaMemcpyDeviceToHost, ctx->d2h_stream));
        if (cost_h) CK(cudaMemcpyAsync(cost_h + off, cost_d, width, cudaMemcpyDeviceToHost, ctx->d2h_stream));
        if (status_h) CK(cudaMemcpyAsync(status_h + off, st_d, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->d2h_stream));
        CK(cudaEventRecord(ctx->ev_d2h[b], ctx->d2h_stream));
    }
    CK(cudaStreamSynchronize(ctx->d2h_stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return KITE_OK;
}

// ---------------------------------------------------------------- sensitivities -------------------
// workspace layout: [stage-state lines of the resident warps][per-group step counters of a rollout]
static size_t sens_state_bytes(long B) {
    // persistent kernel: one private [4 stages][x(13) | u(3)][32 units] line of stage states per RESIDENT warp (work items
    // are claimed dynamically, so every warp of every launched CTA may need its line), independent of B beyond one wave.
    // The stage Jacobians themselves never leave shared memory.
    const long groups = (B + 31) / 32;
    const long warps = std::min(groups + SF_WARPS, sens_fused_max_warps());     // covers any warps-per-CTA <= SF_WARPS
    return sizeof(double) * (size_t)SF_SCRATCH_PER_WARP * (size_t)warps;
}
size_t kite_rk4_sens_work_bytes(long B) {
    if (B <= 0) return 0;
    return sens_state_bytes(B) + (sizeof(int) * (size_t)((B + 31) / 32) + 255) / 256 * 256;
}

static int sens_impl(kite_ctx* ctx, long B, long ld, long N, double h, const double* x, const double* u, double* xn,
                     double* Phi, double* Gamma, void* work) {
    const bool rigid = ctx->model_kind == KITE_MODEL_RIGID_BODY;
    if (ctx->counters.reserve(64)) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
    CK(cudaMemsetAsync(ctx->counters.ptr, 0, 8, ctx->stream));
    SensArgs a{};
    a.K = ctx->K; a.B = B; a.ld = ld; a.N = N; a.rk = make_rk_tab(h); a.x = x; a.u = u; a.xn = xn; a.Phi = Phi; a.Gamma = Gamma;
    a.Sw = (double*)work; a.next_group = (unsigned long long*)ctx->counters.ptr;
    a.done = (int*)((char*)work + sens_state_bytes(B));
    if (N > 1) CK(cudaMemsetAsync(a.done, 0, sizeof(int) * (size_t)((B + 31) / 32), ctx->stream));
    a.status = ctx->status_out;
    if (a.status) CK(cudaMemsetAsync(a.status, 0, sizeof(int32_t) * (size_t)B, ctx->stream));      // the kernel ORs flags in
    // [Phi | Gamma] leave through TMA tensor stores when the output layout allows it (16-byte aligned base and pitch:
    // an even ld; an even B)
    const bool tma_out = !rigid && sens_make_tensor_map(&a.tmPhi, Phi, B, ld, 169, N) &&
                         sens_make_tensor_map(&a.tmGam, Gamma, B, ld, 39, N);
    launch_sens_fused(a, rigid, ctx->K.has_arm != 0, tma_out, ctx->stream);
    LAUNCH_CHECK("k_sens_fused");
    return KITE_OK;
}

int kite_rk4_sens_step(kite_ctx* ctx, long B, long ld, double h, const double* x_d, const double* u_d, double* xn_d,
                       double* Phi_d, double* Gamma_d, void* work_d) {
    if (ctx && B == 0) return KITE_OK;
    if (!ctx || B < 0 || ld < B || !x_d || !xn_d || !Phi_d || !Gamma_d || !work_d)
        return fail(ctx, KITE_ERR_ARG, "kite_rk4_sens_step: bad argument");
    if (!u_d && ctx->model_kind != KITE_MODEL_RIGID_BODY) return fail(ctx, KITE_ERR_ARG, "kite_rk4_sens_step: u_d is null");
    if (B == 0) return KITE_OK;
    CK(cudaSetDevice(ctx->device));
    return sens_impl(ctx, B, ld, 1, h, x_d, u_d ? u_d : x_d, xn_d, Phi_d, Gamma_d, work_d);
}

int kite_rk4_sens_rollout(kite_ctx* ctx, long B, long ld, long N, double h, const double* x0_d, const double* u_d,
                          double* xs_d, double* Phi_d, double* Gamma_d, void* work_d) {
    if (ctx && (B == 0 || N == 0)) return KITE_OK;
    if (!ctx || B < 0 || N < 0 || ld < B || !x0_d || !u_d || !xs_d || !Phi_d || !Gamma_d || !work_d)
        return fail(ctx, KITE_ERR_ARG, "kite_rk4_sens_rollout: bad argument");
    if (B == 0) return KITE_OK;
    CK(cudaSetDevice(ctx->device));
    // The primal recurrence is sequential in k, but only per trajectory: ONE launch walks the (step, group) work items
    // in step-major order, step k of a group waiting for the state its step k - 1 has published (k_sens_fused).
    return sens_impl(ctx, B, ld, N, h, x0_d, u_d, xs_d, Phi_d, Gamma_d, work_d);
}

// ---------------------------------------------------------------- collocation ---------------------
static int colloc_eval_impl(kite_ctx* ctx, long B, long ld, int M, const double* compD_h, double tau, const double* sx_h,
                            const double* su_h, const double* z_d, const double* p_d, double* G_d, double* JX_d, double* JU_d,
                            double* gnorm_d, bool sparse, const char* who) {
    if (ctx && B == 0) return KITE_OK;
    if (!ctx || B < 0 || ld < B || M < 2 || M > 1024 || !compD_h || !sx_h || !su_h || !z_d || !G_d || (sparse && !JX_d))
        return fail(ctx, KITE_ERR_ARG, std::string(who) + ": bad argument");
    if (ctx->model_kind == KITE_MODEL_RIGID_BODY) return fail(ctx, KITE_ERR_STATE, std::string(who) + ": kite models only");
    CK(cudaSetDevice(ctx->device));
    if (ctx->small.reserve(sizeof(double) * (size_t)M * M + 4096)) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
    CK(cudaMemcpyAsync(ctx->small.ptr, compD_h, sizeof(double) * (size_t)M * M, cudaMemcpyHostToDevice, ctx->stream));
    CollocArgs a{};
    a.K = ctx->K; a.B = B; a.ld = ld; a.M = M; a.tau = tau;
    for (int i = 0; i < 15; ++i) { a.sx[i] = sx_h[i]; a.isx[i] = 1.0 / sx_h[i]; }
    for (int i = 0; i < 4; ++i) { a.su[i] = su_h[i]; a.isu[i] = 1.0 / su_h[i]; }
    a.compD = (const double*)ctx->small.ptr;
    a.cd_compact = 0;
    if (M <= 16) {                       // compact rows for the constant bank (summation order = ascending column, as the dense walk)
        bool fits = true;
        for (int k = 0; k < M && fits; ++k) {
            int n = 0;
            for (int l = 0; l < M; ++l)
                if (compD_h[(size_t)k * M + l] != 0.0) {
                    if (n == 8) { fits = false; break; }
                    a.cd_col[k][n] = (signed char)l; a.cd_val[k][n] = compD_h[(size_t)k * M + l]; ++n;
                }
            a.cd_nz[k] = n;
        }
        a.cd_compact = fits ? 1 : 0;
    }
    a.z = z_d; a.p = p_d; a.G = G_d; a.JX = JX_d; a.JU = JU_d; a.gnorm = gnorm_d; a.status = ctx->status_out;
    const int fmt = sparse ? (ctx->K.has_arm ? 2 : 1) : ((JX_d || JU_d) ? 0 : 3);      // no Jacobian output: no Jacobian code
    launch_colloc_eval(a, p_d != nullptr, fmt, ctx->stream);
    LAUNCH_CHECK("k_colloc_eval");
    return KITE_OK;
}

int kite_colloc_eval(kite_ctx* ctx, long B, long ld, int M, const double* compD_h, double tau, const double* sx_h,
                     const double* su_h, const double* z_d, const double* p_d, double* G_d, double* JX_d, double* JU_d,
                     double* gnorm_d) {
    return colloc_eval_impl(ctx, B, ld, M, compD_h, tau, sx_h, su_h, z_d, p_d, G_d, JX_d, JU_d, gnorm_d, false, "kite_colloc_eval");
}

int kite_colloc_nnz_per_node(const kite_ctx* ctx) {
    if (!ctx) return KITE_ERR_ARG;
    return ctx->K.has_arm ? COLLOC_NNZ_ARM : COLLOC_NNZ_NOARM;
}
int kite_colloc_sparsity(const kite_ctx* ctx, int* row_out, int* col_out) {
    if (!ctx || !row_out || !col_out) return KITE_ERR_ARG;
    const CollocTab t = make_colloc_tab(ctx->K.has_arm != 0);
    for (int j = 0; j < 19; ++j)
        for (int i = 0; i < 15; ++i)
            if (t.slot[i][j] >= 0) { row_out[t.slot[i][j]] = i; col_out[t.slot[i][j]] = j; }
    return t.nnz;
}
int kite_colloc_eval_sparse(kite_ctx* ctx, long B, long ld, int M, const double* compD_h, double tau, const double* sx_h,
                            const double* su_h, const double* z_d, const double* p_d, double* G_d, double* JV_d, double* gnorm_d) {
    return colloc_eval_impl(ctx, B, ld, M, compD_h, tau, sx_h, su_h, z_d, p_d, G_d, JV_d, nullptr, gnorm_d, true, "kite_colloc_eval_sparse");
}

int kite_colloc_cost(kite_ctx* ctx, long B, long ld, int P, int S, const double* qw_h, double tau, const double* sx_h,
                     const kite_nmpc_cost* c, const double* z_d, double* cost_d, double* grad_d) {
    if (ctx && B == 0) return KITE_OK;
    if (!ctx || B < 0 || ld < B || P < 1 || S < 1 || S * P + 1 > 1024 || !qw_h || !sx_h || !c || !z_d || !cost_d)
        return fail(ctx, KITE_ERR_ARG, "kite_colloc_cost: bad argument");
    const int M = S * P + 1;
    CK(cudaSetDevice(ctx->device));
    // node weights: node seg*P + m carries tau * w_m; a node shared by two segments carries both (chebyshev.hpp:298-330)
    std::vector<double> wnode((size_t)M, 0.0);
    for (int k = 0; k < S; ++k)
        for (int m = 0; m <= P; ++m) wnode[(size_t)k * P + m] += tau * qw_h[m];
    if (ctx->node_w.reserve(sizeof(double) * 1024)) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
    double* wd = (double*)ctx->node_w.ptr;
    CK(cudaMemcpyAsync(wd, wnode.data(), sizeof(double) * (size_t)M, cudaMemcpyHostToDevice, ctx->stream));
    CostArgs a{};
    a.B = B; a.ld = ld; a.M = M;
    for (int i = 0; i < 3; ++i) { a.sx6[i] = sx_h[6 + i]; a.Q[i] = c->Q[i]; }
    a.sx13 = sx_h[13]; a.isx13 = 1.0 / sx_h[13];
    for (int i = 0; i < 4; ++i) a.R[i] = c->R[i];
    a.W = c->W; a.vref = c->vref_scaled;
    // path = vec( conj(q) (x) [0, P] (x) q ) = M(q)^T P with P = [r cos, r sin, alt]
    const double s0 = c->path_q[0], v1 = c->path_q[1], v2 = c->path_q[2], v3 = c->path_q[3];
    const double Mq[3][3] = {{s0 * s0 + v1 * v1 - v2 * v2 - v3 * v3, 2 * (v1 * v2 - s0 * v3), 2 * (v1 * v3 + s0 * v2)},
                             {2 * (v1 * v2 + s0 * v3), s0 * s0 - v1 * v1 + v2 * v2 - v3 * v3, 2 * (v2 * v3 - s0 * v1)},
                             {2 * (v1 * v3 - s0 * v2), 2 * (v2 * v3 + s0 * v1), s0 * s0 - v1 * v1 - v2 * v2 + v3 * v3}};
    for (int i = 0; i < 3; ++i) {
        a.rc[i] = Mq[0][i] * c->path_radius;
        a.rs[i] = Mq[1][i] * c->path_radius;
        a.ra[i] = Mq[2][i] * c->path_altitude;
    }
    a.wnode = wd; a.z = z_d; a.cost = cost_d; a.grad = grad_d;
    launch_colloc_cost(a, ctx->stream);
    LAUNCH_CHECK("k_colloc_cost");
    return KITE_OK;
}

// ---------------------------------------------------------------- EKF -----------------------------
size_t kite_ekf_work_bytes(long) { return 0; }      // the predict kernel keeps the Jacobian in shared memory

int kite_ekf_predict_batch(kite_ctx* ctx, long B, long ld, double dt, const double* x_d, const double* u_d,
                           const double* P_d, const double* W_h, double* xn_d, double* Pn_d, void* work_d) {
    if (ctx && B == 0) return KITE_OK;
    (void)work_d;
    if (!ctx || B < 0 || ld < B || !x_d || !P_d || !W_h || !xn_d || !Pn_d)
        return fail(ctx, KITE_ERR_ARG, "kite_ekf_predict_batch: bad argument");
    const bool rigid = ctx->model_kind == KITE_MODEL_RIGID_BODY;
    if (!rigid && !u_d) return fail(ctx, KITE_ERR_ARG, "kite_ekf_predict_batch: u_d is null");
    if (P_d == Pn_d) return fail(ctx, KITE_ERR_ARG, "kite_ekf_predict_batch: P_d and Pn_d must not alias");
    if (B == 0) return KITE_OK;
    CK(cudaSetDevice(ctx->device));
    if (ctx->small.reserve(4096)) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
    CK(cudaMemcpyAsync(ctx->small.ptr, W_h, sizeof(double) * 169, cudaMemcpyHostToDevice, ctx->stream));
    if (ctx->counters.reserve(64)) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
    CK(cudaMemsetAsync((char*)ctx->counters.ptr + 8, 0, 8, ctx->stream));
    EkfArgs a{ctx->K, B, ld, dt, make_rk_tab(dt), x_d, u_d, P_d, xn_d, Pn_d, (const double*)ctx->small.ptr,
              (unsigned long long*)((char*)ctx->counters.ptr + 8), ctx->status_out};
    if (ctx->ekf_lines.reserve(ekf_predict_scratch_bytes())) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
    launch_ekf_predict(a, rigid, ctx->K.has_arm != 0, (double*)ctx->ekf_lines.ptr, ctx->stream);
    LAUNCH_CHECK("k_ekf_predict");
    return KITE_OK;
}

int kite_ekf_update_batch(kite_ctx* ctx, long B, long ld, const double* z_d, const double* V_h, double* x_d, double* P_d) {
    if (ctx && B == 0) return KITE_OK;
    if (!ctx || B < 0 || ld < B || !z_d || !V_h || !x_d || !P_d) return fail(ctx, KITE_ERR_ARG, "kite_ekf_update_batch: bad argument");
    if (B == 0) return KITE_OK;
    CK(cudaSetDevice(ctx->device));
    if (ctx->small.reserve(4096)) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
    double* Vd = (double*)ctx->small.ptr + 256;     // keep clear of W staging
    CK(cudaMemcpyAsync(Vd, V_h, sizeof(double) * 49, cudaMemcpyHostToDevice, ctx->stream));
    EkfUpdArgs a{B, ld, z_d, P_d, x_d, Vd, ctx->status_out};          // in place: no staging copy of the covariance
    launch_ekf_update(a, ctx->stream);
    LAUNCH_CHECK("k_ekf_update");
    return KITE_OK;
}

int kite_comm_unique_id(char id_out[128]) {
    NcclApi& n = nccl_api();
    if (!n.ok() || !id_out) return KITE_ERR_NCCL;
    nccl_unique_id_t id;
    if (n.GetUniqueId(&id) != 0) return KITE_ERR_NCCL;
    std::memcpy(id_out, id.internal, 128);
    return KITE_OK;
}
int kite_comm_init(kite_ctx* ctx, int nranks, int rank, const char id[128]) {
    if (!ctx || !id || nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, KITE_ERR_ARG, "kite_comm_init: bad argument");
    NcclApi& n = nccl_api();
    if (!n.ok()) return fail(ctx, KITE_ERR_NCCL, "kite_comm_init: libnccl not found");
    CK(cudaSetDevice(ctx->device));
    nccl_unique_id_t uid; std::memcpy(uid.internal, id, 128);
    int rc = n.CommInitRank(&ctx->comm, nranks, uid, rank);
    if (rc != 0) return fail(ctx, KITE_ERR_NCCL, std::string("ncclCommInitRank: ") + (n.GetErrorString ? n.GetErrorString(rc) : "error"));
    ctx->nranks = nranks; ctx->rank = rank;
    return KITE_OK;
}
int kite_allgather(kite_ctx* ctx, const double* send_d, double* recv_d, long count) {
    if (!ctx || !send_d || !recv_d || count < 0) return fail(ctx, KITE_ERR_ARG, "kite_allgather: bad argument");
    if (!ctx->comm) return fail(ctx, KITE_ERR_STATE, "kite_allgather: communicator not initialised");
    NcclApi& n = nccl_api();
    CK(cudaSetDevice(ctx->device));
    int rc = n.AllGather(send_d, recv_d, (size_t)count, /*ncclFloat64*/ 8, ctx->comm, ctx->stream);
    if (rc != 0) return fail(ctx, KITE_ERR_NCCL, std::string("ncclAllGather: ") + (n.GetErrorString ? n.GetErrorString(rc) : "error"));
    return KITE_OK;
}
int kite_comm_destroy(kite_ctx* ctx) {
    if (!ctx) return KITE_ERR_ARG;
    if (ctx->comm && nccl_api().ok()) { nccl_api().CommDestroy(ctx->comm); ctx->comm = nullptr; }
    return KITE_OK;
}

// ---------------------------------------------------------------- diagnostics ---------------------
int kite_math_selftest(kite_ctx* ctx, long n, const double* x_d, double* out_d, int which) {
    if (!ctx || n < 0 || !x_d || !out_d || which < 0 || which > 6) return fail(ctx, KITE_ERR_ARG, "kite_math_selftest: bad argument");
    if (n == 0) return KITE_OK;
    CK(cudaSetDevice(ctx->device));
    launch_math_selftest(x_d, out_d, n, which, ctx->stream);
    LAUNCH_CHECK("k_math_selftest");
    return KITE_OK;
}
static int fp64_peak_impl(kite_ctx* ctx, int iters, double* tflops_out, bool three_operands) {
    if (!ctx || iters <= 0 || !tflops_out) return fail(ctx, KITE_ERR_ARG, "kite_fp64_peak: bad argument");
    CK(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, ctx->device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    if (ctx->scratch.reserve(sizeof(double) * (size_t)blocks * threads)) return fail(ctx, KITE_ERR_CUDA, "cudaMalloc failed");
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    auto go = [&](int n) {
        if (three_operands) launch_fp64_peak3((double*)ctx->scratch.ptr, n, blocks, threads, ctx->stream);
        else launch_fp64_peak((double*)ctx->scratch.ptr, n, blocks, threads, ctx->stream);
    };
    go(iters / 8 + 1);   // warm-up
    CK(cudaEventRecord(e0, ctx->stream));
    go(iters);
    CK(cudaEventRecord(e1, ctx->stream));
    ctx->launches += 2;
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    const double flops = 2.0 * (double)FP64_PEAK_FMAS_PER_ITER * iters * (double)blocks * threads;
    *tflops_out = flops / (ms * 1e-3) / 1e12;
    return KITE_OK;
}
int kite_fp64_peak(kite_ctx* ctx, int iters, double* tflops_out) { return fp64_peak_impl(ctx, iters, tflops_out, false); }
int kite_fp64_peak_reg3(kite_ctx* ctx, int iters, double* tflops_out) { return fp64_peak_impl(ctx, iters, tflops_out, true); }

}  // extern "C"
