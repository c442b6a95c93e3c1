// ntm_cabi.cu -- the extern "C" boundary declared in include/ntm_mpc.h.
//
// Host-pointer entry points stage through a grow-only device arena owned by the handle:
// H2D copies, kernel launch and D2H copies are all enqueued on the handle's stream, then the
// call blocks on the stream.  *_dev entry points only enqueue.  No exceptions leave this file
// and there is no CPU fallback: without a usable CUDA device ntm_create fails with NTM_ERR_CUDA.
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/ntm_mpc.h"
#include "ntm_kernels.h"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

}  // namespace

struct ntm_handle {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    ntm::DeviceProps props{};
    unsigned char *arena = nullptr;
    size_t arena_bytes = 0, arena_used = 0;
    unsigned int *counter = nullptr;
    double *hscratch = nullptr;      // global LDL' slabs for horizons whose G + H exceed shared memory
    size_t hscratch_bytes = 0;
    double *sv = nullptr;            // two-phase launch: saved loop state (ntm::LoopArgs::sv) ...
    size_t sv_doubles = 0;
    int *lpt = nullptr;              // ... and keys + order + bins of its longest-first work queue
    size_t lpt_ints = 0;
    long long launches = 0;
};

namespace {

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) return fail(NTM_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e__));     \
    } while (0)

#define REQUIRE(cond, msg)                                  \
    do {                                                    \
        if (!(cond)) return fail(NTM_ERR_INVALID, "%s", msg); \
    } while (0)

int check_common(ntm_handle *h, int layout, int S) {
    REQUIRE(h != nullptr, "handle is NULL");
    REQUIRE(layout == NTM_LAYOUT_MATLAB || layout == NTM_LAYOUT_SOA, "unknown layout");
    REQUIRE(S >= 0, "S must be >= 0");
    CU(cudaSetDevice(h->device));
    return NTM_OK;
}

int check_params(const double *params, int pc, int S) {
    REQUIRE(params != nullptr, "params is NULL");
    REQUIRE(pc == 1 || pc == S, "params_count must be 1 or S");
    return NTM_OK;
}

// ---- arena -------------------------------------------------------------------------------------
struct Arena {
    ntm_handle *h;
    size_t need = 0;
    explicit Arena(ntm_handle *hh) : h(hh) {}
    static size_t pad(size_t b) { return (b + 255) & ~(size_t)255; }
    void want(size_t bytes) { need += pad(bytes); }
    int reserve() {
        h->arena_used = 0;
        if (need <= h->arena_bytes) return NTM_OK;
        CU(cudaStreamSynchronize(h->stream));
        if (h->arena) CU(cudaFree(h->arena));
        h->arena = nullptr; h->arena_bytes = 0;
        const size_t want_bytes = need + need / 4;
        cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&h->arena), want_bytes);
        if (e != cudaSuccess) return fail(NTM_ERR_ALLOC, "cudaMalloc(%zu): %s", want_bytes, cudaGetErrorString(e));
        h->arena_bytes = want_bytes;
        return NTM_OK;
    }
    template <typename T>
    T *take(size_t count) {
        T *p = reinterpret_cast<T *>(h->arena + h->arena_used);
        h->arena_used += pad(count * sizeof(T));
        return p;
    }
};

int ensure_hscratch(ntm_handle *h, int N) {
    const size_t need = ntm::hscratch_bytes(h->props, N);
    if (need <= h->hscratch_bytes) return NTM_OK;
    CU(cudaStreamSynchronize(h->stream));
    if (h->hscratch) CU(cudaFree(h->hscratch));
    h->hscratch = nullptr; h->hscratch_bytes = 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&h->hscratch), need);
    if (e != cudaSuccess) return fail(NTM_ERR_ALLOC, "cudaMalloc(%zu): %s", need, cudaGetErrorString(e));
    h->hscratch_bytes = need;
    return NTM_OK;
}

int ensure_lpt(ntm_handle *h, size_t doubles, size_t ints) {
    if (doubles <= h->sv_doubles && ints <= h->lpt_ints) return NTM_OK;
    CU(cudaStreamSynchronize(h->stream));
    if (doubles > h->sv_doubles) {
        if (h->sv) CU(cudaFree(h->sv));
        h->sv = nullptr; h->sv_doubles = 0;
        cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&h->sv), doubles * sizeof(double));
        if (e != cudaSuccess) return fail(NTM_ERR_ALLOC, "cudaMalloc(%zu): %s", doubles * sizeof(double), cudaGetErrorString(e));
        h->sv_doubles = doubles;
    }
    if (ints > h->lpt_ints) {
        if (h->lpt) CU(cudaFree(h->lpt));
        h->lpt = nullptr; h->lpt_ints = 0;
        cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&h->lpt), ints * sizeof(int));
        if (e != cudaSuccess) return fail(NTM_ERR_ALLOC, "cudaMalloc(%zu): %s", ints * sizeof(int), cudaGetErrorString(e));
        h->lpt_ints = ints;
    }
    return NTM_OK;
}

template <typename T>
int h2d(ntm_handle *h, T *dst, const T *src, size_t count) {
    if (count == 0) return NTM_OK;
    CU(cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    return NTM_OK;
}
template <typename T>
int d2h(ntm_handle *h, T *dst, const T *src, size_t count) {
    if (count == 0 || dst == nullptr) return NTM_OK;
    CU(cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyDeviceToHost, h->stream));
    return NTM_OK;
}

#define TRY(expr)                      \
    do {                               \
        int rc__ = (expr);             \
        if (rc__ != NTM_OK) return rc__; \
    } while (0)

// shard copies: see closed_loop_host_impl
template <typename T>
int h2d_shard(ntm_handle *h, int layout, T *dst, const T *src, size_t E, size_t S, size_t S_total, size_t s_off) {
    if (S == 0 || E == 0) return NTM_OK;
    if (layout == NTM_LAYOUT_MATLAB || S == S_total)
        CU(cudaMemcpyAsync(dst, src + (layout == NTM_LAYOUT_MATLAB ? s_off * E : 0), E * S * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    else
        CU(cudaMemcpy2DAsync(dst, S * sizeof(T), src + s_off, S_total * sizeof(T), S * sizeof(T), E, cudaMemcpyHostToDevice, h->stream));
    return NTM_OK;
}
template <typename T>
int d2h_shard(ntm_handle *h, int layout, T *dst, const T *src, size_t E, size_t S, size_t S_total, size_t s_off) {
    if (S == 0 || E == 0 || dst == nullptr) return NTM_OK;
    if (layout == NTM_LAYOUT_MATLAB || S == S_total)
        CU(cudaMemcpyAsync(dst + (layout == NTM_LAYOUT_MATLAB ? s_off * E : 0), src, E * S * sizeof(T), cudaMemcpyDeviceToHost, h->stream));
    else
        CU(cudaMemcpy2DAsync(dst + s_off, S_total * sizeof(T), src, S * sizeof(T), S * sizeof(T), E, cudaMemcpyDeviceToHost, h->stream));
    return NTM_OK;
}

}  // namespace

extern "C" {

const char *ntm_last_error(void) { return g_err; }
int ntm_version(void) { return NTM_VERSION; }

int ntm_create(ntm_handle **out, int device) {
    REQUIRE(out != nullptr, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(NTM_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    REQUIRE(device >= 0 && device < count, "device ordinal out of range");
    CU(cudaSetDevice(device));
    ntm_handle *h = new (std::nothrow) ntm_handle();
    if (!h) return fail(NTM_ERR_ALLOC, "out of host memory");
    h->device = device;
    cudaDeviceProp p;
    e = cudaGetDeviceProperties(&p, device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void **>(&h->counter), 256);
    if (e == cudaSuccess) e = cudaMemset(h->counter, 0, 256);      // work-queue head + exit count; kernels re-arm them
    if (e != cudaSuccess) {
        delete h;
        return fail(NTM_ERR_CUDA, "ntm_create: %s", cudaGetErrorString(e));
    }
    h->stream = h->own_stream;
    h->props.sm_count = p.multiProcessorCount;
    h->props.cc_major = p.major;
    h->props.cc_minor = p.minor;
    h->props.smem_optin = p.sharedMemPerBlockOptin;
    *out = h;
    return NTM_OK;
}

int ntm_destroy(ntm_handle *h) {
    if (!h) return NTM_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->arena) cudaFree(h->arena);
    if (h->counter) cudaFree(h->counter);
    if (h->hscratch) cudaFree(h->hscratch);
    if (h->sv) cudaFree(h->sv);
    if (h->lpt) cudaFree(h->lpt);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return NTM_OK;
}

// The handle's scratch (arena, LDL' slabs, work-queue counter) is shared by everything queued through it, so a handle
// runs on ONE stream at a time: switching streams first drains the stream that is being left.  (Work still queued on the
// old stream could otherwise touch scratch that a call on the new stream re-allocates, or share the work-queue counter.)
int ntm_set_stream(ntm_handle *h, void *cuda_stream) {
    REQUIRE(h != nullptr, "handle is NULL");
    cudaStream_t ns = reinterpret_cast<cudaStream_t>(cuda_stream);
    if (ns != h->stream) {
        CU(cudaSetDevice(h->device));
        CU(cudaStreamSynchronize(h->stream));
    }
    h->stream = ns;
    return NTM_OK;
}

int ntm_reset_stream(ntm_handle *h) {
    REQUIRE(h != nullptr, "handle is NULL");
    if (h->stream != h->own_stream) {
        CU(cudaSetDevice(h->device));
        CU(cudaStreamSynchronize(h->stream));
    }
    h->stream = h->own_stream;
    return NTM_OK;
}

int ntm_sync(ntm_handle *h) {
    REQUIRE(h != nullptr, "handle is NULL");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

int ntm_device_info(ntm_handle *h, int *sm_count, int *cc_major, int *cc_minor) {
    REQUIRE(h != nullptr, "handle is NULL");
    if (sm_count) *sm_count = h->props.sm_count;
    if (cc_major) *cc_major = h->props.cc_major;
    if (cc_minor) *cc_minor = h->props.cc_minor;
    return NTM_OK;
}

long long ntm_launch_count(ntm_handle *h) { return h ? h->launches : -1; }

// ------------------------------------------------------------------------------------------------ rho
int ntm_rho_dev(ntm_handle *h, int layout, int profile, int S, const double *x, const double *params, int pc,
                double *rho1, double *rho2, double *rho3) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(x && rho1 && rho2 && rho3, "NULL array");
    CU(ntm::launch_rho(h->stream, layout, profile, S, x, params, pc, rho1, rho2, rho3, &h->launches));
    return NTM_OK;
}

int ntm_rho(ntm_handle *h, int layout, int profile, int S, const double *x, const double *params, int pc,
            double *rho1, double *rho2, double *rho3) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(x && rho1 && rho2 && rho3, "NULL array");
    const size_t s = (size_t)S;
    Arena A(h);
    A.want(2 * s * 8); A.want((size_t)pc * NTM_NPARAM * 8); A.want(s * 8); A.want(s * 8); A.want(s * 8);
    TRY(A.reserve());
    double *dx = A.take<double>(2 * s), *dp = A.take<double>((size_t)pc * NTM_NPARAM);
    double *d1 = A.take<double>(s), *d2 = A.take<double>(s), *d3 = A.take<double>(s);
    TRY(h2d(h, dx, x, 2 * s)); TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    TRY(ntm_rho_dev(h, layout, profile, S, dx, dp, pc, d1, d2, d3));
    TRY(d2h(h, rho1, d1, s)); TRY(d2h(h, rho2, d2, s)); TRY(d2h(h, rho3, d3, s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ A, B
int ntm_lpv_AB_dev(ntm_handle *h, int layout, int S, const double *rho1, const double *rho2, const double *rho3,
                   const double *params, int pc, double *Aout, double *Bout) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(rho1 && rho2 && rho3 && Aout && Bout, "NULL array");
    CU(ntm::launch_lpv(h->stream, layout, S, rho1, rho2, rho3, params, pc, Aout, Bout, &h->launches));
    return NTM_OK;
}

int ntm_lpv_AB(ntm_handle *h, int layout, int S, const double *rho1, const double *rho2, const double *rho3,
               const double *params, int pc, double *Aout, double *Bout) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(rho1 && rho2 && rho3 && Aout && Bout, "NULL array");
    const size_t s = (size_t)S;
    Arena A(h);
    A.want(s * 8); A.want(s * 8); A.want(s * 8); A.want((size_t)pc * NTM_NPARAM * 8); A.want(4 * s * 8); A.want(2 * s * 8);
    TRY(A.reserve());
    double *d1 = A.take<double>(s), *d2 = A.take<double>(s), *d3 = A.take<double>(s);
    double *dp = A.take<double>((size_t)pc * NTM_NPARAM), *dA = A.take<double>(4 * s), *dB = A.take<double>(2 * s);
    TRY(h2d(h, d1, rho1, s)); TRY(h2d(h, d2, rho2, s)); TRY(h2d(h, d3, rho3, s));
    TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    TRY(ntm_lpv_AB_dev(h, layout, S, d1, d2, d3, dp, pc, dA, dB));
    TRY(d2h(h, Aout, dA, 4 * s)); TRY(d2h(h, Bout, dB, 2 * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ condense
int ntm_condense_dev(ntm_handle *h, int layout, int profile, int S, int N, const double *R1, const double *R2,
                     const double *R3, const double *params, int pc, double *Phi, double *Gamma, double *Lambda) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(R1 && R2 && R3 && Phi && Gamma && Lambda, "NULL array");
    CU(ntm::launch_condense(h->stream, h->props, layout, profile, S, N, R1, R2, R3, params, pc, Phi, Gamma, Lambda,
                            &h->launches));
    return NTM_OK;
}

int ntm_condense(ntm_handle *h, int layout, int profile, int S, int N, const double *R1, const double *R2,
                 const double *R3, const double *params, int pc, double *Phi, double *Gamma, double *Lambda) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(R1 && R2 && R3 && Phi && Gamma && Lambda, "NULL array");
    const size_t s = (size_t)S, n = (size_t)N;
    Arena A(h);
    A.want(n * s * 8); A.want(n * s * 8); A.want(n * s * 8); A.want((size_t)pc * NTM_NPARAM * 8);
    A.want(4 * n * s * 8); A.want(2 * n * n * s * 8); A.want(2 * n * s * 8);
    TRY(A.reserve());
    double *d1 = A.take<double>(n * s), *d2 = A.take<double>(n * s), *d3 = A.take<double>(n * s);
    double *dp = A.take<double>((size_t)pc * NTM_NPARAM);
    double *dPhi = A.take<double>(4 * n * s), *dGam = A.take<double>(2 * n * n * s), *dLam = A.take<double>(2 * n * s);
    TRY(h2d(h, d1, R1, n * s)); TRY(h2d(h, d2, R2, n * s)); TRY(h2d(h, d3, R3, n * s));
    TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    TRY(ntm_condense_dev(h, layout, profile, S, N, d1, d2, d3, dp, pc, dPhi, dGam, dLam));
    TRY(d2h(h, Phi, dPhi, 4 * n * s)); TRY(d2h(h, Gamma, dGam, 2 * n * n * s)); TRY(d2h(h, Lambda, dLam, 2 * n * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ G, F
int ntm_hessian_grad_dev(ntm_handle *h, int layout, int S, int N, const double *Phi, const double *Gamma,
                         const double *Lambda, const double *x, const double *params, int pc, double *G, double *F) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(Phi && Gamma && Lambda && x && G && F, "NULL array");
    CU(ntm::launch_hessian_grad(h->stream, h->props, layout, S, N, Phi, Gamma, Lambda, x, params, pc, G, F,
                                &h->launches));
    return NTM_OK;
}

int ntm_hessian_grad(ntm_handle *h, int layout, int S, int N, const double *Phi, const double *Gamma,
                     const double *Lambda, const double *x, const double *params, int pc, double *G, double *F) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(Phi && Gamma && Lambda && x && G && F, "NULL array");
    const size_t s = (size_t)S, n = (size_t)N;
    Arena A(h);
    A.want(4 * n * s * 8); A.want(2 * n * n * s * 8); A.want(2 * n * s * 8); A.want(2 * s * 8);
    A.want((size_t)pc * NTM_NPARAM * 8); A.want(n * n * s * 8); A.want(n * s * 8);
    TRY(A.reserve());
    double *dPhi = A.take<double>(4 * n * s), *dGam = A.take<double>(2 * n * n * s), *dLam = A.take<double>(2 * n * s);
    double *dx = A.take<double>(2 * s), *dp = A.take<double>((size_t)pc * NTM_NPARAM);
    double *dG = A.take<double>(n * n * s), *dF = A.take<double>(n * s);
    TRY(h2d(h, dPhi, Phi, 4 * n * s)); TRY(h2d(h, dGam, Gamma, 2 * n * n * s)); TRY(h2d(h, dLam, Lambda, 2 * n * s));
    TRY(h2d(h, dx, x, 2 * s)); TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    TRY(ntm_hessian_grad_dev(h, layout, S, N, dPhi, dGam, dLam, dx, dp, pc, dG, dF));
    TRY(d2h(h, G, dG, n * n * s)); TRY(d2h(h, F, dF, n * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ box QP
int ntm_qp_box_dev(ntm_handle *h, int layout, int S, int N, const double *G, const double *F, const double *lb,
                   const double *ub, int bc, double *U, int *iters, int *status) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(G && F && lb && ub && U, "NULL array");
    REQUIRE(bc == 1 || bc == S, "bounds_count must be 1 or S");
    TRY(ensure_hscratch(h, N));
    CU(ntm::launch_qp_box(h->stream, h->props, layout, S, N, G, F, lb, ub, bc, U, iters, status, h->counter,
                          h->hscratch, &h->launches));
    return NTM_OK;
}

int ntm_qp_box(ntm_handle *h, int layout, int S, int N, const double *G, const double *F, const double *lb,
               const double *ub, int bc, double *U, int *iters, int *status) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(G && F && lb && ub && U, "NULL array");
    REQUIRE(bc == 1 || bc == S, "bounds_count must be 1 or S");
    const size_t s = (size_t)S, n = (size_t)N, b = (size_t)bc;
    Arena A(h);
    A.want(n * n * s * 8); A.want(n * s * 8); A.want(n * b * 8); A.want(n * b * 8); A.want(n * s * 8);
    A.want(s * 4); A.want(s * 4);
    TRY(A.reserve());
    double *dG = A.take<double>(n * n * s), *dF = A.take<double>(n * s), *dlb = A.take<double>(n * b);
    double *dub = A.take<double>(n * b), *dU = A.take<double>(n * s);
    int *dit = A.take<int>(s), *dst = A.take<int>(s);
    TRY(h2d(h, dG, G, n * n * s)); TRY(h2d(h, dF, F, n * s)); TRY(h2d(h, dlb, lb, n * b)); TRY(h2d(h, dub, ub, n * b));
    TRY(ntm_qp_box_dev(h, layout, S, N, dG, dF, dlb, dub, bc, dU, dit, dst));
    TRY(d2h(h, U, dU, n * s)); TRY(d2h(h, iters, dit, s)); TRY(d2h(h, status, dst, s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ general-inequality QP
int ntm_qp_ineq_dev(ntm_handle *h, int layout, int S, int N, int M, const double *G, const double *F,
                    const double *lb, const double *ub, int bc, const double *Lg, const double *bg, double *U,
                    int *iters, int *status) {
    TRY(check_common(h, layout, S));
    REQUIRE(M >= 0, "M must be >= 0");
    if (M == 0) return ntm_qp_box_dev(h, layout, S, N, G, F, lb, ub, bc, U, iters, status);
    if (S == 0) return NTM_OK;
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(G && F && lb && ub && U && Lg && bg, "NULL array");
    REQUIRE(bc == 1 || bc == S, "bounds_count must be 1 or S");
    REQUIRE((long long)M * N <= 0x7fffffffLL, "M*N overflows int");
    const cudaError_t e = ntm::launch_qp_ineq(h->stream, h->props, layout, S, N, M, G, F, lb, ub, bc, Lg, bg, U, iters,
                                              status, h->counter, &h->launches);
    REQUIRE(e != cudaErrorInvalidConfiguration, "ntm_qp_ineq: N, M too large for the shared-memory factor pair");
    CU(e);
    return NTM_OK;
}

int ntm_qp_ineq(ntm_handle *h, int layout, int S, int N, int M, const double *G, const double *F, const double *lb,
                const double *ub, int bc, const double *Lg, const double *bg, double *U, int *iters, int *status) {
    TRY(check_common(h, layout, S));
    REQUIRE(M >= 0, "M must be >= 0");
    if (M == 0) return ntm_qp_box(h, layout, S, N, G, F, lb, ub, bc, U, iters, status);
    if (S == 0) return NTM_OK;
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(G && F && lb && ub && U && Lg && bg, "NULL array");
    REQUIRE(bc == 1 || bc == S, "bounds_count must be 1 or S");
    const size_t s = (size_t)S, n = (size_t)N, b = (size_t)bc, m = (size_t)M;
    Arena A(h);
    A.want(n * n * s * 8); A.want(n * s * 8); A.want(n * b * 8); A.want(n * b * 8); A.want(n * s * 8);
    A.want(m * n * s * 8); A.want(m * s * 8); A.want(s * 4); A.want(s * 4);
    TRY(A.reserve());
    double *dG = A.take<double>(n * n * s), *dF = A.take<double>(n * s), *dlb = A.take<double>(n * b);
    double *dub = A.take<double>(n * b), *dU = A.take<double>(n * s);
    double *dL = A.take<double>(m * n * s), *dbg = A.take<double>(m * s);
    int *dit = A.take<int>(s), *dst = A.take<int>(s);
    TRY(h2d(h, dG, G, n * n * s)); TRY(h2d(h, dF, F, n * s)); TRY(h2d(h, dlb, lb, n * b)); TRY(h2d(h, dub, ub, n * b));
    TRY(h2d(h, dL, Lg, m * n * s)); TRY(h2d(h, dbg, bg, m * s));
    TRY(ntm_qp_ineq_dev(h, layout, S, N, M, dG, dF, dlb, dub, bc, dL, dbg, dU, dit, dst));
    TRY(d2h(h, U, dU, n * s)); TRY(d2h(h, iters, dit, s)); TRY(d2h(h, status, dst, s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ plant
int ntm_plant_step_dev(ntm_handle *h, int layout, int profile, int S, const double *x, const double *u,
                       const double *params, int pc, double *xn) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(x && u && xn, "NULL array");
    CU(ntm::launch_plant(h->stream, layout, profile, S, x, u, params, pc, xn, &h->launches));
    return NTM_OK;
}

int ntm_plant_step(ntm_handle *h, int layout, int profile, int S, const double *x, const double *u,
                   const double *params, int pc, double *xn) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(x && u && xn, "NULL array");
    const size_t s = (size_t)S;
    Arena A(h);
    A.want(2 * s * 8); A.want(s * 8); A.want((size_t)pc * NTM_NPARAM * 8); A.want(2 * s * 8);
    TRY(A.reserve());
    double *dx = A.take<double>(2 * s), *du = A.take<double>(s), *dp = A.take<double>((size_t)pc * NTM_NPARAM);
    double *dn = A.take<double>(2 * s);
    TRY(h2d(h, dx, x, 2 * s)); TRY(h2d(h, du, u, s)); TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    TRY(ntm_plant_step_dev(h, layout, profile, S, dx, du, dp, pc, dn));
    TRY(d2h(h, xn, dn, 2 * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ closed loop
static int check_loop(int N, int k_sim, int i_sim, const double *x0, double *xk, double *uk) {
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(k_sim >= 0, "k_sim must be >= 0");
    REQUIRE(i_sim >= 1, "i_sim must be >= 1");
    REQUIRE(x0 && xk && (uk || k_sim == 0), "NULL array");
    return NTM_OK;
}

static int closed_loop_dev_impl(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                                const double *x0, const double *params, int pc, int state_rows, const double *xb,
                                double *xk, double *uk, double *Uk, double *cost, int *inner_iters, int *qp_iters,
                                int *status, int rec_ld = 0, double *rec_status = nullptr) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    TRY(check_loop(N, k_sim, i_sim, x0, xk, uk));
    REQUIRE(state_rows >= NTM_STATE_ROWS_OFF && state_rows <= NTM_STATE_ROWS_FROZEN, "unknown state_rows mode");
    ntm::LoopArgs a = {};
    a.layout = layout; a.flags = profile; a.S = S; a.N = N; a.k_sim = k_sim; a.i_sim = i_sim; a.eps = eps;
    a.x0 = x0; a.params = params; a.params_count = pc;
    a.xk = xk; a.uk = uk; a.Uk = Uk; a.cost = cost; a.inner = inner_iters; a.qpit = qp_iters; a.status = status;
    a.counter = h->counter;
    a.rec_ld = rec_ld; a.rec_status = rec_status;
    a.srows = state_rows;
    if (state_rows != NTM_STATE_ROWS_OFF) {
        REQUIRE(xb, "NULL state bounds");
        a.xmin1 = xb[0]; a.xmax1 = xb[1]; a.xmin2 = xb[2]; a.xmax2 = xb[3];
        REQUIRE(a.xmin1 <= a.xmax1 && a.xmin2 <= a.xmax2, "state bounds: xmin > xmax (or NaN)");
        if (profile & (NTM_PROFILE_GAMMA_I | NTM_PROFILE_DENSE_G)) {
            // rows of a non-literal Gamma are read from the per-warp dense Gamma tile of the tensor-core Hessian build
            REQUIRE(N <= 32, "state rows inside the loop with NTM_PROFILE_GAMMA_I / DENSE_G: N <= 32");
            REQUIRE(ntm::state_rows_dense_smem(N, state_rows) <= h->props.smem_optin,
                    "horizon too long for the state rows in shared memory");
        } else {
            // both N x N factors of the continuation + 4N rows of bookkeeping live in shared memory
            const size_t need = (ntm::state_rows_smem(N));
            REQUIRE(need <= h->props.smem_optin, "horizon too long for the state rows in shared memory");
        }
    }
    TRY(ensure_hscratch(h, N));
    a.hscratch = h->hscratch;
    const size_t svd = ntm::lpt_doubles(h->props, a);      // two-phase launch with a longest-first queue (ntm_kernels.h)
    if (svd != 0) {
        TRY(ensure_lpt(h, svd, 2 * (size_t)S + NTM_LPT_BINS));
        a.sv = h->sv; a.lpt = h->lpt;
    }
    CU(ntm::launch_closed_loop(h->stream, h->props, a, &h->launches));
    return NTM_OK;
}

// Host-pointer closed loop for the scenarios [s_off, s_off + S) of a caller array that holds S_total scenarios.
// MATLAB layout: a shard is a contiguous slice of every array.  SoA layout (scenario fastest): a shard is a column
// band, moved with 2-D copies.  S_total == S, s_off == 0 is the plain single-device call.
static int closed_loop_host_impl(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                                 const double *x0, const double *params, int pc, int state_rows, const double *xb,
                                 double *xk, double *uk, double *Uk, double *cost, int *inner_iters, int *qp_iters,
                                 int *status, int S_total = -1, int s_off = 0) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    if (S_total < 0) S_total = S;
    const int pc_total = pc;                             // 1 (shared block) or S_total
    const int pcl = (pc == 1) ? 1 : S;                   // parameter blocks this shard holds
    REQUIRE(params != nullptr, "params is NULL");
    REQUIRE(pc_total == 1 || pc_total == S_total, "params_count must be 1 or S");
    TRY(check_loop(N, k_sim, i_sim, x0, xk, uk));
    const size_t s = (size_t)S, n = (size_t)N, ks = (size_t)k_sim, st = (size_t)S_total, so = (size_t)s_off;
    Arena A(h);
    A.want(2 * s * 8); A.want((size_t)pcl * NTM_NPARAM * 8); A.want(2 * (ks + 1) * s * 8); A.want(ks * s * 8);
    if (Uk) A.want(n * ks * s * 8);
    A.want(s * 8); A.want(ks * s * 4); A.want(ks * s * 4); A.want(s * 4);
    TRY(A.reserve());
    double *dx0 = A.take<double>(2 * s), *dp = A.take<double>((size_t)pcl * NTM_NPARAM);
    double *dxk = A.take<double>(2 * (ks + 1) * s), *duk = A.take<double>(ks * s);
    double *dUk = Uk ? A.take<double>(n * ks * s) : nullptr;
    double *dcost = A.take<double>(s);
    int *din = A.take<int>(ks * s), *dqp = A.take<int>(ks * s), *dst = A.take<int>(s);
    TRY(h2d_shard(h, layout, dx0, x0, 2, s, st, so));
    if (pc == 1) TRY(h2d(h, dp, params, (size_t)NTM_NPARAM));
    else TRY(h2d_shard(h, layout, dp, params, NTM_NPARAM, s, st, so));
    TRY(closed_loop_dev_impl(h, layout, profile, S, N, k_sim, i_sim, eps, dx0, dp, pcl, state_rows, xb, dxk, duk, dUk,
                             dcost, din, dqp, dst));
    TRY(d2h_shard(h, layout, xk, dxk, 2 * (ks + 1), s, st, so)); TRY(d2h_shard(h, layout, uk, duk, ks, s, st, so));
    if (Uk) TRY(d2h_shard(h, layout, Uk, dUk, n * ks, s, st, so));
    TRY(d2h_shard(h, layout, cost, dcost, 1, s, st, so)); TRY(d2h_shard(h, layout, inner_iters, din, ks, s, st, so));
    TRY(d2h_shard(h, layout, qp_iters, dqp, ks, s, st, so)); TRY(d2h_shard(h, layout, status, dst, 1, s, st, so));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ---- one host process, every visible GPU (the MEX gateway ntm_mpc_batch is single-process by construction) ----------
// Scenarios never interact (NTM_MPC_Sim.m:93-131 has no cross-scenario term), so the batch is cut into contiguous
// shards of ceil(S / G) scenarios, one per device; each device runs on its own pooled handle and host thread and moves
// its shard straight between the caller's arrays and its HBM.  No collective: the "gather" is the D2H copy itself.
namespace {
std::mutex g_pool_mu;
std::vector<ntm_handle *> g_pool;                          // one lazily created handle per device ordinal

int pool_handle(int device, ntm_handle **out) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if ((int)g_pool.size() <= device) g_pool.resize((size_t)device + 1, nullptr);
    if (g_pool[device] == nullptr) TRY(ntm_create(&g_pool[device], device));
    *out = g_pool[device];
    return NTM_OK;
}
}  // namespace

long long ntm_pool_launch_count(int device) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (device < 0 || device >= (int)g_pool.size() || g_pool[device] == nullptr) return -1;
    return g_pool[device]->launches;
}

int ntm_device_count(int *count) {
    REQUIRE(count != nullptr, "count is NULL");
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) return fail(NTM_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    *count = c;
    return NTM_OK;
}

int ntm_mpc_closed_loop_multi(int n_devices, const int *devices, int layout, int profile, int S, int N, int k_sim,
                              int i_sim, double eps, const double *x0, const double *params, int pc, int state_rows,
                              const double *xbounds, double *xk, double *uk, double *Uk, double *cost, int *inner_iters,
                              int *qp_iters, int *status) {
    REQUIRE(layout == NTM_LAYOUT_MATLAB || layout == NTM_LAYOUT_SOA, "unknown layout");
    REQUIRE(S >= 0, "S must be >= 0");
    int visible = 0;
    TRY(ntm_device_count(&visible));
    if (visible == 0) return fail(NTM_ERR_CUDA, "no CUDA device available; this library has no CPU fallback");
    if (n_devices <= 0) n_devices = visible;               // 0 = all visible devices
    REQUIRE(n_devices <= 64, "too many devices");
    std::vector<int> dev((size_t)n_devices);
    for (int g = 0; g < n_devices; ++g) {
        dev[g] = devices ? devices[g] : g;
        REQUIRE(dev[g] >= 0 && dev[g] < visible, "device ordinal out of range");
        for (int q = 0; q < g; ++q) REQUIRE(dev[q] != dev[g], "device listed twice");
    }
    if (S == 0) return NTM_OK;
    REQUIRE(params != nullptr, "params is NULL");
    REQUIRE(pc == 1 || pc == S, "params_count must be 1 or S");
    TRY(check_loop(N, k_sim, i_sim, x0, xk, uk));
    const int per = (S + n_devices - 1) / n_devices;       // SURVEY 8(e): rank g owns [g*per, min(S, (g+1)*per))
    std::vector<ntm_handle *> hs((size_t)n_devices, nullptr);
    for (int g = 0; g < n_devices; ++g) if (g * per < S) TRY(pool_handle(dev[g], &hs[g]));
    std::vector<int> rc((size_t)n_devices, NTM_OK);
    std::vector<std::string> msg((size_t)n_devices);
    auto shard = [&](int g) {
        const int s0 = g * per, sl = (S - s0 < per) ? S - s0 : per;
        rc[g] = closed_loop_host_impl(hs[g], layout, profile, sl, N, k_sim, i_sim, eps, x0, params, pc, state_rows, xbounds,
                                      xk, uk, Uk, cost, inner_iters, qp_iters, status, S, s0);
        if (rc[g] != NTM_OK) msg[g] = g_err;               // g_err is thread-local: carry the text to the caller's thread
    };
    std::vector<std::thread> th;
    for (int g = 1; g < n_devices; ++g) if (hs[g]) th.emplace_back(shard, g);
    shard(0);
    for (auto &t : th) t.join();
    for (int g = 0; g < n_devices; ++g)
        if (rc[g] != NTM_OK) return fail(rc[g], "device %d: %s", dev[g], msg[g].c_str());
    return NTM_OK;
}

// Packed-record variant of the resident entry (scenario-slowest inputs): ONE array `rec` of NTM_REC_DOUBLES(k_sim)
// doubles per scenario = [xk (2(k_sim+1)) | uk (k_sim) | cost | status] -- the block a multi-GPU caller gathers with a
// single collective (SURVEY 8e: "one ncclAllGather of per-scenario outputs").
int ntm_mpc_closed_loop_rec_dev(ntm_handle *h, int profile, int S, int N, int k_sim, int i_sim, double eps,
                                const double *x0, const double *params, int pc, int state_rows, const double *xbounds,
                                double *rec, int *inner_iters, int *qp_iters) {
    TRY(check_common(h, NTM_LAYOUT_MATLAB, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(rec != nullptr, "rec is NULL");
    TRY(check_loop(N, k_sim, i_sim, x0, rec, rec));
    const int ld = NTM_REC_DOUBLES(k_sim);
    return closed_loop_dev_impl(h, NTM_LAYOUT_MATLAB, profile, S, N, k_sim, i_sim, eps, x0, params, pc, state_rows, xbounds,
                                rec, rec + 2 * (k_sim + 1), nullptr, rec + 3 * k_sim + 2, inner_iters, qp_iters, nullptr,
                                ld, rec + 3 * k_sim + 3);
}

int ntm_mpc_closed_loop_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                            const double *x0, const double *params, int pc, double *xk, double *uk, double *Uk,
                            double *cost, int *inner_iters, int *qp_iters, int *status) {
    return closed_loop_dev_impl(h, layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, NTM_STATE_ROWS_OFF, nullptr,
                                xk, uk, Uk, cost, inner_iters, qp_iters, status);
}

int ntm_mpc_closed_loop(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                        const double *x0, const double *params, int pc, double *xk, double *uk, double *Uk,
                        double *cost, int *inner_iters, int *qp_iters, int *status) {
    return closed_loop_host_impl(h, layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, NTM_STATE_ROWS_OFF,
                                 nullptr, xk, uk, Uk, cost, inner_iters, qp_iters, status);
}

int ntm_mpc_closed_loop_sc_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                               const double *x0, const double *params, int pc, int state_rows, const double *xbounds,
                               double *xk, double *uk, double *Uk, double *cost, int *inner_iters, int *qp_iters,
                               int *status) {
    return closed_loop_dev_impl(h, layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, state_rows, xbounds, xk, uk,
                                Uk, cost, inner_iters, qp_iters, status);
}

int ntm_mpc_closed_loop_sc(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                           const double *x0, const double *params, int pc, int state_rows, const double *xbounds,
                           double *xk, double *uk, double *Uk, double *cost, int *inner_iters, int *qp_iters,
                           int *status) {
    return closed_loop_host_impl(h, layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, state_rows, xbounds, xk,
                                 uk, Uk, cost, inner_iters, qp_iters, status);
}

// ------------------------------------------------------------------------------------------------ controller step
// One time step of the fused loop without the plant: k_sim = 1, the caller's records in LoopArgs::sv, ONE launch.
static int check_step(int profile, int N, int i_sim) {
    REQUIRE(!(profile & NTM_PROFILE_TAUE_W), "ntm_mpc_step: NTM_PROFILE_TAUE_W is not supported by the controller step");
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(i_sim >= 1, "i_sim must be >= 1");
    return NTM_OK;
}

int ntm_mpc_step_dev(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                     const double *params, int pc, double *state, double *u, double *U, int *inner_iters, int *qp_iters,
                     int *status) {
    TRY(check_common(h, layout, S));
    TRY(check_step(profile, N, i_sim));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(x && state && u, "NULL array");
    ntm::LoopArgs a = {};
    a.layout = layout; a.S = S; a.N = N; a.k_sim = 1; a.i_sim = i_sim; a.eps = eps;
    a.flags = profile & ~(NTM_PROFILE_PLANT_C | NTM_PROFILE_PLANT_RK4);   // plant-only bits: no effect on the controller
    a.x0 = x; a.params = params; a.params_count = pc;
    a.uk = u; a.Uk = U; a.inner = inner_iters; a.qpit = qp_iters; a.status = status;
    a.counter = h->counter;
    a.sv = state; a.ctl = 1;
    TRY(ensure_hscratch(h, N));
    a.hscratch = h->hscratch;
    CU(ntm::launch_closed_loop(h->stream, h->props, a, &h->launches));
    return NTM_OK;
}

int ntm_mpc_step(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                 const double *params, int pc, double *state, double *u, double *U, int *inner_iters, int *qp_iters,
                 int *status) {
    TRY(check_common(h, layout, S));
    TRY(check_step(profile, N, i_sim));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(x && state && u, "NULL array");
    const size_t s = (size_t)S, n = (size_t)N, ld = (size_t)NTM_CTRL_DOUBLES(N);
    Arena A(h);
    A.want(2 * s * 8); A.want((size_t)pc * NTM_NPARAM * 8); A.want(ld * s * 8); A.want(s * 8);
    if (U) A.want(n * s * 8);
    A.want(s * 4); A.want(s * 4); A.want(s * 4);
    TRY(A.reserve());
    double *dx = A.take<double>(2 * s), *dp = A.take<double>((size_t)pc * NTM_NPARAM), *dst = A.take<double>(ld * s);
    double *du = A.take<double>(s), *dU = U ? A.take<double>(n * s) : nullptr;
    int *din = A.take<int>(s), *dqp = A.take<int>(s), *dstat = A.take<int>(s);
    TRY(h2d(h, dx, x, 2 * s)); TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM)); TRY(h2d(h, dst, state, ld * s));
    TRY(ntm_mpc_step_dev(h, layout, profile, S, N, i_sim, eps, dx, dp, pc, dst, du, dU, din, dqp, dstat));
    TRY(d2h(h, state, dst, ld * s)); TRY(d2h(h, u, du, s)); TRY(d2h(h, U, dU, n * s));
    TRY(d2h(h, inner_iters, din, s)); TRY(d2h(h, qp_iters, dqp, s)); TRY(d2h(h, status, dstat, s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ getWLc
int ntm_getWLc_dev(ntm_handle *h, int layout, int S, int N, const double *bounds, const double *Gamma, const double *Phi,
                   const double *Lambda, double *W, double *L, double *c) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(bounds && Gamma && Phi && Lambda && W && L && c, "NULL array");
    CU(ntm::launch_getwlc(h->stream, h->props, layout, S, N, bounds, Gamma, Phi, Lambda, W, L, c, &h->launches));
    return NTM_OK;
}

int ntm_getWLc(ntm_handle *h, int layout, int S, int N, const double *bounds, const double *Gamma, const double *Phi,
               const double *Lambda, double *W, double *L, double *c) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(bounds && Gamma && Phi && Lambda && W && L && c, "NULL array");
    const size_t s = (size_t)S, n = (size_t)N, r = 6 * n + 4;
    Arena A(h);
    A.want(2 * n * n * s * 8); A.want(4 * n * s * 8); A.want(2 * n * s * 8);
    A.want(r * 2 * s * 8); A.want(r * n * s * 8); A.want(r * s * 8);
    TRY(A.reserve());
    double *dGam = A.take<double>(2 * n * n * s), *dPhi = A.take<double>(4 * n * s), *dLam = A.take<double>(2 * n * s);
    double *dW = A.take<double>(r * 2 * s), *dL = A.take<double>(r * n * s), *dc = A.take<double>(r * s);
    TRY(h2d(h, dGam, Gamma, 2 * n * n * s)); TRY(h2d(h, dPhi, Phi, 4 * n * s)); TRY(h2d(h, dLam, Lambda, 2 * n * s));
    TRY(ntm_getWLc_dev(h, layout, S, N, bounds, dGam, dPhi, dLam, dW, dL, dc));
    TRY(d2h(h, W, dW, r * 2 * s)); TRY(d2h(h, L, dL, r * n * s)); TRY(d2h(h, c, dc, r * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ Monte-Carlo statistics
int ntm_mc_stats_dev(ntm_handle *h, int layout, int S, int k_sim, const double *xk, const double *uk,
                     const double *cost, const int *status, const double *params, int pc, const double *bounds,
                     double w_sup, double hist_max, double *out) {
    TRY(check_common(h, layout, S));
    REQUIRE(k_sim >= 1, "k_sim must be >= 1");
    REQUIRE(bounds && out, "NULL array");
    const double *umin = nullptr, *umax = nullptr;
    int ustride = 0;
    if (S > 0) {
        TRY(check_params(params, pc, S));
        REQUIRE(xk && uk, "NULL array");
        // where umin / umax (slots 8 and 9 of the parameter block) of scenario s live in the caller's layout
        if (pc == 1) { umin = params + 8; umax = params + 9; ustride = 0; }
        else if (layout == NTM_LAYOUT_MATLAB) { umin = params + 8; umax = params + 9; ustride = NTM_NPARAM; }
        else { umin = params + 8 * (size_t)S; umax = params + 9 * (size_t)S; ustride = 1; }
    }
    CU(ntm::launch_mc_stats(h->stream, h->props, layout, S, k_sim, xk, uk, cost, status, umin, umax, ustride, bounds, w_sup,
                            hist_max, out, &h->launches));
    return NTM_OK;
}

// The same reduction with the EC-power box handed over as two compact arrays umin[S], umax[S] (bounds_count = S) or
// one shared pair (bounds_count = 1): in the MATLAB layout the parameter block costs a 128-byte line per scenario for
// these two doubles (ncu: 667 MB of DRAM reads for 534 MB of results at S = 2^20).
int ntm_mc_stats_ub_dev(ntm_handle *h, int layout, int S, int k_sim, const double *xk, const double *uk,
                        const double *cost, const int *status, const double *umin, const double *umax, int bounds_count,
                        const double *bounds, double w_sup, double hist_max, double *out) {
    TRY(check_common(h, layout, S));
    REQUIRE(k_sim >= 1, "k_sim must be >= 1");
    REQUIRE(bounds && out, "NULL array");
    if (S > 0) {
        REQUIRE(xk && uk && umin && umax, "NULL array");
        REQUIRE(bounds_count == 1 || bounds_count == S, "bounds_count must be 1 or S");
    }
    CU(ntm::launch_mc_stats(h->stream, h->props, layout, S, k_sim, xk, uk, cost, status, umin, umax, bounds_count == 1 ? 0 : 1,
                            bounds, w_sup, hist_max, out, &h->launches));
    return NTM_OK;
}

int ntm_mc_stats(ntm_handle *h, int layout, int S, int k_sim, const double *xk, const double *uk, const double *cost,
                 const int *status, const double *params, int pc, const double *bounds, double w_sup,
                 double hist_max, double *out) {
    TRY(check_common(h, layout, S));
    REQUIRE(k_sim >= 1, "k_sim must be >= 1");
    REQUIRE(bounds && out, "NULL array");
    if (S > 0) {
        TRY(check_params(params, pc, S));
        REQUIRE(xk && uk, "NULL array");
    }
    const size_t s = (size_t)S, k = (size_t)k_sim;
    Arena A(h);
    A.want(2 * (k + 1) * s * 8 + 8); A.want(k * s * 8 + 8); A.want(s * 8 + 8); A.want(s * 4 + 8);
    A.want((size_t)pc * NTM_NPARAM * 8 + 8); A.want(NTM_MC_NSTAT * 8);
    TRY(A.reserve());
    double *dx = A.take<double>(2 * (k + 1) * s + 1), *du = A.take<double>(k * s + 1), *dc = A.take<double>(s + 1);
    int *dst = A.take<int>(s + 2);
    double *dp = A.take<double>((size_t)(S > 0 ? pc : 0) * NTM_NPARAM + 1), *dout = A.take<double>(NTM_MC_NSTAT);
    if (S > 0) {
        TRY(h2d(h, dx, xk, 2 * (k + 1) * s)); TRY(h2d(h, du, uk, k * s));
        if (cost) TRY(h2d(h, dc, cost, s));
        if (status) TRY(h2d(h, dst, status, s));
        TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    }
    TRY(ntm_mc_stats_dev(h, layout, S, k_sim, dx, du, cost ? dc : nullptr, status ? dst : nullptr, dp, pc, bounds, w_sup,
                         hist_max, dout));
    TRY(d2h(h, out, dout, (size_t)NTM_MC_NSTAT));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ fp64 peak
int ntm_fp64_peak(ntm_handle *h, int iters, double *tflops_dfma, double *ms_out) {
    REQUIRE(h != nullptr, "handle is NULL");
    REQUIRE(iters > 0, "iters must be > 0");
    CU(cudaSetDevice(h->device));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    double *out = reinterpret_cast<double *>(h->counter) + 8;
    CU(ntm::launch_fp64_peak(h->stream, h->props, iters / 8 + 1, out, &h->launches));   // warm-up
    CU(cudaEventRecord(e0, h->stream));
    CU(ntm::launch_fp64_peak(h->stream, h->props, iters, out, &h->launches));
    CU(cudaEventRecord(e1, h->stream));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    const double flops = 2.0 * 64.0 * (double)iters * 256.0 * (double)h->props.sm_count * 8.0;
    if (tflops_dfma) *tflops_dfma = flops / (ms * 1e-3) / 1e12;
    if (ms_out) *ms_out = ms;
    return NTM_OK;
}

}  // extern "C"

int ntm_dmma_peak(ntm_handle *h, int iters, double *tflops_dmma, double *ms_out) {
    REQUIRE(h != nullptr, "handle is NULL");
    REQUIRE(iters > 0, "iters must be > 0");
    CU(cudaSetDevice(h->device));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    double *out = reinterpret_cast<double *>(h->counter) + 8;
    CU(ntm::launch_dmma_peak(h->stream, h->props, iters / 8 + 1, out, &h->launches));   // warm-up
    CU(cudaEventRecord(e0, h->stream));
    CU(ntm::launch_dmma_peak(h->stream, h->props, iters, out, &h->launches));
    CU(cudaEventRecord(e1, h->stream));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    // 8 DMMA.8x8x4 per warp and iteration, 2*8*8*4 flops each, 8 warps per CTA, 8 CTAs per SM
    const double flops = 512.0 * 8.0 * (double)iters * 8.0 * (double)h->props.sm_count * 8.0;
    if (tflops_dmma) *tflops_dmma = flops / (ms * 1e-3) / 1e12;
    if (ms_out) *ms_out = ms;
    return NTM_OK;
}
