// ntm_cabi.cu -- the extern "C" boundary declared in include/ntm_mpc.h.
//
// Host-pointer entry points stage through a grow-only device arena owned by the handle:
// H2D copies, kernel launch and D2H copies are all enqueued on the handle's stream, then the
// call blocks on the stream.  *_dev entry points only enqueue.  Every entry checks all of its
// arguments before it allocates, copies or launches anything.  No exceptions leave this file
// and there is no CPU fallback: without a usable CUDA device ntm_create fails with NTM_ERR_CUDA.
#include <algorithm>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <type_traits>
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
    size_t arena_bytes = 0;
    unsigned int *counter = nullptr;
    double *hscratch = nullptr;      // global LDL' slabs for horizons whose G + H exceed shared memory
    size_t hscratch_bytes = 0;
    double *sv = nullptr;            // two-phase launch: saved loop state (ntm::LoopArgs::sv) ...
    size_t sv_bytes = 0;
    int *lpt = nullptr;              // ... and keys + order + bins of its longest-first work queue
    size_t lpt_bytes = 0;
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

#define TRY(expr)                      \
    do {                               \
        int rc__ = (expr);             \
        if (rc__ != NTM_OK) return rc__; \
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

// Grows a handle-owned device buffer to `bytes` unless it already holds `need`; it never shrinks.  Work still queued on
// the handle's stream may use the old buffer, so the stream is drained before it is freed.
template <typename T>
int grow(ntm_handle *h, T *&buf, size_t &have, size_t need, size_t bytes) {
    if (need <= have) return NTM_OK;
    CU(cudaStreamSynchronize(h->stream));
    if (buf) CU(cudaFree(buf));
    buf = nullptr; have = 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&buf), bytes);
    if (e != cudaSuccess) return fail(NTM_ERR_ALLOC, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    have = bytes;
    return NTM_OK;
}
template <typename T>
int grow(ntm_handle *h, T *&buf, size_t &have, size_t bytes) { return grow(h, buf, have, bytes, bytes); }

// ---- arena -------------------------------------------------------------------------------------
// The buffers of one host-pointer call, carved from the handle's grow-only device arena.  A call declares them once, in a
// layout callback of take<T>(count) calls; reserve runs it twice, to size the arena and to hand the buffers out, so the
// size cannot disagree with what is handed out.
class Arena {
  public:
    explicit Arena(ntm_handle *hh) : h(hh) {}
    template <typename F>
    int reserve(F layout) {
        base = nullptr; used = 0;                        // sizing pass: take() returns NULL
        layout(*this);
        TRY(grow(h, h->arena, h->arena_bytes, used, used + used / 4));
        base = h->arena; used = 0;
        layout(*this);
        return NTM_OK;
    }
    template <typename T>
    T *take(size_t count) {
        T *p = base ? reinterpret_cast<T *>(base + used) : nullptr;
        used += (count * sizeof(T) + 255) & ~(size_t)255;
        return p;
    }

  private:
    ntm_handle *h;
    unsigned char *base = nullptr;
    size_t used = 0;
};

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

// shard copies: see fused_host
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

// ---- fused calls: closed loop, perturbed loop, controller step -------------------------------------------------------
// A fused call is the ntm::LoopArgs of its launch.  Its entry fills in the caller's arrays (NULL = not passed) and its
// mode: srows, ctl with the controller records in sv, pert with the plant in pp, rec_ld and rec_status.  check_fused
// checks it, then the dev path launches it as it is and the host path stages its arrays first.

ntm::LoopArgs loop_args(int layout, int profile, int S, int N, int k_sim, int i_sim, double eps, const double *x0,
                        const double *params, int pc, int state_rows, double *xk, double *uk, double *Uk, double *cost,
                        int *inner, int *qpit, int *status) {
    ntm::LoopArgs a = {};
    a.layout = layout; a.flags = profile; a.S = S; a.N = N; a.k_sim = k_sim; a.i_sim = i_sim; a.eps = eps;
    a.x0 = x0; a.params = params; a.params_count = pc; a.srows = state_rows;
    a.xk = xk; a.uk = uk; a.Uk = Uk; a.cost = cost; a.inner = inner; a.qpit = qpit; a.status = status;
    return a;
}

// One time step of the fused loop without the plant: k_sim = 1, x the measured state, the caller's records in sv, u and U
// in uk and Uk.
ntm::LoopArgs step_args(int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                        const double *params, int pc, int state_rows, double *state, double *u, double *U, int *inner,
                        int *qpit, int *status) {
    ntm::LoopArgs a = loop_args(layout, profile, S, N, 1, i_sim, eps, x, params, pc, state_rows, nullptr, u, U, nullptr,
                                inner, qpit, status);
    a.sv = state; a.ctl = 1;
    return a;
}

// The fused loop with the plant of ntm_plant_step on its own block and profile bits, d_k and v_k.
ntm::LoopArgs perturbed_args(int layout, int profile, int S, int N, int k_sim, int i_sim, double eps, const double *x0,
                             const double *params, int pc, int state_rows, const double *plant_params, int ppc,
                             int plant_profile, const double *w, const double *v, double *xk, double *uk, double *Uk,
                             double *cost, int *inner, int *qpit, int *status) {
    ntm::LoopArgs a = loop_args(layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, state_rows, xk, uk, Uk, cost,
                                inner, qpit, status);
    a.pp = {plant_params, w, v, ppc, plant_profile};
    a.pert = 1;
    return a;
}

// Every rule of a fused call.  It also sets what the rules decide: the state box from xb (on the host), the profile the
// controller runs (a step and the perturbed loop ignore the plant-only bits) and the plant's parameter count when
// plant_params is NULL (the controller's block).  At S == 0 a loop checks nothing beyond handle, layout and S; a
// controller step checks everything but its parameters and arrays.  params_count (and plant_params_count) is 1 or
// S_total, the scenarios of the caller's arrays, of which `a` may be a shard.
int check_fused(ntm_handle *h, ntm::LoopArgs &a, const double *xb, int S_total) {
    TRY(check_common(h, a.layout, a.S));
    if (a.S == 0 && !a.ctl) return NTM_OK;
    if (a.ctl || a.pert) {
        REQUIRE(!(a.flags & NTM_PROFILE_TAUE_W), "ntm_mpc_step: NTM_PROFILE_TAUE_W is not supported by the controller step");
        a.flags &= ~(NTM_PROFILE_PLANT_C | NTM_PROFILE_PLANT_RK4);
    }
    REQUIRE(a.N >= 1 && a.N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(a.k_sim >= 0, "k_sim must be >= 0");
    REQUIRE(a.i_sim >= 1, "i_sim must be >= 1");
    REQUIRE(a.srows >= NTM_STATE_ROWS_OFF && a.srows <= NTM_STATE_ROWS_FROZEN, "unknown state_rows mode");
    if (a.srows != NTM_STATE_ROWS_OFF) {
        REQUIRE(xb, "NULL state bounds");
        a.xmin1 = xb[0]; a.xmax1 = xb[1]; a.xmin2 = xb[2]; a.xmax2 = xb[3];
        REQUIRE(a.xmin1 <= a.xmax1 && a.xmin2 <= a.xmax2, "state bounds: xmin > xmax (or NaN)");
        // The rows of a non-literal Gamma are read from the per-warp dense Gamma tile of the tensor-core Hessian build;
        // with the literal Gamma both N x N factors of the continuation + 4N rows of bookkeeping live in shared memory.
        const bool dense = a.flags & (NTM_PROFILE_GAMMA_I | NTM_PROFILE_DENSE_G);
        REQUIRE(!dense || a.N <= 32, "state rows inside the loop with NTM_PROFILE_GAMMA_I / DENSE_G: N <= 32");
        REQUIRE((dense ? ntm::state_rows_dense_smem(a.N, a.srows) : ntm::state_rows_smem(a.N)) <= h->props.smem_optin,
                "horizon too long for the state rows in shared memory");
    }
    if (a.S == 0) return NTM_OK;
    TRY(check_params(a.params, a.params_count, S_total));
    REQUIRE(a.rec_ld == 0 || a.xk, "rec is NULL");
    REQUIRE(a.x0 && (a.ctl ? a.sv : a.xk) && (a.uk || a.k_sim == 0), "NULL array");
    if (a.pert) {
        if (!a.pp.pparams) a.pp.pparams_count = a.params_count;
        REQUIRE(a.pp.pparams_count == 1 || a.pp.pparams_count == S_total, "plant_params_count must be 1 or S");
        REQUIRE(!(a.pp.pflags & ~(NTM_PROFILE_RHO1_SQ | NTM_PROFILE_PLANT_C | NTM_PROFILE_PLANT_RK4 | NTM_PROFILE_TAUE_W)),
                "plant_profile: only RHO1_SQ, PLANT_C, PLANT_RK4 and TAUE_W act on the plant");
    }
    return NTM_OK;
}

// Launches a checked fused call on device arrays, with the handle's work-queue counter, LDL' scratch and, when the launch
// runs in two phases, its saved loop state and longest-first queue.
int launch_fused(ntm_handle *h, ntm::LoopArgs a) {
    if (a.pert && !a.pp.pparams) a.pp.pparams = a.params;
    a.counter = h->counter;
    TRY(grow(h, h->hscratch, h->hscratch_bytes, ntm::hscratch_bytes(h->props, a.N)));
    a.hscratch = h->hscratch;
    const size_t svd = ntm::lpt_doubles(h->props, a);      // two-phase launch with a longest-first queue (ntm_kernels.h)
    int *lpt = nullptr;
    if (svd != 0) {
        TRY(grow(h, h->sv, h->sv_bytes, svd * sizeof(double)));
        TRY(grow(h, h->lpt, h->lpt_bytes, (2 * (size_t)a.S + NTM_LPT_BINS) * sizeof(int)));
        a.sv = h->sv; lpt = h->lpt;
    }
    CU(ntm::launch_closed_loop(h->stream, h->props, a, lpt, &h->launches));
    return NTM_OK;
}

enum Dir { IN, OUT, INOUT };

// The arrays a host-pointer fused call stages, the caller's in `a` beside their device copies in `d`:
// f(caller's, copy, elements per scenario, direction, one block for every scenario).  The only place their sizes are
// written.
template <typename F>
void fused_arrays(const ntm::LoopArgs &a, ntm::LoopArgs &d, F f) {
    const size_t n = (size_t)a.N, ks = (size_t)a.k_sim;
    f(a.x0, d.x0, 2, IN, false);
    f(a.params, d.params, NTM_NPARAM, IN, a.params_count == 1);
    f(a.pp.pparams, d.pp.pparams, NTM_NPARAM, IN, a.pp.pparams_count == 1);
    f(a.pp.dist, d.pp.dist, 2 * ks, IN, false);
    f(a.pp.noise, d.pp.noise, 2 * ks, IN, false);
    f(a.sv, d.sv, (size_t)NTM_CTRL_DOUBLES(a.N), INOUT, false);
    f(a.xk, d.xk, 2 * (ks + 1), OUT, false);
    f(a.uk, d.uk, ks, OUT, false);
    f(a.Uk, d.Uk, n * ks, OUT, false);
    f(a.cost, d.cost, 1, OUT, false);
    f(a.inner, d.inner, ks, OUT, false);
    f(a.qpit, d.qpit, ks, OUT, false);
    f(a.status, d.status, 1, OUT, false);
}

// Host-pointer fused call for the scenarios [s_off, s_off + a.S) of caller arrays that hold S_total scenarios, `a`
// checked: copies every array the caller passed to the arena, launches on the copies, copies the outputs back and waits.
// MATLAB layout: a shard is a contiguous slice of every array.  SoA layout (scenario fastest): a shard is a column band,
// moved with 2-D copies.  A parameter count of 1 is one block for every scenario.
int fused_host(ntm_handle *h, const ntm::LoopArgs &a, int S_total, int s_off) {
    const size_t s = (size_t)a.S, st = (size_t)S_total, so = (size_t)s_off;
    ntm::LoopArgs d = a;
    TRY(Arena(h).reserve([&](Arena &A) {
        fused_arrays(a, d, [&](auto src, auto &dst, size_t E, Dir, bool shared) {
            if (src) dst = A.take<std::remove_pointer_t<decltype(src)>>(shared ? E : E * s);
        });
    }));
    int rc = NTM_OK;
    fused_arrays(a, d, [&](auto src, auto dst, size_t E, Dir dir, bool shared) {
        using T = std::remove_const_t<std::remove_pointer_t<decltype(src)>>;
        T *to = const_cast<T *>(dst);                      // the arena copy of an input
        if (rc == NTM_OK && src && dir != OUT)
            rc = shared ? h2d(h, to, src, E) : h2d_shard(h, a.layout, to, src, E, s, st, so);
    });
    TRY(rc);
    if (d.params_count == S_total) d.params_count = a.S;   // the blocks of this shard
    if (d.pp.pparams_count == S_total) d.pp.pparams_count = a.S;
    TRY(launch_fused(h, d));
    fused_arrays(a, d, [&](auto src, auto dst, size_t E, Dir dir, bool) {
        if constexpr (!std::is_const_v<std::remove_pointer_t<decltype(src)>>)   // inputs are const
            if (rc == NTM_OK && dir != IN) rc = d2h_shard(h, a.layout, src, dst, E, s, st, so);
    });
    TRY(rc);
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

int fused_dev_call(ntm_handle *h, ntm::LoopArgs a, const double *xb) {
    TRY(check_fused(h, a, xb, a.S));
    return a.S == 0 ? NTM_OK : launch_fused(h, a);
}

int fused_host_call(ntm_handle *h, ntm::LoopArgs a, const double *xb) {
    TRY(check_fused(h, a, xb, a.S));
    return a.S == 0 ? NTM_OK : fused_host(h, a, a.S, 0);
}

// ---- per-call operations: one check each, called by its host and its device entry ------------------------------------

int check_rho(ntm_handle *h, int layout, int S, const double *x, const double *params, int pc, const double *rho1,
              const double *rho2, const double *rho3) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(x && rho1 && rho2 && rho3, "NULL array");
    return NTM_OK;
}

int check_lpv(ntm_handle *h, int layout, int S, const double *rho1, const double *rho2, const double *rho3,
              const double *params, int pc, const double *A, const double *B) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(rho1 && rho2 && rho3 && A && B, "NULL array");
    return NTM_OK;
}

int check_condense(ntm_handle *h, int layout, int S, int N, const double *R1, const double *R2, const double *R3,
                   const double *params, int pc, const double *Phi, const double *Gamma, const double *Lambda) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(R1 && R2 && R3 && Phi && Gamma && Lambda, "NULL array");
    return NTM_OK;
}

int check_hessian_grad(ntm_handle *h, int layout, int S, int N, const double *Phi, const double *Gamma,
                       const double *Lambda, const double *x, const double *params, int pc, const double *G,
                       const double *F) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(Phi && Gamma && Lambda && x && G && F, "NULL array");
    return NTM_OK;
}

int check_qp_box(ntm_handle *h, int layout, int S, int N, const double *G, const double *F, const double *lb,
                 const double *ub, int bc, const double *U) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(G && F && lb && ub && U, "NULL array");
    REQUIRE(bc == 1 || bc == S, "bounds_count must be 1 or S");
    return NTM_OK;
}

// M == 0 passes here and is ntm_qp_box's to check
int check_qp_ineq(ntm_handle *h, int layout, int S, int N, int M, const double *G, const double *F, const double *lb,
                  const double *ub, int bc, const double *Lg, const double *bg, const double *U) {
    TRY(check_common(h, layout, S));
    REQUIRE(M >= 0, "M must be >= 0");
    if (M == 0 || S == 0) return NTM_OK;
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(G && F && lb && ub && U && Lg && bg, "NULL array");
    REQUIRE(bc == 1 || bc == S, "bounds_count must be 1 or S");
    REQUIRE((long long)M * N <= 0x7fffffffLL, "M*N overflows int");
    REQUIRE(ntm::qp_ineq_groups(h->props, N, M) > 0, "ntm_qp_ineq: N, M too large for the shared-memory factor pair");
    return NTM_OK;
}

int check_plant(ntm_handle *h, int layout, int S, const double *x, const double *u, const double *params, int pc,
                const double *xn) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(x && u && xn, "NULL array");
    return NTM_OK;
}

int check_getwlc(ntm_handle *h, int layout, int S, int N, const double *bounds, const double *Gamma, const double *Phi,
                 const double *Lambda, const double *W, const double *L, const double *c) {
    TRY(check_common(h, layout, S));
    if (S == 0) return NTM_OK;
    REQUIRE(N >= 1 && N <= NTM_MAX_HORIZON, "N out of range [1, NTM_MAX_HORIZON]");
    REQUIRE(bounds && Gamma && Phi && Lambda && W && L && c, "NULL array");
    return NTM_OK;
}

// S == 0 passes here and still reduces (to empty statistics)
int check_mc_stats(ntm_handle *h, int layout, int S, int k_sim, const double *xk, const double *uk, const double *params,
                   int pc, const double *bounds, const double *out) {
    TRY(check_common(h, layout, S));
    REQUIRE(k_sim >= 1, "k_sim must be >= 1");
    REQUIRE(bounds && out, "NULL array");
    if (S == 0) return NTM_OK;
    TRY(check_params(params, pc, S));
    REQUIRE(xk && uk, "NULL array");
    return NTM_OK;
}

// launch_mc_stats with umin / umax read where they live (slots 8 and 9 of the parameter block) in the caller's layout
int mc_stats_launch(ntm_handle *h, int layout, int S, int k_sim, const double *xk, const double *uk, const double *cost,
                    const int *status, const double *params, int pc, const double *bounds, double w_sup, double hist_max,
                    double *out) {
    const double *umin = nullptr, *umax = nullptr;
    int ustride = 0;
    if (S > 0) {
        if (pc == 1) { umin = params + 8; umax = params + 9; ustride = 0; }
        else if (layout == NTM_LAYOUT_MATLAB) { umin = params + 8; umax = params + 9; ustride = NTM_NPARAM; }
        else { umin = params + 8 * (size_t)S; umax = params + 9 * (size_t)S; ustride = 1; }
    }
    CU(ntm::launch_mc_stats(h->stream, h->props, layout, S, k_sim, xk, uk, cost, status, umin, umax, ustride, bounds, w_sup,
                            hist_max, out, &h->launches));
    return NTM_OK;
}

// Times `launch` (after a warm-up of an eighth of its iterations) with events on the handle's stream; `flops` per
// iteration and SM.
int time_peak(ntm_handle *h, int iters, cudaError_t (*launch)(cudaStream_t, const ntm::DeviceProps &, int, double *, long long *),
              double flops, double *tflops, double *ms_out) {
    REQUIRE(h != nullptr, "handle is NULL");
    REQUIRE(iters > 0, "iters must be > 0");
    CU(cudaSetDevice(h->device));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    double *out = reinterpret_cast<double *>(h->counter) + 8;
    CU(launch(h->stream, h->props, iters / 8 + 1, out, &h->launches));   // warm-up
    CU(cudaEventRecord(e0, h->stream));
    CU(launch(h->stream, h->props, iters, out, &h->launches));
    CU(cudaEventRecord(e1, h->stream));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (tflops) *tflops = flops * (double)iters * (double)h->props.sm_count / (ms * 1e-3) / 1e12;
    if (ms_out) *ms_out = ms;
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
    TRY(check_rho(h, layout, S, x, params, pc, rho1, rho2, rho3));
    if (S == 0) return NTM_OK;
    CU(ntm::launch_rho(h->stream, layout, profile, S, x, params, pc, rho1, rho2, rho3, &h->launches));
    return NTM_OK;
}

int ntm_rho(ntm_handle *h, int layout, int profile, int S, const double *x, const double *params, int pc,
            double *rho1, double *rho2, double *rho3) {
    TRY(check_rho(h, layout, S, x, params, pc, rho1, rho2, rho3));
    if (S == 0) return NTM_OK;
    const size_t s = (size_t)S;
    double *dx, *dp, *d1, *d2, *d3;
    TRY(Arena(h).reserve([&](Arena &A) {
        dx = A.take<double>(2 * s); dp = A.take<double>((size_t)pc * NTM_NPARAM);
        d1 = A.take<double>(s); d2 = A.take<double>(s); d3 = A.take<double>(s);
    }));
    TRY(h2d(h, dx, x, 2 * s)); TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    CU(ntm::launch_rho(h->stream, layout, profile, S, dx, dp, pc, d1, d2, d3, &h->launches));
    TRY(d2h(h, rho1, d1, s)); TRY(d2h(h, rho2, d2, s)); TRY(d2h(h, rho3, d3, s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ A, B
int ntm_lpv_AB_dev(ntm_handle *h, int layout, int S, const double *rho1, const double *rho2, const double *rho3,
                   const double *params, int pc, double *Aout, double *Bout) {
    TRY(check_lpv(h, layout, S, rho1, rho2, rho3, params, pc, Aout, Bout));
    if (S == 0) return NTM_OK;
    CU(ntm::launch_lpv(h->stream, layout, S, rho1, rho2, rho3, params, pc, Aout, Bout, &h->launches));
    return NTM_OK;
}

int ntm_lpv_AB(ntm_handle *h, int layout, int S, const double *rho1, const double *rho2, const double *rho3,
               const double *params, int pc, double *Aout, double *Bout) {
    TRY(check_lpv(h, layout, S, rho1, rho2, rho3, params, pc, Aout, Bout));
    if (S == 0) return NTM_OK;
    const size_t s = (size_t)S;
    double *d1, *d2, *d3, *dp, *dA, *dB;
    TRY(Arena(h).reserve([&](Arena &A) {
        d1 = A.take<double>(s); d2 = A.take<double>(s); d3 = A.take<double>(s);
        dp = A.take<double>((size_t)pc * NTM_NPARAM); dA = A.take<double>(4 * s); dB = A.take<double>(2 * s);
    }));
    TRY(h2d(h, d1, rho1, s)); TRY(h2d(h, d2, rho2, s)); TRY(h2d(h, d3, rho3, s));
    TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    CU(ntm::launch_lpv(h->stream, layout, S, d1, d2, d3, dp, pc, dA, dB, &h->launches));
    TRY(d2h(h, Aout, dA, 4 * s)); TRY(d2h(h, Bout, dB, 2 * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ condense
int ntm_condense_dev(ntm_handle *h, int layout, int profile, int S, int N, const double *R1, const double *R2,
                     const double *R3, const double *params, int pc, double *Phi, double *Gamma, double *Lambda) {
    TRY(check_condense(h, layout, S, N, R1, R2, R3, params, pc, Phi, Gamma, Lambda));
    if (S == 0) return NTM_OK;
    CU(ntm::launch_condense(h->stream, h->props, layout, profile, S, N, R1, R2, R3, params, pc, Phi, Gamma, Lambda,
                            &h->launches));
    return NTM_OK;
}

int ntm_condense(ntm_handle *h, int layout, int profile, int S, int N, const double *R1, const double *R2,
                 const double *R3, const double *params, int pc, double *Phi, double *Gamma, double *Lambda) {
    TRY(check_condense(h, layout, S, N, R1, R2, R3, params, pc, Phi, Gamma, Lambda));
    if (S == 0) return NTM_OK;
    const size_t s = (size_t)S, n = (size_t)N;
    double *d1, *d2, *d3, *dp, *dPhi, *dGam, *dLam;
    TRY(Arena(h).reserve([&](Arena &A) {
        d1 = A.take<double>(n * s); d2 = A.take<double>(n * s); d3 = A.take<double>(n * s);
        dp = A.take<double>((size_t)pc * NTM_NPARAM);
        dPhi = A.take<double>(4 * n * s); dGam = A.take<double>(2 * n * n * s); dLam = A.take<double>(2 * n * s);
    }));
    TRY(h2d(h, d1, R1, n * s)); TRY(h2d(h, d2, R2, n * s)); TRY(h2d(h, d3, R3, n * s));
    TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    CU(ntm::launch_condense(h->stream, h->props, layout, profile, S, N, d1, d2, d3, dp, pc, dPhi, dGam, dLam,
                            &h->launches));
    TRY(d2h(h, Phi, dPhi, 4 * n * s)); TRY(d2h(h, Gamma, dGam, 2 * n * n * s)); TRY(d2h(h, Lambda, dLam, 2 * n * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ G, F
int ntm_hessian_grad_dev(ntm_handle *h, int layout, int S, int N, const double *Phi, const double *Gamma,
                         const double *Lambda, const double *x, const double *params, int pc, double *G, double *F) {
    TRY(check_hessian_grad(h, layout, S, N, Phi, Gamma, Lambda, x, params, pc, G, F));
    if (S == 0) return NTM_OK;
    CU(ntm::launch_hessian_grad(h->stream, h->props, layout, S, N, Phi, Gamma, Lambda, x, params, pc, G, F,
                                &h->launches));
    return NTM_OK;
}

int ntm_hessian_grad(ntm_handle *h, int layout, int S, int N, const double *Phi, const double *Gamma,
                     const double *Lambda, const double *x, const double *params, int pc, double *G, double *F) {
    TRY(check_hessian_grad(h, layout, S, N, Phi, Gamma, Lambda, x, params, pc, G, F));
    if (S == 0) return NTM_OK;
    const size_t s = (size_t)S, n = (size_t)N;
    double *dPhi, *dGam, *dLam, *dx, *dp, *dG, *dF;
    TRY(Arena(h).reserve([&](Arena &A) {
        dPhi = A.take<double>(4 * n * s); dGam = A.take<double>(2 * n * n * s); dLam = A.take<double>(2 * n * s);
        dx = A.take<double>(2 * s); dp = A.take<double>((size_t)pc * NTM_NPARAM);
        dG = A.take<double>(n * n * s); dF = A.take<double>(n * s);
    }));
    TRY(h2d(h, dPhi, Phi, 4 * n * s)); TRY(h2d(h, dGam, Gamma, 2 * n * n * s)); TRY(h2d(h, dLam, Lambda, 2 * n * s));
    TRY(h2d(h, dx, x, 2 * s)); TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    CU(ntm::launch_hessian_grad(h->stream, h->props, layout, S, N, dPhi, dGam, dLam, dx, dp, pc, dG, dF, &h->launches));
    TRY(d2h(h, G, dG, n * n * s)); TRY(d2h(h, F, dF, n * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ box QP
int ntm_qp_box_dev(ntm_handle *h, int layout, int S, int N, const double *G, const double *F, const double *lb,
                   const double *ub, int bc, double *U, int *iters, int *status) {
    TRY(check_qp_box(h, layout, S, N, G, F, lb, ub, bc, U));
    if (S == 0) return NTM_OK;
    TRY(grow(h, h->hscratch, h->hscratch_bytes, ntm::hscratch_bytes(h->props, N)));
    CU(ntm::launch_qp_box(h->stream, h->props, layout, S, N, G, F, lb, ub, bc, U, iters, status, h->counter,
                          h->hscratch, &h->launches));
    return NTM_OK;
}

int ntm_qp_box(ntm_handle *h, int layout, int S, int N, const double *G, const double *F, const double *lb,
               const double *ub, int bc, double *U, int *iters, int *status) {
    TRY(check_qp_box(h, layout, S, N, G, F, lb, ub, bc, U));
    if (S == 0) return NTM_OK;
    const size_t s = (size_t)S, n = (size_t)N, b = (size_t)bc;
    double *dG, *dF, *dlb, *dub, *dU;
    int *dit, *dst;
    TRY(Arena(h).reserve([&](Arena &A) {
        dG = A.take<double>(n * n * s); dF = A.take<double>(n * s); dlb = A.take<double>(n * b);
        dub = A.take<double>(n * b); dU = A.take<double>(n * s);
        dit = A.take<int>(s); dst = A.take<int>(s);
    }));
    TRY(h2d(h, dG, G, n * n * s)); TRY(h2d(h, dF, F, n * s)); TRY(h2d(h, dlb, lb, n * b)); TRY(h2d(h, dub, ub, n * b));
    TRY(grow(h, h->hscratch, h->hscratch_bytes, ntm::hscratch_bytes(h->props, N)));
    CU(ntm::launch_qp_box(h->stream, h->props, layout, S, N, dG, dF, dlb, dub, bc, dU, dit, dst, h->counter,
                          h->hscratch, &h->launches));
    TRY(d2h(h, U, dU, n * s)); TRY(d2h(h, iters, dit, s)); TRY(d2h(h, status, dst, s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ general-inequality QP
int ntm_qp_ineq_dev(ntm_handle *h, int layout, int S, int N, int M, const double *G, const double *F,
                    const double *lb, const double *ub, int bc, const double *Lg, const double *bg, double *U,
                    int *iters, int *status) {
    TRY(check_qp_ineq(h, layout, S, N, M, G, F, lb, ub, bc, Lg, bg, U));
    if (M == 0) return ntm_qp_box_dev(h, layout, S, N, G, F, lb, ub, bc, U, iters, status);
    if (S == 0) return NTM_OK;
    CU(ntm::launch_qp_ineq(h->stream, h->props, layout, S, N, M, G, F, lb, ub, bc, Lg, bg, U, iters, status, h->counter,
                           &h->launches));
    return NTM_OK;
}

int ntm_qp_ineq(ntm_handle *h, int layout, int S, int N, int M, const double *G, const double *F, const double *lb,
                const double *ub, int bc, const double *Lg, const double *bg, double *U, int *iters, int *status) {
    TRY(check_qp_ineq(h, layout, S, N, M, G, F, lb, ub, bc, Lg, bg, U));
    if (M == 0) return ntm_qp_box(h, layout, S, N, G, F, lb, ub, bc, U, iters, status);
    if (S == 0) return NTM_OK;
    const size_t s = (size_t)S, n = (size_t)N, b = (size_t)bc, m = (size_t)M;
    double *dG, *dF, *dlb, *dub, *dU, *dL, *dbg;
    int *dit, *dst;
    TRY(Arena(h).reserve([&](Arena &A) {
        dG = A.take<double>(n * n * s); dF = A.take<double>(n * s); dlb = A.take<double>(n * b);
        dub = A.take<double>(n * b); dU = A.take<double>(n * s);
        dL = A.take<double>(m * n * s); dbg = A.take<double>(m * s);
        dit = A.take<int>(s); dst = A.take<int>(s);
    }));
    TRY(h2d(h, dG, G, n * n * s)); TRY(h2d(h, dF, F, n * s)); TRY(h2d(h, dlb, lb, n * b)); TRY(h2d(h, dub, ub, n * b));
    TRY(h2d(h, dL, Lg, m * n * s)); TRY(h2d(h, dbg, bg, m * s));
    CU(ntm::launch_qp_ineq(h->stream, h->props, layout, S, N, M, dG, dF, dlb, dub, bc, dL, dbg, dU, dit, dst, h->counter,
                           &h->launches));
    TRY(d2h(h, U, dU, n * s)); TRY(d2h(h, iters, dit, s)); TRY(d2h(h, status, dst, s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ plant
int ntm_plant_step_dev(ntm_handle *h, int layout, int profile, int S, const double *x, const double *u,
                       const double *params, int pc, double *xn) {
    TRY(check_plant(h, layout, S, x, u, params, pc, xn));
    if (S == 0) return NTM_OK;
    CU(ntm::launch_plant(h->stream, layout, profile, S, x, u, params, pc, xn, &h->launches));
    return NTM_OK;
}

int ntm_plant_step(ntm_handle *h, int layout, int profile, int S, const double *x, const double *u,
                   const double *params, int pc, double *xn) {
    TRY(check_plant(h, layout, S, x, u, params, pc, xn));
    if (S == 0) return NTM_OK;
    const size_t s = (size_t)S;
    double *dx, *du, *dp, *dn;
    TRY(Arena(h).reserve([&](Arena &A) {
        dx = A.take<double>(2 * s); du = A.take<double>(s); dp = A.take<double>((size_t)pc * NTM_NPARAM);
        dn = A.take<double>(2 * s);
    }));
    TRY(h2d(h, dx, x, 2 * s)); TRY(h2d(h, du, u, s)); TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    CU(ntm::launch_plant(h->stream, layout, profile, S, dx, du, dp, pc, dn, &h->launches));
    TRY(d2h(h, xn, dn, 2 * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ closed loop
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
    const int per = (S + n_devices - 1) / n_devices;       // SURVEY 8(e): rank g owns [g*per, min(S, (g+1)*per))
    const int shards = (S + per - 1) / per;
    std::vector<ntm_handle *> hs((size_t)shards, nullptr);
    std::vector<ntm::LoopArgs> as((size_t)shards);
    for (int g = 0; g < shards; ++g) {                     // every shard is checked before any is copied
        TRY(pool_handle(dev[g], &hs[g]));
        as[g] = loop_args(layout, profile, std::min(per, S - g * per), N, k_sim, i_sim, eps, x0, params, pc, state_rows,
                          xk, uk, Uk, cost, inner_iters, qp_iters, status);
        TRY(check_fused(hs[g], as[g], xbounds, S));
    }
    std::vector<int> rc((size_t)shards, NTM_OK);
    std::vector<std::string> msg((size_t)shards);
    auto shard = [&](int g) -> int {
        CU(cudaSetDevice(hs[g]->device));                  // the current device is per host thread
        return fused_host(hs[g], as[g], S, g * per);
    };
    auto run = [&](int g) {
        rc[g] = shard(g);
        if (rc[g] != NTM_OK) msg[g] = g_err;               // g_err is thread-local: carry the text to the caller's thread
    };
    std::vector<std::thread> th;
    for (int g = 1; g < shards; ++g) th.emplace_back(run, g);
    run(0);
    for (auto &t : th) t.join();
    for (int g = 0; g < shards; ++g)
        if (rc[g] != NTM_OK) return fail(rc[g], "device %d: %s", dev[g], msg[g].c_str());
    return NTM_OK;
}

// Packed-record variant of the resident entry (scenario-slowest inputs): ONE array `rec` of NTM_REC_DOUBLES(k_sim)
// doubles per scenario = [xk (2(k_sim+1)) | uk (k_sim) | cost | status] -- the block a multi-GPU caller gathers with a
// single collective (SURVEY 8e: "one ncclAllGather of per-scenario outputs").
int ntm_mpc_closed_loop_rec_dev(ntm_handle *h, int profile, int S, int N, int k_sim, int i_sim, double eps,
                                const double *x0, const double *params, int pc, int state_rows, const double *xbounds,
                                double *rec, int *inner_iters, int *qp_iters) {
    ntm::LoopArgs a = loop_args(NTM_LAYOUT_MATLAB, profile, S, N, k_sim, i_sim, eps, x0, params, pc, state_rows, rec,
                                nullptr, nullptr, nullptr, inner_iters, qp_iters, nullptr);
    a.rec_ld = NTM_REC_DOUBLES(k_sim);
    if (rec) { a.uk = rec + 2 * (k_sim + 1); a.cost = rec + 3 * k_sim + 2; a.rec_status = rec + 3 * k_sim + 3; }
    return fused_dev_call(h, a, xbounds);
}

int ntm_mpc_closed_loop_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                            const double *x0, const double *params, int pc, double *xk, double *uk, double *Uk,
                            double *cost, int *inner_iters, int *qp_iters, int *status) {
    return fused_dev_call(h, loop_args(layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, NTM_STATE_ROWS_OFF, xk,
                                       uk, Uk, cost, inner_iters, qp_iters, status), nullptr);
}

int ntm_mpc_closed_loop(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                        const double *x0, const double *params, int pc, double *xk, double *uk, double *Uk,
                        double *cost, int *inner_iters, int *qp_iters, int *status) {
    return fused_host_call(h, loop_args(layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, NTM_STATE_ROWS_OFF, xk,
                                        uk, Uk, cost, inner_iters, qp_iters, status), nullptr);
}

int ntm_mpc_closed_loop_sc_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                               const double *x0, const double *params, int pc, int state_rows, const double *xbounds,
                               double *xk, double *uk, double *Uk, double *cost, int *inner_iters, int *qp_iters,
                               int *status) {
    return fused_dev_call(h, loop_args(layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, state_rows, xk, uk, Uk,
                                       cost, inner_iters, qp_iters, status), xbounds);
}

int ntm_mpc_closed_loop_sc(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim, double eps,
                           const double *x0, const double *params, int pc, int state_rows, const double *xbounds,
                           double *xk, double *uk, double *Uk, double *cost, int *inner_iters, int *qp_iters,
                           int *status) {
    return fused_host_call(h, loop_args(layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, state_rows, xk, uk, Uk,
                                        cost, inner_iters, qp_iters, status), xbounds);
}

// ------------------------------------------------------------------------------------------------ controller step
int ntm_mpc_step_dev(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                     const double *params, int pc, double *state, double *u, double *U, int *inner_iters, int *qp_iters,
                     int *status) {
    return fused_dev_call(h, step_args(layout, profile, S, N, i_sim, eps, x, params, pc, NTM_STATE_ROWS_OFF, state, u, U,
                                       inner_iters, qp_iters, status), nullptr);
}

int ntm_mpc_step(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                 const double *params, int pc, double *state, double *u, double *U, int *inner_iters, int *qp_iters,
                 int *status) {
    return fused_host_call(h, step_args(layout, profile, S, N, i_sim, eps, x, params, pc, NTM_STATE_ROWS_OFF, state, u, U,
                                        inner_iters, qp_iters, status), nullptr);
}

int ntm_mpc_step_sc_dev(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                        const double *params, int pc, int state_rows, const double *xbounds, double *state, double *u,
                        double *U, int *inner_iters, int *qp_iters, int *status) {
    return fused_dev_call(h, step_args(layout, profile, S, N, i_sim, eps, x, params, pc, state_rows, state, u, U,
                                       inner_iters, qp_iters, status), xbounds);
}

int ntm_mpc_step_sc(ntm_handle *h, int layout, int profile, int S, int N, int i_sim, double eps, const double *x,
                    const double *params, int pc, int state_rows, const double *xbounds, double *state, double *u,
                    double *U, int *inner_iters, int *qp_iters, int *status) {
    return fused_host_call(h, step_args(layout, profile, S, N, i_sim, eps, x, params, pc, state_rows, state, u, U,
                                        inner_iters, qp_iters, status), xbounds);
}

// ------------------------------------------------------------------------------------------------ perturbed plant
int ntm_mpc_closed_loop_perturbed_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim,
                                      double eps, const double *x0, const double *params, int pc,
                                      const double *plant_params, int ppc, int plant_profile, const double *w,
                                      const double *v, double *xk, double *uk, double *Uk, double *cost,
                                      int *inner_iters, int *qp_iters, int *status) {
    return fused_dev_call(h, perturbed_args(layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, NTM_STATE_ROWS_OFF,
                                            plant_params, ppc, plant_profile, w, v, xk, uk, Uk, cost, inner_iters,
                                            qp_iters, status), nullptr);
}

int ntm_mpc_closed_loop_perturbed(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim,
                                  double eps, const double *x0, const double *params, int pc,
                                  const double *plant_params, int ppc, int plant_profile, const double *w,
                                  const double *v, double *xk, double *uk, double *Uk, double *cost, int *inner_iters,
                                  int *qp_iters, int *status) {
    return fused_host_call(h, perturbed_args(layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, NTM_STATE_ROWS_OFF,
                                             plant_params, ppc, plant_profile, w, v, xk, uk, Uk, cost, inner_iters,
                                             qp_iters, status), nullptr);
}

int ntm_mpc_closed_loop_perturbed_sc_dev(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim,
                                         double eps, const double *x0, const double *params, int pc, int state_rows,
                                         const double *xbounds, const double *plant_params, int ppc, int plant_profile,
                                         const double *w, const double *v, double *xk, double *uk, double *Uk,
                                         double *cost, int *inner_iters, int *qp_iters, int *status) {
    return fused_dev_call(h, perturbed_args(layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, state_rows,
                                            plant_params, ppc, plant_profile, w, v, xk, uk, Uk, cost, inner_iters,
                                            qp_iters, status), xbounds);
}

int ntm_mpc_closed_loop_perturbed_sc(ntm_handle *h, int layout, int profile, int S, int N, int k_sim, int i_sim,
                                     double eps, const double *x0, const double *params, int pc, int state_rows,
                                     const double *xbounds, const double *plant_params, int ppc, int plant_profile,
                                     const double *w, const double *v, double *xk, double *uk, double *Uk, double *cost,
                                     int *inner_iters, int *qp_iters, int *status) {
    return fused_host_call(h, perturbed_args(layout, profile, S, N, k_sim, i_sim, eps, x0, params, pc, state_rows,
                                             plant_params, ppc, plant_profile, w, v, xk, uk, Uk, cost, inner_iters,
                                             qp_iters, status), xbounds);
}

// ------------------------------------------------------------------------------------------------ getWLc
int ntm_getWLc_dev(ntm_handle *h, int layout, int S, int N, const double *bounds, const double *Gamma, const double *Phi,
                   const double *Lambda, double *W, double *L, double *c) {
    TRY(check_getwlc(h, layout, S, N, bounds, Gamma, Phi, Lambda, W, L, c));
    if (S == 0) return NTM_OK;
    CU(ntm::launch_getwlc(h->stream, h->props, layout, S, N, bounds, Gamma, Phi, Lambda, W, L, c, &h->launches));
    return NTM_OK;
}

int ntm_getWLc(ntm_handle *h, int layout, int S, int N, const double *bounds, const double *Gamma, const double *Phi,
               const double *Lambda, double *W, double *L, double *c) {
    TRY(check_getwlc(h, layout, S, N, bounds, Gamma, Phi, Lambda, W, L, c));
    if (S == 0) return NTM_OK;
    const size_t s = (size_t)S, n = (size_t)N, r = 6 * n + 4;
    double *dGam, *dPhi, *dLam, *dW, *dL, *dc;
    TRY(Arena(h).reserve([&](Arena &A) {
        dGam = A.take<double>(2 * n * n * s); dPhi = A.take<double>(4 * n * s); dLam = A.take<double>(2 * n * s);
        dW = A.take<double>(r * 2 * s); dL = A.take<double>(r * n * s); dc = A.take<double>(r * s);
    }));
    TRY(h2d(h, dGam, Gamma, 2 * n * n * s)); TRY(h2d(h, dPhi, Phi, 4 * n * s)); TRY(h2d(h, dLam, Lambda, 2 * n * s));
    CU(ntm::launch_getwlc(h->stream, h->props, layout, S, N, bounds, dGam, dPhi, dLam, dW, dL, dc, &h->launches));
    TRY(d2h(h, W, dW, r * 2 * s)); TRY(d2h(h, L, dL, r * n * s)); TRY(d2h(h, c, dc, r * s));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ Monte-Carlo statistics
int ntm_mc_stats_dev(ntm_handle *h, int layout, int S, int k_sim, const double *xk, const double *uk,
                     const double *cost, const int *status, const double *params, int pc, const double *bounds,
                     double w_sup, double hist_max, double *out) {
    TRY(check_mc_stats(h, layout, S, k_sim, xk, uk, params, pc, bounds, out));
    return mc_stats_launch(h, layout, S, k_sim, xk, uk, cost, status, params, pc, bounds, w_sup, hist_max, out);
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
    TRY(check_mc_stats(h, layout, S, k_sim, xk, uk, params, pc, bounds, out));
    const size_t s = (size_t)S, k = (size_t)k_sim;
    double *dx, *du, *dc, *dp, *dout;
    int *dst;
    TRY(Arena(h).reserve([&](Arena &A) {
        dx = A.take<double>(2 * (k + 1) * s + 1); du = A.take<double>(k * s + 1); dc = A.take<double>(s + 1);
        dst = A.take<int>(s + 2);
        dp = A.take<double>((size_t)(S > 0 ? pc : 0) * NTM_NPARAM + 1); dout = A.take<double>(NTM_MC_NSTAT);
    }));
    if (S > 0) {
        TRY(h2d(h, dx, xk, 2 * (k + 1) * s)); TRY(h2d(h, du, uk, k * s));
        if (cost) TRY(h2d(h, dc, cost, s));
        if (status) TRY(h2d(h, dst, status, s));
        TRY(h2d(h, dp, params, (size_t)pc * NTM_NPARAM));
    }
    TRY(mc_stats_launch(h, layout, S, k_sim, dx, du, cost ? dc : nullptr, status ? dst : nullptr, dp, pc, bounds, w_sup,
                        hist_max, dout));
    TRY(d2h(h, out, dout, (size_t)NTM_MC_NSTAT));
    CU(cudaStreamSynchronize(h->stream));
    return NTM_OK;
}

// ------------------------------------------------------------------------------------------------ fp64 peak
int ntm_fp64_peak(ntm_handle *h, int iters, double *tflops_dfma, double *ms_out) {
    // 64 DFMA (2 flops each) per thread and iteration, 256 threads per CTA, 8 CTAs per SM
    return time_peak(h, iters, ntm::launch_fp64_peak, 2.0 * 64.0 * 256.0 * 8.0, tflops_dfma, ms_out);
}

int ntm_dmma_peak(ntm_handle *h, int iters, double *tflops_dmma, double *ms_out) {
    // 8 DMMA.8x8x4 per warp and iteration, 2*8*8*4 flops each, 8 warps per CTA, 8 CTAs per SM
    return time_peak(h, iters, ntm::launch_dmma_peak, 512.0 * 8.0 * 8.0 * 8.0, tflops_dmma, ms_out);
}

}  // extern "C"
