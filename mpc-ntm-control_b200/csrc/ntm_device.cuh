// ntm_device.cuh -- device-side building blocks of the LPV-MPC hot path (sm_100a, fp64).
//
// One *group* of GW warps owns one scenario; thread j of the group owns horizon index j (MATLAB
// index j+1): row j of the Hessian, input U(j+1), stage j of the rollout.  GW = 1 (N <= 32: pure
// warp-synchronous code, shuffles, several scenarios per CTA) or GW = 2/4 (N <= 64/128: one CTA per
// scenario).  Everything a scenario needs between two HBM touches lives in shared memory / registers.
//
// Reference lines implemented here (relative to the upstream tree):
//   rho1.m:2 | rhos.m:18, rho2.m:2, rho3.m:2-3                    -> schedule()
//   A.m:2, B.m:2                                                   -> schedule() (hoisted coefficients)
//   Rho_to_PhiGammaLambda.m:17-52 + NTM_MPC_Sim.m:72-73,120-121    -> build_GF_toeplitz / build_GF_dense
//   NTM_MPC_Sim.m:97 (quadprog, input-box rows only)               -> qp_solve (primal active set, warm started)
//   NTM_MPC_Sim.m:110-117                                          -> rollout in run_scenario (ntm_kernels.cu)
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include "../../include/ntm_mpc.h"

namespace ntm {

struct Params {
    double c_a11, c_a21, a22, c_b, C1, C2, wmarg2, w_dep, umin, umax, r1, r2, q11, q12, q22;
    double inv_wdep;   // 1 / w_dep, filled by load_params_shared (slot 15 of the block is reserved, so sizeof matches)
};

// element e of scenario s in an array of E doubles per scenario
__device__ __forceinline__ size_t elem(int layout, int S, int E, int s, int e) {
    return layout == NTM_LAYOUT_SOA ? (size_t)e * (size_t)S + (size_t)s : (size_t)s * (size_t)E + (size_t)e;
}

__device__ __forceinline__ Params load_params(const double *__restrict__ p, int layout, int count, int s) {
    const int ss = (count == 1) ? 0 : s;
    const int SS = (count == 1) ? 1 : count;
    Params P;
    P.c_a11 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 0));
    P.c_a21 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 1));
    P.a22 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 2));
    P.c_b = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 3));
    P.C1 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 4));
    P.C2 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 5));
    P.wmarg2 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 6));
    P.w_dep = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 7));
    P.umin = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 8));
    P.umax = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 9));
    P.r1 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 10));
    P.r2 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 11));
    P.q11 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 12));
    P.q12 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 13));
    P.q22 = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 14));
    P.inv_wdep = 1.0 / P.w_dep;
    return P;
}

// cooperative variant: thread p < 15 of the group fetches parameter p into shared memory
__device__ __forceinline__ void load_params_shared(Params *dst, const double *__restrict__ p, int layout, int count, int s,
                                                   int j) {
    const int ss = (count == 1) ? 0 : s;
    const int SS = (count == 1) ? 1 : count;
    if (j < 15) reinterpret_cast<double *>(dst)[j] = __ldg(p + elem(layout, SS, NTM_NPARAM, ss, j));
    if (j == 15) dst->inv_wdep = 1.0 / __ldg(p + elem(layout, SS, NTM_NPARAM, ss, 7));
}

// rho1.m:2 (rhos.m:18 with NTM_PROFILE_RHO1_SQ), rho2.m:2, rho3.m:2-3.  IEEE divisions, no fast-math:
// omega = 0 and the pole of rho3 propagate Inf/NaN exactly like the interpreter would.
// FAST_WS (fused kernel only): wstar = w * (1/w_dep) with the reciprocal hoisted per scenario -- one division less
// per stage and inner iteration, <= 1 ulp away from rho3.m:2; the API kernels keep the division.
template <bool FAST_WS = false>
__device__ __forceinline__ void rho_of(const Params &P, int flags, double w, double om, double &r1, double &r2,
                                       double &r3) {
    r1 = (flags & NTM_PROFILE_RHO1_SQ) ? 1.0 / (w * w + P.wmarg2) : 1.0 / (w + P.wmarg2);
    r2 = (w * w) / om;
    const double ws = FAST_WS ? w * P.inv_wdep : w / P.w_dep;
    r3 = (0.25 + 0.24 * ws) / (1.0 + 1.5 * ws + 0.43 * (ws * ws) + 0.64 * (ws * ws * ws));
}

// A.m:2 / B.m:2 with hoisted coefficients: a11 = c_a11*rho1 + 1, a21 = c_a21*rho2, b = c_b*rho3.
__device__ __forceinline__ void lpv_of(const Params &P, double r1, double r2, double r3, double &a11, double &a21,
                                       double &b) {
    a11 = P.c_a11 * r1 + 1.0;
    a21 = P.c_a21 * r2;
    b = P.c_b * r3;
}

template <bool FAST_WS = false>
__device__ __forceinline__ void schedule(const Params &P, int flags, double w, double om, double &a11, double &a21,
                                         double &b) {
    double r1, r2, r3;
    rho_of<FAST_WS>(P, flags, w, om, r1, r2, r3);
    lpv_of(P, r1, r2, r3, a11, a21, b);
}

// ------------------------------------------------------------------------------------------------
// Group primitives.  GW == 1: warp shuffles / ballots only.  GW > 1: the CTA is the group.
// ------------------------------------------------------------------------------------------------
template <int GW>
struct Group {
    static constexpr int T = 32 * GW;

    __device__ static __forceinline__ void sync() {
        if constexpr (GW == 1) __syncwarp();
        else __syncthreads();
    }

    // deterministic sum over the group (fixed butterfly order)
    __device__ static __forceinline__ double sum(double v, double *red) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if constexpr (GW > 1) {
            __syncthreads();
            if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
            __syncthreads();
            v = red[0];
#pragma unroll
            for (int i = 1; i < GW; ++i) v += red[i];
        }
        return v;
    }

    __device__ static __forceinline__ int count(bool p, int *ired) {
        int c = __popc(__ballot_sync(0xffffffffu, p));
        if constexpr (GW > 1) {
            __syncthreads();
            if ((threadIdx.x & 31) == 0) ired[threadIdx.x >> 5] = c;
            __syncthreads();
            c = ired[0];
#pragma unroll
            for (int i = 1; i < GW; ++i) c += ired[i];
        }
        return c;
    }

    // exclusive prefix count of p over the group (thread order) and the total
    __device__ static __forceinline__ int prefix(bool p, int *ired, int &total) {
        const unsigned b = __ballot_sync(0xffffffffu, p);
        const unsigned lane = threadIdx.x & 31;
        int pre = __popc(b & ((1u << lane) - 1u));
        int tot = __popc(b);
        if constexpr (GW > 1) {
            const int w = threadIdx.x >> 5;
            __syncthreads();
            if (lane == 0) ired[w] = tot;
            __syncthreads();
            tot = 0;
#pragma unroll
            for (int i = 0; i < GW; ++i) {
                const int c = ired[i];
                if (i < w) pre += c;
                tot += c;
            }
        }
        total = tot;
        return pre;
    }

    // largest thread index j with p true, -1 if none
    __device__ static __forceinline__ int maxidx(bool p, int j, int *ired) {
        const unsigned b = __ballot_sync(0xffffffffu, p);
        int m = b ? (int)(j - (int)(threadIdx.x & 31)) + (31 - __clz(b)) : -1;
        if constexpr (GW > 1) {
            __syncthreads();
            if ((threadIdx.x & 31) == 0) ired[threadIdx.x >> 5] = m;
            __syncthreads();
            m = ired[0];
#pragma unroll
            for (int i = 1; i < GW; ++i) m = max(m, ired[i]);
        }
        return m;
    }

    // minimum of v over the group and the lowest thread index attaining it (NaNs are ignored; index -1
    // when every value is NaN)
    __device__ static __forceinline__ double argmin(double v, int j, double *red, int *ired, int &jmin) {
        double m = v;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, o));
        const unsigned b = __ballot_sync(0xffffffffu, v == m);
        int idx = b ? (int)(j - (int)(threadIdx.x & 31)) + (__ffs(b) - 1) : -1;
        if constexpr (GW > 1) {
            __syncthreads();
            if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = m; ired[threadIdx.x >> 5] = idx; }
            __syncthreads();
            m = red[0]; idx = ired[0];
#pragma unroll
            for (int i = 1; i < GW; ++i) {
                const double mi = red[i];
                const int ii = ired[i];
                if (ii >= 0 && (idx < 0 || mi < m)) { m = mi; idx = ii; }
            }
        }
        jmin = idx;
        return m;
    }

    // value held by thread 0 of the group
    __device__ static __forceinline__ double bcast0(double v, double *red) {
        if constexpr (GW == 1) return __shfl_sync(0xffffffffu, v, 0);
        else {
            __syncthreads();
            if (threadIdx.x == 0) red[0] = v;
            __syncthreads();
            return red[0];
        }
    }
    __device__ static __forceinline__ int bcast0(int v, int *ired) {
        if constexpr (GW == 1) return __shfl_sync(0xffffffffu, v, 0);
        else {
            __syncthreads();
            if (threadIdx.x == 0) ired[0] = v;
            __syncthreads();
            return ired[0];
        }
    }
    // value held by thread src of the group
    __device__ static __forceinline__ int bcast_from(int v, int src, int *ired) {
        if constexpr (GW == 1) return __shfl_sync(0xffffffffu, v, src);
        else {
            __syncthreads();
            if ((int)threadIdx.x == src) ired[0] = v;
            __syncthreads();
            return ired[0];
        }
    }
    __device__ static __forceinline__ bool any(bool p, int *ired) { return count(p, ired) > 0; }
    __device__ static __forceinline__ bool all(bool p, int *ired) {
        if constexpr (GW == 1) return __all_sync(0xffffffffu, p) != 0;
        else return count(!p, ired) == 0;
    }
};

// ------------------------------------------------------------------------------------------------
// Per-group shared-memory work area.  16-byte aligned vector arrays first (double2 / 2 x double2
// accesses), then the odd-pitched matrices.
// ------------------------------------------------------------------------------------------------
struct Work {
    double2 *cand;   // [2N] QP start candidates, entry k = {lb_k, ub_k | u(t-2)_k, u(t-1)_k}
    double2 *P12;    // [N]  p_d = first column of A_d...A_1
    double2 *QP12;   // [2N] Q*p_d, zero padded beyond N (dense sweep: row buffer of Q*Gamma(i,:))
    double2 *QE12;   // [2N] Q*(v_i - r), zero padded beyond N
    double *GamS;    // dense Gamma staging for the tensor-core contraction (non-literal Gamma index, N <= 32) or NULL:
                     // column c at GamS[c*ldgam + k], ceil8(N) columns, pitch 4 mod 8 doubles, zero padded
    int ldgam;
    double *G;       // N x ldg, full symmetric
    double *H;       // hcap x (hcap|1) LDL' workspace for free sets of up to hcap variables (shared memory)
    double *Hbig;    // N x ldg slab in global memory for the rare larger free sets (NULL when hcap == N)
    double *a11s, *a21s, *bbs;   // per-stage LPV entries (current rho)
    double *qv;      // b_i*U_i + C1
    double *uv, *sol;            // QP vectors
    double *red;     // 8 doubles of reduction scratch
    Params *prm;     // this scenario's parameter block (kept in shared memory to spare ~30 registers)
    int *idx;        // free-set index list
    int *ired;       // 8 ints of reduction scratch
    int ldg, hcap;
};

__host__ __device__ inline int odd_ld(int N) { return N | 1; }

// bytes (multiple of 16) of one group's work area with an LDL' workspace for free sets of up to hcap variables
__host__ __device__ inline int gam_pitch(int N) {
    int ld = (2 * N + 3) & ~3;
    while ((ld & 7) != 4) ++ld;
    return ld;
}

// dense Gamma on the tensor cores, multi-warp groups: Gamma streams through a chunk buffer of NTM_DCH rows (8 stages),
// column c at GamS[c * NTM_DLD + k]; ceil8(N + 1) columns (column N carries v = Phi x + Lambda - R)
#define NTM_DCH 16
#define NTM_DLD (NTM_DCH + 4)
__host__ __device__ inline size_t gam_doubles(int N, int gam) {
    if (gam == 1) return (size_t)((N + 7) & ~7) * gam_pitch(N);
    if (gam == 2) return (size_t)((N + 1 + 7) & ~7) * NTM_DLD;
    return 0;
}
__host__ __device__ inline size_t work_bytes(int N, int hcap, int gam = 0) {
    const size_t ld = (size_t)odd_ld(N);
    const size_t dbl = 14 * (size_t)N + (size_t)N * ld + (size_t)hcap * odd_ld(hcap) + 6 * (size_t)N + 8 + 16 +
                       gam_doubles(N, gam);
    const size_t ints = (size_t)N + 8;
    size_t b = dbl * 8 + ints * 4;
    return (b + 15) & ~(size_t)15;
}

__device__ inline Work carve(unsigned char *base, int N, int hcap, double *hbig, int gam = 0) {
    Work w;
    const int ld = odd_ld(N);
    double2 *v = reinterpret_cast<double2 *>(base);
    w.cand = v; v += 2 * N; w.P12 = v; v += N; w.QP12 = v; v += 2 * N; w.QE12 = v; v += 2 * N;
    w.GamS = nullptr; w.ldgam = gam_pitch(N);
    if (gam) { w.GamS = reinterpret_cast<double *>(v); v += gam_doubles(N, gam) / 2; if (gam == 2) w.ldgam = NTM_DLD; }
    double *d = reinterpret_cast<double *>(v);
    w.ldg = ld; w.hcap = hcap;
    w.G = d; d += (size_t)N * ld;
    w.H = d; d += (size_t)hcap * odd_ld(hcap);
    w.Hbig = hbig;
    w.a11s = d; d += N; w.a21s = d; d += N; w.bbs = d; d += N;
    w.qv = d; d += N; w.uv = d; d += N; w.sol = d; d += N;
    w.red = d; d += 8;
    w.prm = reinterpret_cast<Params *>(d); d += 16;
    int *ip = reinterpret_cast<int *>(d);
    w.idx = ip; ip += N;
    w.ired = ip;
    return w;
}

// ------------------------------------------------------------------------------------------------
// LDL' factor + solve of the m x m SPD system H*sol = sol (in place), group-cooperative:
// thread a < m owns row a.  Lower triangle holds the running Schur complement, the upper triangle
// receives L'.  Returns true (group-uniform) on a non-positive pivot (numerical breakdown).
// The caller must have synchronised after filling H and sol.
// ------------------------------------------------------------------------------------------------
template <int GW>
__device__ bool ldl_solve(int m, int a, double *__restrict__ H, int ldh, double *__restrict__ sol) {
    using Gp = Group<GW>;
    const bool own = a < m;
    double ya = own ? sol[a] : 0.0;
    double inv_a = 0.0;
    bool bad = false;
    for (int k = 0; k < m; ++k) {
        Gp::sync();
        const double d = H[k * ldh + k];
        const bool ok = d > 0.0;
        bad |= !ok;
        const double inv = ok ? 1.0 / d : 0.0;
        const double yk = sol[k];
        if (a == k) inv_a = inv;
        if constexpr (GW == 1) {
            if (own && a > k) {                              // thread a updates its own row
                const double l = H[a * ldh + k] * inv;
                for (int b = k + 1; b <= a; ++b) H[a * ldh + b] = fma(-l, H[b * ldh + k], H[a * ldh + b]);
                H[k * ldh + a] = l;
                ya = fma(-l, yk, ya);
                sol[a] = ya;
            }
        } else {
            // trailing update spread over the whole CTA: warp w takes rows k+1+w, k+1+w+GW, ... eight at a time (the
            // rows of a batch share the column-k loads and give the shared-memory pipeline independent work to hide
            // its latency: there is only one warp per scheduler here); lanes run along the rows
            const int wid = a >> 5, lane = a & 31;
            constexpr int RB = 8;
            for (int r0 = k + 1 + wid; r0 < m; r0 += RB * GW) {
                double l[RB];
                int rmax = r0;
#pragma unroll
                for (int q = 0; q < RB; ++q) {
                    const int r = r0 + q * GW;
                    l[q] = (r < m) ? H[r * ldh + k] * inv : 0.0;
                    if (r < m) rmax = r;
                }
                for (int b = k + 1 + lane; b <= rmax; b += 32) {
                    const double hb = H[b * ldh + k];
                    double h[RB];
#pragma unroll
                    for (int q = 0; q < RB; ++q) {
                        const int r = r0 + q * GW;
                        h[q] = (r < m && b <= r) ? H[r * ldh + b] : 0.0;
                    }
#pragma unroll
                    for (int q = 0; q < RB; ++q) {
                        const int r = r0 + q * GW;
                        if (r < m && b <= r) H[r * ldh + b] = fma(-l[q], hb, h[q]);
                    }
                }
            }
            if (own && a > k) ya = fma(-(H[a * ldh + k] * inv), yk, ya);
            Gp::sync();                                      // column k is read-only until every row is done
            if (own && a > k) { H[k * ldh + a] = H[a * ldh + k] * inv; sol[a] = ya; }
        }
    }
    Gp::sync();
    double za = ya * inv_a;
    if (own) sol[a] = za;
    for (int k = m - 1; k >= 1; --k) {
        Gp::sync();
        const double xk = sol[k];
        if (a < k) {
            za = fma(-H[a * ldh + k], xk, za);
            sol[a] = za;
        }
    }
    Gp::sync();
    return bad;
}

// ------------------------------------------------------------------------------------------------
// Maintaining the factorisation across active-set iterations.  ldl_solve leaves L' in the strict UPPER triangle
// (U[k][a] = l_ak, a > k: thread a owns column a) and D on the diagonal; the strict lower triangle is scratch.
//   ldl_apply   solve with the stored factor                      (2m barrier steps, no trailing update)
//   ldl_append  a variable joins the free set: new last row of L   (m steps)
//   ldl_delete  the variable at position p leaves: rank-one update of the trailing factor (Gill-Golub-Murray-
//               Saunders C1, alpha = d_p > 0 so it is stable), then rows/columns close up through the scratch half
// An active-set iteration therefore costs O(m) barrier steps of O(1) work per thread instead of an O(m) x O(m)
// refactorisation -- the difference between 35 k and 170 k scenario-steps/s at N = 100.
// ------------------------------------------------------------------------------------------------
template <int GW>
__device__ void ldl_apply(int m, int a, const double *__restrict__ H, int ldh, double *__restrict__ sol) {
    using Gp = Group<GW>;
    const bool own = a < m;
    double ya = own ? sol[a] : 0.0;
    for (int k = 0; k + 1 < m; ++k) {
        Gp::sync();
        const double yk = sol[k];
        if (own && a > k) { ya = fma(-H[k * ldh + a], yk, ya); sol[a] = ya; }
    }
    Gp::sync();
    double za = 0.0;
    if (own) { const double d = H[a * ldh + a]; za = (d > 0.0) ? ya / d : 0.0; sol[a] = za; }
    for (int k = m - 1; k >= 1; --k) {
        Gp::sync();
        const double xk = sol[k];
        if (a < k) { za = fma(-H[a * ldh + k], xk, za); sol[a] = za; }
    }
    Gp::sync();
}

// ga = Hessian(idx[a], v) for a < m (this thread's entry of the new column), gvv = Hessian(v, v); wv: scratch vector.
// Returns true when the new pivot is not positive (numerical breakdown).
template <int GW>
__device__ bool ldl_append(int m, int a, double *__restrict__ H, int ldh, double ga, double gvv, double *__restrict__ wv,
                           double *red) {
    using Gp = Group<GW>;
    const bool own = a < m;
    double ya = own ? ga : 0.0;
    if (own) wv[a] = ya;
    for (int k = 0; k + 1 < m; ++k) {
        Gp::sync();
        const double yk = wv[k];
        if (own && a > k) { ya = fma(-H[k * ldh + a], yk, ya); wv[a] = ya; }
    }
    double la = 0.0;
    if (own) { const double d = H[a * ldh + a]; la = (d > 0.0) ? ya / d : 0.0; }
    const double dn = gvv - Gp::sum(own ? ya * la : 0.0, red);
    if (own) H[a * ldh + m] = la;
    if (a == m) H[m * ldh + m] = dn;
    Gp::sync();
    return !(dn > 0.0);
}

template <int GW>
__device__ void ldl_delete(int m, int a, int p, double *__restrict__ H, int ldh, double *__restrict__ wv,
                           double *__restrict__ dv) {
    using Gp = Group<GW>;
    const bool in = a < m;
    double wa = (in && a > p) ? H[p * ldh + a] : 0.0;
    double alpha = H[p * ldh + p];
    if (in) wv[a] = wa;
    double dpend = 0.0;
    bool pend = false;
    for (int jj = p + 1; jj < m; ++jj) {
        Gp::sync();
        if (pend) { H[a * ldh + a] = dpend; pend = false; }     // a == jj-1: nobody reads that diagonal any more
        const double wj = wv[jj], dj = H[jj * ldh + jj];
        const double dnew = fma(alpha * wj, wj, dj);
        const double beta = (alpha * wj) / dnew;
        alpha = alpha * (dj / dnew);
        if (a == jj) { dpend = dnew; pend = true; }
        if (in && a > jj) {
            double la = H[jj * ldh + a];
            wa = fma(-wj, la, wa);
            la = fma(beta, wa, la);
            H[jj * ldh + a] = la;
            wv[a] = wa;
        }
    }
    Gp::sync();
    if (pend) H[a * ldh + a] = dpend;
    // close up: U[k][c] -> U[k'][c'] with every index above p shifted down by one, through the lower triangle
    if (in && a != p) {
        const int a2 = a - (a > p);
        for (int k = 0; k < a; ++k) {
            if (k == p) continue;
            H[a2 * ldh + (k - (k > p))] = H[k * ldh + a];
        }
        dv[a2] = H[a * ldh + a];
    }
    Gp::sync();
    if (a < m - 1) {
        for (int k = 0; k < a; ++k) H[k * ldh + a] = H[a * ldh + k];
        H[a * ldh + a] = dv[a];
    }
    Gp::sync();
}

// ------------------------------------------------------------------------------------------------
// Box QP  min 1/2 U'GU + F'U, lb <= U <= ub  -- exact primal active-set method (free block solved by
// LDL', ratio test to the first blocking bound, most negative relative multiplier leaves), started
// from the best of four candidate vertices/partitions by objective value: all-lower, all-upper and
// the two previous solutions of this scenario.  The reference's quasi-LPV inner iteration
// (NTM_MPC_Sim.m:94-128) often runs into a period-2 limit cycle between bang-bang patterns, so
// "the solution before last" is usually the right partition and the method stops after one check.
// The candidate pass also yields the exact gradient and its scale |F| + |G||u| at every candidate, so
// in that common case the whole solve is ONE pass over G.
// (Block principal pivoting was tried first: it cycles on these Hessians, cond 1e6..1e11.)
// Bound components of the result are exactly lb/ub (the reference's 1e-14 stop rule compares bits).
// ------------------------------------------------------------------------------------------------
#define NTM_QP_EPS_G 1e-13
#define NTM_QP_CAREFUL_IT 16

struct QpHist {
    double u1, u2;   // this thread's component of the last / second-to-last solution
    int s1, s2;      // and its partition state there (-1 at lb, +1 at ub, 0 free)
    int n;           // number of valid history entries (0..2); 3 = two entries AND a warm QP of this scenario needed more than
                     // NTM_QP_CAREFUL_IT active-set iterations (one-warp groups: selects the start rule, sticky)
};

template <int GW>
__device__ int qp_solve(int N, int j, const Work &w, double Fj, double lbj, double ubj, QpHist &hist, double &Uout,
                        int max_iter, int &iters_out, int *slow_out = nullptr) {
    using Gp = Group<GW>;
    const bool act = j < N;
    const int ldg = w.ldg;
    const bool pinned = !(ubj > lbj);          // degenerate box (or NaN bounds): stays at lb
    const double INF = __longlong_as_double(0x7ff0000000000000LL);

    // ---- cold start on a long horizon: offer the clipped unconstrained minimiser as a candidate (interior
    //      solutions would otherwise cost one active-set iteration per freed variable)
    if (GW > 1 && hist.n == 0) {
        double *H = (N <= w.hcap) ? w.H : w.Hbig;
        const int ldh = (N <= w.hcap) ? odd_ld(w.hcap) : ldg;
        if (act) {
            for (int a = 0; a < N; ++a) H[a * ldh + j] = w.G[a * ldg + j];
            w.sol[j] = -Fj;
        }
        Gp::sync();
        const bool bad = ldl_solve<GW>(N, j, H, ldh, w.sol);
        const double un = act ? w.sol[j] : 0.0;
        const bool usable = !Gp::any(act && !isfinite(un), w.ired) && !bad;
        if (usable) {
            hist.u2 = fmin(fmax(un, lbj), ubj);
            hist.s2 = (un <= lbj) ? -1 : ((un >= ubj) ? 1 : 0);
            hist.u1 = hist.u2; hist.s1 = hist.s2;
            hist.n = 2;                         // occupies the two history slots until real solutions arrive
        }
        Gp::sync();
    }
    // ---- start.  (1) The two previous solutions: one pass over G gives the exact gradient G*c + F and its
    //      scale |F| + |G||c| at both; if one of them is a vertex whose multipliers have the right sign it IS the
    //      (unique) minimiser and the solve is over.  (2) Otherwise add all-lower / all-upper and start the
    //      active-set iterations from the candidate with the lowest objective.
    const double cu2 = (hist.n >= 2) ? hist.u2 : lbj, cu1 = (hist.n >= 1) ? hist.u1 : lbj;
    double g2 = 0.0, g3 = 0.0, s2 = 0.0, s3 = 0.0;
    int state = -1;
    double u = lbj, g = Fj, sc = fabs(Fj);
    bool solved = false;
    if (hist.n >= 1) {
        if (act) w.cand[2 * j + 1] = make_double2(cu2, cu1);
        Gp::sync();
        if (act) {
            const double *gp = w.G + j;
            const double2 *cp = w.cand + 1;
#pragma unroll 2
            for (int k = 0; k < N; ++k, gp += ldg, cp += 2) {
                const double gk = *gp, ga = fabs(gk);
                const double2 cb = *cp;
                g2 = fma(gk, cb.x, g2); g3 = fma(gk, cb.y, g3);
                s2 = fma(ga, fabs(cb.x), s2); s3 = fma(ga, fabs(cb.y), s3);
            }
        }
        {   // last solution first
            const double t = g3 + Fj, sa = s3 + fabs(Fj);
            const bool ok = !act || pinned || (hist.s1 < 0 && t >= -NTM_QP_EPS_G * sa) || (hist.s1 > 0 && -t >= -NTM_QP_EPS_G * sa);
            if (Gp::all(ok, w.ired)) { solved = true; state = pinned ? -1 : hist.s1; u = cu1; g = t; sc = sa; }
        }
        if (!solved && hist.n >= 2) {
            const double t = g2 + Fj, sa = s2 + fabs(Fj);
            const bool ok = !act || pinned || (hist.s2 < 0 && t >= -NTM_QP_EPS_G * sa) || (hist.s2 > 0 && -t >= -NTM_QP_EPS_G * sa);
            if (Gp::all(ok, w.ired)) { solved = true; state = pinned ? -1 : hist.s2; u = cu2; g = t; sc = sa; }
        }
    }
    bool exact = true;                          // g, sc are the exact gradient / scale at u
    if (slow_out != nullptr && !solved) ++*slow_out;    // this QP takes the active-set path (cost key of the scenario)
    if (GW == 1 && !solved && hist.n == 2) {
        // One-warp groups with a history: start from the better of the two previous solutions and leave all-lower /
        // all-upper out -- a QP that misses the vertex test has interior components that move a little at every
        // re-linearisation, and its predecessors are far better starts than a corner of the box; skipping the second
        // pass over G and two of the four objective sums takes ~0.3 us off the ~5 us such a QP costs a lone warp.
        // NOT for a scenario one of whose warm QPs ran long (hist.n == 3, sticky): scenario 62,420 of config 3 flips
        // ~10 bang-bang switches per QP, and from a previous solution that costs 27 iterations per QP instead of 11
        // from the best corner (5.3 against 2.8 ms alone -- the scenario that ends the slowest 8-GPU shard of config 3).
        const double q2 = Gp::sum(act ? cu2 * fma(0.5, g2, Fj) : 0.0, w.red);
        const double q3 = Gp::sum(act ? cu1 * fma(0.5, g3, Fj) : 0.0, w.red);
        if (q3 <= q2) { state = hist.s1; u = cu1; g = g3 + Fj; sc = s3; }
        else { state = hist.s2; u = cu2; g = g2 + Fj; sc = s2; }
        sc += fabs(Fj);
        if (pinned) { state = -1; u = lbj; }
    } else if (!solved) {
        double g0 = 0.0, g1 = 0.0, s0 = 0.0, s1 = 0.0;
        if (act) w.cand[2 * j] = make_double2(lbj, ubj);
        Gp::sync();
        if (act) {
            const double *gp = w.G + j;
            const double2 *cp = w.cand;
#pragma unroll 2
            for (int k = 0; k < N; ++k, gp += ldg, cp += 2) {
                const double gk = *gp, ga = fabs(gk);
                const double2 ca = *cp;
                g0 = fma(gk, ca.x, g0); g1 = fma(gk, ca.y, g1);
                s0 = fma(ga, fabs(ca.x), s0); s1 = fma(ga, fabs(ca.y), s1);
            }
        }
        const double q0 = Gp::sum(act ? lbj * fma(0.5, g0, Fj) : 0.0, w.red);
        const double q1 = Gp::sum(act ? ubj * fma(0.5, g1, Fj) : 0.0, w.red);
        double qb = q0;
        state = -1; u = lbj; g = g0 + Fj; sc = s0;
        if (q1 < qb) { qb = q1; state = 1; u = ubj; g = g1 + Fj; sc = s1; }
        if (hist.n >= 2) {
            const double q2 = Gp::sum(act ? cu2 * fma(0.5, g2, Fj) : 0.0, w.red);
            if (q2 < qb) { qb = q2; state = hist.s2; u = cu2; g = g2 + Fj; sc = s2; }
        }
        if (hist.n >= 1) {
            const double q3 = Gp::sum(act ? cu1 * fma(0.5, g3, Fj) : 0.0, w.red);
            if (q3 < qb) { qb = q3; state = hist.s1; u = cu1; g = g3 + Fj; sc = s3; }
        }
        sc += fabs(Fj);
        if (pinned) { state = -1; u = lbj; }
    }

    int status = solved ? NTM_SCN_OK : NTM_SCN_QP_ITER_CAP, it = 1;
    bool broke = false;
    if (!solved && GW > 1) {
        // Long horizons: the factorisation of the free block is MAINTAINED across iterations (append / rank-one delete).
        // free list in factor order; `pos` is this thread's variable's position in it (-1: at a bound)
        int m;
        int pos = Gp::prefix(act && state == 0, w.ired, m);
        if (!(act && state == 0)) pos = -1;
        if (pos >= 0) w.idx[pos] = j;
        double *H = (m <= w.hcap) ? w.H : w.Hbig;                // big free sets live in the global slab
        int ldh = (m <= w.hcap) ? odd_ld(w.hcap) : ldg;
        bool factored = false, refined = false;
        int nops = 0;                                            // factor updates since the last full factorisation
        Gp::sync();
        for (it = 1; it <= max_iter; ++it) {
            if (m > 0) {
                if (pos >= 0) w.sol[pos] = -g;
                if (!factored || nops >= 32) {                   // (re)factorise the free block, fused with the solve
                    if (j < m) {
                        const int cb = w.idx[j];
                        for (int a = 0; a < m; ++a) H[a * ldh + j] = w.G[w.idx[a] * ldg + cb];
                    }
                    Gp::sync();
                    broke |= ldl_solve<GW>(m, j, H, ldh, w.sol);
                    factored = true; nops = 0;
                } else {
                    Gp::sync();
                    ldl_apply<GW>(m, j, H, ldh, w.sol);
                }
                const double pj = (pos >= 0) ? w.sol[pos] : 0.0;   // Newton step on the face
                double aj = INF;
                if (pos >= 0) {
                    if (pj < 0.0) aj = (lbj - u) / pj;
                    else if (pj > 0.0) aj = (ubj - u) / pj;
                }
                int jblk;
                const double amin = Gp::argmin(aj, j, w.red, w.ired, jblk);
                const bool blocked = amin < 1.0;
                const double alpha = blocked ? fmax(amin, 0.0) : 1.0;
                if (pos >= 0) u = fma(alpha, pj, u);
                exact = false;
                if (blocked) {                                   // a bound blocks: fix it, stay on the arc
                    if (act) {
                        double dg = 0.0;
                        for (int a = 0; a < m; ++a) dg = fma(w.G[w.idx[a] * ldg + j], w.sol[a], dg);
                        g = fma(alpha, dg, g);
                    }
                    if (j == jblk) { state = (pj < 0.0) ? -1 : 1; u = (pj < 0.0) ? lbj : ubj; w.ired[7] = pos; }
                    Gp::sync();
                    const int p = w.ired[7];
                    ldl_delete<GW>(m, j, p, H, ldh, w.uv, w.sol);
                    int moved = -1;
                    if (j > p && j < m) moved = w.idx[j];
                    Gp::sync();
                    if (moved >= 0) w.idx[j - 1] = moved;
                    if (pos == p) pos = -1; else if (pos > p) --pos;
                    --m; ++nops;
                    Gp::sync();
                    continue;
                }
            }
            // minimiser on the current face: exact gradient and its scale, then the bound multipliers
            if (!exact) {
                if (act) w.uv[j] = u;
                Gp::sync();
                double t = Fj, sa = fabs(Fj);
                if (act) {
                    const double *gp = w.G + j;
#pragma unroll 2
                    for (int k = 0; k < N; ++k, gp += ldg) {
                        const double gk = *gp, uk = w.uv[k];
                        t = fma(gk, uk, t);
                        sa = fma(fabs(gk), fabs(uk), sa);
                    }
                }
                g = t; sc = sa; exact = true;
            }
            // the step came from an updated factor: if the free gradient is not at rounding level, refine once with a
            // fresh factorisation (one more Newton step = iterative refinement)
            if (nops > 0 && !refined) {
                if (Gp::any(pos >= 0 && fabs(g) > 1e-9 * sc, w.ired)) { factored = false; refined = true; continue; }
            }
            double lam = INF;
            if (act && !pinned) {
                if (state < 0) lam = g / sc;
                else if (state > 0) lam = -g / sc;
            }
            int jw;
            const double lmin = Gp::argmin(lam, j, w.red, w.ired, jw);
            if (!(lmin < -NTM_QP_EPS_G)) { status = NTM_SCN_OK; break; }
            // variable jw leaves its bound: append it to the factorisation
            if (m + 1 > w.hcap && H == w.H) {                    // outgrew the shared-memory workspace: move to the slab
                if (j < m) for (int k = 0; k <= j; ++k) w.Hbig[k * ldg + j] = H[k * ldh + j];
                H = w.Hbig; ldh = ldg;
                Gp::sync();
            }
            if (factored && m > 0) {
                const double ga = (j < m) ? w.G[w.idx[j] * ldg + jw] : 0.0;
                const bool bad = ldl_append<GW>(m, j, H, ldh, ga, w.G[jw * ldg + jw], w.uv, w.red);
                if (bad) factored = false;                       // numerically singular direction: rebuild next time
                ++nops;
            } else factored = false;
            if (j == jw) { state = 0; pos = m; w.idx[m] = j; }
            ++m;
            Gp::sync();
        }
    }
    if constexpr (GW == 1) {
        // Short horizons (one warp): free sets are a handful of variables, refactorising each iteration is cheapest.
        for (it = 1; !solved && it <= max_iter; ++it) {
            const bool isfree = act && state == 0;
            int m;
            const int pos = Gp::prefix(isfree, w.ired, m);
            if (m > 0) {
                if (isfree) { w.idx[pos] = j; w.sol[pos] = -g; }
                Gp::sync();
                double *H = (m <= w.hcap) ? w.H : w.Hbig;                // big free sets spill to the global slab
                const int ldh = (m <= w.hcap) ? odd_ld(w.hcap) : ldg;
                if (j < m) {
                    const int cb = w.idx[j];
                    for (int a = 0; a < m; ++a) H[a * ldh + j] = w.G[w.idx[a] * ldg + cb];
                }
                Gp::sync();
                broke |= ldl_solve<GW>(m, j, H, ldh, w.sol);              // sol[0..m) = Newton step on the face
                const double pj = isfree ? w.sol[pos] : 0.0;
                double aj = INF;
                if (isfree) {
                    if (pj < 0.0) aj = (lbj - u) / pj;
                    else if (pj > 0.0) aj = (ubj - u) / pj;
                }
                int jblk;
                const double amin = Gp::argmin(aj, j, w.red, w.ired, jblk);
                const bool blocked = amin < 1.0;
                const double alpha = blocked ? fmax(amin, 0.0) : 1.0;
                if (isfree) u = fma(alpha, pj, u);
                exact = false;
                if (blocked) {                                           // a bound blocks: fix it, stay on the arc
                    if (act) {
                        double dg = 0.0;
                        for (int a = 0; a < m; ++a) dg = fma(w.G[w.idx[a] * ldg + j], w.sol[a], dg);
                        g = fma(alpha, dg, g);
                    }
                    if (j == jblk) { state = (pj < 0.0) ? -1 : 1; u = (pj < 0.0) ? lbj : ubj; }
                    Gp::sync();
                    continue;
                }
            }
            // minimiser on the current face: exact gradient and its scale, then the bound multipliers
            if (!exact) {
                if (act) w.uv[j] = u;
                Gp::sync();
                double t = Fj, sa = fabs(Fj);
                if (act) {
                    const double *gp = w.G + j;
    #pragma unroll 2
                    for (int k = 0; k < N; ++k, gp += ldg) {
                        const double gk = *gp, uk = w.uv[k];
                        t = fma(gk, uk, t);
                        sa = fma(fabs(gk), fabs(uk), sa);
                    }
                }
                g = t; sc = sa; exact = true;
            }
            double lam = INF;
            if (act && !pinned) {
                if (state < 0) lam = g / sc;
                else if (state > 0) lam = -g / sc;
            }
            int jw;
            const double lmin = Gp::argmin(lam, j, w.red, w.ired, jw);
            if (!(lmin < -NTM_QP_EPS_G)) { status = NTM_SCN_OK; break; }
            if (j == jw) state = 0;
            Gp::sync();
        }
    }
    if (it > max_iter) it = max_iter;
    // a pinned variable (lbj == ubj) has one value either way; its state is the side the gradient points to, which is
    // what the literal kernels map back to U: b * [umin, umax] can round to one y although umin < umax
    if (pinned) state = (g < 0.0) ? 1 : -1;
    const bool nonfinite = Gp::any(act && !(isfinite(u) && isfinite(g)), w.ired);
    double Uj = (state < 0) ? lbj : ((state > 0) ? ubj : fmin(fmax(u, lbj), ubj));
    if (nonfinite) Uj = nan("");               // IEEE-faithful: a non-finite Hessian/gradient poisons the step
    if (nonfinite || broke) status = NTM_SCN_NONFINITE;
    hist.u2 = hist.u1; hist.s2 = hist.s1;
    hist.u1 = Uj; hist.s1 = state;
    hist.n = (GW == 1 && hist.n >= 2 && it > NTM_QP_CAREFUL_IT) ? 3 : max(hist.n, min(hist.n + 1, 2));
    Gp::sync();
    Uout = Uj;
    iters_out = it;
    return status;
}

// ------------------------------------------------------------------------------------------------
// General-inequality QP  min 1/2 U'GU + F'U,  lb <= U <= ub,  Lg U <= bg  -- what NTM_MPC_Sim.m:97 hands to quadprog
// once getWLc.m's state rows are kept (SURVEY 8(f)-1).  qp_solve gives the minimiser over the box; when it violates a
// general row it is a dual-feasible start (an "S-pair") for a Goldfarb-Idnani dual active-set continuation in scaled
// variables t = (U - lb)/(ub - lb), rows divided by their 1-norm:
//     J (n x n, J'HJ = I) and R (q x q upper triangular, J1'N = R) are kept in shared memory;
//     the most violated row/bound n+ enters:  d = J'n+,  z = J2 d2,  r = R^{-1} d1,
//     t2 = violation/|d2|^2 (full step),  t1 = min_{r_k>0} u_k/r_k (a multiplier hits zero first: that constraint
//     leaves, Givens rotations restore R), no step possible = infeasible (quadprog exitflag -2).
// The start factor comes from ONE Cholesky of the permuted scaled Hessian (free variables first, the variables on
// their bounds last) and the inverse of its factor: with that order J2 has zero rows at the fixed variables and R can be
// read off J.  Thread j owns variable j, row j of J, row/column j of R and multiplier position j.
// ------------------------------------------------------------------------------------------------
struct IneqWork {
    double *t, *d, *r, *mu, *nv, *rg, *x, *colv;   // [N] each
    double *rs;                                    // [M] row 1-norms in scaled variables (0: empty row)
    int *aset;                                     // [N] constraint at active position k: j (lower), N+j (upper), 2N+i
    int *ord;                                      // [N] start permutation
    int *tmpi;                                     // [N] general rows carried over a factor rebuild
    int *gact;                                     // [M] general row i active
};

__host__ __device__ inline size_t ineq_bytes(int N, int M) {
    const size_t b = (8 * (size_t)N + (size_t)M) * 8 + (3 * (size_t)N + (size_t)M) * 4;
    return (b + 15) & ~(size_t)15;
}

__device__ inline IneqWork carve_ineq(unsigned char *base, int N, int M) {
    IneqWork q;
    double *d = reinterpret_cast<double *>(base);
    q.t = d; d += N; q.d = d; d += N; q.r = d; d += N; q.mu = d; d += N; q.nv = d; d += N; q.rg = d; d += N;
    q.x = d; d += N; q.colv = d; d += N; q.rs = d; d += M;
    int *ip = reinterpret_cast<int *>(d);
    q.aset = ip; ip += N; q.ord = ip; ip += N; q.tmpi = ip; ip += N; q.gact = ip;
    return q;
}

#define NTM_QP_INEQ_TOL 1e-9
#define NTM_QP_STUCK_TOL 1e-6

// Row providers: M rows a_i'U <= b_i.  ncol(i) = number of leading columns that can be non-zero.
struct GlobalRows {                                  // ntm_qp_ineq: caller-supplied dense rows in global memory
    const double *__restrict__ Lg, *__restrict__ bg;
    int layout, S, s, M, N;
    __device__ __forceinline__ int count() const { return M; }
    __device__ __forceinline__ int ncol(int) const { return N; }
    __device__ __forceinline__ double coef(int i, int c) const { return Lg[elem(layout, S, M * N, s, i + M * c)]; }
    __device__ __forceinline__ double rhs(int i) const { return bg[elem(layout, S, M, s, i)]; }
    // pass 1: rs[i] = 1-norm of row i in scaled variables; true if an empty row has a negative right-hand side
    __device__ __forceinline__ bool scales(int j, int T, const double *rg, double *rs) const {
        bool bad = false;
        for (int i = j; i < M; i += T) {
            double a1 = 0.0;
            for (int c = 0; c < N; ++c) a1 = fma(fabs(coef(i, c)), rg[c], a1);
            rs[i] = a1;
            if (a1 == 0.0 && rhs(i) < 0.0) bad = true;
        }
        return bad;
    }
    // pass 2: this thread's most violated inactive row at x (normalised), merged into (vbest, idbest)
    __device__ __forceinline__ void most_violated(int j, int T, const double *x, const double *rs, const int *gact,
                                                  double &vbest, int &idbest) const {
        for (int i = j; i < M; i += T) {
            const double rsi = rs[i];
            if (rsi == 0.0 || gact[i]) continue;
            double acc = -rhs(i);
            for (int c = 0; c < N; ++c) acc = fma(coef(i, c), x[c], acc);
            acc /= rsi;
            if (acc > vbest) { vbest = acc; idbest = 2 * N + i; }
        }
    }
};
// Fused loop, literal Gamma, QP variables y = b .* U: the state rows of getWLc.m (Mi/MN blocks :9-12,25 through
// Mcal*Gamma :57) for predicted state i+1 are  xmin <= f_i + sum_{c<=i} p_{i-c} cs_c y_c <= xmax  with p_d the first
// column of A_d...A_1 and f = Phi*x_k + Lambda (the right-hand side c + W*x_k of NTM_MPC_Sim.m:97).  Refreshed rows:
// p = the current condensation (w.P12), cs = NULL (1).  Frozen rows (the script builds L, W, c once, :74): p, f from
// the offline build and cs_c = b0 / b_c, because the variables carry the CURRENT b.
// Row 4i+q: q = 0: -w <= -xmin(1), 1: -omega <= -xmin(2), 2: w <= xmax(1), 3: omega <= xmax(2).
struct StateRows {
    const double2 *P12, *fs;
    const double *cs;
    double xmin1, xmax1, xmin2, xmax2;
    int N;
    __device__ __forceinline__ int count() const { return 4 * N; }
    __device__ __forceinline__ int ncol(int r) const { return (r >> 2) + 1; }
    __device__ __forceinline__ double coef(int r, int c) const {
        const int i = r >> 2;
        if (c > i) return 0.0;
        const double2 p = P12[i - c];
        double v = (r & 1) ? p.y : p.x;
        if (cs) v *= cs[c];
        return (r & 2) ? v : -v;
    }
    __device__ __forceinline__ double rhs(int r) const {
        const double2 f = fs[r >> 2];
        switch (r & 3) {
            case 0: return f.x - xmin1;
            case 1: return f.y - xmin2;
            case 2: return xmax1 - f.x;
            default: return xmax2 - f.y;
        }
    }
    // The four rows of predicted state i share one coefficient pair per column (+-p.x, +-p.y), so both passes walk the
    // states, not the rows: one thread per state, i + 1 columns, a quarter of the loads of the generic loops.  Same
    // summation order per row as the generic passes (c ascending), so the numbers do not depend on the path.
    __device__ __forceinline__ bool scales(int j, int T, const double *rg, double *rs) const {
        bool bad = false;
        for (int i = j; i < N; i += T) {
            double aw = 0.0, ao = 0.0;
            const double2 *p = P12 + i;
            for (int c = 0; c <= i; ++c, --p) {
                const double2 pc = *p;
                const double g = cs ? cs[c] * rg[c] : rg[c];
                aw = fma(fabs(pc.x), fabs(g), aw);
                ao = fma(fabs(pc.y), fabs(g), ao);
            }
            rs[4 * i] = aw; rs[4 * i + 1] = ao; rs[4 * i + 2] = aw; rs[4 * i + 3] = ao;
            const double2 f = fs[i];
            if (aw == 0.0 && (f.x - xmin1 < 0.0 || xmax1 - f.x < 0.0)) bad = true;
            if (ao == 0.0 && (f.y - xmin2 < 0.0 || xmax2 - f.y < 0.0)) bad = true;
        }
        return bad;
    }
    __device__ __forceinline__ void most_violated(int j, int T, const double *x, const double *rs, const int *gact,
                                                  double &vbest, int &idbest) const {
        for (int i = j; i < N; i += T) {
            double sw = 0.0, so = 0.0;
            const double2 *p = P12 + i;
            for (int c = 0; c <= i; ++c, --p) {
                const double2 pc = *p;
                const double xc = cs ? cs[c] * x[c] : x[c];
                sw = fma(pc.x, xc, sw);
                so = fma(pc.y, xc, so);
            }
            const double2 f = fs[i];
            const double aw = rs[4 * i], ao = rs[4 * i + 1];
            const double v[4] = {(xmin1 - f.x) - sw, (xmin2 - f.y) - so, (f.x - xmax1) + sw, (f.y - xmax2) + so};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double a = (q & 1) ? ao : aw;
                if (a == 0.0 || gact[4 * i + q]) continue;
                if (!(v[q] > vbest * a)) continue;             // v/a > vbest <=> v > vbest*a (a > 0): only winners are divided
                const double acc = v[q] / a;
                if (acc > vbest) { vbest = acc; idbest = 2 * N + 4 * i + q; }
            }
        }
    }
};

// Fused loop, ANY Gamma index (NTM_PROFILE_GAMMA_I / DENSE_G, one-warp groups), QP variables U: the same rows read from
// the dense Gamma tile the tensor-core Hessian build keeps in shared memory (build_GF_dense_dmma: column c at
// Gam + c*ldm, state i in rows 2i, 2i+1) -- getWLc.m:57  L = Mcal*Gamma + Ecal with Gamma as Rho_to_PhiGammaLambda.m:26-40
// wrote it.  Refreshed rows: the current tile; frozen rows (:74): a copy of the offline tile.  Row numbering as StateRows.
struct DenseRows {
    const double *Gam;
    int ldm;
    const double2 *fs;
    double xmin1, xmax1, xmin2, xmax2;
    int N;
    __device__ __forceinline__ int count() const { return 4 * N; }
    __device__ __forceinline__ int ncol(int r) const { return (r >> 2) + 1; }
    __device__ __forceinline__ double coef(int r, int c) const {
        const int i = r >> 2;
        if (c > i) return 0.0;
        const double v = Gam[(size_t)c * ldm + 2 * i + (r & 1)];
        return (r & 2) ? v : -v;
    }
    __device__ __forceinline__ double rhs(int r) const {
        const double2 f = fs[r >> 2];
        switch (r & 3) {
            case 0: return f.x - xmin1;
            case 1: return f.y - xmin2;
            case 2: return xmax1 - f.x;
            default: return xmax2 - f.y;
        }
    }
    __device__ __forceinline__ bool scales(int j, int T, const double *rg, double *rs) const {
        bool bad = false;
        for (int i = j; i < N; i += T) {
            double aw = 0.0, ao = 0.0;
            const double *p = Gam + 2 * i;
            for (int c = 0; c <= i; ++c, p += ldm) {
                const double2 pc = *reinterpret_cast<const double2 *>(p);
                aw = fma(fabs(pc.x), fabs(rg[c]), aw);
                ao = fma(fabs(pc.y), fabs(rg[c]), ao);
            }
            rs[4 * i] = aw; rs[4 * i + 1] = ao; rs[4 * i + 2] = aw; rs[4 * i + 3] = ao;
            const double2 f = fs[i];
            if (aw == 0.0 && (f.x - xmin1 < 0.0 || xmax1 - f.x < 0.0)) bad = true;
            if (ao == 0.0 && (f.y - xmin2 < 0.0 || xmax2 - f.y < 0.0)) bad = true;
        }
        return bad;
    }
    __device__ __forceinline__ void most_violated(int j, int T, const double *x, const double *rs, const int *gact,
                                                  double &vbest, int &idbest) const {
        for (int i = j; i < N; i += T) {
            double sw = 0.0, so = 0.0;
            const double *p = Gam + 2 * i;
            for (int c = 0; c <= i; ++c, p += ldm) {
                const double2 pc = *reinterpret_cast<const double2 *>(p);
                sw = fma(pc.x, x[c], sw);
                so = fma(pc.y, x[c], so);
            }
            const double2 f = fs[i];
            const double aw = rs[4 * i], ao = rs[4 * i + 1];
            const double v[4] = {(xmin1 - f.x) - sw, (xmin2 - f.y) - so, (f.x - xmax1) + sw, (f.y - xmax2) + so};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double a = (q & 1) ? ao : aw;
                if (a == 0.0 || gact[4 * i + q]) continue;
                if (!(v[q] > vbest * a)) continue;
                const double acc = v[q] / a;
                if (acc > vbest) { vbest = acc; idbest = 2 * N + 4 * i + q; }
            }
        }
    }
};

struct ExtWork {                 // extra per-group shared memory of the fused kernel's EXT instantiation
    double2 *fs;                 // [N] free response Phi*x_k + Lambda of the rows
    double2 *P0;                 // [N] frozen rows: p_d of the offline build
    double2 *Phi0;               // [N] frozen rows: first column of Phi's blocks, offline build
    double2 *Lam0;               // [N] frozen rows: Lambda of the offline build
    double *cs;                  // [N] frozen rows: b0 / b_c
};
__host__ __device__ inline size_t ext_bytes(int N) { return (((size_t)N * (4 * 16 + 8)) + 15) & ~(size_t)15; }
__device__ inline ExtWork carve_ext(unsigned char *base, int N) {
    ExtWork x;
    double2 *d = reinterpret_cast<double2 *>(base);
    x.fs = d; d += N; x.P0 = d; d += N; x.Phi0 = d; d += N; x.Lam0 = d; d += N;
    x.cs = reinterpret_cast<double *>(d);
    return x;
}

// Uj: in = this thread's component of the box minimiser (qp_solve), out = the solution.  Overwrites w.G (-> J) and
// w.H (-> R; needs hcap == N).  vst_out: -1 / +1 = this thread's variable ends on its lower / upper bound, 0 = inside.
//
// regen: group-cooperative callable that puts the Hessian back into w.G (the continuation has overwritten it with J).
// With it, J and R are REBUILT from the current active set -- Cholesky of the permuted Hessian for the active bounds,
// then the active general rows re-join one by one -- every NTM_QP_REFACTOR_EVERY factor updates and whenever the
// maintained factors say "no step possible": exitflag -2 is only reported by factors that are fresh.  (Measured need:
// N = 72, dozens of nearly parallel state rows, cond(G) ~ 1e10, 300+ Givens updates -> a false infeasible.)
#define NTM_QP_REFACTOR_EVERY 96
struct NoRegen {
    static constexpr bool available = false;
    __device__ __forceinline__ void operator()() const {}
};
template <class F>
struct RegenFn {
    F f;
    static constexpr bool available = true;
    __device__ __forceinline__ void operator()() const { f(); }
};
template <class F>
__device__ __forceinline__ RegenFn<F> make_regen(F f) { return RegenFn<F>{f}; }

// WARM START (round 2; rows numbered 4*state + q only: StateRows / DenseRows).  warm_mask >= 0 offers the active set of an
// earlier QP of the same scenario -- warm_vst = this thread's variable on its lower / upper bound / free, bit q of
// warm_mask = row 4j + q active -- instead of the box minimiser: J, R are built for that set (bounds from the permuted
// Cholesky factor, rows join by one reflector each: no search, no step), the minimiser ON the set and its multipliers
// follow from two triangular solves, and if every multiplier is non-negative that is a dual-feasible start (an
// "S-pair") from which the iteration continues -- usually straight to "nothing violated".  Consecutive QPs of a step
// alternate between two active sets (the period-2 cycle of the inner iteration: 96 % of the QPs of the binding-box
// sample end on the active set of the QP before last), so this replaces 12-20 dual iterations by none.  A negative
// multiplier (below -1e-12 of their sum: with cond(G) up to 1e11 a constraint kept on a slightly negative multiplier moves
// the answer visibly) returns NTM_QP_WARM_FAILED with w.G destroyed: the caller restores the Hessian and calls again cold.
// Tried on top and removed: a VERTEX TEST without any factor of the Hessian (LU of the active rows on the free
// variables, multipliers from its transpose, KKT check) -- 5-13 % faster, 2,300 more instructions in a kernel that
// waits on instruction fetch, and one false accept at 1e-10 on the consistent profile (2 % off in one input).
#define NTM_QP_WARM_FAILED (-1)
template <int GW, class Rows, class Regen = NoRegen>
__device__ int qp_ineq_continue(int N, const Rows &rows, int j, const Work &w, const IneqWork &q, double Fj, double lbj,
                                double ubj, double &Uj, int max_iter, int &iters, int *vst_out = nullptr,
                                const Regen &regen = Regen(), int warm_vst = 0, int warm_mask = -1) {
    const int M = rows.count();
    using Gp = Group<GW>;
    const bool act = j < N;
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    const int ldj = w.ldg, ldr = odd_ld(N);
    double *J = w.G, *R = w.H;
    const bool pinned = !(ubj > lbj);
    const double rgj = pinned ? 1.0 : (ubj - lbj);
    const double hbj = pinned ? 0.0 : 1.0;                     // upper bound of the scaled variable
    int vst = 0;
    if (act) vst = (Uj >= ubj && !pinned) ? 1 : ((Uj <= lbj || pinned) ? -1 : 0);
    double tj = (vst == 1) ? 1.0 : ((vst == -1) ? 0.0 : (Uj - lbj) / rgj);
    if (act) { q.rg[j] = rgj; q.x[j] = Uj; }
    for (int i = j; i < M; i += Gp::T) q.gact[i] = 0;
    Gp::sync();
    // row scales; an empty row is a pure feasibility statement 0 <= bg_i
    const bool bad_row = rows.scales(j, Gp::T, q.rg, q.rs);
    if (vst_out) *vst_out = vst;
    if (Gp::any(bad_row, w.ired)) return NTM_SCN_INFEASIBLE;

    int nact = 0;                 // q of the description: number of active constraints (group-uniform)
    int age = 0;                  // factor updates since J and R were last built from scratch
    bool have_factor = false;
    int status = NTM_SCN_QP_ITER_CAP;
    int it = iters;
    bool warm = warm_mask >= 0;   // group-uniform: the caller passes -1 on every thread for a cold call
    int warm_ngen = 0;
    double gtil = 0.0;            // warm start: this thread's component of the scaled gradient at t = 0
    if (warm) {
        vst = act ? (pinned ? -1 : warm_vst) : 0;
        tj = (vst == 1) ? hbj : 0.0;
        if (act) q.x[j] = lbj;
        for (int qq = 0; qq < 4; ++qq) {                        // the offered rows, bit by bit (order: q, then state)
            const bool has = act && ((warm_mask >> qq) & 1);
            int tot;
            const int pos = Gp::prefix(has, w.ired, tot);
            if (has && warm_ngen + pos < N) { q.tmpi[warm_ngen + pos] = 2 * N + 4 * j + qq; q.r[warm_ngen + pos] = 0.0; q.gact[4 * j + qq] = 1; }
            warm_ngen = min(warm_ngen + tot, N);
            Gp::sync();
        }
    }

    // this thread's component of the normal of constraint pid (GI convention n't >= b)
    auto normal_of = [&](int pid) -> double {
        if (!act) return 0.0;
        if (pid < N) return (j == pid) ? 1.0 : 0.0;
        if (pid < 2 * N) return (j == pid - N) ? -1.0 : 0.0;
        return -rows.coef(pid - 2 * N, j) * rgj / q.rs[pid - 2 * N];
    };
    // (J' n)_j for constraint pid; q.nv holds the normal (needed for general rows only)
    auto jt_normal = [&](int pid) -> double {
        double dj = 0.0;
        if (act) {
            if (pid < N) dj = J[(size_t)pid * ldj + j];
            else if (pid < 2 * N) dj = -J[(size_t)(pid - N) * ldj + j];
            else for (int row = 0; row < N; ++row) dj = fma(J[(size_t)row * ldj + j], q.nv[row], dj);
        }
        return dj;
    };
    // constraint pid joins at position nact: ONE Householder reflector H = I - beta v v' turns d2 = q.d[nact..N) into
    // delta e1 (q.d visible to all, dj = q.d[j], dd2 = |d2|^2 > 0) and J2 <- J2 H is two passes over this thread's row.
    // (Round 1 used a chain of N - 1 - nact Givens rotations: a square root and two divisions each, executed serially by
    // every lane -- half of the instructions of a dual iteration.)  v = d2 - delta e1 with delta = -sign(d2_0) |d2|, so
    // v_0 = d2_0 - delta never cancels and beta = 2 / v'v = 1 / (|d2| (|d2| + |d2_0|)).
    auto append = [&](int pid, double dj, double muval, double dd2) {
        double delta = (nact < N) ? q.d[nact] : 0.0;
        if (N - nact > 1) {
            const double alpha = delta, nrm = sqrt(dd2);
            delta = (alpha >= 0.0) ? -nrm : nrm;
            const double v0 = alpha - delta;
            const double beta = 1.0 / (nrm * (nrm + fabs(alpha)));
            if (act) {
                double *Jr = J + (size_t)j * ldj;
                double t = Jr[nact] * v0;
                for (int c = nact + 1; c < N; ++c) t = fma(Jr[c], q.d[c], t);
                t *= beta;
                Jr[nact] = fma(-t, v0, Jr[nact]);
                for (int c = nact + 1; c < N; ++c) Jr[c] = fma(-t, q.d[c], Jr[c]);
            }
        }
        if (j < nact) R[j * ldr + nact] = dj;
        if (j == nact) { R[nact * ldr + nact] = delta; q.aset[nact] = pid; q.mu[nact] = muval; }
        ++nact;
    };
    // J and R from scratch.  fresh: the start from the box minimiser (multipliers = its gradient, no general row is
    // active yet, w.G still holds the Hessian).  Otherwise: the current multipliers are kept, regen() restores the
    // Hessian, the active bounds come from the Cholesky factor and the active general rows re-join one by one.
    // mode 0 = fresh, 1 = rebuild, 2 = warm start: like a rebuild, but w.G still holds the Hessian (no regen), the rows
    // to join are the offered ones (q.tmpi[0..warm_ngen)) and every multiplier is computed afterwards
    auto build_factor = [&](int mode) -> int {
        const bool fresh = mode == 0;
        int ngen = 0;
        double gj = 0.0;
        if (mode != 1) {                                   // gradient at q.x: the box minimiser, or lb for the warm start
            if (act) {
                gj = Fj;
                for (int l = 0; l < N; ++l) gj = fma(w.G[j * w.ldg + l], q.x[l], gj);
                gj *= rgj;
            }
            if (mode == 2) { gtil = gj; ngen = warm_ngen; if (act) q.d[j] = 0.0; Gp::sync(); }
        } else {
            const int id = (j < nact) ? q.aset[j] : -1;
            const double mj = (j < nact) ? q.mu[j] : 0.0;
            const bool isgen = id >= 2 * N;
            const int kg = Gp::prefix(isgen, w.ired, ngen);
            Gp::sync();
            if (j < nact) {
                if (isgen) { q.tmpi[kg] = id; q.r[kg] = mj; }
                else q.d[id < N ? id : id - N] = mj;           // bound multipliers by variable
            }
            Gp::sync();
            regen();
            Gp::sync();
        }
        int nfix = 0, nfree = 0;
        const int kfix = Gp::prefix(act && vst != 0, w.ired, nfix);
        const int kfree = Gp::prefix(act && vst == 0, w.ired, nfree);
        Gp::sync();
        if (act) {
            if (vst != 0) {
                q.ord[N - 1 - kfix] = j;
                q.aset[kfix] = (vst == -1) ? j : N + j;
                q.mu[kfix] = fresh ? fmax((vst == -1) ? gj : -gj, 0.0) : q.d[j];
            } else {
                q.ord[kfree] = j;
            }
        }
        nact = nfix;
        Gp::sync();
        if (act) {                                         // permuted scaled Hessian, lower triangle, into R's buffer
            const int oa = q.ord[j];
            const double ra = q.rg[oa];
            for (int b = 0; b <= j; ++b) {
                const int ob = q.ord[b];
                R[j * ldr + b] = ra * w.G[oa * w.ldg + ob] * q.rg[ob];
            }
        }
        bool broke = false;
        for (int c = 0; c < N; ++c) {
            Gp::sync();
            const double dcc = R[c * ldr + c];
            if (!(dcc > 0.0) || !(dcc < INF)) { broke = true; break; }      // group-uniform (same word read)
            const double ilc = rsqrt(dcc);                  // one reciprocal root per step: l_cc = d * ilc, column scaled by ilc
            double la = 0.0;
            if (act && j > c) { la = R[j * ldr + c] * ilc; q.colv[j] = la; }
            Gp::sync();
            if (act && j > c) {
                R[j * ldr + c] = la;
                for (int b = c + 1; b <= j; ++b) R[j * ldr + b] = fma(-la, q.colv[b], R[j * ldr + b]);
            } else if (j == c) {
                R[c * ldr + c] = dcc * ilc;
                q.nv[c] = ilc;                             // 1 / l_cc for the inverse below (q.nv is free here)
            }
        }
        if (broke) return (int)NTM_SCN_NONFINITE;
        Gp::sync();
        if (act) {                                         // column j of the inverse factor -> row ord[j] of J, columns flipped
            double *Jr = J + (size_t)q.ord[j] * ldj;
            for (int a = 0; a < N; ++a) {
                double val = 0.0;
                if (a == j) val = q.nv[j];
                else if (a > j) {
                    double acc = 0.0;
                    for (int m = j; m < a; ++m) acc = fma(R[a * ldr + m], Jr[N - 1 - m], acc);
                    val = -acc * q.nv[a];
                }
                Jr[N - 1 - a] = val;
            }
        }
        Gp::sync();
        if (j < nact)                                      // R(i,k) = sigma_k * J(f_k, i), i <= k
            for (int k = j; k < nact; ++k) {
                const int id = q.aset[k];
                const double v = J[(size_t)(id < N ? id : id - N) * ldj + j];
                R[j * ldr + k] = (id < N) ? v : -v;
            }
        if (act) q.t[j] = tj;
        for (int g = 0; g < ngen; ++g) {                   // the general rows that were active re-join
            Gp::sync();
            const int pid = q.tmpi[g];
            if (act) q.nv[j] = normal_of(pid);
            Gp::sync();
            const double dj = jt_normal(pid);
            if (act) q.d[j] = dj;
            const double dd2 = Gp::sum((act && j >= nact) ? dj * dj : 0.0, w.red);
            const double dd = Gp::sum(act ? dj * dj : 0.0, w.red);
            Gp::sync();
            if (!(dd2 > 1e-18 * dd) || nact >= N) {         // numerically dependent on the ones before it: it leaves
                if (j == 0) q.gact[pid - 2 * N] = 0;
                continue;
            }
            append(pid, dj, q.r[g], dd2);
        }
        Gp::sync();
        age = 0;
        return (int)NTM_SCN_OK;
    };

    // build_factor has ONE call site (after the search): the start from the box minimiser, the periodic rebuild and the
    // rebuild after "no step possible" on aged factors all pass through it.  (Three inlined copies were 2,000 of the
    // fused kernel's 12,500 instructions, and that kernel waits on instruction fetch: profiles/README.md, round 2.)
    bool rebuild = false;
    for (;;) {
        double vmax = 0.0;
        int pid = -1;
        if (!warm) {
            // ---- most violated constraint (normalised): bounds of this thread's variable, then its share of the rows
            double vbest = -INF;
            int idbest = -1;
            if (act) {
                if (vst != -1) { vbest = -tj; idbest = j; }
                if (vst != 1 && tj - hbj > vbest) { vbest = tj - hbj; idbest = N + j; }
            }
            rows.most_violated(j, Gp::T, q.x, q.rs, q.gact, vbest, idbest);
            int owner;
            vmax = -Gp::argmin(-vbest, j, w.red, w.ired, owner);
            if (owner < 0 || !(vmax == vmax)) { status = NTM_SCN_NONFINITE; break; }
            if (vmax <= NTM_QP_INEQ_TOL) { status = NTM_SCN_OK; break; }
            if (it >= max_iter) break;
            ++it;
            pid = Gp::bcast_from(idbest, owner, w.ired);
        }

        if (!have_factor || (Regen::available && (rebuild || age >= NTM_QP_REFACTOR_EVERY))) {
            const int bs = build_factor(warm ? 2 : (have_factor ? 1 : 0));   // 0: start factor from the box solution
            if (bs != NTM_SCN_OK) { if (warm) return NTM_QP_WARM_FAILED; status = bs; break; }
            have_factor = true; rebuild = false;
            Gp::sync();
        }

        if (warm) {
            // ---- minimiser on the offered set W (N_W't = b_W) and its multipliers, t = J y:
            //      y1 = R^-T b_W,  y2 = -(J'f)_2,  mu = R^-1 (y1 + (J'f)_1),  f = the scaled gradient at t = 0
            warm = false;
            if (act) q.nv[j] = gtil;
            Gp::sync();
            const double cj = jt_normal(2 * N);                       // (J'f)_j
            double bk = 0.0;                                         // right-hand side of the constraint at position j
            if (j < nact) {
                const int id = q.aset[j];
                if (id >= 2 * N) {
                    const int i = id - 2 * N, nc = rows.ncol(i);
                    double acc = -rows.rhs(i);
                    for (int c = 0; c < nc; ++c) acc = fma(rows.coef(i, c), q.x[c], acc);     // q.x = lb
                    bk = acc / q.rs[i];
                } else if (id >= N) bk = -q.t[id - N];               // upper bound: -t >= -hb
            }
            double accf = bk;
            for (int i = 0; i < nact; ++i) {                         // forward substitution R'y1 = b_W
                if (j == i) q.d[i] = accf / R[i * ldr + i];
                Gp::sync();
                if (j > i && j < nact) accf = fma(-R[i * ldr + j], q.d[i], accf);
            }
            if (act && j >= nact) q.d[j] = -cj;
            Gp::sync();
            double tw = 0.0;
            if (act) for (int c = 0; c < N; ++c) tw = fma(J[(size_t)j * ldj + c], q.d[c], tw);
            double acc = (j < nact) ? q.d[j] + cj : 0.0;
            const double rdiag = (j < nact) ? 1.0 / R[j * ldr + j] : 0.0;
            Gp::sync();
            for (int k = nact - 1; k >= 0; --k) {
                if (j == k) q.r[k] = acc * rdiag;
                Gp::sync();
                if (j < k) acc = fma(-R[j * ldr + k], q.r[k], acc);
            }
            Gp::sync();
            const double muj = (j < nact) ? q.r[j] : 0.0;
            const double musum = Gp::sum(fabs(muj), w.red);
            const bool badmu = (j < nact && !(muj >= -1e-12 * musum)) || (act && !(tw == tw)) || !(musum < INF);
            if (Gp::any(badmu, w.ired)) return NTM_QP_WARM_FAILED;    // not dual feasible: the caller starts cold
            if (j < nact) q.mu[j] = fmax(muj, 0.0);
            if (act) {
                tj = (vst == 1) ? hbj : ((vst == -1) ? 0.0 : tw);
                q.x[j] = (vst == 1) ? ubj : ((vst == -1) ? lbj : fma(rgj, tj, lbj));
            }
            Gp::sync();
            continue;                                                // look for violated constraints from here
        }

        // ---- entering normal
        if (act) q.nv[j] = normal_of(pid);
        double up = 0.0;
        bool infeasible = false, capped = false, stale = false;
        for (;;) {
            Gp::sync();
            const double dj = jt_normal(pid);
            if (act) q.d[j] = dj;
            const double dd2 = Gp::sum((act && j >= nact) ? dj * dj : 0.0, w.red);
            const double dd = Gp::sum(act ? dj * dj : 0.0, w.red);
            Gp::sync();
            // r = R^{-1} d1 (column-oriented back substitution; the reciprocal diagonal comes first, one division per
            // lane in parallel instead of one per step of the chain)
            double acc = dj;
            const double rdiag = (j < nact) ? 1.0 / R[j * ldr + j] : 0.0;
            for (int k = nact - 1; k >= 0; --k) {
                if (j == k) q.r[k] = acc * rdiag;
                Gp::sync();
                if (j < k) acc = fma(-R[j * ldr + k], q.r[k], acc);
            }
            Gp::sync();
            const double rj = (j < nact) ? q.r[j] : 0.0;
            int ldrop;
            const double t1 = Gp::argmin((j < nact && rj > 0.0) ? q.mu[j] / rj : INF, j, w.red, w.ired, ldrop);
            const bool zero = !(dd2 > 1e-18 * dd) || nact >= N;
            const double t2 = zero ? INF : vmax / dd2;
            const double tau = fmin(t1, t2);
            if (!(tau < INF)) {
                // no step possible: believed only from factors that are fresh
                if (Regen::available && age > 0) stale = true; else infeasible = true;
                break;
            }
            if (!zero && act) {
                double zj = 0.0;
                for (int c = nact; c < N; ++c) zj = fma(J[(size_t)j * ldj + c], q.d[c], zj);
                tj = fma(tau, zj, tj);
            }
            if (j < nact) q.mu[j] = fmax(fma(-tau, rj, q.mu[j]), 0.0);
            up += tau;
            if (t2 <= t1) {
                // ---- full step: the constraint joins
                append(pid, dj, up, dd2);
                if (pid < N) { if (j == pid) { vst = -1; tj = 0.0; } }
                else if (pid < 2 * N) { if (j == pid - N) { vst = 1; tj = hbj; } }
                else if (j == 0) q.gact[pid - 2 * N] = 1;
                ++age;
                break;
            }
            // ---- partial step: the constraint at position ldrop leaves
            vmax = zero ? vmax : fma(-tau, dd2, vmax);
            {
                const int id = q.aset[ldrop];
                Gp::sync();
                if (id < N) { if (j == id) vst = 0; }
                else if (id < 2 * N) { if (j == id - N) vst = 0; }
                else if (j == 0) q.gact[id - 2 * N] = 0;
                if (j < nact) for (int c = ldrop; c < nact - 1; ++c) R[j * ldr + c] = R[j * ldr + c + 1];
                int as = 0; double ms = 0.0;
                if (j >= ldrop && j < nact - 1) { as = q.aset[j + 1]; ms = q.mu[j + 1]; }
                Gp::sync();
                if (j >= ldrop && j < nact - 1) { q.aset[j] = as; q.mu[j] = ms; }
                for (int k = ldrop; k < nact - 1; ++k) {
                    Gp::sync();
                    const double a = R[k * ldr + k], b = R[(k + 1) * ldr + k];
                    Gp::sync();
                    if (b == 0.0) continue;
                    const double ir = rsqrt(fma(a, a, b * b));             // one reciprocal root instead of a root and two divisions
                    const double cs = a * ir, sn = b * ir;
                    if (j >= k && j < nact - 1) {
                        const double xx = R[k * ldr + j], yy = R[(k + 1) * ldr + j];
                        R[k * ldr + j] = fma(cs, xx, sn * yy);
                        R[(k + 1) * ldr + j] = fma(cs, yy, -sn * xx);
                    }
                    if (act) {
                        const double xx = J[(size_t)j * ldj + k], yy = J[(size_t)j * ldj + k + 1];
                        J[(size_t)j * ldj + k] = fma(cs, xx, sn * yy);
                        J[(size_t)j * ldj + k + 1] = fma(cs, yy, -sn * xx);
                    }
                }
                --nact;
                ++age;
            }
            if (++it >= max_iter) { capped = true; break; }
        }
        if (infeasible) {
            // No step possible on fresh factors.  A row that cannot join AND is violated by no more than
            // NTM_QP_STUCK_TOL of its range is rounding, not infeasibility.
            status = (vmax <= NTM_QP_STUCK_TOL) ? NTM_SCN_OK : NTM_SCN_INFEASIBLE;
            break;
        }
        if (capped) break;
        Gp::sync();
        if (act) q.x[j] = (vst == 1) ? ubj : ((vst == -1) ? lbj : fma(rgj, tj, lbj));
        Gp::sync();
        if (stale) rebuild = true;                             // rebuild J, R from the active set and look again
    }
    if (act) {
        Uj = (vst == 1) ? ubj : ((vst == -1) ? lbj : fma(rgj, tj, lbj));
        if (!(Uj == Uj) && status == NTM_SCN_OK) status = NTM_SCN_NONFINITE;
    }
    if (vst_out) *vst_out = vst;
    iters = it;
    return status;
}

// ------------------------------------------------------------------------------------------------
// Affine stage maps z -> A z + k with A = [a 0; c s] (A.m:2 is lower triangular), composed by a
// warp-level Kogge-Stone scan: lane i ends with M_i o ... o M_0.  Used for the free response
// (Phi*x + Lambda, Rho_to_PhiGammaLambda.m:20-22,49-52), the columns p_d of the literal Gamma and the
// rollout NTM_MPC_Sim.m:112-113 -- 5 dependent stages instead of N.
// ------------------------------------------------------------------------------------------------
struct Aff { double a, c, k1, k2; };           // the (2,2) entry of a composed block is a22^length: tracked outside

// L after E; sL = (2,2) entry of L's linear part
__device__ __forceinline__ Aff aff_compose(const Aff &L, const Aff &E, double sL) {
    Aff r;
    r.a = L.a * E.a;
    r.c = fma(L.c, E.a, sL * E.c);
    r.k1 = fma(L.a, E.k1, L.k1);
    r.k2 = fma(L.c, E.k1, fma(sL, E.k2, L.k2));
    return r;
}

__device__ __forceinline__ Aff aff_shfl_up(const Aff &m, int off) {
    Aff r;
    r.a = __shfl_up_sync(0xffffffffu, m.a, off);
    r.c = __shfl_up_sync(0xffffffffu, m.c, off);
    r.k1 = __shfl_up_sync(0xffffffffu, m.k1, off);
    r.k2 = __shfl_up_sync(0xffffffffu, m.k2, off);
    return r;
}

// Inclusive prefix over lanes 0..N-1.  A lane that still composes at stage `off` holds a full block of `off`
// stages, so its (2,2) entry is the warp-uniform a22^off -- no need to carry it through the shuffles.
__device__ __forceinline__ Aff aff_scan(Aff m, int lane, int N, double a22) {
    double sq = a22;
    for (int off = 1; off < N; off <<= 1) {
        const Aff e = aff_shfl_up(m, off);
        if (lane >= off) m = aff_compose(m, e, sq);
        sq *= sq;
    }
    return m;
}

__device__ __forceinline__ Aff aff_exclusive(const Aff &inc, int lane) {
    Aff e = aff_shfl_up(inc, 1);
    if (lane == 0) { e.a = 1.0; e.c = 0.0; e.k1 = 0.0; e.k2 = 0.0; }
    return e;
}

// ------------------------------------------------------------------------------------------------
// G, F for the literal Gamma (Rho_to_PhiGammaLambda.m:32, index i-j).  There
//     Gamma(i,j) = b_j * p_{i-j},   p_d = first column of A_d*...*A_1, p_0 = e1,
// so G(j,l) = 2 b_j b_l * T[N-j][j-l] with the running correlation sums
//     T[m][e] = sum_{d<=m} p_d' Q p_{d+e}
// -- O(N^2) work instead of the O(N^3) contraction Gamma'*Omega*Gamma (NTM_MPC_Sim.m:120).
// F = 2 Gamma' Omega (Phi x + Lambda - R) uses v_i = A_i v_{i-1} + C, v_0 = x (== Phi*x + Lambda,
// Rho_to_PhiGammaLambda.m:20-22,49-52) and F_l = 2 b_l sum_d p_d' Q (v_{l+d} - r)  (:121).
// Thread j: lag j of T, entry j of F.  a11/a21 are this thread's stage entries (also in w.a11s/w.a21s
// for the serial chain of the multi-warp groups).
// The b factors never enter the loop: the QP is solved in the variables y_j = b_j U_j, whose Hessian is the bare
// table 2T and whose gradient is F_l / b_l.  Writes Gy(j,l) = 2 T[N-j][j-l] (both triangles) and returns Fy_j;
// run_scenario scales the box to b_j*[umin, umax] and maps the solution back (bound components stay exact).
// ------------------------------------------------------------------------------------------------
template <int GW>
__device__ double build_GF_toeplitz(int N, int j, const Work &w, const Params &P, double a11, double a21, double sE,
                                    double xF1, double xF2) {
    using Gp = Group<GW>;
    const bool act = j < N;
    double myp1 = 0.0, myp2 = 0.0, mye1 = 0.0, mye2 = 0.0;
    if constexpr (GW == 1) {
        Aff m;                                           // sE = a22^j: (2,2) entry of the exclusive prefix
        m.a = act ? a11 : 1.0; m.c = act ? a21 : 0.0;
        m.k1 = act ? P.C1 : 0.0; m.k2 = act ? P.C2 : 0.0;
        const Aff inc = aff_scan(m, j, N, P.a22);
        const Aff exc = aff_exclusive(inc, j);
        myp1 = exc.a; myp2 = exc.c;
        mye1 = fma(inc.a, xF1, inc.k1) - P.r1;
        mye2 = fma(inc.c, xF1, fma(sE * P.a22, xF2, inc.k2)) - P.r2;
    } else {
        double p1 = 1.0, p2 = 0.0, v1 = xF1, v2 = xF2;
        for (int d = 0; d < N; ++d) {
            if (d == j) { myp1 = p1; myp2 = p2; }
            const double a = w.a11s[d], c = w.a21s[d];
            const double nv1 = fma(a, v1, P.C1);
            const double nv2 = fma(P.a22, v2, fma(c, v1, P.C2));
            v1 = nv1; v2 = nv2;
            if (d == j) { mye1 = v1 - P.r1; mye2 = v2 - P.r2; }
            const double np1 = a * p1;
            const double np2 = fma(c, p1, P.a22 * p2);
            p1 = np1; p2 = np2;
        }
    }
    if (act) {
        w.P12[j] = make_double2(myp1, myp2);
        w.QP12[j] = make_double2(2.0 * (P.q11 * myp1 + P.q12 * myp2), 2.0 * (P.q12 * myp1 + P.q22 * myp2));
        w.QE12[j] = make_double2(2.0 * (P.q11 * mye1 + P.q12 * mye2), 2.0 * (P.q12 * mye1 + P.q22 * mye2));
    }
    Gp::sync();
    double Fj = 0.0;
    if (act) {
        double accF = 0.0, accG = 0.0;
        const double2 *pp = w.P12, *qp = w.QP12 + j, *qe = w.QE12 + j;
        const int step = w.ldg + 1;
        double *grow = w.G + (N - 1) * w.ldg + (N - 1 - j);      // G[jj][ll], jj = N-1-m, ll = jj-j
        double *gcol = w.G + (N - 1 - j) * w.ldg + (N - 1);      // G[ll][jj]
        const int mmax = N - j;                                  // ll >= 0  <=>  m < N - j
        // One-warp groups: every lane runs N steps (QP12 / QE12 are zero beyond N, so the sums stop growing by
        // themselves) and only the stores are predicated: with the per-lane trip count N - j the warp ran the 4-deep
        // unrolled body AND a remainder loop (27.6 -> 27.0 ms on config 3).  Multi-warp groups keep their own count.
        const int mtrip = (GW == 1) ? N : mmax;
        for (int m = 0; m < mtrip; ++m) {
            const double2 p = pp[m], a = qp[m], e = qe[m];
            accF = fma(p.x, e.x, accF); accF = fma(p.y, e.y, accF);
            accG = fma(p.x, a.x, accG); accG = fma(p.y, a.y, accG);
            if (m < mmax) { *grow = accG; *gcol = accG; }
            grow -= step; gcol -= step;
        }
        Fj = accF;
    }
    Gp::sync();
    return Fj;
}

// ------------------------------------------------------------------------------------------------
// G, F by a row sweep over the dense Gamma -- any gamma_index (Rho_to_PhiGammaLambda.m:26-40).
// Thread j carries column j of Gamma down the rows (block(i,j) = A_k*block(i-1,j), k = i-j or i),
// publishes Q*block into a row buffer and accumulates G(j,l), l<=j, and F_j.  Gamma itself is
// never stored.  O(N^3/3) FMA pairs.
// ------------------------------------------------------------------------------------------------
template <int GW>
__device__ double build_GF_dense(int N, int j, const Work &w, const Params &P, int flags, double xF1, double xF2) {
    using Gp = Group<GW>;
    const bool act = j < N;
    const bool gi = (flags & NTM_PROFILE_GAMMA_I) != 0;
    double g1 = 0.0, g2 = 0.0, accF = 0.0, v1 = xF1, v2 = xF2;
    for (int i = 0; i < N; ++i) {
        const double a = w.a11s[i], c = w.a21s[i];
        const double nv1 = fma(a, v1, P.C1);
        const double nv2 = fma(P.a22, v2, fma(c, v1, P.C2));
        v1 = nv1; v2 = nv2;
        const double e1 = v1 - P.r1, e2 = v2 - P.r2;
        const double qe1 = P.q11 * e1 + P.q12 * e2, qe2 = P.q12 * e1 + P.q22 * e2;
        const bool on = act && j <= i;
        if (on) {
            if (j == i) { g1 = w.bbs[i]; g2 = 0.0; }
            else {
                const int k = gi ? i : (i - j - 1);
                const double aa = w.a11s[k], cc = w.a21s[k];
                const double n1 = aa * g1;
                const double n2 = fma(cc, g1, P.a22 * g2);
                g1 = n1; g2 = n2;
            }
            w.QP12[j] = make_double2(P.q11 * g1 + P.q12 * g2, P.q12 * g1 + P.q22 * g2);
            accF = fma(g1, qe1, fma(g2, qe2, accF));
        }
        Gp::sync();
        if (on) {
            double *row = w.G + j * w.ldg;
            if (j == i) { for (int l = 0; l <= j; ++l) { const double2 q = w.QP12[l]; row[l] = fma(g1, q.x, g2 * q.y); } }
            else { for (int l = 0; l <= j; ++l) { const double2 q = w.QP12[l]; row[l] += fma(g1, q.x, g2 * q.y); } }
        }
        Gp::sync();
    }
    if (act) {
        for (int l = 0; l <= j; ++l) {
            const double val = 2.0 * w.G[j * w.ldg + l];
            w.G[j * w.ldg + l] = val;
            w.G[l * w.ldg + j] = val;
        }
    }
    Gp::sync();
    return 2.0 * accF;
}

// mma.sync.aligned.m8n8k4 on the FP64 tensor cores (SASS: DMMA.8x8x4).  Fragments: A[row = lane>>2][col = lane&3],
// B[row = lane&3][col = lane>>2], C[row = lane>>2][cols 2*(lane&3), +1].
__device__ __forceinline__ void dmma_m8n8k4(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// ------------------------------------------------------------------------------------------------
// Dense Gamma on the tensor cores (one-warp groups, any Gamma index): lane j writes column j of Gamma into the
// group's staging tile by its recurrence (Rho_to_PhiGammaLambda.m:26-40), then G = 2 Gamma' Omega Gamma is formed
// tile by tile with DMMA (Omega = I (x) Q applied on the fly: the partner of row k is k^1) and F_j by a dot product
// with Omega (Phi x + Lambda - R).  ~600 warp instructions at N = 20 against ~4000 for the scalar row sweep.
// ------------------------------------------------------------------------------------------------
__device__ inline double build_GF_dense_dmma(int N, int j, const Work &w, const Params &P, int flags, double a11, double a21,
                                      double sE, double xF1, double xF2) {
    using Gp = Group<1>;
    const bool act = j < N;
    const bool gi = (flags & NTM_PROFILE_GAMMA_I) != 0;
    const int ldm = w.ldgam, Kp = (2 * N + 3) & ~3, nt = (N + 7) >> 3;
    // Omega (Phi x + Lambda - R) from the scan of the stage maps (as in the literal path)
    {
        Aff m;
        m.a = act ? a11 : 1.0; m.c = act ? a21 : 0.0;
        m.k1 = act ? P.C1 : 0.0; m.k2 = act ? P.C2 : 0.0;
        const Aff inc = aff_scan(m, j, N, P.a22);
        const double e1 = fma(inc.a, xF1, inc.k1) - P.r1;
        const double e2 = fma(inc.c, xF1, fma(sE * P.a22, xF2, inc.k2)) - P.r2;
        if (act) w.QE12[j] = make_double2(P.q11 * e1 + P.q12 * e2, P.q12 * e1 + P.q22 * e2);
    }
    if (act) {
        double *col = w.GamS + j * ldm;
        double g1 = 0.0, g2 = 0.0;
        for (int i = 0; i < N; ++i) {
            if (i == j) { g1 = w.bbs[j]; g2 = 0.0; }
            else if (i > j) {
                const int k = gi ? i : (i - j - 1);
                const double aa = w.a11s[k], cc = w.a21s[k];
                const double n2 = fma(cc, g1, P.a22 * g2);
                g1 = aa * g1; g2 = n2;
            }
            *reinterpret_cast<double2 *>(col + 2 * i) = make_double2(g1, g2);
        }
    }
    Gp::sync();
    double Fj = 0.0;
    if (act) {
        const double2 *cj = reinterpret_cast<const double2 *>(w.GamS + j * ldm);
        double f0 = 0.0, f1 = 0.0;
        for (int i = 0; i < N; ++i) { const double2 gm = cj[i], qe = w.QE12[i]; f0 = fma(gm.x, qe.x, f0); f1 = fma(gm.y, qe.y, f1); }
        Fj = 2.0 * (f0 + f1);
    }
    const int g = j >> 2, t4 = j & 3;
    const double qs = (t4 & 1) ? P.q22 : P.q11, q12 = P.q12;
    for (int tm = 0; tm < nt; ++tm) {
        for (int tn = 0; tn <= tm; ++tn) {
            const double *ap = w.GamS + (size_t)(tm * 8 + g) * ldm + t4;
            const double *bp = w.GamS + (size_t)(tn * 8 + g) * ldm + t4;
            const double *bq = w.GamS + (size_t)(tn * 8 + g) * ldm + (t4 ^ 1);
            double c0 = 0.0, c1 = 0.0;
#pragma unroll 2
            for (int k0 = 0; k0 < Kp; k0 += 4) {
                const double a = ap[k0];
                const double b = fma(qs, bp[k0], q12 * bq[k0]);
                dmma_m8n8k4(c0, c1, a, b);
            }
            const int r = tm * 8 + g, cc = tn * 8 + 2 * t4;
            if (r < N) {
                if (cc < N && cc <= r) { w.G[r * w.ldg + cc] = 2.0 * c0; w.G[cc * w.ldg + r] = 2.0 * c0; }
                if (cc + 1 < N && cc + 1 <= r) { w.G[r * w.ldg + cc + 1] = 2.0 * c1; w.G[(cc + 1) * w.ldg + r] = 2.0 * c1; }
            }
        }
    }
    Gp::sync();
    return Fj;
}

// ------------------------------------------------------------------------------------------------
// Dense Gamma on the tensor cores, multi-warp groups (33 <= N, ceil8(N + 1) <= 32 GW columns and <= NTM_DMAXT tiles per
// warp: N <= 63 for two warps, N <= 103 for four) -- BASELINE config 5's "dense Gamma'QGamma contraction on FP64 tensor
// cores" inside the fused loop (any Gamma index; round 1 ran the scalar row sweep build_GF_dense here).  Thread c carries
// column c of Gamma down the rows by its recurrence (Rho_to_PhiGammaLambda.m:26-40), thread N the vector
// v = Phi x + Lambda - R (:20-22, 49-52; NTM_MPC_Sim.m:121), eight stages (16 rows) at a time into the chunk buffer; the
// warps then contract the chunk, G += Gamma_chunk' Omega Gamma_chunk, on 8 x 8 tiles of the lower triangle with
// mma.sync.m8n8k4.f64 (Omega applied to the B fragment on the fly: the partner row of a (w, omega) pair is k ^ 1).
// Accumulators stay in registers over all chunks (2 doubles per tile and lane); row N of the product is F.
// ------------------------------------------------------------------------------------------------
#define NTM_DMAXT 23
template <int GW>
__device__ double build_GF_dense_dmma_long(int N, int j, const Work &w, const Params &P, int flags, double xF1, double xF2) {
    using Gp = Group<GW>;
    constexpr int T = Gp::T;
    const bool gi = (flags & NTM_PROFILE_GAMMA_I) != 0;
    const int Np = (N + 1 + 7) & ~7, nt = Np >> 3, ntile = nt * (nt + 1) / 2;
    const int lane = j & 31, wid = j >> 5, g = lane >> 2, t4 = lane & 3;
    const int dpart = (t4 ^ 1) - t4;
    const double qs = (t4 & 1) ? P.q22 : P.q11, q12 = P.q12;
    double *__restrict__ Gs = w.GamS;
    double acc[NTM_DMAXT][2];
#pragma unroll
    for (int q = 0; q < NTM_DMAXT; ++q) { acc[q][0] = 0.0; acc[q][1] = 0.0; }
    double g1 = 0.0, g2 = 0.0;                               // this thread's column of Gamma (j < N) ...
    double v1 = xF1, v2 = xF2;                               // ... or the free response (j == N)
    for (int i0 = 0; i0 < N; i0 += NTM_DCH / 2) {
        Gp::sync();                                          // the previous chunk has been contracted
        if (j < Np) {
            double *col = Gs + (size_t)j * NTM_DLD;
#pragma unroll
            for (int ii = 0; ii < NTM_DCH / 2; ++ii) {
                const int i = i0 + ii;
                double o1 = 0.0, o2 = 0.0;
                if (i < N) {
                    if (j < N) {
                        if (i == j) { g1 = w.bbs[j]; g2 = 0.0; }
                        else if (i > j) {
                            const int k = gi ? i : (i - j - 1);
                            const double aa = w.a11s[k], cc = w.a21s[k];
                            const double n2 = fma(cc, g1, P.a22 * g2);
                            g1 = aa * g1; g2 = n2;
                        }
                        o1 = g1; o2 = g2;
                    } else if (j == N) {
                        const double aa = w.a11s[i], cc = w.a21s[i];
                        const double nv1 = fma(aa, v1, P.C1);
                        const double nv2 = fma(P.a22, v2, fma(cc, v1, P.C2));
                        v1 = nv1; v2 = nv2;
                        o1 = v1 - P.r1; o2 = v2 - P.r2;
                    }
                }
                *reinterpret_cast<double2 *>(col + 2 * ii) = make_double2(o1, o2);
            }
        }
        Gp::sync();
#pragma unroll
        for (int q = 0; q < NTM_DMAXT; ++q) {
            const int t = wid + GW * q;
            if (t < ntile) {
                int tm = 0, rem = t;
                while (rem > tm) { rem -= tm + 1; ++tm; }
                const double *ap = Gs + (size_t)(8 * tm + g) * NTM_DLD + t4;
                const double *bp = Gs + (size_t)(8 * rem + g) * NTM_DLD + t4;
#pragma unroll
                for (int k0 = 0; k0 < NTM_DCH; k0 += 4) {
                    const double a = ap[k0];
                    const double b = fma(qs, bp[k0], q12 * bp[k0 + dpart]);
                    dmma_m8n8k4(acc[q][0], acc[q][1], a, b);
                }
            }
        }
    }
    Gp::sync();
    // G (both triangles, exactly symmetric) and F out of the accumulators; F travels through w.sol
#pragma unroll
    for (int q = 0; q < NTM_DMAXT; ++q) {
        const int t = wid + GW * q;
        if (t < ntile) {
            int tm = 0, rem = t;
            while (rem > tm) { rem -= tm + 1; ++tm; }
            const int r = 8 * tm + g, cc = 8 * rem + 2 * t4;
            const double v0 = 2.0 * acc[q][0], v1o = 2.0 * acc[q][1];
            if (r < N) {
                if (cc < N && cc <= r) { w.G[r * w.ldg + cc] = v0; w.G[cc * w.ldg + r] = v0; }
                if (cc + 1 < N && cc + 1 <= r) { w.G[r * w.ldg + cc + 1] = v1o; w.G[(cc + 1) * w.ldg + r] = v1o; }
            } else if (r == N) {
                if (cc < N) w.sol[cc] = v0;
                if (cc + 1 < N) w.sol[cc + 1] = v1o;
            }
        }
    }
    Gp::sync();
    const double Fj = (j < N) ? w.sol[j] : 0.0;
    Gp::sync();
    return Fj;
}

// DENSE is a compile-time property of the kernel instantiation (the launcher picks it from the profile bits), so the
// literal kernel carries no dense-Gamma code at all and vice versa (instruction-cache footprint of the hot loop).
template <int GW, bool DENSE>
__device__ __forceinline__ double build_GF(int N, int j, const Work &w, const Params &P, int flags, double a11,
                                           double a21, double sE, double xF1, double xF2) {
    if constexpr (DENSE) {
        if constexpr (GW == 1) {
            if (w.GamS != nullptr) return build_GF_dense_dmma(N, j, w, P, flags, a11, a21, sE, xF1, xF2);
        } else {
            if (w.GamS != nullptr) return build_GF_dense_dmma_long<GW>(N, j, w, P, flags, xF1, xF2);
        }
        return build_GF_dense<GW>(N, j, w, P, flags, xF1, xF2);
    } else {
        return build_GF_toeplitz<GW>(N, j, w, P, a11, a21, sE, xF1, xF2);
    }
}

}  // namespace ntm
