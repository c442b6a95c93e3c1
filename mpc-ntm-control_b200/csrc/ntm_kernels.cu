// ntm_kernels.cu -- hand-written sm_100a kernels of the LPV-MPC hot path and their launchers.
//
//   closed_loop_kernel<GW>   NTM_MPC_Sim.m:63-73 + 80-131, fused and persistent: one group of GW warps per
//                            scenario pulls scenarios from a work queue and keeps rho, G, F, U and the QP
//                            partition on chip for all k_sim steps; HBM sees x0/params in and xk/uk/... out.
//   condense_kernel<GW>      Rho_to_PhiGammaLambda.m, materialising Phi/Gamma/Lambda (HBM-write bound).
//   hessian_grad_kernel<GW>  NTM_MPC_Sim.m:72-73 for arbitrary dense Phi/Gamma/Lambda.
//   qp_box_kernel<GW>        NTM_MPC_Sim.m:97 (box rows only) for arbitrary SPD G.
//   rho/lpv/plant kernels    rho1-3.m, A.m, B.m, NTM_MPC_Sim.m:130, one thread per scenario.
#include <climits>
#include <cstdint>
#include <cstdlib>
#include <map>
#include <mutex>
#include <tuple>
#include <utility>
#include <vector>
#include "ntm_device.cuh"
#include "ntm_kernels.h"
#include "ntm_loop.cuh"

namespace ntm {

// =================================================================================================
// elementwise kernels (one thread per scenario)
// =================================================================================================
__global__ void rho_kernel(int layout, int flags, int S, const double *__restrict__ x,
                           const double *__restrict__ params, int pc, double *__restrict__ r1o,
                           double *__restrict__ r2o, double *__restrict__ r3o) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const Params P = load_params(params, layout, pc, s);
    const double w = x[elem(layout, S, 2, s, 0)], om = x[elem(layout, S, 2, s, 1)];
    double r1, r2, r3;
    rho_of(P, flags, w, om, r1, r2, r3);
    r1o[s] = r1; r2o[s] = r2; r3o[s] = r3;
}

__global__ void lpv_kernel(int layout, int S, const double *__restrict__ r1, const double *__restrict__ r2,
                           const double *__restrict__ r3, const double *__restrict__ params, int pc,
                           double *__restrict__ A, double *__restrict__ B) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const Params P = load_params(params, layout, pc, s);
    double a11, a21, b;
    lpv_of(P, r1[s], r2[s], r3[s], a11, a21, b);
    A[elem(layout, S, 4, s, 0)] = a11;
    A[elem(layout, S, 4, s, 1)] = a21;
    A[elem(layout, S, 4, s, 2)] = 0.0;
    A[elem(layout, S, 4, s, 3)] = P.a22;
    B[elem(layout, S, 2, s, 0)] = b;
    B[elem(layout, S, 2, s, 1)] = 0.0;
}

// RK4 as a template parameter (keeps the option's code out of the Euler kernel).  ncu: DRAM traffic is 152 B per
// scenario -- the whole 128-byte parameter line comes in although the plant needs 8 of its 16 doubles -- at 5.2 TB/s,
// 80 % of the copy peak; more resident CTAs (40 registers, 6 per SM) measured slower (69 % against 77 %).
template <bool RK4>
__global__ void __launch_bounds__(256, 4)
plant_kernel(int layout, int flags, int S, const double *__restrict__ x, const double *__restrict__ u,
             const double *__restrict__ params, int pc, double *__restrict__ xn) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const Params P = load_params(params, layout, pc, s);
    double nw, nom;
    const double w = x[elem(layout, S, 2, s, 0)], om = x[elem(layout, S, 2, s, 1)];
    if constexpr (RK4) {                                 // the cold options: RK4 and / or tau_E(w)
        const double ctau = (flags & NTM_PROFILE_TAUE_W)
                                ? __ldg(params + elem(layout, pc == 1 ? 1 : pc, NTM_NPARAM, pc == 1 ? 0 : s, 15)) : 0.0;
        plant_exact(P, flags, P.a22, ctau, w, om, u[s], nw, nom);   // the fused loop's rounding (ntm_loop.cuh)
    } else plant_euler(P, flags, w, om, u[s], nw, nom);
    xn[elem(layout, S, 2, s, 0)] = nw;
    xn[elem(layout, S, 2, s, 1)] = nom;
}

// =================================================================================================
// getWLc.m: L = Mcal*Gamma + Ecal, W = -Dcal - Mcal*Phi, c = Ccal - Mcal*Lambda.  Mcal/Ecal/Dcal are sign/selection
// matrices, so every output row is +-(one row of Gamma/Phi/Lambda) or a constant: a pure gather, one thread per
// output element, HBM-bound.  Row r = 6*i + q for stage i < N (q: -u, +u, -x1, -x2, +x1, +x2), then 4 terminal rows.
// =================================================================================================
struct WLcBounds { double xmax1, xmax2, xmin1, xmin2, umax, umin; };

// element (r, col) of scenario s: col 0..N-1 = L, N..N+1 = W, N+2 = c
__device__ __forceinline__ void wlc_element(int layout, int S, int N, int R, const WLcBounds &b, const double *__restrict__ Gam,
                                            const double *__restrict__ Phi, const double *__restrict__ Lam,
                                            double *__restrict__ W, double *__restrict__ L, double *__restrict__ c, int s,
                                            int col, int r) {
    // which state row of X = [x_1; ...; x_N] this constraint row looks at (xb < 0: none), with which sign
    int i, q, xb = -1, comp = 0;
    double sgn = 0.0, cc;
    if (r < 6 * N) {
        i = r / 6; q = r - 6 * i;
        if (q >= 2) { comp = (q - 2) & 1; sgn = (q < 4) ? -1.0 : 1.0; xb = i - 1; }     // block 0 constrains x_0 itself
        cc = (q == 0) ? -b.umin : (q == 1) ? b.umax : (q == 2) ? -b.xmin1 : (q == 3) ? -b.xmin2 : (q == 4) ? b.xmax1 : b.xmax2;
    } else {
        i = N; q = r - 6 * N;
        comp = q & 1; sgn = (q < 2) ? -1.0 : 1.0; xb = N - 1;
        cc = (q == 0) ? -b.xmin1 : (q == 1) ? -b.xmin2 : (q == 2) ? b.xmax1 : b.xmax2;
    }
    if (col < N) {                                            // L
        double v = (xb >= 0) ? sgn * Gam[elem(layout, S, 2 * N * N, s, col * 2 * N + 2 * xb + comp)] : 0.0;
        if (r < 6 * N && col == i) { if (q == 0) v += -1.0; else if (q == 1) v += 1.0; }   // Ecal
        L[elem(layout, S, R * N, s, col * R + r)] = (v == 0.0) ? 0.0 : v;   // -1 * 0 above the diagonal: +0, like the other kernels
    } else if (col < N + 2) {                                 // W = -Dcal - Mcal*Phi
        const int wc = col - N;
        double v = (xb >= 0) ? -sgn * Phi[elem(layout, S, 4 * N, s, wc * 2 * N + 2 * xb + comp)] : 0.0;
        if (r < 6 && q >= 2 && comp == wc) v += -sgn;         // -Dcal: Mi acts on x_0 in block 0
        W[elem(layout, S, R * 2, s, wc * R + r)] = (v == 0.0) ? 0.0 : v;
    } else {                                                  // c = Ccal - Mcal*Lambda
        const double v = (xb >= 0) ? cc - sgn * Lam[elem(layout, S, 2 * N, s, 2 * xb + comp)] : cc;
        c[elem(layout, S, R, s, r)] = v;
    }
}

__global__ void getwlc_kernel(int layout, int S, int N, WLcBounds b, const double *__restrict__ Gam,
                              const double *__restrict__ Phi, const double *__restrict__ Lam, double *__restrict__ W,
                              double *__restrict__ L, double *__restrict__ c) {
    const int R = 6 * N + 4;
    const int per = R * (N + 3);                                  // L (N cols) + W (2 cols) + c (1 col) per scenario
    // one CTA per scenario (grid-stride); (col, r) advance by running counters: no integer division per element
    for (int s = blockIdx.x; s < S; s += gridDim.x)
    for (int e = threadIdx.x, col = (int)threadIdx.x / R, r = (int)threadIdx.x - col * R; e < per; e += blockDim.x) {
        if (e != (int)threadIdx.x) { r += blockDim.x; while (r >= R) { r -= R; ++col; } }
        wlc_element(layout, S, N, R, b, Gam, Phi, Lam, W, L, c, s, col, r);
    }
}

// SoA layout (scenario index fastest): thread = scenario (so every warp access is 256 contiguous bytes), blockIdx.y =
// one (column, stage) pair: two loads of the Gamma/Phi/Lambda block row, the stage's six constraint rows out.  (Round 1
// let one thread walk all (N+3)(6N+4) elements of its scenario through the generic per-element routine: ~40 instructions
// per element and 14 warps per SM in flight -- 34 % of the copy peak.)  Same values, bit for bit.
__global__ void __launch_bounds__(128)
getwlc_soa_kernel(int S, int N, WLcBounds b, const double *__restrict__ Gam, const double *__restrict__ Phi,
                  const double *__restrict__ Lam, double *__restrict__ W, double *__restrict__ L, double *__restrict__ c) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int R = 6 * N + 4;
    const size_t Ss = (size_t)S;
    const int col = (int)blockIdx.y / (N + 1), i = (int)blockIdx.y - col * (N + 1);    // stage N = the 4 terminal rows
    const int xb = (i == 0) ? -1 : (i - 1);
    double x1 = 0.0, x2 = 0.0, sc = 1.0;
    double *dst;
    if (col < N) {
        if (xb >= 0) { x1 = __ldg(Gam + ((size_t)col * 2 * N + 2 * xb) * Ss + s); x2 = __ldg(Gam + ((size_t)col * 2 * N + 2 * xb + 1) * Ss + s); }
        dst = L + (size_t)col * R * Ss + s;
    } else if (col < N + 2) {
        if (xb >= 0) { x1 = __ldg(Phi + ((size_t)(col - N) * 2 * N + 2 * xb) * Ss + s); x2 = __ldg(Phi + ((size_t)(col - N) * 2 * N + 2 * xb + 1) * Ss + s); }
        dst = W + (size_t)(col - N) * R * Ss + s; sc = -1.0;
    } else {
        if (xb >= 0) { x1 = __ldg(Lam + (size_t)(2 * xb) * Ss + s); x2 = __ldg(Lam + (size_t)(2 * xb + 1) * Ss + s); }
        dst = c + s; sc = -1.0;
    }
    const double m1 = sc * x1, m2 = sc * x2;
    double lo1 = -m1, lo2 = -m2, hi1 = m1, hi2 = m2, u1 = 0.0, u2 = 0.0;
    if (col < N) {
        if (i < N && col == i) { u1 = -1.0; u2 = 1.0; }                                   // Ecal
    } else if (col < N + 2) {
        if (i == 0) {                                                                      // -Dcal: block 0 constrains x_0
            const int wc = col - N;
            lo1 = wc == 0 ? 1.0 : 0.0; lo2 = wc == 1 ? 1.0 : 0.0; hi1 = wc == 0 ? -1.0 : 0.0; hi2 = wc == 1 ? -1.0 : 0.0;
        }
    } else {
        u1 = -b.umin; u2 = b.umax;
        lo1 = -b.xmin1 + lo1; lo2 = -b.xmin2 + lo2; hi1 = b.xmax1 + hi1; hi2 = b.xmax2 + hi2;
    }
    if (lo1 == 0.0) lo1 = 0.0; if (lo2 == 0.0) lo2 = 0.0; if (hi1 == 0.0) hi1 = 0.0; if (hi2 == 0.0) hi2 = 0.0;   // +0, like the other paths
    if (i < N) {
        double *d = dst + (size_t)(6 * i) * Ss;
        d[0] = u1; d[Ss] = u2; d[2 * Ss] = lo1; d[3 * Ss] = lo2; d[4 * Ss] = hi1; d[5 * Ss] = hi2;
    } else {
        double *d = dst + (size_t)(6 * N) * Ss;
        d[0] = lo1; d[Ss] = lo2; d[2 * Ss] = hi1; d[3 * Ss] = hi2;
    }
}

// MATLAB layout, 16-byte aligned: one thread per (column, stage) writes the stage's six constraint rows as three
// double2 stores from ONE double2 load of the Gamma/Phi/Lambda block row -- ~2.5 instructions per output element
// instead of ~40 in the generic per-element kernel above.  Column index: 0..N-1 = L, N..N+1 = W, N+2 = c.
__global__ void __launch_bounds__(256)
getwlc_vec_kernel(int S, int N, WLcBounds b, const double *__restrict__ Gam, const double *__restrict__ Phi,
                  const double *__restrict__ Lam, double *__restrict__ W, double *__restrict__ L, double *__restrict__ c) {
    const int R = 6 * N + 4, NC = N + 3;
    const int per = NC * (N + 1);                                  // (column, stage) pairs; stage N = the 4 terminal rows
    for (int s = blockIdx.x; s < S; s += gridDim.x) {
        const double *gam = Gam + (size_t)s * 2 * N * N, *phi = Phi + (size_t)s * 4 * N, *lam = Lam + (size_t)s * 2 * N;
        for (int e = threadIdx.x, col = (int)threadIdx.x / (N + 1), i = (int)threadIdx.x - col * (N + 1); e < per; e += blockDim.x) {
            if (e != (int)threadIdx.x) { i += blockDim.x; while (i > N) { i -= N + 1; ++col; } }
            // the block row of X = [x_1..x_N] this stage constrains: stage 0 constrains x_0 itself (none), stage i>0 x_i, terminal x_N
            const int xb = (i == 0) ? -1 : (i - 1);
            double2 xr = make_double2(0.0, 0.0);                  // the two entries (w, omega rows) of that block row in this column
            double *dst;
            double sc = 1.0;                                       // W and c carry Mcal with a minus sign
            if (col < N) {
                if (xb >= 0) xr = __ldg(reinterpret_cast<const double2 *>(gam + (size_t)col * 2 * N + 2 * xb));
                dst = L + (size_t)s * R * N + (size_t)col * R;
            } else if (col < N + 2) {
                if (xb >= 0) xr = __ldg(reinterpret_cast<const double2 *>(phi + (size_t)(col - N) * 2 * N + 2 * xb));
                dst = W + (size_t)s * R * 2 + (size_t)(col - N) * R; sc = -1.0;
            } else {
                if (xb >= 0) xr = __ldg(reinterpret_cast<const double2 *>(lam + 2 * xb));
                dst = c + (size_t)s * R; sc = -1.0;
            }
            const double m1 = sc * xr.x, m2 = sc * xr.y;           // +-(Mcal-selected entries): rows are [-x; +x]
            double2 lo, hi, uu = make_double2(0.0, 0.0);
            lo = make_double2(-m1, -m2); hi = make_double2(m1, m2);
            if (col < N) {
                if (i < N && col == i) uu = make_double2(-1.0, 1.0);                      // Ecal
            } else if (col < N + 2) {
                if (i == 0) {                                      // -Dcal: block 0 constrains x_0
                    const int wc = col - N;
                    lo = make_double2(wc == 0 ? 1.0 : 0.0, wc == 1 ? 1.0 : 0.0);
                    hi = make_double2(wc == 0 ? -1.0 : 0.0, wc == 1 ? -1.0 : 0.0);
                }
            } else {
                uu = make_double2(-b.umin, b.umax);
                lo = make_double2(-b.xmin1 + lo.x, -b.xmin2 + lo.y); hi = make_double2(b.xmax1 + hi.x, b.xmax2 + hi.y);
            }
            // exact zeros instead of -0.0 where nothing is selected (matches the per-element kernel bit for bit)
            if (lo.x == 0.0) lo.x = 0.0; if (lo.y == 0.0) lo.y = 0.0; if (hi.x == 0.0) hi.x = 0.0; if (hi.y == 0.0) hi.y = 0.0;
            if (i < N) {
                double2 *d2 = reinterpret_cast<double2 *>(dst + 6 * i);
                d2[0] = uu; d2[1] = lo; d2[2] = hi;
            } else {
                double2 *d2 = reinterpret_cast<double2 *>(dst + 6 * N);
                d2[0] = lo; d2[1] = hi;
            }
        }
    }
}

cudaError_t launch_getwlc(cudaStream_t st, const DeviceProps &dp, int layout, int S, int N, const double *bounds,
                          const double *Gam, const double *Phi, const double *Lam, double *W, double *L, double *c,
                          long long *launches) {
    if (S <= 0) return cudaSuccess;
    WLcBounds b = {bounds[0], bounds[1], bounds[2], bounds[3], bounds[4], bounds[5]};
    const long long cap = (long long)dp.sm_count * 64;
    const bool aligned = ((reinterpret_cast<uintptr_t>(Gam) | reinterpret_cast<uintptr_t>(Phi) | reinterpret_cast<uintptr_t>(Lam) |
                           reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(L) | reinterpret_cast<uintptr_t>(c)) & 15) == 0;
    if (layout == NTM_LAYOUT_MATLAB && aligned)
        getwlc_vec_kernel<<<(int)(S < cap ? S : cap), 256, 0, st>>>(S, N, b, Gam, Phi, Lam, W, L, c);
    else if (layout == NTM_LAYOUT_SOA)
        getwlc_soa_kernel<<<dim3((unsigned)((S + 127) / 128), (unsigned)((N + 3) * (N + 1))), 128, 0, st>>>(S, N, b, Gam, Phi, Lam, W, L, c);
    else
        getwlc_kernel<<<(int)(S < cap ? S : cap), 256, 0, st>>>(layout, S, N, b, Gam, Phi, Lam, W, L, c);
    ++*launches;
    return cudaGetLastError();
}

// =================================================================================================
// box QP on caller-supplied G, F
// =================================================================================================
template <int GW>
__global__ void __launch_bounds__(GW == 1 ? 256 : 32 * GW)
qp_box_kernel(int layout, int S, int N, const double *__restrict__ G, const double *__restrict__ F,
              const double *__restrict__ lb, const double *__restrict__ ub, int bc, double *__restrict__ U,
              int *__restrict__ iters, int *__restrict__ status, unsigned int *counter, unsigned int gbytes,
              double *hscratch, int hcap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using Gp = Group<GW>;
    const int gib = (GW == 1) ? (int)(threadIdx.x >> 5) : 0;
    const int j = (GW == 1) ? (int)(threadIdx.x & 31) : (int)threadIdx.x;
    const int gpb = (GW == 1) ? (int)(blockDim.x >> 5) : 1;
    double *hbig = hscratch + ((size_t)blockIdx.x * gpb + gib) * N * odd_ld(N);
    const Work w = carve(smem_raw + (size_t)gib * gbytes, N, hcap, hbig);
    for (;;) {
        int s = 0;
        if (j == 0) s = (int)atomicAdd(counter, 1u);
        s = Gp::bcast0(s, w.ired);
        if (s >= S) break;
        for (int e = j; e < N * N; e += Gp::T) {
            const int col = e / N, row = e - col * N;
            w.G[row * w.ldg + col] = G[elem(layout, S, N * N, s, e)];
        }
        double Fj = 0.0, lbj = 0.0, ubj = 0.0;
        if (j < N) {
            Fj = F[elem(layout, S, N, s, j)];
            const int sb = (bc == 1) ? 0 : s, Sb = (bc == 1) ? 1 : S;
            lbj = lb[elem(layout, Sb, N, sb, j)];
            ubj = ub[elem(layout, Sb, N, sb, j)];
        }
        Gp::sync();
        int nit = 0;
        double Uj = 0.0;
        QpHist hist = {0.0, 0.0, -1, -1, 0};
        const int st = qp_solve<GW>(N, j, w, Fj, lbj, ubj, hist, Uj, 10 * N + 20, nit);
        if (j < N) U[elem(layout, S, N, s, j)] = Uj;
        if (j == 0) {
            if (iters) iters[s] = nit;
            if (status) status[s] = st;
        }
        Gp::sync();
    }
    if (j == 0) {
        const unsigned int groups = gridDim.x * ((GW == 1) ? (blockDim.x >> 5) : 1);
        __threadfence();
        if (atomicAdd(counter + 1, 1u) == groups - 1) { counter[0] = 0u; counter[1] = 0u; __threadfence(); }
    }
}

// =================================================================================================
// NTM_MPC_Sim.m:97 with the state rows of getWLc.m kept: box QP + M general rows per scenario.
// =================================================================================================
template <int GW>
__global__ void __launch_bounds__(GW == 1 ? 128 : 32 * GW)
qp_ineq_kernel(int layout, int S, int N, int M, const double *__restrict__ G, const double *__restrict__ F,
               const double *__restrict__ lb, const double *__restrict__ ub, int bc, const double *__restrict__ Lg,
               const double *__restrict__ bg, double *__restrict__ U, int *__restrict__ iters,
               int *__restrict__ status, unsigned int *counter, unsigned int gbytes, unsigned int wbytes) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using Gp = Group<GW>;
    const int gib = (GW == 1) ? (int)(threadIdx.x >> 5) : 0;
    const int j = (GW == 1) ? (int)(threadIdx.x & 31) : (int)threadIdx.x;
    const Work w = carve(smem_raw + (size_t)gib * gbytes, N, N, nullptr);
    const IneqWork q = carve_ineq(smem_raw + (size_t)gib * gbytes + wbytes, N, M);
    for (;;) {
        int s = 0;
        if (j == 0) s = (int)atomicAdd(counter, 1u);
        s = Gp::bcast0(s, w.ired);
        if (s >= S) break;
        for (int e = j; e < N * N; e += Gp::T) {
            const int col = e / N, row = e - col * N;
            w.G[row * w.ldg + col] = G[elem(layout, S, N * N, s, e)];
        }
        double Fj = 0.0, lbj = 0.0, ubj = 0.0;
        if (j < N) {
            Fj = F[elem(layout, S, N, s, j)];
            const int sb = (bc == 1) ? 0 : s, Sb = (bc == 1) ? 1 : S;
            lbj = lb[elem(layout, Sb, N, sb, j)];
            ubj = ub[elem(layout, Sb, N, sb, j)];
        }
        Gp::sync();
        int nit = 0;
        double Uj = 0.0;
        QpHist hist = {0.0, 0.0, -1, -1, 0};
        int st = qp_solve<GW>(N, j, w, Fj, lbj, ubj, hist, Uj, 10 * N + 20, nit);
        if (st == NTM_SCN_OK && M > 0)
        {
            const GlobalRows rows = {Lg, bg, layout, S, s, M, N};
            const auto regen = make_regen([&]() {              // the Hessian comes back from global memory
                for (int e = j; e < N * N; e += Gp::T) {
                    const int col = e / N, row = e - col * N;
                    w.G[row * w.ldg + col] = G[elem(layout, S, N * N, s, e)];
                }
            });
            st = qp_ineq_continue<GW>(N, rows, j, w, q, Fj, lbj, ubj, Uj, nit + 20 * (N + M) + 50, nit, nullptr, regen);
        }
        if (j < N) U[elem(layout, S, N, s, j)] = Uj;
        if (j == 0) {
            if (iters) iters[s] = nit;
            if (status) status[s] = st;
        }
        Gp::sync();
    }
    if (j == 0) {
        const unsigned int groups = gridDim.x * ((GW == 1) ? (blockDim.x >> 5) : 1);
        __threadfence();
        if (atomicAdd(counter + 1, 1u) == groups - 1) { counter[0] = 0u; counter[1] = 0u; __threadfence(); }
    }
}

// =================================================================================================
// materialising condensation: Rho -> Phi, Gamma, Lambda
// =================================================================================================
#define NTM_COND_RC 16        // block rows per staged chunk of the index-i Gamma on long horizons (power of two)
template <int GW>
__global__ void __launch_bounds__(GW == 1 ? 256 : 32 * GW)
condense_kernel(int layout, int flags, int S, int N, const double *__restrict__ R1, const double *__restrict__ R2,
                const double *__restrict__ R3, const double *__restrict__ params, int pc, double *__restrict__ Phi,
                double *__restrict__ Gam, double *__restrict__ Lam, int vec_ok, int stage_tiles) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using Gp = Group<GW>;
    const int gpb = (GW == 1) ? (int)(blockDim.x >> 5) : 1;
    const int gib = (GW == 1) ? (int)(threadIdx.x >> 5) : 0;
    const int j = (GW == 1) ? (int)(threadIdx.x & 31) : (int)threadIdx.x;
    double *a11s = reinterpret_cast<double *>(smem_raw) + (size_t)gib * 4 * N;     // 4N keeps every warp's slice 16-byte aligned
    double *a21s = a11s + N, *bbs = a21s + N;
    const bool gi = (flags & NTM_PROFILE_GAMMA_I) != 0;
    const bool act = j < N;
    double2 *stage = stage_tiles ? reinterpret_cast<double2 *>(reinterpret_cast<double *>(smem_raw) + (size_t)gpb * 4 * N) : nullptr;
    if constexpr (GW == 1) {
        // Literal Gamma, MATLAB layout, one warp per scenario: Gamma(i,c) = b_c * p_{i-c} (Toeplitz in the block index),
        // Phi_i / Lambda_i / p_i all come out of ONE warp scan of the stage maps, and every output array is then
        // written with consecutive 16-byte stores per lane (full 512-byte lines per warp instruction).
        if (!gi && vec_ok) {
            double2 *P12 = reinterpret_cast<double2 *>(a11s);      // reuses a11s/a21s (2N doubles, 16-byte aligned)
            for (int s = blockIdx.x * gpb + gib; s < S; s += gridDim.x * gpb) {
                const Params P = load_params(params, layout, pc, s);
                Aff m;
                double b = 0.0;
                m.a = 1.0; m.c = 0.0; m.k1 = 0.0; m.k2 = 0.0;
                if (act) {
                    lpv_of(P, __ldg(R1 + (size_t)s * N + j), __ldg(R2 + (size_t)s * N + j), __ldg(R3 + (size_t)s * N + j),
                           m.a, m.c, b);
                    m.k1 = P.C1; m.k2 = P.C2;
                }
                const Aff inc = aff_scan(m, j, N, P.a22);
                const Aff exc = aff_exclusive(inc, j);
                double sI = P.a22;
                for (int t = 0; t < j && t < N; ++t) sI *= P.a22;    // a22^(j+1)
                __syncwarp();
                if (act) {
                    P12[j] = make_double2(exc.a, exc.c);
                    bbs[j] = b;
                    double2 *phi = reinterpret_cast<double2 *>(Phi + (size_t)s * 4 * N);
                    phi[j] = make_double2(inc.a, inc.c);
                    phi[N + j] = make_double2(0.0, sI);
                    reinterpret_cast<double2 *>(Lam + (size_t)s * 2 * N)[j] = make_double2(inc.k1, inc.k2);
                }
                __syncwarp();
                double2 *gam = reinterpret_cast<double2 *>(Gam + (size_t)s * 2 * N * N);
                int c = j / N, i = j - c * N;                       // block t = c*N + i, t = j, j+32, ...
                const int dc = 32 / N, di = 32 - dc * N;
                for (int t = j; t < N * N; t += 32) {
                    double2 v = make_double2(0.0, 0.0);
                    if (i >= c) {
                        const double2 p = P12[i - c];
                        const double bc = bbs[c];
                        v = make_double2(bc * p.x, bc * p.y);
                    }
                    gam[t] = v;
                    c += dc; i += di;
                    if (i >= N) { i -= N; ++c; }
                }
            }
            return;
        }
        if (gi && vec_ok && stage != nullptr) {
            // Gamma(i,c) = A_i * Gamma(i-1,c) has no Toeplitz structure: lane c runs its column recurrence into a
            // per-warp staging tile of this CTA, then the warp copies the tile out with consecutive 16-byte stores.
            double2 *tile = stage + (size_t)gib * N * N;
            for (int s = blockIdx.x * gpb + gib; s < S; s += gridDim.x * gpb) {
                const Params P = load_params(params, layout, pc, s);
                Aff m;
                double b = 0.0;
                m.a = 1.0; m.c = 0.0; m.k1 = 0.0; m.k2 = 0.0;
                if (act) {
                    lpv_of(P, __ldg(R1 + (size_t)s * N + j), __ldg(R2 + (size_t)s * N + j), __ldg(R3 + (size_t)s * N + j),
                           m.a, m.c, b);
                    m.k1 = P.C1; m.k2 = P.C2;
                }
                const Aff inc = aff_scan(m, j, N, P.a22);
                double sI = P.a22;
                for (int t = 0; t < j && t < N; ++t) sI *= P.a22;
                __syncwarp();
                if (act) {
                    a11s[j] = m.a; a21s[j] = m.c;
                    double2 *phi = reinterpret_cast<double2 *>(Phi + (size_t)s * 4 * N);
                    phi[j] = make_double2(inc.a, inc.c);
                    phi[N + j] = make_double2(0.0, sI);
                    reinterpret_cast<double2 *>(Lam + (size_t)s * 2 * N)[j] = make_double2(inc.k1, inc.k2);
                }
                __syncwarp();
                if (act) {
                    double g1 = 0.0, g2 = 0.0;
                    for (int i = 0; i < N; ++i) {
                        if (i == j) { g1 = b; g2 = 0.0; }
                        else if (i > j) {
                            const double aa = a11s[i], cc = a21s[i];
                            const double n2 = fma(cc, g1, P.a22 * g2);
                            g1 = aa * g1; g2 = n2;
                        }
                        tile[j * N + i] = make_double2(g1, g2);
                    }
                }
                __syncwarp();
                double2 *gam = reinterpret_cast<double2 *>(Gam + (size_t)s * 2 * N * N);
                for (int t = j; t < N * N; t += 32) gam[t] = tile[t];
            }
            return;
        }
    } else {
        // Same idea for long horizons (one CTA per scenario): the prefix products come from the serial chain every
        // thread runs redundantly (N cheap steps against 2N^2 doubles to write), then the whole CTA generates Gamma in
        // output order with 16-byte stores.
        if (!gi && vec_ok) {
            double2 *P12 = reinterpret_cast<double2 *>(a11s);
            const int T = 32 * GW;
            for (int s = blockIdx.x; s < S; s += gridDim.x) {
                const Params P = load_params(params, layout, pc, s);
                double a11 = 1.0, a21 = 0.0, b = 0.0;
                __syncthreads();                                     // previous scenario's readers are done with P12 / bbs
                if (act) {
                    lpv_of(P, __ldg(R1 + (size_t)s * N + j), __ldg(R2 + (size_t)s * N + j), __ldg(R3 + (size_t)s * N + j), a11, a21, b);
                    P12[j] = make_double2(a11, a21);                // stage entries first, replaced by the prefix below
                    bbs[j] = b;
                }
                __syncthreads();
                double f11 = 1.0, f21 = 0.0, f22 = 1.0, l1 = 0.0, l2 = 0.0;      // Phi_i (lower triangular), Lambda_i
                double e11 = 1.0, e21 = 0.0, m11 = 0, m21 = 0, m22 = 0, ml1 = 0, ml2 = 0;
                for (int i = 0; i < N; ++i) {
                    const double2 ac = P12[i];
                    if (i == j) { e11 = f11; e21 = f21; }            // exclusive prefix: p_j
                    const double n21 = fma(ac.y, f11, P.a22 * f21);
                    f11 = ac.x * f11; f21 = n21; f22 = P.a22 * f22;
                    const double nl2 = fma(ac.y, l1, P.a22 * l2) + P.C2;
                    l1 = ac.x * l1 + P.C1; l2 = nl2;
                    if (i == j) { m11 = f11; m21 = f21; m22 = f22; ml1 = l1; ml2 = l2; }
                }
                __syncthreads();
                if (act) {
                    P12[j] = make_double2(e11, e21);
                    double2 *phi = reinterpret_cast<double2 *>(Phi + (size_t)s * 4 * N);
                    phi[j] = make_double2(m11, m21);
                    phi[N + j] = make_double2(0.0, m22);
                    reinterpret_cast<double2 *>(Lam + (size_t)s * 2 * N)[j] = make_double2(ml1, ml2);
                }
                __syncthreads();
                double2 *gam = reinterpret_cast<double2 *>(Gam + (size_t)s * 2 * N * N);
                int c = j / N, i = j - c * N;
                const int dc = T / N, di = T - dc * N;
                for (int t = j; t < N * N; t += T) {
                    double2 v = make_double2(0.0, 0.0);
                    if (i >= c) {
                        const double2 p = P12[i - c];
                        const double bc = bbs[c];
                        v = make_double2(bc * p.x, bc * p.y);
                    }
                    gam[t] = v;
                    c += dc; i += di;
                    if (i >= N) { i -= N; ++c; }
                }
            }
            return;
        }
        if (gi && vec_ok && stage != nullptr) {
            // Index i, long horizons: thread c carries column c of Gamma down the block rows (A_i * Gamma(i-1,c), no
            // Toeplitz structure to generate from) in chunks of NTM_COND_RC rows into a CTA tile of odd pitch, and the
            // CTA copies each chunk out as 256-byte column segments.  Writing straight from the recurrence is a
            // 2N-double stride between neighbouring threads: 18-20 % of the HBM peak.
            constexpr int RC = NTM_COND_RC, PITCH = NTM_COND_RC + 1;
            const int T = 32 * GW;
            for (int s = blockIdx.x; s < S; s += gridDim.x) {
                const Params P = load_params(params, layout, pc, s);
                double b = 0.0;
                __syncthreads();                                     // previous scenario's readers are done with a11s / a21s
                if (act) {
                    double a11, a21;
                    lpv_of(P, __ldg(R1 + (size_t)s * N + j), __ldg(R2 + (size_t)s * N + j), __ldg(R3 + (size_t)s * N + j), a11, a21, b);
                    a11s[j] = a11; a21s[j] = a21;
                }
                __syncthreads();
                double f11 = 1.0, f21 = 0.0, f22 = 1.0, l1 = 0.0, l2 = 0.0;      // Phi_i (lower triangular), Lambda_i
                double m11 = 0, m21 = 0, m22 = 0, ml1 = 0, ml2 = 0;
                for (int i = 0; i < N; ++i) {
                    const double aa = a11s[i], cc = a21s[i];
                    const double n21 = fma(cc, f11, P.a22 * f21);
                    f11 = aa * f11; f21 = n21; f22 = P.a22 * f22;
                    const double nl2 = fma(cc, l1, P.a22 * l2) + P.C2;
                    l1 = aa * l1 + P.C1; l2 = nl2;
                    if (i == j) { m11 = f11; m21 = f21; m22 = f22; ml1 = l1; ml2 = l2; }
                }
                if (act) {
                    double2 *phi = reinterpret_cast<double2 *>(Phi + (size_t)s * 4 * N);
                    phi[j] = make_double2(m11, m21);
                    phi[N + j] = make_double2(0.0, m22);
                    reinterpret_cast<double2 *>(Lam + (size_t)s * 2 * N)[j] = make_double2(ml1, ml2);
                }
                double2 *gam = reinterpret_cast<double2 *>(Gam + (size_t)s * 2 * N * N);
                double g1 = 0.0, g2 = 0.0;
                for (int i0 = 0; i0 < N; i0 += RC) {
                    const int rows = (N - i0) < RC ? (N - i0) : RC;
                    if (act) {
                        double2 *col = stage + (size_t)j * PITCH;
                        for (int r = 0; r < rows; ++r) {
                            const int i = i0 + r;
                            if (i == j) { g1 = b; g2 = 0.0; }
                            else if (i > j) {
                                const double aa = a11s[i], cc = a21s[i];
                                const double n2 = fma(cc, g1, P.a22 * g2);
                                g1 = aa * g1; g2 = n2;
                            }
                            col[r] = make_double2(g1, g2);
                        }
                    }
                    __syncthreads();
                    for (int e = j; e < N * RC; e += T) {
                        const int c = e / RC, r = e - c * RC;        // RC is a power of two
                        if (r < rows) gam[(size_t)c * N + i0 + r] = stage[(size_t)c * PITCH + r];
                    }
                    __syncthreads();
                }
            }
            return;
        }
    }
    for (int s = blockIdx.x * gpb + gib; s < S; s += gridDim.x * gpb) {
        const Params P = load_params(params, layout, pc, s);
        if (act) {
            double a11, a21, b;
            lpv_of(P, R1[elem(layout, S, N, s, j)], R2[elem(layout, S, N, s, j)], R3[elem(layout, S, N, s, j)], a11,
                   a21, b);
            a11s[j] = a11; a21s[j] = a21; bbs[j] = b;
        }
        Gp::sync();
        // Phi_i = A_i Phi_{i-1} (lower triangular), Lambda_i = A_i Lambda_{i-1} + C   (:17-22, :47-52)
        double f11 = 1.0, f21 = 0.0, f22 = 1.0, l1 = 0.0, l2 = 0.0;
        double m11 = 0, m21 = 0, m22 = 0, ml1 = 0, ml2 = 0;
        for (int i = 0; i < N; ++i) {
            const double aa = a11s[i], cc = a21s[i];
            const double n21 = fma(cc, f11, P.a22 * f21);
            f11 = aa * f11; f21 = n21; f22 = P.a22 * f22;
            const double nl2 = fma(cc, l1, P.a22 * l2) + P.C2;
            l1 = aa * l1 + P.C1; l2 = nl2;
            if (i == j) { m11 = f11; m21 = f21; m22 = f22; ml1 = l1; ml2 = l2; }
        }
        if (act) {
            Phi[elem(layout, S, 4 * N, s, 2 * j)] = m11;
            Phi[elem(layout, S, 4 * N, s, 2 * j + 1)] = m21;
            Phi[elem(layout, S, 4 * N, s, 2 * N + 2 * j)] = 0.0;
            Phi[elem(layout, S, 4 * N, s, 2 * N + 2 * j + 1)] = m22;
            Lam[elem(layout, S, 2 * N, s, 2 * j)] = ml1;
            Lam[elem(layout, S, 2 * N, s, 2 * j + 1)] = ml2;
            // Gamma column j (:26-40)
            double g1 = 0.0, g2 = 0.0;
            const int EG = 2 * N * N;
            for (int i = 0; i < N; ++i) {
                if (i == j) { g1 = bbs[j]; g2 = 0.0; }
                else if (i > j) {
                    const int k = gi ? i : (i - j - 1);
                    const double aa = a11s[k], cc = a21s[k];
                    const double n2 = fma(cc, g1, P.a22 * g2);
                    g1 = aa * g1; g2 = n2;
                }
                const int e = j * 2 * N + 2 * i;
                if (vec_ok) {
                    *reinterpret_cast<double2 *>(Gam + (size_t)s * EG + e) = make_double2(g1, g2);
                } else {
                    Gam[elem(layout, S, EG, s, e)] = g1;
                    Gam[elem(layout, S, EG, s, e + 1)] = g2;
                }
            }
        }
        Gp::sync();
    }
}

// =================================================================================================
// G = 2 Gamma' Omega Gamma, F = 2 Gamma' Omega (Phi x + Lambda - R) for dense caller-supplied matrices
// =================================================================================================
template <int GW>
__global__ void __launch_bounds__(32 * GW)
hessian_grad_kernel(int layout, int S, int N, int CH, const double *__restrict__ Phi, const double *__restrict__ Gam,
                    const double *__restrict__ Lam, const double *__restrict__ x, const double *__restrict__ params,
                    int pc, double *__restrict__ G, double *__restrict__ F) {
    // Gamma is streamed through shared memory in chunks of CH block rows; the lower triangle of G is
    // accumulated in shared memory and written out coalesced at the end.
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int T = 32 * GW;
    const int j = threadIdx.x;
    const int ldg = odd_ld(N), ldc = 2 * CH + 1;
    double *Gs = reinterpret_cast<double *>(smem_raw);   // N x ldg, lower triangle
    double *Cs = Gs + (size_t)N * ldg;                   // chunk: column c at Cs[c*ldc + k], k < 2*CH
    double *Es = Cs + (size_t)N * ldc;                   // Omega*(Phi x + Lambda - R), 2N
    for (int s = blockIdx.x; s < S; s += gridDim.x) {
        const Params P = load_params(params, layout, pc, s);
        const int EG = 2 * N * N;
        const double xw = x[elem(layout, S, 2, s, 0)], xo = x[elem(layout, S, 2, s, 1)];
        for (int i = j; i < N; i += T) {
            const double v1 = Phi[elem(layout, S, 4 * N, s, 2 * i)] * xw + Phi[elem(layout, S, 4 * N, s, 2 * N + 2 * i)] * xo +
                              Lam[elem(layout, S, 2 * N, s, 2 * i)] - P.r1;
            const double v2 = Phi[elem(layout, S, 4 * N, s, 2 * i + 1)] * xw +
                              Phi[elem(layout, S, 4 * N, s, 2 * N + 2 * i + 1)] * xo +
                              Lam[elem(layout, S, 2 * N, s, 2 * i + 1)] - P.r2;
            Es[2 * i] = P.q11 * v1 + P.q12 * v2;
            Es[2 * i + 1] = P.q12 * v1 + P.q22 * v2;
        }
        double accF = 0.0;
        for (int c0 = 0; c0 < N; c0 += CH) {
            const int ch = min(CH, N - c0);
            __syncthreads();
            for (int e = j; e < N * 2 * ch; e += T) {
                const int c = e / (2 * ch), k = e - c * 2 * ch;
                Cs[c * ldc + k] = Gam[elem(layout, S, EG, s, c * 2 * N + 2 * c0 + k)];
            }
            __syncthreads();
            if (j < N) {
                const double *cj = Cs + j * ldc;
                for (int k = 0; k < 2 * ch; ++k) accF = fma(cj[k], Es[2 * c0 + k], accF);
                for (int l = 0; l <= j; ++l) {
                    const double *cl = Cs + l * ldc;
                    double acc = 0.0;
                    for (int i = 0; i < ch; ++i) {
                        const double g1 = cj[2 * i], g2 = cj[2 * i + 1];
                        acc = fma(P.q11 * g1 + P.q12 * g2, cl[2 * i], acc);
                        acc = fma(P.q12 * g1 + P.q22 * g2, cl[2 * i + 1], acc);
                    }
                    if (c0 == 0) Gs[j * ldg + l] = acc;
                    else Gs[j * ldg + l] += acc;
                }
            }
        }
        __syncthreads();
        if (j < N) F[elem(layout, S, N, s, j)] = 2.0 * accF;
        for (int e = j; e < N * N; e += T) {
            const int col = e / N, row = e - col * N;
            const double v = (row >= col) ? Gs[row * ldg + col] : Gs[col * ldg + row];
            G[elem(layout, S, N * N, s, e)] = 2.0 * v;
        }
        __syncthreads();
    }
}

// =================================================================================================
// Long horizons (N > 32): the same contraction G = 2 Gamma' (Omega Gamma) on the FP64 tensor cores.
// Gamma (2N x N, column-major) is staged once in shared memory with a pitch that is 4 mod 8 doubles (conflict-free
// fragment loads); each warp owns 8x8 tiles of the lower triangle of G and walks K = 2N in steps of 4 with
// mma.sync.m8n8k4.f64 (SASS: DMMA.8x8x4).  Omega = I (x) Q is applied on the fly to the B fragment: rows 2i, 2i+1 of
// Gamma are one block row, so the partner element sits at row ^ 1 of the same column.
// =================================================================================================
__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }
template <int NKEEP>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;\n" ::"n"(NKEEP) : "memory"); }

#define NTM_DMMA_KC 56          // rows of Gamma per shared-memory chunk = the pitch: 8 mod 16 doubles, conflict-free LDS.128

// A warp owns 2x2 SUPER-TILES of the lower triangle.  History of the operand path (profiles/README.md):
//   * one 8x8 tile per warp-step, fragments by LDS.64: 3 shared-memory loads per DMMA, shared-memory pipe at 68 %;
//   * 2x2 super-tiles, Omega applied per fragment: 1.5 loads + a DMUL/DFMA pair per DMMA, 47 % of the DMMA peak;
//     ncu: 39 % of the instructions and half of the stall samples sat in the per-element staging loops.
// Now: (1) two copies of the chunk sit in shared memory, Gamma (A operands) and Omega*Gamma (B operands; Omega =
// I (x) Q mixes rows 2i, 2i+1, and the thread that copied a 16-byte row pair transforms exactly that pair, so there is no
// barrier between copy and transform).  (2) The contraction index is permuted inside every group of 8 rows -- k-slot t4
// of two consecutive DMMAs takes rows 2*t4 and 2*t4 + 1 -- so ONE LDS.128 per fragment feeds two DMMAs: per 8 rows a
// super-tile issues 4 LDS.128 and 8 DMMAs, nothing else.  (3) The chunk buffers are dense (pitch == rows == 56), so
// the copy and transform loops walk pair p = tid, tid + 256, ... with no index arithmetic on the shared side.
// K = 2N = 200 is 56 + 56 + 56 + 32: no nearly empty last chunk.
// Measured and rejected (profiles/README.md, round 2): a double buffer with 40-row chunks (2.01 ms against 1.91), Omega
// applied in registers without the second copy and one barrier per chunk (bulk copies 2.19, cp.async 2.11), a half-period
// stagger of the two CTAs of an SM (2.25), dealing the super-tiles to the warps by cost (2.05; 1.78 against 1.75 after the
// predicated DMMAs were gone), 16 warps and one CTA per SM with the raw chunk double buffered (2.22 against 1.89).
// F rides along: v = Phi x + Lambda - R is staged as column N of the chunk, and row N of the extended product
// [Gamma v]' Omega [Gamma v] is F / 2.
// 8 warps per CTA: two CTAs per SM fill each other's copy waits.
template <int MAXST>   // MAXST super-tiles per warp: ceil(nst (nst + 1) / 2 / WARPS), nst = ceil(ceil8(N + 1) / 16)
__global__ void __launch_bounds__(256, MAXST <= 4 ? 2 : 1)
hessian_grad_dmma_kernel(int layout, int S, int N, const double *__restrict__ Phi, const double *__restrict__ Gam,
                         const double *__restrict__ Lam, const double *__restrict__ x, const double *__restrict__ params,
                         int pc, double *__restrict__ G, double *__restrict__ F) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int WARPS = 8, T = 32 * WARPS, KC = NTM_DMMA_KC, ldc = KC, KH = KC / 2;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int Np = (N + 1 + 7) & ~7;                       // at least one spare column: column N carries v
    const int K2 = 2 * N, VP = K2 + 4;                     // a Vs buffer: v (2N), then q11, q12, q22 of its scenario
    double *Ga = reinterpret_cast<double *>(smem_raw);     // the raw chunk: column c at Ga[c*ldc + k], k < KC
    double *Qs = Ga + (size_t)Np * ldc;                    // the current chunk times Omega
    double *Vs = Qs + (size_t)Np * ldc;                    // two buffers (this scenario / the next one)
    unsigned char *stab = reinterpret_cast<unsigned char *>(Vs + 2 * VP);   // super-tile t -> (sm, sn)
    const int EG = 2 * N * N;
    const int nt = Np >> 3, nst = (nt + 1) >> 1, nsuper = nst * (nst + 1) / 2;
    for (int t = tid; t < nsuper; t += T) {
        int sm = 0, rem = t;
        while (rem > sm) { rem -= sm + 1; ++sm; }
        stab[2 * t] = (unsigned char)sm; stab[2 * t + 1] = (unsigned char)rem;
    }
    const int g = lane >> 2, t4 = lane & 3;
    // 16-byte copies: MATLAB layout (a column of Gamma is contiguous), 16-byte aligned base; 2N and the chunk start are even
    const bool vec16 = layout == NTM_LAYOUT_MATLAB && (reinterpret_cast<uintptr_t>(Gam) & 15) == 0;
    // v = Phi x + Lambda - R of scenario sc, entries 2*tid, 2*tid + 1 (N <= 128 < T).  Two call sites (the first scenario,
    // and the prefetch of the next one inside the chunk loop): explicitly rounded operations, so that the compiler cannot
    // contract the two copies into FMAs differently and give a scenario other bits as a CTA's second scenario.
    auto vpair = [&](int sc, double &v0, double &v1) {
        const Params P = load_params(params, layout, pc, sc);
        const double xw = x[elem(layout, S, 2, sc, 0)], xo = x[elem(layout, S, 2, sc, 1)];
        const int i = tid;
        v0 = __dsub_rn(__dadd_rn(__fma_rn(Phi[elem(layout, S, 4 * N, sc, 2 * i)], xw,
                                          __dmul_rn(Phi[elem(layout, S, 4 * N, sc, 2 * N + 2 * i)], xo)),
                                 Lam[elem(layout, S, 2 * N, sc, 2 * i)]), P.r1);
        v1 = __dsub_rn(__dadd_rn(__fma_rn(Phi[elem(layout, S, 4 * N, sc, 2 * i + 1)], xw,
                                          __dmul_rn(Phi[elem(layout, S, 4 * N, sc, 2 * N + 2 * i + 1)], xo)),
                                 Lam[elem(layout, S, 2 * N, sc, 2 * i + 1)]), P.r2);
    };
    auto qstore = [&](int sc, double *vb) {
        if (tid == T - 1) {
            const Params P = load_params(params, layout, pc, sc);
            vb[K2] = P.q11; vb[K2 + 1] = P.q12; vb[K2 + 2] = P.q22;
        }
    };
    int s = blockIdx.x;
    if (s >= S) return;
    int vp = 0;
    if (tid < N) { double v0, v1; vpair(s, v0, v1); Vs[2 * tid] = v0; Vs[2 * tid + 1] = v1; }
    qstore(s, Vs);
    constexpr int QT = T / KH, RT = T - QT * KH;
    const int h_first = tid % KH;
    const unsigned off_first = (unsigned)(tid / KH) * K2 + 2 * h_first;
    // Gamma row pairs of chunk kc of scenario sc -> dst: pair p = c * KH + k/2 sits at doubles 2p, 2p + 1; the source offset
    // c * 2N + k is tracked incrementally.  Rows beyond 2N (last chunk only) are zero-filled, so the Omega pass needs no
    // row test.  The Omega pass of the same thread walks the same pairs.
    auto issue = [&](int sc, int kc, double *dst) {
        const int hrows = min(KC, K2 - kc) >> 1;
        int h = h_first;
        unsigned off = off_first;
        const double *src = Gam + (size_t)sc * EG + kc;
        const unsigned step = QT * K2 + 2 * RT, wrap = K2 - 2 * KH;
        for (int p = tid; p < N * KH; p += T) {
            if (h < hrows) {
                if (vec16) cp_async16(dst + 2 * p, src + off);
                else {
                    const int c = off / K2, k = off - c * K2;
                    cp_async8(dst + 2 * p, Gam + elem(layout, S, EG, sc, c * K2 + kc + k));
                    cp_async8(dst + 2 * p + 1, Gam + elem(layout, S, EG, sc, c * K2 + kc + k + 1));
                }
            } else *reinterpret_cast<double2 *>(dst + 2 * p) = make_double2(0.0, 0.0);
            h += RT; off += step;
            if (h >= KH) { h -= KH; off += wrap; }
        }
    };
    for (; s < S; s += gridDim.x) {
        const int sn = s + gridDim.x;
        const double *vs = Vs + vp * VP;
        double acc[MAXST][4][2];                            // [super-tile][(r0,c0), (r1,c0), (r0,c1), (r1,c1)]
#pragma unroll
        for (int i = 0; i < MAXST; ++i)
#pragma unroll
            for (int q = 0; q < 4; ++q) { acc[i][q][0] = 0.0; acc[i][q][1] = 0.0; }
        for (int kc = 0; kc < K2; kc += KC) {
            const int rows = min(KC, K2 - kc);              // even
            const int kend = (rows + 7) & ~7;               // rows [rows, kend) are zero, the rest of the chunk is not read
            const bool last = kc + KC >= K2;
            double nv0 = 0.0, nv1 = 0.0;
            __syncthreads();                                // everyone is done with the previous chunk; Vs visible
            issue(s, kc, Ga);
            if (last && sn < S && tid < N) vpair(sn, nv0, nv1);
            cp_async_wait_all();
            const double q11 = vs[K2], q12 = vs[K2 + 1], q22 = vs[K2 + 2];
            // Omega image of the pairs this thread copied itself (visible to it after the wait)
#pragma unroll 4
            for (int p = tid; p < N * KH; p += T) {
                const double2 gg = *reinterpret_cast<const double2 *>(Ga + 2 * p);
                *reinterpret_cast<double2 *>(Qs + 2 * p) = make_double2(fma(q11, gg.x, q12 * gg.y), fma(q22, gg.y, q12 * gg.x));
            }
            // the v column and the padding columns: plain stores, both images
            for (int p = N * KH + tid; p < Np * KH; p += T) {
                const int c = p / KH, k = 2 * (p - c * KH);
                const bool vcol = (c == N) && (k < rows);
                const double g0 = vcol ? vs[kc + k] : 0.0, g1 = vcol ? vs[kc + k + 1] : 0.0;
                *reinterpret_cast<double2 *>(Ga + 2 * p) = make_double2(g0, g1);
                *reinterpret_cast<double2 *>(Qs + 2 * p) = make_double2(fma(q11, g0, q12 * g1), fma(q22, g1, q12 * g0));
            }
            if (last && sn < S) {
                double *vn = Vs + (vp ^ 1) * VP;
                if (tid < N) { vn[2 * tid] = nv0; vn[2 * tid + 1] = nv1; }
                qstore(sn, vn);
            }
            __syncthreads();
#pragma unroll
            for (int i = 0; i < MAXST; ++i) {
                const int st = wid + WARPS * i;
                if (st < nsuper) {
                    const int sm = stab[2 * st], sn2 = stab[2 * st + 1];
                    const bool diag = sm == sn2;
                    const bool row1 = 2 * sm + 1 < nt;      // the super-tile has a second tile row / column
                    const bool col1 = 2 * sn2 + 1 < nt;
                    const double *r0 = Ga + (size_t)(16 * sm + g) * ldc + 2 * t4;
                    const double *c0 = Qs + (size_t)(16 * sn2 + g) * ldc + 2 * t4;
                    const double *r1 = row1 ? r0 + 8 * ldc : r0;
                    const double *c1 = col1 ? c0 + 8 * ldc : c0;
                    // Four loop bodies, selected OUTSIDE the k loop: a DMMA that is issued with its predicate off still holds
                    // the tensor pipe for its 16 cycles (tools/ubench/dmma_sweep.cu), and at N = 100 the last super-tile row
                    // has one tile row only -- predicated, that was 15 % of the DMMAs issued.
                    if (diag && row1) {                     // (r0,c0), (r1,c0), (r1,c1)
#pragma unroll 2
                        for (int k0 = 0; k0 < kend; k0 += 8) {
                            const double2 a0 = *reinterpret_cast<const double2 *>(r0 + k0), a1 = *reinterpret_cast<const double2 *>(r1 + k0);
                            const double2 b0 = *reinterpret_cast<const double2 *>(c0 + k0), b1 = *reinterpret_cast<const double2 *>(c1 + k0);
                            dmma_m8n8k4(acc[i][0][0], acc[i][0][1], a0.x, b0.x);
                            dmma_m8n8k4(acc[i][1][0], acc[i][1][1], a1.x, b0.x);
                            dmma_m8n8k4(acc[i][3][0], acc[i][3][1], a1.x, b1.x);
                            dmma_m8n8k4(acc[i][0][0], acc[i][0][1], a0.y, b0.y);
                            dmma_m8n8k4(acc[i][1][0], acc[i][1][1], a1.y, b0.y);
                            dmma_m8n8k4(acc[i][3][0], acc[i][3][1], a1.y, b1.y);
                        }
                    } else if (diag) {                      // (r0,c0) only
#pragma unroll 2
                        for (int k0 = 0; k0 < kend; k0 += 8) {
                            const double2 a0 = *reinterpret_cast<const double2 *>(r0 + k0), b0 = *reinterpret_cast<const double2 *>(c0 + k0);
                            dmma_m8n8k4(acc[i][0][0], acc[i][0][1], a0.x, b0.x);
                            dmma_m8n8k4(acc[i][0][0], acc[i][0][1], a0.y, b0.y);
                        }
                    } else if (row1) {                      // all four tiles (col1 always holds below the diagonal)
#pragma unroll 2
                        for (int k0 = 0; k0 < kend; k0 += 8) {
                            const double2 a0 = *reinterpret_cast<const double2 *>(r0 + k0), a1 = *reinterpret_cast<const double2 *>(r1 + k0);
                            const double2 b0 = *reinterpret_cast<const double2 *>(c0 + k0), b1 = *reinterpret_cast<const double2 *>(c1 + k0);
                            dmma_m8n8k4(acc[i][0][0], acc[i][0][1], a0.x, b0.x);
                            dmma_m8n8k4(acc[i][2][0], acc[i][2][1], a0.x, b1.x);
                            dmma_m8n8k4(acc[i][1][0], acc[i][1][1], a1.x, b0.x);
                            dmma_m8n8k4(acc[i][3][0], acc[i][3][1], a1.x, b1.x);
                            dmma_m8n8k4(acc[i][0][0], acc[i][0][1], a0.y, b0.y);
                            dmma_m8n8k4(acc[i][2][0], acc[i][2][1], a0.y, b1.y);
                            dmma_m8n8k4(acc[i][1][0], acc[i][1][1], a1.y, b0.y);
                            dmma_m8n8k4(acc[i][3][0], acc[i][3][1], a1.y, b1.y);
                        }
                    } else {                                // (r0,c0), (r0,c1)
#pragma unroll 2
                        for (int k0 = 0; k0 < kend; k0 += 8) {
                            const double2 a0 = *reinterpret_cast<const double2 *>(r0 + k0);
                            const double2 b0 = *reinterpret_cast<const double2 *>(c0 + k0), b1 = *reinterpret_cast<const double2 *>(c1 + k0);
                            dmma_m8n8k4(acc[i][0][0], acc[i][0][1], a0.x, b0.x);
                            dmma_m8n8k4(acc[i][2][0], acc[i][2][1], a0.x, b1.x);
                            dmma_m8n8k4(acc[i][0][0], acc[i][0][1], a0.y, b0.y);
                            dmma_m8n8k4(acc[i][2][0], acc[i][2][1], a0.y, b1.y);
                        }
                    }
                }
            }
        }
        vp ^= 1;
        // results: element e of this scenario sits at base + e * es in either layout (one multiply per store instead of the
        // generic index function: the stores were a quarter of a warp's instructions outside the k loops)
        const bool soa = layout == NTM_LAYOUT_SOA;
        const size_t es = soa ? (size_t)S : 1;
        double *Gb = G + (soa ? (size_t)s : (size_t)s * N * N), *Fb = F + (soa ? (size_t)s : (size_t)s * N);
#pragma unroll
        for (int i = 0; i < MAXST; ++i) {
            const int st = wid + WARPS * i;
            if (st < nsuper) {
                const int sm = stab[2 * st], sn2 = stab[2 * st + 1];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int tm = 2 * sm + (q & 1), tn = 2 * sn2 + (q >> 1);
                    if (tm >= nt || tn >= nt || tn > tm) continue;
                    const int r = tm * 8 + g, cc = tn * 8 + 2 * t4;
                    const double v0 = 2.0 * acc[i][q][0], v1 = 2.0 * acc[i][q][1];
                    if (r < N) {                           // lower part only (diagonal tiles hold both), mirrored: exactly symmetric
                        double *pd = Gb + (size_t)(cc * N + r) * es, *pm = Gb + (size_t)(r * N + cc) * es;
                        if (cc < N && cc <= r) { *pd = v0; *pm = v0; }
                        if (cc + 1 < N && cc + 1 <= r) { pd[(size_t)N * es] = v1; pm[es] = v1; }
                    } else if (r == N) {                   // the v row: F = 2 v' Omega Gamma
                        if (cc < N) Fb[(size_t)cc * es] = v0;
                        if (cc + 1 < N) Fb[(size_t)(cc + 1) * es] = v1;
                    }
                }
            }
        }
    }
}

// Short horizons (N <= 32) on the tensor cores too: one warp per scenario, the whole Gamma (K = 2N <= 64 rows) of a
// scenario in the warp's own shared-memory slice.  This entry point is HBM-bound (9.7 KB per scenario at N = 20), so
// the job is to keep loads in flight.  ncu on the first version (46 % of the HBM peak): 1750 warp instructions per
// scenario, and a staging loop whose load -> shared-store dependency left ONE 16-byte load per lane in flight
// (long-scoreboard stalls on top).  Now:
//   * Gamma is staged with cp.async into a double-buffered slice: the copy of scenario s+1 is issued before the
//     tensor-core pass over scenario s, no register dependency, ~12 requests per lane in flight;
//   * F rides on the tensor cores: v = Phi x + Lambda - R is staged as column N of the tile (Np = ceil8(N + 1), so
//     there is always a spare column), and row N of the extended product [Gamma v]' Omega [Gamma v] is F / 2;
//   * the k loop is outermost: per 4 rows the NT A fragments and the NT Omega-transformed B fragments are loaded once
//     and feed all NT (NT + 1) / 2 lower-triangle tiles (accumulators in registers);
//   * staging walks (column, row pair) incrementally -- no integer division per element.
template <int NT>                                                  // NT = ceil((N + 1) / 8) tile rows
__global__ void __launch_bounds__(128, NT <= 3 ? 3 : 1)
hessian_grad_dmma_warp_kernel(int S, int N, int ld, const double *__restrict__ Phi, const double *__restrict__ Gam,
                              const double *__restrict__ Lam, const double *__restrict__ x, const double *__restrict__ params,
                              int pc, double *__restrict__ G, double *__restrict__ F, int aligned16) {
    // MATLAB layout only (the launcher falls back to the scalar kernel otherwise); aligned16: Gam and G are 16-byte aligned
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    constexpr int Np = NT * 8;
    const int Kp = (2 * N + 3) & ~3;
    const size_t slice = (size_t)Np * ld;
    double *buf0 = reinterpret_cast<double *>(smem_raw) + (size_t)wid * 2 * slice;     // column c at buf[c*ld + k]
    const int EG = 2 * N * N;
    const int g = lane >> 2, t4 = lane & 3;
    const bool vec = aligned16 && !(N & 1);
    const int stride = gridDim.x * wpb;

    // asynchronous copy of Gamma(:,:,s) into columns 0..N-1 of dst (one commit group per scenario).  A lane's element
    // index advances by 32 per request: (column, row) move by the precomputed quotient / remainder, branch-free (the
    // first version normalised with a while loop: 16 % of the kernel's instructions).
    const int per_col = vec ? N : 2 * N;                           // requests per column: double2 or double
    const int dq = 32 / per_col, dr = 32 % per_col;
    const int c_first = lane / per_col, k_first = lane % per_col;
    auto stage = [&](int s, double *dst) {
        const double *gsrc = Gam + (size_t)s * EG;
        int c = c_first, k = k_first;
        if (vec) {
            const double2 *src = reinterpret_cast<const double2 *>(gsrc) + lane;
            while (c < N) {
                cp_async16(dst + c * ld + 2 * k, src);
                src += 32; c += dq; k += dr;
                const bool wrap = k >= per_col;
                k -= wrap ? per_col : 0; c += wrap ? 1 : 0;
            }
        } else {
            const double *src = gsrc + lane;
            while (c < N) {
                cp_async8(dst + c * ld + k, src);
                src += 32; c += dq; k += dr;
                const bool wrap = k >= per_col;
                k -= wrap ? per_col : 0; c += wrap ? 1 : 0;
            }
        }
        cp_async_commit();
    };
    // columns N+1 .. Np-1 are padding that nothing ever dirties (the G staging area N*N + N <= N*ld stays inside the
    // Gamma columns): zero them once, in both buffers
    for (int e = lane; e < 2 * (Np - N - 1) * ld; e += 32) {
        const int b = e / ((Np - N - 1) * ld), r = e - b * (Np - N - 1) * ld;
        buf0[(size_t)b * slice + (size_t)(N + 1) * ld + r] = 0.0;
    }

    int s = blockIdx.x * wpb + wid;
    int cur = 0;
    if (s < S) stage(s, buf0);
    for (; s < S; s += stride, cur ^= 1) {
        double *Gs = buf0 + (size_t)cur * slice;
        const int sn = s + stride;
        if (sn < S) stage(sn, buf0 + (size_t)(cur ^ 1) * slice);   // the other buffer was drained in the previous pass
        const Params P = load_params(params, NTM_LAYOUT_MATLAB, pc, s);
        {
            // v (column N) and zero rows 2N..Kp-1 of the Gamma columns: the slice doubles as the G staging area, so those
            // rows are rewritten for every scenario (plain stores: disjoint from what cp.async writes)
            const double xw = __ldg(x + 2 * (size_t)s), xo = __ldg(x + 2 * (size_t)s + 1);
            const double *ph = Phi + (size_t)s * 4 * N, *lm = Lam + (size_t)s * 2 * N;
            double *vc = Gs + N * ld;
            for (int i = lane; i < Kp / 2; i += 32) {
                double v1 = 0.0, v2 = 0.0;
                if (i < N) {
                    v1 = __ldg(ph + 2 * i) * xw + __ldg(ph + 2 * N + 2 * i) * xo + __ldg(lm + 2 * i) - P.r1;
                    v2 = __ldg(ph + 2 * i + 1) * xw + __ldg(ph + 2 * N + 2 * i + 1) * xo + __ldg(lm + 2 * i + 1) - P.r2;
                }
                vc[2 * i] = v1; vc[2 * i + 1] = v2;
            }
            for (int k = 2 * N + lane; k < Kp; k += 32)           // Kp - 2N <= 2 padding rows of the Gamma columns
                for (int c = 0; c < N; ++c) Gs[c * ld + k] = 0.0;
        }
        if (sn < S) cp_async_wait_group<1>(); else cp_async_wait_group<0>();     // this scenario's Gamma has landed
        __syncwarp();
        const double qs = (t4 & 1) ? P.q22 : P.q11;
        double acc[NT * (NT + 1) / 2][2];                          // kept in registers until Gamma is dead
#pragma unroll
        for (int ti = 0; ti < NT * (NT + 1) / 2; ++ti) { acc[ti][0] = 0.0; acc[ti][1] = 0.0; }
        {
            const double *fp = Gs + (size_t)g * ld + t4;           // fragment element of tile row 0: row g of the tile, k = t4
            const int tstride = 8 * ld;
#pragma unroll 2
            for (int k0 = 0; k0 < Kp; k0 += 4) {
                double af[NT], bf[NT];
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    const double *q = fp + t * tstride + k0;
                    const double own = q[0], partner = q[(t4 ^ 1) - t4];     // the other row of the (w, omega) pair
                    af[t] = own;
                    bf[t] = fma(qs, own, P.q12 * partner);                     // Omega = I (x) Q applied on the fly
                }
#pragma unroll
                for (int tm = 0; tm < NT; ++tm)
#pragma unroll
                    for (int tn = 0; tn <= tm; ++tn) dmma_m8n8k4(acc[tm * (tm + 1) / 2 + tn][0], acc[tm * (tm + 1) / 2 + tn][1], af[tm], bf[tn]);
            }
        }
        __syncwarp();                                              // every lane is done reading Gamma: reuse the slice for G
        double *Go = Gs;                                           // N x N, column-major like the output; F behind it
        double *Fo = Gs + N * N;
#pragma unroll
        for (int tm = 0; tm < NT; ++tm) {
#pragma unroll
            for (int tn = 0; tn <= tm; ++tn) {
                const int ti = tm * (tm + 1) / 2 + tn;
                const int r = tm * 8 + g, cc = tn * 8 + 2 * t4;
                if (r < N) {
                    if (cc < N && cc <= r) { Go[cc * N + r] = 2.0 * acc[ti][0]; Go[r * N + cc] = 2.0 * acc[ti][0]; }
                    if (cc + 1 < N && cc + 1 <= r) { Go[(cc + 1) * N + r] = 2.0 * acc[ti][1]; Go[r * N + cc + 1] = 2.0 * acc[ti][1]; }
                } else if (r == N) {                               // the v row: F = 2 * v' Omega Gamma
                    if (cc < N) Fo[cc] = 2.0 * acc[ti][0];
                    if (cc + 1 < N) Fo[cc + 1] = 2.0 * acc[ti][1];
                }
            }
        }
        __syncwarp();
        double *gdst = G + (size_t)s * N * N;
        if (vec) {
            for (int e = lane; e < N * N / 2; e += 32) reinterpret_cast<double2 *>(gdst)[e] = *reinterpret_cast<const double2 *>(Go + 2 * e);
        } else {
            for (int e = lane; e < N * N; e += 32) gdst[e] = Go[e];
        }
        if (lane < N) F[(size_t)s * N + lane] = Fo[lane];
        __syncwarp();                                              // the slice is free for the copy issued in the next pass
    }
}

// =================================================================================================
// Monte-Carlo back end: reduction of a batch of closed-loop results (SURVEY 8f-3).  One warp per scenario (lane =
// time sample, so the trajectory reads are contiguous in the MATLAB layout), per-CTA partials in shared memory,
// one atomic per statistic and CTA.  HBM-bound: 8*(3*k_sim + 3) + 4 bytes per scenario.
// =================================================================================================
__device__ __forceinline__ void atomic_min_f64(double *addr, double v) {
    unsigned long long *a = reinterpret_cast<unsigned long long *>(addr);
    unsigned long long old = *a;
    while (__longlong_as_double((long long)old) > v) {
        const unsigned long long seen = atomicCAS(a, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}
__device__ __forceinline__ void atomic_max_f64(double *addr, double v) {
    unsigned long long *a = reinterpret_cast<unsigned long long *>(addr);
    unsigned long long old = *a;
    while (__longlong_as_double((long long)old) < v) {
        const unsigned long long seen = atomicCAS(a, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}

struct McBounds { double xmin1, xmax1, xmin2, xmax2, w_sup, hist_max; };

__global__ void mc_stats_init_kernel(double *out) {
    const int i = threadIdx.x;
    if (i < NTM_MC_NSTAT) {
        const double inf = __longlong_as_double(0x7ff0000000000000LL);
        out[i] = (i == 6 || i == 10) ? inf : ((i == 7 || i == 11) ? -inf : 0.0);
    }
}

// per-thread accumulators, indexed like out[0..21]; reduced once per warp at the end of the kernel
struct McAcc {
    // Sums and extrema are doubles; everything that counts (13 of the 22 statistics) is an integer while a thread
    // accumulates -- a predicated integer add instead of a 64-bit select + DADD, and 12 registers instead of 26 -- and
    // becomes a double in fold(), once, before the reduction.  Per-thread counts stay far below 2^31 (a thread sees
    // S / (resident threads) scenarios of K samples).
    double v[22];
    int n_st0, n_st1, n_st2, n_st3, n_sup, s_first, n_first, n_lo, n_hi, n_w, n_om, n_ok;
    __device__ void init() {
        const double inf = __longlong_as_double(0x7ff0000000000000LL);
#pragma unroll
        for (int i = 0; i < 22; ++i) v[i] = 0.0;
        v[6] = inf; v[10] = inf; v[7] = -inf; v[11] = -inf;
        n_st0 = n_st1 = n_st2 = n_st3 = n_sup = s_first = n_first = n_lo = n_hi = n_w = n_om = n_ok = 0;
    }
    __device__ __forceinline__ void count_status(int st) {
        n_st0 += (st == NTM_SCN_OK) ? 1 : 0; n_st1 += (st == NTM_SCN_QP_ITER_CAP) ? 1 : 0;
        n_st2 += (st == NTM_SCN_NONFINITE) ? 1 : 0; n_st3 += (st > NTM_SCN_NONFINITE) ? 1 : 0;
    }
    __device__ void scalars(int st, double c, double wf, int K, const McBounds &b, int *hist) {
        v[4] += c; v[5] = fma(c, c, v[5]); v[6] = fmin(v[6], c); v[7] = fmax(v[7], c);
        v[8] += wf; v[9] = fma(wf, wf, v[9]); v[10] = fmin(v[10], wf); v[11] = fmax(v[11], wf);
        n_sup += (wf < b.w_sup) ? 1 : 0;
        n_ok += 1;                                           // [17] and [21] are K per included scenario
        int bin = (wf > 0.0 && b.hist_max > 0.0) ? (int)(wf / b.hist_max * NTM_MC_NBINS) : 0;
        bin = bin < 0 ? 0 : (bin >= NTM_MC_NBINS ? NTM_MC_NBINS - 1 : bin);
        atomicAdd(&hist[bin], 1);
    }
    __device__ __forceinline__ void sample(double u, double w, double om, double umin, double umax, const McBounds &b) {
        n_lo += (u <= umin) ? 1 : 0; n_hi += (u >= umax) ? 1 : 0; v[18] += u;
        n_w += (w < b.xmin1 || w > b.xmax1) ? 1 : 0;
        n_om += (om < b.xmin2 || om > b.xmax2) ? 1 : 0;
    }
    __device__ __forceinline__ void first_below(int first) { s_first += first; n_first += (first != 0) ? 1 : 0; }
    __device__ void fold(int K) {
        v[0] += (double)n_st0; v[1] += (double)n_st1; v[2] += (double)n_st2; v[3] += (double)n_st3;
        v[12] += (double)n_sup; v[13] += (double)s_first; v[14] += (double)n_first;
        v[15] += (double)n_lo; v[16] += (double)n_hi; v[19] += (double)n_w; v[20] += (double)n_om;
        v[17] += (double)n_ok * (double)K; v[21] += (double)n_ok * (double)K;
        n_st0 = n_st1 = n_st2 = n_st3 = n_sup = s_first = n_first = n_lo = n_hi = n_w = n_om = n_ok = 0;
    }
};

__device__ void mc_finish(McAcc &a, int K, double *acc, int *hist, double *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    a.fold(K);
#pragma unroll
    for (int i = 0; i < 22; ++i) {
        double x = a.v[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double y = __shfl_xor_sync(0xffffffffu, x, o);
            x = (i == 6 || i == 10) ? fmin(x, y) : ((i == 7 || i == 11) ? fmax(x, y) : x + y);
        }
        if (lane == 0) {
            if (i == 6 || i == 10) atomic_min_f64(&acc[i], x);
            else if (i == 7 || i == 11) atomic_max_f64(&acc[i], x);
            else atomicAdd(&acc[i], x);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < NTM_MC_NSTAT; i += blockDim.x) {
        if (i >= 22) { if (hist[i - 22]) atomicAdd(&out[i], (double)hist[i - 22]); continue; }
        const double x = acc[i];
        if (i == 6 || i == 10) atomic_min_f64(&out[i], x);
        else if (i == 7 || i == 11) atomic_max_f64(&out[i], x);
        else if (x != 0.0) atomicAdd(&out[i], x);
    }
}

__device__ __forceinline__ void mc_shared_init(double *acc, int *hist) {
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    for (int i = threadIdx.x; i < 22; i += blockDim.x) acc[i] = (i == 6 || i == 10) ? inf : ((i == 7 || i == 11) ? -inf : 0.0);
    for (int i = threadIdx.x; i < NTM_MC_NBINS; i += blockDim.x) hist[i] = 0;
    __syncthreads();
}

// MATLAB layout, fallback for trajectories too long for the staged kernel below: lanes = time samples.  Each warp takes
// 32 scenarios per round: the per-scenario scalars (cost, final width, status, bounds) lane-parallel over the
// scenarios, then the trajectories one scenario at a time with fully coalesced rows (20 of 32 lanes busy at
// k_sim = 20, one dependent round trip per scenario: 19 % of the HBM peak).
__global__ void __launch_bounds__(256)
mc_stats_matlab_lanes_kernel(int S, int K, const double *__restrict__ xk, const double *__restrict__ uk,
                       const double *__restrict__ cost, const int *__restrict__ status,
                       const double *__restrict__ params, const double *__restrict__ umaxp, int pc, McBounds b, double *__restrict__ out) {
    __shared__ double acc[22];
    __shared__ int hist[NTM_MC_NBINS];
    mc_shared_init(acc, hist);
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const size_t EX = 2 * ((size_t)K + 1);
    McAcc a; a.init();
    for (long long base = ((long long)blockIdx.x * wpb + wib) * 32; base < S; base += (long long)gridDim.x * wpb * 32) {
        const long long s = base + lane;
        const bool valid = s < S;
        const int st = valid ? (status ? status[s] : 0) : NTM_SCN_NONFINITE;
        if (valid) a.count_status(st);
        const bool ok = valid && st < NTM_SCN_NONFINITE;      // non-finite and infeasible (NaN from the failing step on) are only counted
        double umin = 0.0, umax = 0.0;
        if (ok) {
            umin = params[(size_t)s * (size_t)pc]; umax = umaxp[(size_t)s * (size_t)pc];
            a.scalars(st, cost ? cost[s] : 0.0, xk[(size_t)s * EX + 2 * (size_t)K], K, b, hist);
        }
        const unsigned okmask = __ballot_sync(0xffffffffu, ok);
        for (int i = 0; i < 32; ++i) {
            if (!((okmask >> i) & 1u)) continue;
            const double um = __shfl_sync(0xffffffffu, umin, i), uM = __shfl_sync(0xffffffffu, umax, i);
            const double *ur = uk + (size_t)(base + i) * K, *xr = xk + (size_t)(base + i) * EX + 2;
            int first = 0;
            for (int k0 = 0; k0 < K; k0 += 32) {
                const int k = k0 + lane;
                bool below = false;
                if (k < K) {
                    const double w = xr[2 * k], om = xr[2 * k + 1];
                    a.sample(ur[k], w, om, um, uM, b);
                    below = w < b.w_sup;
                }
                const unsigned m = __ballot_sync(0xffffffffu, below);
                if (first == 0 && m) first = k0 + __ffs(m);
            }
            if (lane == i) a.first_below(first);
        }
    }
    mc_finish(a, K, acc, hist, out);
}

// MATLAB layout, staged: the trajectories of 32 consecutive scenarios are ONE contiguous block of 32 * 2(K+1) doubles
// (xk) and one of 32 * K (uk).  A warp copies both blocks to its shared-memory slice with 8-byte cp.async -- fully
// coalesced, ~60 independent requests per lane in flight -- into rows of odd pitch, then every lane walks its own
// scenario conflict-free, exactly like the SoA kernel.

__global__ void __launch_bounds__(128)
mc_stats_matlab_kernel(int S, int K, const double *__restrict__ xk, const double *__restrict__ uk,
                       const double *__restrict__ cost, const int *__restrict__ status,
                       const double *__restrict__ params, const double *__restrict__ umaxp, int pc, McBounds b, double *__restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double acc[22];
    __shared__ int hist[NTM_MC_NBINS];
    mc_shared_init(acc, hist);
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int EX = 2 * (K + 1), EXP = EX | 1, KP = K | 1;
    double *xs = reinterpret_cast<double *>(smem_raw) + (size_t)wib * 32 * (EXP + KP);
    double *us = xs + 32 * EXP;
    const int xdq = 32 / EX, xdr = 32 % EX, xr0 = lane / EX, xc0 = lane % EX;
    const int Kd = K > 0 ? K : 1;
    const int udq = 32 / Kd, udr = 32 % Kd, ur0 = K > 0 ? lane / Kd : 32, uc0 = lane % Kd;
    McAcc a; a.init();
    for (long long base = ((long long)blockIdx.x * wpb + wib) * 32; base < S; base += (long long)gridDim.x * wpb * 32) {
        const int nv = (int)((S - base) < 32 ? (S - base) : 32);
        __syncwarp();                                          // the previous tile has been consumed
        {
            // a lane's element index advances by 32 per request: (row, column) move by quotient / remainder, branch-free
            const double *src = xk + (size_t)base * EX + lane;
            int r = xr0, c = xc0;
            while (r < nv) {
                cp_async8(xs + r * EXP + c, src);
                src += 32; r += xdq; c += xdr;
                const bool wrap = c >= EX;
                c -= wrap ? EX : 0; r += wrap ? 1 : 0;
            }
            src = uk + (size_t)base * K + lane;
            r = ur0; c = uc0;
            while (r < nv) {
                cp_async8(us + r * KP + c, src);
                src += 32; r += udq; c += udr;
                const bool wrap = c >= K;
                c -= wrap ? K : 0; r += wrap ? 1 : 0;
            }
        }
        const long long s = base + lane;
        const bool valid = s < S;
        const int st = valid ? (status ? status[s] : 0) : NTM_SCN_NONFINITE;
        const bool ok = valid && st < NTM_SCN_NONFINITE;      // non-finite and infeasible (NaN from the failing step on) are only counted
        double umin = 0.0, umax = 0.0, cs = 0.0;
        if (ok) {
            umin = params[(size_t)s * (size_t)pc]; umax = umaxp[(size_t)s * (size_t)pc];
            cs = cost ? cost[s] : 0.0;
        }
        cp_async_wait_all();
        __syncwarp();
        if (valid) a.count_status(st);
        if (ok) {
            const double *xr = xs + lane * EXP + 2, *ur = us + lane * KP;
            a.scalars(st, cs, xr[2 * K - 2], K, b, hist);
            int first = 0;
            for (int k = 0; k < K; ++k) {
                const double w = xr[2 * k], om = xr[2 * k + 1];
                a.sample(ur[k], w, om, umin, umax, b);
                if (first == 0 && w < b.w_sup) first = k + 1;
            }
            a.first_below(first);
        }
    }
    mc_finish(a, K, acc, hist, out);
}

// SoA layout: the scenario index is fastest, so one thread per scenario reads coalesced and walks the time axis.
__global__ void __launch_bounds__(256, 3)
mc_stats_soa_kernel(int S, int K, const double *__restrict__ xk, const double *__restrict__ uk,
                    const double *__restrict__ cost, const int *__restrict__ status, const double *__restrict__ params, const double *__restrict__ umaxp,
                    int pc, McBounds b, double *__restrict__ out) {
    __shared__ double acc[22];
    __shared__ int hist[NTM_MC_NBINS];
    mc_shared_init(acc, hist);
    McAcc a; a.init();
    const size_t Ss = (size_t)S;
    for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < S; s += (long long)gridDim.x * blockDim.x) {
        const int st = status ? status[s] : 0;
        a.count_status(st);
        if (st >= NTM_SCN_NONFINITE) continue;                  // non-finite / infeasible: counted only
        const double umin = params[(size_t)s * (size_t)pc], umax = umaxp[(size_t)s * (size_t)pc];
        a.scalars(st, cost ? cost[s] : 0.0, xk[2 * (size_t)K * Ss + s], K, b, hist);
        int first = 0;
        // chunks of 4 time samples: 12 independent loads are issued before the first one is consumed (with a plain
        // unrolled loop the compiler interleaved loads and dependent accumulator updates); 4 keeps the kernel at 80
        // registers = 3 CTAs per SM
        for (int k0 = 0; k0 < K; k0 += 4) {
            double uu[4], ww[4], oo[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int k = (k0 + i < K) ? k0 + i : K - 1;
                uu[i] = __ldg(uk + (size_t)k * Ss + s);
                ww[i] = __ldg(xk + (2 * (size_t)k + 2) * Ss + s);
                oo[i] = __ldg(xk + (2 * (size_t)k + 3) * Ss + s);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (k0 + i < K) {
                    a.sample(uu[i], ww[i], oo[i], umin, umax, b);
                    if (first == 0 && ww[i] < b.w_sup) first = k0 + i + 1;
                }
            }
        }
        a.first_below(first);
    }
    mc_finish(a, K, acc, hist, out);
}

// =================================================================================================
// FP64 pipe microbenchmark: 8 independent register-resident DFMA chains per thread
// =================================================================================================
__global__ void __launch_bounds__(256) fp64_peak_kernel(int iters, double *out) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    const double r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == 12345.678) out[0] = r;   // keeps the chains alive without a store in the common case
}

// =================================================================================================
// launchers
// =================================================================================================
static inline int gw_for(int N) { return N <= 32 ? 1 : (N <= 64 ? 2 : 4); }

// Shared-memory LDL' capacity: the closed loop sees bang-bang solutions with a handful of free variables, so a
// small workspace buys occupancy; caller-supplied QPs (ntm_qp_box) may be interior, so they get the full N when
// it fits.  Larger free sets use the group's global slab.
static inline int hcap_loop(const DeviceProps &dp, int N, int gam = 0) {
    if (gw_for(N) == 1) {
        // One-warp groups: the largest capacity that costs no resident CTA (4 warps per CTA, 1 KB reserve per CTA, at most
        // the 5 CTAs per SM the registers allow): N = 20 -> 20, N = 24 -> 16, N = 32 -> 20 -- so that the global slab is
        // only touched where shared memory really runs out.  (Measured: no effect on config 3 -- its free sets stay
        // below 12; what makes a scenario slow there is that EVERY one of its 200 QPs takes the active-set path, ~5 us
        // alone against ~1 us for the vertex test: tools/heavy_probe.py, 1.65 ms against a median of 0.62 ms.)
        if (N <= 12) return N;
        const size_t sm = 228 * 1024;
        auto occ = [&](int h) { const size_t per = work_bytes(N, h, gam) * 4 + 1024; const int o = (int)(sm / per); return o < 5 ? o : 5; };
        const int base = occ(12);
        int h = N;
        while (h > 12 && occ(h) < base) h -= 4;
        return h < 12 ? 12 : h;
    }
    return (work_bytes(N, N, gam) + 1024 <= dp.smem_optin) ? N : 16;    // long horizons do see large free sets
}
static inline int hcap_qp(const DeviceProps &dp, int N) {
    const int gw = gw_for(N);
    const size_t per_block = work_bytes(N, N) * (gw == 1 ? 4 : 1);
    return (per_block + 1024 <= dp.smem_optin) ? N : 16;
}
// upper bound on simultaneously resident groups (one global slab each)
static inline int max_groups(const DeviceProps &dp, int N) { return dp.sm_count * (gw_for(N) == 1 ? 32 : 4); }

size_t state_rows_smem(int N) {
    return (work_bytes(N, N, false) + ineq_bytes(N, 4 * N) + ext_bytes(N)) * (gw_for(N) == 1 ? 4 : 1);
}
// one group's share with a non-literal Gamma index (one-warp groups only): + the dense Gamma tile, + its frozen copy
size_t state_rows_dense_smem(int N, int srows) {
    return work_bytes(N, N, 1) + ineq_bytes(N, 4 * N) + ext_bytes(N) + (srows == 2 ? gam_doubles(N, 1) * sizeof(double) : 0);
}

int qp_ineq_groups(const DeviceProps &dp, int N, int M) {
    const size_t gbytes = work_bytes(N, N) + ineq_bytes(N, M);
    int wpb = (gw_for(N) == 1) ? 4 : 1;
    while (wpb > 1 && gbytes * wpb + 1024 > dp.smem_optin) wpb >>= 1;
    return gbytes * wpb + 1024 <= dp.smem_optin ? wpb : 0;
}

size_t hscratch_bytes(const DeviceProps &dp, int N) {
    return (size_t)max_groups(dp, N) * N * odd_ld(N) * sizeof(double);
}

cudaError_t launch_rho(cudaStream_t st, int layout, int flags, int S, const double *x, const double *params, int pc,
                       double *r1, double *r2, double *r3, long long *launches) {
    if (S <= 0) return cudaSuccess;
    rho_kernel<<<(S + 255) / 256, 256, 0, st>>>(layout, flags, S, x, params, pc, r1, r2, r3);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_lpv(cudaStream_t st, int layout, int S, const double *r1, const double *r2, const double *r3,
                       const double *params, int pc, double *A, double *B, long long *launches) {
    if (S <= 0) return cudaSuccess;
    lpv_kernel<<<(S + 255) / 256, 256, 0, st>>>(layout, S, r1, r2, r3, params, pc, A, B);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_plant(cudaStream_t st, int layout, int flags, int S, const double *x, const double *u,
                         const double *params, int pc, double *xn, long long *launches) {
    if (S <= 0) return cudaSuccess;
    if (flags & (NTM_PROFILE_PLANT_RK4 | NTM_PROFILE_TAUE_W)) plant_kernel<true><<<(S + 255) / 256, 256, 0, st>>>(layout, flags, S, x, u, params, pc, xn);
    else plant_kernel<false><<<(S + 255) / 256, 256, 0, st>>>(layout, flags, S, x, u, params, pc, xn);
    ++*launches;
    return cudaGetLastError();
}

// The dynamic-shared-memory attribute is PROCESS-WIDE per kernel and device, so it is only ever raised: once per
// (kernel, device) to the device's opt-in maximum, under a lock.  (Caching "the last size this thread set" and skipping the
// call let a second host thread lower the attribute under the first one's feet: its next launch then failed with
// cudaErrorInvalidValue.)  The occupancy answer depends on the launch's own size only and stays cached per thread.
cudaError_t raise_smem_attribute(const void *fn, int dev, size_t smem_optin) {
    static std::mutex mu;
    static std::vector<std::pair<const void *, int>> done;
    std::lock_guard<std::mutex> lk(mu);
    for (const auto &d : done) if (d.first == fn && d.second == dev) return cudaSuccess;
    cudaFuncAttributes fa;                                 // static + dynamic shared memory share the opt-in limit
    cudaError_t e = cudaFuncGetAttributes(&fa, fn);
    if (e != cudaSuccess) return e;
    const size_t room = smem_optin > fa.sharedSizeBytes ? smem_optin - fa.sharedSizeBytes : 0;
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)room);
    if (e == cudaSuccess) done.emplace_back(fn, dev);
    return e;
}

template <typename K>
static cudaError_t persistent_geometry(K kernel, const DeviceProps &dp, int block, size_t smem, int groups_needed,
                                       int groups_per_block, int *grid) {
    // The occupancy query costs several microseconds of host time -- a visible part of a single-scenario MPC step --
    // so the answers are cached per thread, keyed by (kernel, block, shared memory, device).
    static thread_local std::map<std::tuple<const void *, int, size_t, int>, int> cache;
    if (smem > dp.smem_optin) return cudaErrorInvalidConfiguration;
    const void *fn = reinterpret_cast<const void *>(kernel);
    int dev = 0;
    cudaGetDevice(&dev);
    const auto key = std::make_tuple(fn, block, smem, dev);
    auto hit = cache.find(key);
    if (hit == cache.end()) {
        cudaError_t e = raise_smem_attribute(fn, dev, dp.smem_optin);
        if (e != cudaSuccess) return e;
        int occ = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, block, smem);
        if (e != cudaSuccess) return e;
        hit = cache.emplace(key, occ).first;
    }
    const int occ = hit->second;
    if (occ < 1) return cudaErrorInvalidConfiguration;
    const long long cap = (long long)occ * dp.sm_count;
    const long long need = ((long long)groups_needed + groups_per_block - 1) / groups_per_block;
    *grid = (int)(need < cap ? need : cap);
    if (*grid < 1) *grid = 1;
    return cudaSuccess;
}

// Launch of a persistent kernel whose groups (groups_per_block per CTA) pull work from a queue: as many CTAs as are
// resident at once, at most those the groups need, and at most group_cap groups (one global LDL' slab each).
template <typename... P, typename... A>
static cudaError_t launch_persistent(cudaStream_t st, const DeviceProps &dp, void (*kernel)(P...), int block, size_t smem,
                                     int groups, int groups_per_block, int group_cap, long long *launches, A... args) {
    int grid = 1;
    const cudaError_t e = persistent_geometry(kernel, dp, block, smem, groups, groups_per_block, &grid);
    if (e != cudaSuccess) return e;
    if (grid * groups_per_block > group_cap) grid = group_cap / groups_per_block;
    kernel<<<grid, block, smem, st>>>(args...);
    ++*launches;
    return cudaGetLastError();
}

// ---- two-phase launch: counting sort of the phase-A cost keys, largest key first -----------------------------------
__global__ void lpt_hist_kernel(int S, const int *__restrict__ key, int *__restrict__ bins) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < S) atomicAdd(bins + key[s], 1);
}
__global__ void lpt_scan_kernel(int *__restrict__ bins) {         // one thread: counts -> start offsets (descending key), in place
    int off = 0;
    for (int b = NTM_LPT_BINS - 1; b >= 0; --b) { const int c = bins[b]; bins[b] = off; off += c; }
}
__global__ void lpt_scatter_kernel(int S, const int *__restrict__ key, int *__restrict__ bins, int *__restrict__ perm) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < S) perm[atomicAdd(bins + key[s], 1)] = s;               // the order inside a bin does not matter
}

static inline bool lpt_enabled() {
    static const char *env = getenv("NTM_LPT");
    return env == nullptr || atoi(env) != 0;
}
// Worth it when the launch runs more than one "round" of resident warps and the state fits a sane buffer; one-warp box
// loop on the literal Gamma with F from x0 (the headline instantiation) only.
size_t lpt_doubles(const DeviceProps &dp, const LoopArgs &a) {
    if (!lpt_enabled() || gw_for(a.N) != 1 || a.srows != 0 || a.ctl || a.pert || a.k_sim < 4) return 0;
    if (a.flags & (NTM_PROFILE_GAMMA_I | NTM_PROFILE_DENSE_G | NTM_PROFILE_PLANT_RK4 | NTM_PROFILE_TAUE_W | NTM_PROFILE_F_XK)) return 0;
    // Measured (profiles/README.md, round 2): -8..9 % at 16 k-64 k scenarios, -20 % with the eps_break stop rule.  At 8,192
    // (2.8 rounds of resident warps) it is a wash -- the eight 8,192-scenario shards of config 3 take 4.7-7.2 ms (mean 5.54)
    // as one launch and 4.7-7.0 ms (mean 5.39) in two phases: step 0 does not see the scenarios that turn slow later, and
    // one scenario that needs 2.6 ms ALONE bounds its shard either way.  So: from 2.5 rounds of resident warps.
    if ((long long)a.S < (long long)dp.sm_count * 20 * 5 / 2) return 0;
    if (a.S > (1 << 18)) return 0;                                 // 0.5 GB of saved state at most; beyond that the tail is < 1 %
    return (size_t)a.S * NTM_CTRL_DOUBLES(a.N);
}

// Every closed_loop_kernel instantiation of this translation unit; the long-horizon ones are in ntm_loop_long.cu.
static const LoopKernel kLoopKernels[] = {
    // one-warp groups (N <= 32); the controller step on the box QP is their runtime mode LoopArgs::ctl
    {{1, false, EXT_BOX, 0, false}, closed_loop_kernel<1, false, EXT_BOX>},
    {{1, true, EXT_BOX, 0, false}, closed_loop_kernel<1, true, EXT_BOX>},
    {{1, false, EXT_COLD_PLANT, 0, false}, closed_loop_kernel<1, false, EXT_COLD_PLANT>},
    {{1, true, EXT_COLD_PLANT, 0, false}, closed_loop_kernel<1, true, EXT_COLD_PLANT>},
    {{1, false, EXT_STATE_ROWS, 0, false}, closed_loop_kernel<1, false, EXT_STATE_ROWS>},
    {{1, true, EXT_STATE_ROWS, 0, false}, closed_loop_kernel<1, true, EXT_STATE_ROWS>},
    {{1, false, EXT_STATE_ROWS, 0, true}, closed_loop_kernel<1, false, EXT_STATE_ROWS, 0, true>},
    {{1, true, EXT_STATE_ROWS, 0, true}, closed_loop_kernel<1, true, EXT_STATE_ROWS, 0, true>},
    {{1, false, EXT_PERTURBED, 0, false}, closed_loop_kernel<1, false, EXT_PERTURBED>},
    {{1, true, EXT_PERTURBED, 0, false}, closed_loop_kernel<1, true, EXT_PERTURBED>},
    {{1, false, EXT_PERTURBED_ROWS, 0, false}, closed_loop_kernel<1, false, EXT_PERTURBED_ROWS>},
    {{1, true, EXT_PERTURBED_ROWS, 0, false}, closed_loop_kernel<1, true, EXT_PERTURBED_ROWS>},
    // multi-warp groups, dense Gamma
    {{2, true, EXT_BOX, 0, false}, closed_loop_kernel<2, true, EXT_BOX>},
    {{4, true, EXT_BOX, 0, false}, closed_loop_kernel<4, true, EXT_BOX>},
    {{2, true, EXT_BOX, 0, true}, closed_loop_kernel<2, true, EXT_BOX, 0, true>},
    {{4, true, EXT_BOX, 0, true}, closed_loop_kernel<4, true, EXT_BOX, 0, true>},
    {{2, true, EXT_COLD_PLANT, 0, false}, closed_loop_kernel<2, true, EXT_COLD_PLANT>},
    {{4, true, EXT_COLD_PLANT, 0, false}, closed_loop_kernel<4, true, EXT_COLD_PLANT>},
    {{2, true, EXT_PERTURBED, 0, false}, closed_loop_kernel<2, true, EXT_PERTURBED>},
    {{4, true, EXT_PERTURBED, 0, false}, closed_loop_kernel<4, true, EXT_PERTURBED>},
    // multi-warp groups, literal Gamma, state rows
    {{2, false, EXT_STATE_ROWS, 0, false}, closed_loop_kernel<2, false, EXT_STATE_ROWS>},
    {{4, false, EXT_STATE_ROWS, 0, false}, closed_loop_kernel<4, false, EXT_STATE_ROWS>},
    {{2, false, EXT_STATE_ROWS, 0, true}, closed_loop_kernel<2, false, EXT_STATE_ROWS, 0, true>},
    {{4, false, EXT_STATE_ROWS, 0, true}, closed_loop_kernel<4, false, EXT_STATE_ROWS, 0, true>},
    {{2, false, EXT_PERTURBED_ROWS, 0, false}, closed_loop_kernel<2, false, EXT_PERTURBED_ROWS>},
    {{4, false, EXT_PERTURBED_ROWS, 0, false}, closed_loop_kernel<4, false, EXT_PERTURBED_ROWS>},
};
static_assert(sizeof(kLoopKernels) / sizeof(kLoopKernels[0]) == 26, "kLoopKernels: one entry per instantiation");

// The launch of one fused call: the instantiation and its shape.
struct LoopRoute {
    LoopKey key;
    bool lng;                      // in kLongLoopKernels (ntm_loop_long.cu)
    int block, groups_per_block, group_cap;
    size_t smem, gbytes;           // dynamic shared memory per CTA / per group
};

// Every rule that picks the closed_loop_kernel instantiation of a call, and its launch shape.  Sets the launcher-owned
// fields of a: hcap, gam, wbytes, qbytes, rows_warm.
static cudaError_t route_closed_loop(const DeviceProps &dp, LoopArgs &a, LoopRoute &r) {
    const int gw = gw_for(a.N);
    const bool dense = (a.flags & (NTM_PROFILE_GAMMA_I | NTM_PROFILE_DENSE_G)) != 0;
    // the headline instantiations carry none of the cold options
    const int ext = a.pert ? (a.srows != 0 ? EXT_PERTURBED_ROWS : EXT_PERTURBED)
                  : a.srows != 0 ? EXT_STATE_ROWS
                  : (a.flags & (NTM_PROFILE_PLANT_RK4 | NTM_PROFILE_TAUE_W)) ? EXT_COLD_PLANT : EXT_BOX;
    // long horizons, literal Gamma, box QP: the sweep tableau, in registers while N + 1 fits 7 x 15 blocks, else in shared
    // memory (LV = 1)
    r.lng = gw > 1 && !dense && ext != EXT_STATE_ROWS && ext != EXT_PERTURBED_ROWS;
    // the controller step is a runtime mode of the one-warp box kernels and its own instantiation (CTL) wherever that mode
    // would cost registers (DESIGN section 4.8)
    const bool ctl = a.ctl != 0 && (ext == EXT_STATE_ROWS || (gw > 1 && ext == EXT_BOX));
    r.key = {gw, dense, ext, (r.lng && a.N + 1 > NTM_TS * 15) ? 1 : 0, ctl};
    // dense Gamma on the FP64 tensor cores: a full staging tile per warp (one-warp groups), a 16-row chunk buffer for the
    // multi-warp groups whose ceil8(N + 1) columns fit the group's threads and NTM_DMAXT tiles per warp (N <= 63 / 103)
    a.gam = 0;
    if (dense && gw == 1) a.gam = 1;
    else if (dense && a.srows == 0) {
        const int Np = (a.N + 1 + 7) & ~7, nt = Np >> 3;
        if (Np <= 32 * gw && (nt * (nt + 1) / 2 + gw - 1) / gw <= NTM_DMAXT) a.gam = 2;
    }
    a.hcap = hcap_loop(dp, a.N, a.gam);
    {
        static const char *env = getenv("NTM_ROWS_WARM");  // diagnostic: 0 = every state-row QP starts cold
        a.rows_warm = (env == nullptr || atoi(env) != 0) ? 1 : 0;
    }
    size_t gbytes = work_bytes(a.N, a.hcap, a.gam);
    int gpb = gw == 1 ? 4 : 1;                               // groups (= scenarios) per CTA
    if (a.srows != 0) {
        if (a.srows < 0 || a.srows > 2) return cudaErrorInvalidValue;
        if (dense && gw != 1) return cudaErrorInvalidValue;   // rows of a non-literal Gamma are read from the per-warp tile: N <= 32
        a.hcap = a.N;                                    // the continuation keeps R in the LDL' buffer: full size
        a.gam = dense ? 1 : 0;
        const size_t wb = work_bytes(a.N, a.N, a.gam);
        a.wbytes = (unsigned int)wb;
        a.qbytes = (unsigned int)(wb + ineq_bytes(a.N, 4 * a.N));
        gbytes = a.qbytes + ext_bytes(a.N);
        if (dense && a.srows == 2) gbytes += gam_doubles(a.N, 1) * sizeof(double);   // frozen rows: the offline tile
        while (gpb > 1 && gbytes * gpb > dp.smem_optin) --gpb;
        if (gbytes * gpb > dp.smem_optin) return cudaErrorInvalidValue;
    }
    r.block = 32 * gw * gpb;
    r.groups_per_block = gpb;
    r.group_cap = max_groups(dp, a.N);
    if (r.lng) {                                           // one CTA per scenario, no global LDL' slabs
        gbytes = work_bytes_long(a.N);
        r.group_cap = INT_MAX;
    }
    r.gbytes = gbytes;
    r.smem = gbytes * gpb;
    return cudaSuccess;
}

cudaError_t launch_closed_loop(cudaStream_t st, const DeviceProps &dp, const LoopArgs &a, int *lpt, long long *launches) {
    if (a.S <= 0) return cudaSuccess;
    if (a.hscratch == nullptr) return cudaErrorInvalidValue;
    LoopArgs aa = a;
    aa.k_begin = 0; aa.k_end = a.k_sim; aa.lpt_key = nullptr; aa.perm = nullptr;
    LoopRoute r;
    cudaError_t e = route_closed_loop(dp, aa, r);
    if (e != cudaSuccess) return e;
    const LoopKernelFn fn = r.lng ? find_long_loop_kernel(r.key) : find_loop_kernel(kLoopKernels, r.key);
    if (fn == nullptr) return cudaErrorInvalidDeviceFunction;
    // a.counter[0..1] are zero: armed at creation, re-armed by each launch
    auto launch = [&] {
        return launch_persistent(st, dp, fn, r.block, r.smem, a.S, r.groups_per_block, r.group_cap, launches, aa,
                                 (unsigned int)r.gbytes);
    };
    if (lpt != nullptr && a.sv != nullptr && lpt_doubles(dp, a) != 0) {
        // phase A: time step 0 of every scenario (state + cost key), counting sort, phase B: the rest, longest first.
        // lpt_doubles admits the headline instantiation <1, false, EXT_BOX> only.
        int *key = lpt, *perm = lpt + a.S, *bins = lpt + 2 * (size_t)a.S;
        e = cudaMemsetAsync(bins, 0, NTM_LPT_BINS * sizeof(int), st);
        if (e != cudaSuccess) return e;
        aa.k_begin = 0; aa.k_end = 1; aa.lpt_key = key;
        e = launch();
        if (e != cudaSuccess) return e;
        lpt_hist_kernel<<<(a.S + 255) / 256, 256, 0, st>>>(a.S, key, bins);
        lpt_scan_kernel<<<1, 1, 0, st>>>(bins);
        lpt_scatter_kernel<<<(a.S + 255) / 256, 256, 0, st>>>(a.S, key, bins, perm);
        *launches += 3;
        aa.k_begin = 1; aa.k_end = a.k_sim; aa.lpt_key = nullptr; aa.perm = perm;
    }
    return launch();
}

cudaError_t launch_qp_box(cudaStream_t st, const DeviceProps &dp, int layout, int S, int N, const double *G,
                          const double *F, const double *lb, const double *ub, int bc, double *U, int *iters,
                          int *status, unsigned int *counter, double *hscratch, long long *launches) {
    if (S <= 0) return cudaSuccess;
    if (hscratch == nullptr) return cudaErrorInvalidValue;
    const int gw = gw_for(N), wpb = gw == 1 ? 4 : 1;
    const int hcap = hcap_qp(dp, N);
    const size_t gbytes = work_bytes(N, hcap);
    const auto kernel = gw == 1 ? qp_box_kernel<1> : (gw == 2 ? qp_box_kernel<2> : qp_box_kernel<4>);
    // counter[0..1] are zero: armed at creation, re-armed by each launch
    return launch_persistent(st, dp, kernel, 32 * gw * wpb, gbytes * wpb, S, wpb, max_groups(dp, N), launches, layout, S,
                             N, G, F, lb, ub, bc, U, iters, status, counter, (unsigned int)gbytes, hscratch, hcap);
}

// returns cudaErrorInvalidConfiguration when N x N factor pair + row scales do not fit in shared memory
cudaError_t launch_qp_ineq(cudaStream_t st, const DeviceProps &dp, int layout, int S, int N, int M, const double *G,
                           const double *F, const double *lb, const double *ub, int bc, const double *Lg,
                           const double *bg, double *U, int *iters, int *status, unsigned int *counter,
                           long long *launches) {
    if (S <= 0) return cudaSuccess;
    const int gw = gw_for(N);
    const size_t wbytes = work_bytes(N, N);
    const size_t gbytes = wbytes + ineq_bytes(N, M);
    const int wpb = qp_ineq_groups(dp, N, M);
    if (wpb == 0) return cudaErrorInvalidConfiguration;
    const auto kernel = gw == 1 ? qp_ineq_kernel<1> : (gw == 2 ? qp_ineq_kernel<2> : qp_ineq_kernel<4>);
    return launch_persistent(st, dp, kernel, 32 * gw * wpb, gbytes * wpb, S, wpb, INT_MAX, launches, layout, S, N, M, G,
                             F, lb, ub, bc, Lg, bg, U, iters, status, counter, (unsigned int)gbytes, (unsigned int)wbytes);
}

// umin / umax of scenario s are umin[s * ustride] / umax[s * ustride] (ustride 0: one shared pair)
cudaError_t launch_mc_stats(cudaStream_t st, const DeviceProps &dp, int layout, int S, int k_sim, const double *xk,
                            const double *uk, const double *cost, const int *status, const double *umin, const double *umax,
                            int ustride, const double *bounds, double w_sup, double hist_max, double *out, long long *launches) {
    const double *params = umin;                           // the kernels call the pair (params, umaxp) with stride pc
    const double *umaxp = umax;
    const int pc = ustride;
    mc_stats_init_kernel<<<1, 64, 0, st>>>(out);
    ++*launches;
    if (S > 0) {
        const McBounds b = {bounds[0], bounds[1], bounds[2], bounds[3], w_sup, hist_max};
        if (layout == NTM_LAYOUT_MATLAB) {
            const size_t per_warp = (size_t)32 * ((2 * ((size_t)k_sim + 1) | 1) + ((size_t)k_sim | 1)) * sizeof(double);
            const size_t budget = dp.smem_optin > 2048 ? dp.smem_optin - 2048 : 0;
            if (per_warp <= budget) {                                  // staged kernel: as many warps per CTA as fit, at most 4
                int wpb = (int)(budget / 3 / per_warp);                // aim at 3 CTAs per SM
                wpb = wpb < 1 ? 1 : (wpb > 4 ? 4 : wpb);
                const size_t smem = per_warp * wpb;
                int dev_ = 0; cudaGetDevice(&dev_);
                cudaError_t e = raise_smem_attribute(reinterpret_cast<const void *>(mc_stats_matlab_kernel), dev_, dp.smem_optin);
                if (e != cudaSuccess) return e;
                int occ = 1;
                e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mc_stats_matlab_kernel, 32 * wpb, smem);
                if (e != cudaSuccess) return e;
                const long long need = ((long long)S + 32 * wpb - 1) / (32 * wpb), cap = (long long)dp.sm_count * (occ < 1 ? 1 : occ);
                mc_stats_matlab_kernel<<<(int)(need < cap ? need : cap), 32 * wpb, smem, st>>>(S, k_sim, xk, uk, cost, status, params, umaxp, pc, b, out);
            } else {
                const long long need = ((long long)S + 255) / 256, cap = (long long)dp.sm_count * 8;
                mc_stats_matlab_lanes_kernel<<<(int)(need < cap ? need : cap), 256, 0, st>>>(S, k_sim, xk, uk, cost, status, params, umaxp, pc, b, out);
            }
        } else {
            const long long need = ((long long)S + 255) / 256, cap = (long long)dp.sm_count * 8;
            mc_stats_soa_kernel<<<(int)(need < cap ? need : cap), 256, 0, st>>>(S, k_sim, xk, uk, cost, status, params, umaxp, pc, b, out);
        }
        ++*launches;
    }
    return cudaGetLastError();
}

// SoA layout (scenario index fastest): one THREAD per scenario.  Every load and store of a warp is then 256 contiguous
// bytes (32 consecutive scenarios of one element), the recurrences of Rho_to_PhiGammaLambda.m:17-52 run in registers and
// the per-stage LPV entries sit in thread-local arrays.  (The group-per-scenario kernel above wrote this layout with a
// stride of S doubles between neighbouring lanes: 6 % of the HBM peak.)
template <int MAXN>                                      // capacity of the thread-local stage arrays (32 keeps the stack at 768 bytes)
__global__ void __launch_bounds__(128)
condense_soa_kernel(int flags, int S, int N, const double *__restrict__ R1, const double *__restrict__ R2,
                    const double *__restrict__ R3, const double *__restrict__ params, int pc, double *__restrict__ Phi,
                    double *__restrict__ Gam, double *__restrict__ Lam) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const size_t Ss = (size_t)S;
    const Params P = load_params(params, NTM_LAYOUT_SOA, pc, s);
    const bool gi = (flags & NTM_PROFILE_GAMMA_I) != 0;
    // The stage entries are RE-LOADED from the rho arrays wherever they are needed (coalesced, L2-resident: 3N doubles
    // per scenario) instead of being kept in thread-local arrays: ncu showed 880 MB of local-memory loads per launch
    // going to DRAM (the arrays of 64 resident warps do not fit L1), 0.87 GB read for 0.13 GB of input.
    auto a11_of = [&](int k) { double a, c, b; lpv_of(P, __ldg(R1 + (size_t)k * Ss + s), 0.0, 0.0, a, c, b); return a; };
    auto a21_of = [&](int k) { double a, c, b; lpv_of(P, 0.0, __ldg(R2 + (size_t)k * Ss + s), 0.0, a, c, b); return c; };
    auto bb_of = [&](int k) { double a, c, b; lpv_of(P, 0.0, 0.0, __ldg(R3 + (size_t)k * Ss + s), a, c, b); return b; };
    // Phi_i = A_i Phi_{i-1} (lower triangular), Lambda_i = A_i Lambda_{i-1} + C   (:17-22, :47-52)
    double f11 = 1.0, f21 = 0.0, f22 = 1.0, l1 = 0.0, l2 = 0.0;
    double *phi = Phi + s, *lam = Lam + s;
    for (int i = 0; i < N; ++i) {
        const double aa = a11_of(i), cc = a21_of(i);
        const double n21 = fma(cc, f11, P.a22 * f21);
        f11 = aa * f11; f21 = n21; f22 = P.a22 * f22;
        const double nl2 = fma(cc, l1, P.a22 * l2) + P.C2;
        l1 = aa * l1 + P.C1; l2 = nl2;
        phi[(size_t)(2 * i) * Ss] = f11;
        phi[(size_t)(2 * i + 1) * Ss] = f21;
        phi[(size_t)(2 * N + 2 * i) * Ss] = 0.0;
        phi[(size_t)(2 * N + 2 * i + 1) * Ss] = f22;
        lam[(size_t)(2 * i) * Ss] = l1;
        lam[(size_t)(2 * i + 1) * Ss] = l2;
    }
    // Gamma column c (:26-40): block (c,c) = B_c, below it A_k * previous with k = i (intent) or i - c - 1 (literal :32)
    double *gam = Gam + s;
    for (int c = 0; c < N; ++c) {
        double g1 = 0.0, g2 = 0.0;
        double *col = gam + (size_t)c * 2 * N * Ss;
        for (int i = 0; i < N; ++i) {
            if (i == c) { g1 = bb_of(c); g2 = 0.0; }
            else if (i > c) {
                const int k = gi ? i : (i - c - 1);
                const double aa = a11_of(k), cc = a21_of(k);
                const double n2 = fma(cc, g1, P.a22 * g2);
                g1 = aa * g1; g2 = n2;
            }
            col[(size_t)(2 * i) * Ss] = g1;
            col[(size_t)(2 * i + 1) * Ss] = g2;
        }
    }
}

cudaError_t launch_condense(cudaStream_t st, const DeviceProps &dp, int layout, int flags, int S, int N,
                            const double *R1, const double *R2, const double *R3, const double *params, int pc,
                            double *Phi, double *Gam, double *Lam, long long *launches) {
    if (S <= 0) return cudaSuccess;
    const int gw = gw_for(N);
    const int vec_ok = (layout == NTM_LAYOUT_MATLAB) && (((reinterpret_cast<uintptr_t>(Gam) | reinterpret_cast<uintptr_t>(Phi) |
                                                            reinterpret_cast<uintptr_t>(Lam)) & 15) == 0);
    if (layout == NTM_LAYOUT_SOA) {
        if (N <= 32) condense_soa_kernel<32><<<(S + 127) / 128, 128, 0, st>>>(flags, S, N, R1, R2, R3, params, pc, Phi, Gam, Lam);
        else condense_soa_kernel<NTM_MAX_HORIZON><<<(S + 127) / 128, 128, 0, st>>>(flags, S, N, R1, R2, R3, params, pc, Phi, Gam, Lam);
        ++*launches;
        return cudaGetLastError();
    }
    if (gw == 1) {
        const int wpb = 8;
        const int stage_tiles = (flags & NTM_PROFILE_GAMMA_I) && vec_ok;      // per-warp N x N double2 staging tiles
        const size_t smem = (size_t)wpb * 4 * N * sizeof(double) + (stage_tiles ? (size_t)wpb * N * N * sizeof(double2) : 0);
        long long need = ((long long)S + wpb - 1) / wpb;
        const long long cap = (long long)dp.sm_count * 32;
        const int grid = (int)(need < cap ? need : cap);
        if (smem > 48 * 1024) {
            int dev_ = 0; cudaGetDevice(&dev_);
            cudaError_t e = raise_smem_attribute(reinterpret_cast<const void *>(condense_kernel<1>), dev_, dp.smem_optin);
            if (e != cudaSuccess) return e;
        }
        condense_kernel<1><<<grid, 32 * wpb, smem, st>>>(layout, flags, S, N, R1, R2, R3, params, pc, Phi, Gam, Lam, vec_ok, stage_tiles);
    } else {
        const int stage_tiles = (flags & NTM_PROFILE_GAMMA_I) && vec_ok;      // one N x (RC + 1) double2 chunk tile per CTA
        const size_t smem = (size_t)4 * N * sizeof(double) + (stage_tiles ? (size_t)N * (NTM_COND_RC + 1) * sizeof(double2) : 0);
        const long long cap = (long long)dp.sm_count * 16;
        const int grid = (int)(S < cap ? S : cap);
        if (gw == 2) condense_kernel<2><<<grid, 64, smem, st>>>(layout, flags, S, N, R1, R2, R3, params, pc, Phi, Gam, Lam, vec_ok, stage_tiles);
        else condense_kernel<4><<<grid, 128, smem, st>>>(layout, flags, S, N, R1, R2, R3, params, pc, Phi, Gam, Lam, vec_ok, stage_tiles);
    }
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_hessian_grad(cudaStream_t st, const DeviceProps &dp, int layout, int S, int N, const double *Phi,
                                const double *Gam, const double *Lam, const double *x, const double *params, int pc,
                                double *G, double *F, long long *launches) {
    if (S <= 0) return cudaSuccess;
    const int gw = gw_for(N);
    int grid = 1;
    cudaError_t e;
    if (N > 32) {                                            // FP64 tensor-core path
        const int Np = (N + 1 + 7) & ~7, nt = Np >> 3, nst = (nt + 1) >> 1, nsuper = nst * (nst + 1) / 2;
        // the raw chunk and its Omega image, two v buffers, the super-tile table
        const size_t smem_d = (2 * (size_t)Np * NTM_DMMA_KC + 2 * (2 * N + 4)) * sizeof(double) + 2 * (size_t)nsuper + 16;
        const int maxst = (nsuper + 7) / 8;                  // 8 warps per CTA
#define NTM_LAUNCH_HD(M)                                                                                     \
    do {                                                                                                     \
        e = persistent_geometry(hessian_grad_dmma_kernel<M>, dp, 256, smem_d, S, 1, &grid);                  \
        if (e != cudaSuccess) return e;                                                                      \
        hessian_grad_dmma_kernel<M><<<grid, 256, smem_d, st>>>(layout, S, N, Phi, Gam, Lam, x, params, pc, G, F); \
    } while (0)
        if (maxst <= 2) NTM_LAUNCH_HD(2); else if (maxst <= 4) NTM_LAUNCH_HD(4); else if (maxst == 5) NTM_LAUNCH_HD(5);
        else NTM_LAUNCH_HD(6);
#undef NTM_LAUNCH_HD
        ++*launches;
        return cudaGetLastError();
    }
    if (layout == NTM_LAYOUT_MATLAB) {                       // N <= 32: one warp per scenario, tensor cores, 8 scenarios per CTA
        const int Np = (N + 1 + 7) & ~7, Kp = (2 * N + 3) & ~3;  // one spare column for v = Phi x + Lambda - R (F on the tensor cores)
        int ld = Kp;
        while ((ld & 7) != 4) ++ld;
        size_t slice = (size_t)Np * ld;
        if (slice < (size_t)N * N + N) slice = (size_t)N * N + N;  // the slice is reused as the G, F staging area
        (void)slice;
        const int wpb = 4;                                       // warps per CTA, each with a double-buffered slice
        const size_t smem_w = (size_t)wpb * 2 * ((size_t)Np * ld) * sizeof(double);
        const int aligned = ((reinterpret_cast<uintptr_t>(Gam) | reinterpret_cast<uintptr_t>(G)) & 15) == 0;
        const int NT = Np >> 3;
#define NTM_LAUNCH_HW(T)                                                                                              \
    do {                                                                                                              \
        e = persistent_geometry(hessian_grad_dmma_warp_kernel<T>, dp, 32 * wpb, smem_w, S, wpb, &grid);               \
        if (e != cudaSuccess) return e;                                                                               \
        hessian_grad_dmma_warp_kernel<T><<<grid, 32 * wpb, smem_w, st>>>(S, N, ld, Phi, Gam, Lam, x, params, pc, G, F, aligned); \
    } while (0)
        if (NT == 1) NTM_LAUNCH_HW(1); else if (NT == 2) NTM_LAUNCH_HW(2); else if (NT == 3) NTM_LAUNCH_HW(3);
        else if (NT == 4) NTM_LAUNCH_HW(4); else NTM_LAUNCH_HW(5);
#undef NTM_LAUNCH_HW
        ++*launches;
        return cudaGetLastError();
    }
    const int CH = N <= 32 ? N : 16;
    const size_t smem = ((size_t)N * odd_ld(N) + (size_t)N * (2 * CH + 1) + 2 * N) * sizeof(double);
    if (gw == 1) {
        e = persistent_geometry(hessian_grad_kernel<1>, dp, 32, smem, S, 1, &grid);
        if (e != cudaSuccess) return e;
        hessian_grad_kernel<1><<<grid, 32, smem, st>>>(layout, S, N, CH, Phi, Gam, Lam, x, params, pc, G, F);
    } else if (gw == 2) {
        e = persistent_geometry(hessian_grad_kernel<2>, dp, 64, smem, S, 1, &grid);
        if (e != cudaSuccess) return e;
        hessian_grad_kernel<2><<<grid, 64, smem, st>>>(layout, S, N, CH, Phi, Gam, Lam, x, params, pc, G, F);
    } else {
        e = persistent_geometry(hessian_grad_kernel<4>, dp, 128, smem, S, 1, &grid);
        if (e != cudaSuccess) return e;
        hessian_grad_kernel<4><<<grid, 128, smem, st>>>(layout, S, N, CH, Phi, Gam, Lam, x, params, pc, G, F);
    }
    ++*launches;
    return cudaGetLastError();
}

// FP64 tensor-core microbenchmark: 8 independent register-resident DMMA.8x8x4 accumulator chains per warp
__global__ void __launch_bounds__(256) dmma_peak_kernel(int iters, double *out) {
    double c[8][2];
#pragma unroll
    for (int u = 0; u < 8; ++u) { c[u][0] = threadIdx.x * 1e-3 + u; c[u][1] = c[u][0] + 0.5; }
    const double a = 1.0000001 * ((threadIdx.x & 3) == 0 ? 1.0 : 1e-9), b = 0.9999999 * ((threadIdx.x & 3) == 0 ? 1.0 : 1e-9);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) dmma_m8n8k4(c[u][0], c[u][1], a, b);
    }
    double r = 0.0;
#pragma unroll
    for (int u = 0; u < 8; ++u) r += c[u][0] + c[u][1];
    if (r == 12345.678) out[0] = r;   // keeps the chains alive without a store in the common case
}

cudaError_t launch_dmma_peak(cudaStream_t st, const DeviceProps &dp, int iters, double *out, long long *launches) {
    dmma_peak_kernel<<<dp.sm_count * 8, 256, 0, st>>>(iters, out);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_fp64_peak(cudaStream_t st, const DeviceProps &dp, int iters, double *out, long long *launches) {
    fp64_peak_kernel<<<dp.sm_count * 8, 256, 0, st>>>(iters, out);
    ++*launches;
    return cudaGetLastError();
}

}  // namespace ntm
