// ntm_long.cuh -- long horizons (N > 32) of the fused loop, literal Gamma, EC-power box QP (NTM_MPC_Sim.m:97,119-121).
//
// Round 1 solved these QPs (60-99 free variables out of N = 100) with an LDL' factor of the free block that was kept
// up to date by chains of barrier-separated O(1) steps (2m for a solve, m for an append, m for a delete): ~460 k cycles
// per re-linearisation, one CTA per SM (80 KB Hessian + 80 KB factor), 1.9 % of the FP64 roofline.  Here the solver
// state is ONE symmetric *sweep tableau*, packed lower-triangular in shared memory, and every active-set step is a
// rank-one update of it -- O(N^2 / threads) independent FMAs per thread between two barriers, no substitution chains:
//
//     T = [ G  g ]   (N+1) x (N+1),  g = G u + F at the current point u.
//         [ g' . ]
//   sweep(k), k joins the free set F:   T(i,j) -= T(i,k) T(k,j) / T(k,k),  T(i,k) /= T(k,k),  T(k,k) = -1/T(k,k)
//   after sweeping F:  T_FF = -inv(G_FF),  T_BF = G_BF inv(G_FF),  T_BB = the Schur complement, and the border row
//   holds  y_F = inv(G_FF) g_F  (minus the Newton step to the minimiser on the face) and  y_B = g_B - G_BF inv(G_FF) g_F
//   (the bound multipliers AT that minimiser).  So the ratio test and the multiplier test read the border row, a
//   partial step alpha scales y_F by (1 - alpha), a blocking variable leaves by the reverse sweep and a released bound
//   joins by a sweep: no mat-vec and no triangular solve inside the iteration.
// G itself is not kept: the literal Hessian is Gy(j,l) = 2 T[N-1-j][j-l] (build_GF_toeplitz) and the exact gradient
// that certifies the answer is evaluated in Gamma form from the N columns p_d (two triangular convolutions), so a
// scenario needs 42 KB + vectors instead of 160 KB and three CTAs share an SM.
// Accuracy: pivots of an SPD matrix in any order are positive; the tableau only PROPOSES the partition and the step --
// the stop test uses the exact gradient, and a failed test re-derives the border row from it (iterative refinement) or
// rebuilds the tableau from the stage entries.
#pragma once
#include "ntm_device.cuh"

namespace ntm {

// packed lower triangle, row r holds r + 1 entries and starts at an even offset (16-byte aligned double2 accesses)
__host__ __device__ __forceinline__ int tri_off(int r) { return 2 * ((r + 1) >> 1) * ((r + 2) >> 1); }

__host__ __device__ inline int tile_pcn(int N) { return (((N + 1 + 6) / 7) * 7 + 9) & ~1; }   // NTM_TS = 7 blocks, padded

__host__ __device__ inline size_t work_bytes_long(int N) {
    // T: tri_off(N + 1) | vectors: cand 4N, P12 2N, QP12 4N, QE12 4N (double2 arrays) | pc, pcs: N + 3 each (even) |
    // a11s a21s bbs qv uv sol: 6N | red 8 | prm 16 | ints: idx N + 8
    const size_t dbl = (size_t)tri_off(N + 1) + 14 * (size_t)N + 2 * (size_t)((N + 4) & ~1) + 6 * (size_t)N + 8 + 16 +
                       3 * (size_t)tile_pcn(N) + (size_t)((N + 1) & ~1);
    const size_t b = dbl * 8 + ((size_t)N + 8) * 4;
    return (b + 15) & ~(size_t)15;
}

struct LongWork : Work {
    double *pc, *pcs;          // pivot column and pivot column / pivot, N + 2 entries (+ zero padding)
    double *tpcb, *tybuf, *tgbuf;   // register-tile variant: column buffers (2 x tpcn), published border row, seed gradient
    int tpcn;
};

__device__ inline LongWork carve_long(unsigned char *base, int N) {
    LongWork w;
    double2 *v = reinterpret_cast<double2 *>(base);
    w.G = reinterpret_cast<double *>(v); v += tri_off(N + 1) / 2;                   // the tableau
    w.cand = v; v += 2 * N; w.P12 = v; v += N; w.QP12 = v; v += 2 * N; w.QE12 = v; v += 2 * N;
    const int pcn = (N + 4) & ~1;
    w.pc = reinterpret_cast<double *>(v); v += pcn / 2;
    w.pcs = reinterpret_cast<double *>(v); v += pcn / 2;
    w.tpcn = tile_pcn(N);
    w.tpcb = reinterpret_cast<double *>(v); v += w.tpcn;                             // 2 buffers
    w.tybuf = reinterpret_cast<double *>(v); v += w.tpcn / 2;
    w.tgbuf = reinterpret_cast<double *>(v); v += ((N + 1) & ~1) / 2;
    w.GamS = nullptr; w.ldgam = 0; w.ldg = 0; w.hcap = 0; w.H = nullptr; w.Hbig = nullptr;
    double *d = reinterpret_cast<double *>(v);
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
// Literal Hessian into the packed tableau: T(jj, ll) = Gy(jj, ll) = 2 sum_{d <= N-1-jj} p_d' Q p_{d + jj - ll}, jj >= ll
// (Rho_to_PhiGammaLambda.m:28-40 with index i-j, NTM_MPC_Sim.m:120), and Fy_j (:121).  Same arithmetic and summation
// order as build_GF_toeplitz; one store per entry.  Thread j: lag j of the table, entry j of F.
// ------------------------------------------------------------------------------------------------
template <int GW>
__device__ double build_GF_toeplitz_packed(int N, int j, const LongWork &w, const Params &P, double xF1, double xF2) {
    using Gp = Group<GW>;
    const bool act = j < N;
    double myp1 = 0.0, myp2 = 0.0, mye1 = 0.0, mye2 = 0.0;
    {
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
        const int mmax = N - j;
        for (int m = 0; m < mmax; ++m) {
            const double2 p = pp[m], a = qp[m], e = qe[m];
            accF = fma(p.x, e.x, accF); accF = fma(p.y, e.y, accF);
            accG = fma(p.x, a.x, accG); accG = fma(p.y, a.y, accG);
            const int jj = N - 1 - m;
            w.G[tri_off(jj) + (jj - j)] = accG;
        }
        Fj = accF;
    }
    Gp::sync();
    return Fj;
}

// ------------------------------------------------------------------------------------------------
// One pivot of the tableau (n1 = N + 1 rows).  forward: variable k joins the swept set; !forward: it leaves.
// Returns false (group-uniform) when the pivot has the wrong sign or is not finite (numerical breakdown; nothing is
// changed).  3 barriers; the rank-one pass folds row r with row n1-1-r so that every work unit has n1 + 1 entries, two
// threads per unit, 16-byte accesses.
// ------------------------------------------------------------------------------------------------
template <int GW>
__device__ bool tab_pivot(int n1, int k, bool forward, const LongWork &w, int tid) {
    using Gp = Group<GW>;
    constexpr int NT = Gp::T;
    double *__restrict__ T = w.G;
    const double d = T[tri_off(k) + k];
    if (forward ? !(d > 0.0 && d < 1.7e308) : !(d < 0.0 && d > -1.7e308)) return false;   // same word for everyone
    const double inv = 1.0 / d;
    double mycs[2];
    // 1. extract column k (symmetric access) and its scaled copy; entry k itself is zeroed for the pass
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int i = tid + q * NT;
        mycs[q] = 0.0;
        if (i < n1) {
            const double c = (i >= k) ? T[tri_off(i) + k] : T[tri_off(k) + i];
            const double cs = c * inv;
            mycs[q] = cs;
            w.pc[i] = (i == k) ? 0.0 : c;
            w.pcs[i] = (i == k) ? 0.0 : cs;
        } else if (i < n1 + 2) {
            w.pc[i] = 0.0; w.pcs[i] = 0.0;                    // padding read by the last double2 of a row
        }
    }
    Gp::sync();
    // 2. T(i,j) -= c_i * cs_j over the lower triangle
    {
        const int half = (n1 + 1) >> 1;                       // folded work units: rows (u, n1-1-u)
        const double2 *__restrict__ cs2 = reinterpret_cast<const double2 *>(w.pcs);
        for (int wu = tid; wu < 2 * half; wu += NT) {
            const int u = wu >> 1, q = wu & 1;
            const int rA = u, rB = n1 - 1 - u;
            {
                const double ci = w.pc[rA];
                double2 *__restrict__ row = reinterpret_cast<double2 *>(T + tri_off(rA));
                const int nch = (rA + 2) >> 1;                // double2 chunks of row rA (r + 1 entries, padded even)
                for (int c = q; c < nch; c += 2) {
                    double2 t = row[c];
                    const double2 s = cs2[c];
                    t.x = fma(-ci, s.x, t.x); t.y = fma(-ci, s.y, t.y);
                    row[c] = t;
                }
            }
            if (rB != rA) {
                const double ci = w.pc[rB];
                double2 *__restrict__ row = reinterpret_cast<double2 *>(T + tri_off(rB));
                const int nch = (rB + 2) >> 1;
                for (int c = 1 - q; c < nch; c += 2) {        // the other parity: the two threads of a unit stay balanced
                    double2 t = row[c];
                    const double2 s = cs2[c];
                    t.x = fma(-ci, s.x, t.x); t.y = fma(-ci, s.y, t.y);
                    row[c] = t;
                }
            }
        }
    }
    Gp::sync();
    // 3. the pivot column itself
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int i = tid + q * NT;
        if (i < n1) {
            if (i == k) T[tri_off(k) + k] = -inv;
            else {
                const double v = forward ? mycs[q] : -mycs[q];
                if (i > k) T[tri_off(i) + k] = v; else T[tri_off(k) + i] = v;
            }
        }
    }
    Gp::sync();
    return true;
}

// gout_j = (Gy v)_j for v = w.uv[0..N) in Gamma form: z_i = sum_{c <= i} p_{i-c} v_c, (Gy v)_l = sum_{i >= l} (2 Q p_{i-l})' z_i
// (w.P12, w.QP12 of the current condensation; w.QE12 is free after the build and holds z).  Caller adds Fy.
template <int GW>
__device__ double gamma_form_Gv(int N, int j, const LongWork &w) {
    using Gp = Group<GW>;
    const bool act = j < N;
    if (act) {
        double z1 = 0.0, z2 = 0.0;
        const double2 *pp = w.P12 + j;
        const double *vv = w.uv;
        for (int c = 0; c <= j; ++c, --pp) {
            const double2 p = *pp;
            const double v = vv[c];
            z1 = fma(p.x, v, z1); z2 = fma(p.y, v, z2);
        }
        w.QE12[j] = make_double2(z1, z2);
    }
    Gp::sync();
    double g = 0.0;
    if (act) {
        const double2 *qp = w.QP12, *zz = w.QE12 + j;
        for (int m = 0; m < N - j; ++m) {
            const double2 a = qp[m], z = zz[m];
            g = fma(a.x, z.x, g); g = fma(a.y, z.y, g);
        }
    }
    Gp::sync();
    return g;
}

// t_j = sum_{k : msk_k != 0} T(j,k) * vec_k over the N x N part of the packed tableau (row-owner, symmetric access)
__device__ __forceinline__ double tab_row_dot(int N, int j, const double *__restrict__ T, const double *__restrict__ vec) {
    double t0 = 0.0, t1 = 0.0;
    const double *row = T + tri_off(j);
    int k = 0;
    for (; k + 1 <= j; k += 2) { t0 = fma(row[k], vec[k], t0); t1 = fma(row[k + 1], vec[k + 1], t1); }
    for (; k <= j; ++k) t0 = fma(row[k], vec[k], t0);
    for (k = j + 1; k < N; ++k) t1 = fma(T[tri_off(k) + j], vec[k], t1);
    return t0 + t1;
}

#define NTM_LONG_REFINE_TOL 1e-9
#define NTM_LONG_MAX_REPAIRS 4

// ------------------------------------------------------------------------------------------------
// Box QP  min 1/2 y'Gy y + Fy'y, lb <= y <= ub  with Gy in w.G as left by build_GF_toeplitz_packed.  Same contract as
// qp_solve (bound components exactly lb/ub, history of the last two solutions as warm starts, unique minimiser of a
// strictly convex problem).  regen() rebuilds w.G (= Gy) from the stage entries.  Overwrites w.G.
// ------------------------------------------------------------------------------------------------
template <int GW, class Regen>
__device__ int qp_solve_long(int N, int j, const LongWork &w, double Fj, double lbj, double ubj, QpHist &hist, double &Uout,
                             int max_iter, int &iters_out, const Regen &regen) {
    using Gp = Group<GW>;
    const bool act = j < N;
    const int n1 = N + 1;
    const bool pinned = !(ubj > lbj);
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    double *__restrict__ T = w.G;
    double *yrow = T + tri_off(N);                      // border row: y_0 .. y_{N-1}, corner
    int status = NTM_SCN_QP_ITER_CAP, it = 0;
    bool broke = false;

    // ---- one pass over T = Gy: gradient at the candidate points and a fixed gradient scale for this QP
    //      sc_j = |F_j| + sum_k |G_jk| max(|lb_k|, |ub_k|)  (rounding level of any gradient component inside the box)
    const double cu1 = (hist.n >= 1) ? hist.u1 : lbj, cu2 = (hist.n >= 2) ? hist.u2 : lbj;
    if (act) {
        w.cand[2 * j] = make_double2(lbj, ubj);
        w.cand[2 * j + 1] = make_double2(cu2, cu1);
    }
    Gp::sync();
    double g0 = 0.0, g1 = 0.0, g2 = 0.0, g3 = 0.0, sc = 0.0;
    if (act) {
        const double *row = T + tri_off(j);
        for (int k = 0; k < N; ++k) {
            const double gk = (k <= j) ? row[k] : T[tri_off(k) + j];
            const double2 ca = w.cand[2 * k], cb = w.cand[2 * k + 1];
            g0 = fma(gk, ca.x, g0); g1 = fma(gk, ca.y, g1);
            g2 = fma(gk, cb.x, g2); g3 = fma(gk, cb.y, g3);
            sc = fma(fabs(gk), fmax(fabs(ca.x), fabs(ca.y)), sc);
        }
        sc += fabs(Fj);
    }
    // ---- cold start: the clipped unconstrained minimiser as a candidate (all variables swept once)
    if (hist.n == 0) {
        if (act) yrow[j] = g0 + Fj;
        if (j == 0) yrow[N] = 0.0;
        Gp::sync();
        bool ok = true;
        for (int k = 0; k < N && ok; ++k) ok = tab_pivot<GW>(n1, k, true, w, j);
        double un = act ? lbj - yrow[j] : 0.0;
        ok = ok && !Gp::any(act && !isfinite(un), w.ired);
        if (ok) {
            hist.u2 = fmin(fmax(un, lbj), ubj);
            hist.s2 = (un <= lbj) ? -1 : ((un >= ubj) ? 1 : 0);
            hist.u1 = hist.u2; hist.s1 = hist.s2;
            hist.n = 2;
        }
        Gp::sync();
        regen();
        Gp::sync();
        if (ok) {                                       // gradient of the new candidate (history slots 2 and 3 are the same point)
            if (act) w.uv[j] = hist.u2;
            Gp::sync();
            const double t = act ? tab_row_dot(N, j, T, w.uv) : 0.0;
            g2 = t; g3 = t;
            Gp::sync();
        }
    }
    const double c2v = (hist.n >= 2) ? hist.u2 : lbj, c3v = (hist.n >= 1) ? hist.u1 : lbj;
    // ---- start: the candidate with the lowest objective (all-lower, all-upper, the two previous solutions)
    int state = -1;
    double u = lbj, g = g0 + Fj;
    {
        const double q0 = Gp::sum(act ? lbj * fma(0.5, g0, Fj) : 0.0, w.red);
        const double q1 = Gp::sum(act ? ubj * fma(0.5, g1, Fj) : 0.0, w.red);
        double qb = q0;
        if (q1 < qb) { qb = q1; state = 1; u = ubj; g = g1 + Fj; }
        if (hist.n >= 2) {
            const double q2 = Gp::sum(act ? c2v * fma(0.5, g2, Fj) : 0.0, w.red);
            if (q2 < qb) { qb = q2; state = hist.s2; u = c2v; g = g2 + Fj; }
        }
        if (hist.n >= 1) {
            const double q3 = Gp::sum(act ? c3v * fma(0.5, g3, Fj) : 0.0, w.red);
            if (q3 < qb) { qb = q3; state = hist.s1; u = c3v; g = g3 + Fj; }
        }
        if (pinned) { state = -1; u = lbj; }
    }

    // sweeps every free variable of the current partition into a fresh tableau whose border row holds g
    auto enter_partition = [&](double gj) -> bool {
        if (act) { yrow[j] = gj; w.idx[j] = state; }
        if (j == 0) yrow[N] = 0.0;
        Gp::sync();
        bool ok = true;
        for (int k = 0; k < N; ++k) {
            if (w.idx[k] != 0) continue;                                  // uniform: same word
            if (!tab_pivot<GW>(n1, k, true, w, j)) {                      // dependent direction: the variable stays where it is
                ok = false;
                if (j == k) { state = (u - lbj <= ubj - u) ? -1 : 1; u = (state < 0) ? lbj : ubj; }
            }
        }
        return ok;
    };
    broke |= !enter_partition(g);

    int repairs = 0, since_build = 0;
    bool stuck = false;                                  // this thread's variable could not be pivoted in (kept on its bound)
    for (it = 1; it <= max_iter; ++it) {
        const bool isfree = act && state == 0;
        const double yj = act ? yrow[j] : 0.0;
        const bool anyfree = Gp::any(isfree, w.ired);
        if (anyfree) {
            const double pj = -yj;                                        // Newton step to the minimiser on the face
            double aj = INF;
            if (isfree) {
                if (pj < 0.0) aj = (lbj - u) / pj;
                else if (pj > 0.0) aj = (ubj - u) / pj;
            }
            int jblk;
            const double amin = Gp::argmin(aj, j, w.red, w.ired, jblk);
            if (amin < 1.0) {                                             // a bound blocks: partial step, the variable leaves
                const double alpha = fmax(amin, 0.0);
                if (isfree) {
                    u = fma(alpha, pj, u);
                    yrow[j] = (1.0 - alpha) * yj;
                }
                if (j == jblk) { state = (pj < 0.0) ? -1 : 1; u = (pj < 0.0) ? lbj : ubj; }
                Gp::sync();
                if (!tab_pivot<GW>(n1, jblk, false, w, j)) { broke = true; break; }
                ++since_build;
                continue;
            }
            if (isfree) { u += pj; yrow[j] = 0.0; }                       // full step: u is the minimiser on the face
        }
        // bound multipliers at the face minimiser, as the tableau sees them
        double lam = INF;
        if (act && !pinned && !stuck) {
            if (state < 0) lam = yj / sc;
            else if (state > 0) lam = -yj / sc;
        }
        int jw;
        const double lmin = Gp::argmin(lam, j, w.red, w.ired, jw);
        if (lmin < -NTM_QP_EPS_G) {                                       // variable jw leaves its bound
            Gp::sync();
            if (tab_pivot<GW>(n1, jw, true, w, j)) { if (j == jw) state = 0; }
            else if (j == jw) stuck = true;                               // numerically dependent direction: stays on its bound
            ++since_build;
            continue;
        }
        // ---- the tableau says optimal: certify with the exact gradient (Gamma form), repair if it disagrees
        if (act) w.uv[j] = u;
        Gp::sync();
        const double ge = gamma_form_Gv<GW>(N, j, w) + Fj;
        bool bad = false;
        if (act && !pinned) {
            if (state == 0) bad = fabs(ge) > NTM_LONG_REFINE_TOL * sc;
            else bad = ((state < 0) ? ge : -ge) < -NTM_QP_EPS_G * sc;
        }
        if (!Gp::any(bad, w.ired)) { status = NTM_SCN_OK; g = ge; break; }
        if (repairs >= NTM_LONG_MAX_REPAIRS) { status = NTM_SCN_OK; g = ge; break; }   // as good as fp64 gets here
        ++repairs;
        if (repairs >= 2 || since_build > 3 * N) {
            // rebuild the tableau from the stage entries and re-enter the partition at the current point
            regen();
            Gp::sync();
            broke |= !enter_partition(ge);
            since_build = 0;
        } else {
            // border row from the exact gradient: y_F = -T_FF g_F, y_B = g_B - T_BF g_F
            if (act) w.sol[j] = (state == 0) ? ge : 0.0;
            Gp::sync();
            const double t = act ? tab_row_dot(N, j, T, w.sol) : 0.0;
            Gp::sync();
            if (act) yrow[j] = (state == 0) ? -t : ge - t;
            Gp::sync();
        }
    }
    if (it > max_iter) it = max_iter;
    // a pinned variable (lbj == ubj) has one value either way; its state is the side the gradient points to, which is
    // what the literal kernels map back to U: b * [umin, umax] can round to one y although umin < umax
    if (pinned) state = (g < 0.0) ? 1 : -1;
    const bool nonfinite = Gp::any(act && !(isfinite(u) && isfinite(g)), w.ired);
    double Uj = (state < 0) ? lbj : ((state > 0) ? ubj : fmin(fmax(u, lbj), ubj));
    if (nonfinite) Uj = nan("");
    if (nonfinite || broke) status = NTM_SCN_NONFINITE;
    hist.u2 = hist.u1; hist.s2 = hist.s1;
    hist.u1 = Uj; hist.s1 = state;
    hist.n = min(hist.n + 1, 2);
    Gp::sync();
    Uout = Uj;
    iters_out = it;
    return status;
}


// =================================================================================================
// Register-resident tableau.  The shared-memory tableau above moves 3 x 41 KB through the shared-memory pipe per pivot
// (read T, read the scaled column, write T: one FMA per 24 bytes) and three CTAs on an SM simply queue up behind that
// pipe (measured: 205 k scenario-steps/s at N = 100, no overlap between the CTAs).  Here the (N+1) x (N+1) symmetric
// tableau is cut into TS x TS blocks, thread I(I+1)/2 + J keeps block (I, J), I >= J, in REGISTERS (49 doubles), and
// a pivot is: the owners of block column / block row K publish the pivot column (one double per row) to shared
// memory, one barrier, every thread reads the 7 + 7 entries its block needs and does 49 independent FMAs.  Shared
// memory traffic per pivot: 128 x 14 doubles instead of 15,000; barriers per pivot: 1 (the column buffer is
// double-buffered).  Tableau index 0 is the border (gradient) row -- a compile-time register index for its owners --,
// index v + 1 is QP variable v.  The Hessian Gy stays intact in shared memory (packed): it seeds the blocks, gives the
// exact gradient that certifies the answer, and makes a rebuild a reload.
// =================================================================================================
#define NTM_TS 7

struct Tile {
    double t[NTM_TS][NTM_TS];
};

// block coordinates of thread tid: tid = I (I + 1) / 2 + J, 0 <= J <= I < nb; I = -1 when the thread holds no block
__device__ inline void tile_coords(int tid, int nb, int &I, int &J) {
    int i = (int)((sqrtf(8.0f * (float)tid + 1.0f) - 1.0f) * 0.5f);
    while ((i + 1) * (i + 2) / 2 <= tid) ++i;
    while (i * (i + 1) / 2 > tid) --i;
    I = i; J = tid - i * (i + 1) / 2;
    if (I >= nb) { I = -1; J = -1; }
}

struct TileWork {
    double *pcb;       // 2 x pcn doubles: pivot column, double-buffered
    double *ybuf;      // pcn doubles: published border row
    double *gbuf;      // N doubles: gradient that seeds the border row
    int pcn;
};

// tableau entry (a, b) of the UNSWEPT tableau: border = gradient (index 0), Gy at (a-1, b-1); 0 outside
__device__ __forceinline__ double seed_entry(int a, int b, int n1, const double *__restrict__ Gy, const double *__restrict__ gb) {
    if (a < b) { const int t = a; a = b; b = t; }
    if (a >= n1) return 0.0;
    if (b == 0) return (a == 0) ? 0.0 : gb[a - 1];
    return Gy[tri_off(a - 1) + (b - 1)];
}

__device__ __forceinline__ void tile_load(Tile &tl, int I, int J, int n1, const double *__restrict__ Gy,
                                          const double *__restrict__ gb) {
    if (I < 0) return;
    // lower part of the block straight from the packed Hessian (a >= b there, so no symmetric swap): row a-1 of Gy is
    // contiguous; column 0 of the blocks (I, 0) is the border (gradient); the upper part of a diagonal block mirrors
#pragma unroll
    for (int r = 0; r < NTM_TS; ++r) {
        const int a = NTM_TS * I + r;
        const bool in = a < n1 && a >= 1;
        const double *row = Gy + (in ? tri_off(a - 1) : 0) + NTM_TS * J - 1;
#pragma unroll
        for (int c = 0; c < NTM_TS; ++c) {
            double v = 0.0;
            if (c == 0 && J == 0) v = in ? gb[a - 1] : 0.0;                   // tableau column 0
            else if (in && NTM_TS * J + c <= a) v = row[c];                  // Gy(a-1, b-1), b <= a
            tl.t[r][c] = v;
        }
    }
    if (I == J) {
#pragma unroll
        for (int r = 0; r < NTM_TS; ++r)
#pragma unroll
            for (int c = r + 1; c < NTM_TS; ++c) tl.t[r][c] = tl.t[c][r];
    }
}

// One pivot on tableau index k.  np = number of pivots done so far in this QP (selects the column buffer).
// Returns false (uniform) on a pivot of the wrong sign / non-finite; the tableau is then unchanged.
template <int GW>
__device__ __forceinline__ bool tile_pivot(Tile &tl, int I, int J, int k, bool forward, const TileWork &tw, int &np) {
    using Gp = Group<GW>;
    const int K = k / NTM_TS, kc = k - K * NTM_TS;
    double *__restrict__ pc = tw.pcb + (np & 1) * tw.pcn;
    ++np;
    if (I >= 0) {
        if (J == K) {                                   // block column K: T(TS*I + r, k) = t[r][kc]
            double *dst = pc + NTM_TS * I;
            switch (kc) {
#define NTM_CASE(q) case q: _Pragma("unroll") for (int r = 0; r < NTM_TS; ++r) dst[r] = tl.t[r][q]; break;
                NTM_CASE(0) NTM_CASE(1) NTM_CASE(2) NTM_CASE(3) NTM_CASE(4) NTM_CASE(5) NTM_CASE(6)
#undef NTM_CASE
            }
            if (I == K) {                               // the pivot itself: d and 1/d go to the two spare slots (one division per
                const double dd = dst[kc];              // pivot, not one per thread).  The column entry k is published as -+1:
                pc[tw.pcn - 2] = dd;                    // times sg = +-1/d that IS the new T(k,k) = -1/d, so the rewrite of
                pc[tw.pcn - 1] = 1.0 / dd;              // column / row k below needs no select; whatever the rank-one pass
                dst[kc] = forward ? -1.0 : 1.0;         // leaves in row and column k is overwritten by that rewrite
            }
        } else if (I == K) {                            // block row K (J < K): T(k, TS*J + c) = t[kc][c]
            double *dst = pc + NTM_TS * J;
            switch (kc) {
#define NTM_CASE(q) case q: _Pragma("unroll") for (int c = 0; c < NTM_TS; ++c) dst[c] = tl.t[q][c]; break;
                NTM_CASE(0) NTM_CASE(1) NTM_CASE(2) NTM_CASE(3) NTM_CASE(4) NTM_CASE(5) NTM_CASE(6)
#undef NTM_CASE
            }
        }
    }
    Gp::sync();
    const double d = pc[tw.pcn - 2];
    if (forward ? !(d > 0.0 && d < 1.7e308) : !(d < 0.0 && d > -1.7e308)) { --np; Gp::sync(); return false; }
    if (I >= 0) {
        const double inv = pc[tw.pcn - 1];                        // 1 / d, computed once by the owner of the pivot's block
        const double sg = forward ? inv : -inv;
        double ci[NTM_TS], cj[NTM_TS];
#pragma unroll
        for (int r = 0; r < NTM_TS; ++r) ci[r] = pc[NTM_TS * I + r];
#pragma unroll
        for (int c = 0; c < NTM_TS; ++c) cj[c] = pc[NTM_TS * J + c];
        double am[NTM_TS], bs[NTM_TS];                            // -c_i, c_j / d
#pragma unroll
        for (int r = 0; r < NTM_TS; ++r) am[r] = -ci[r];
#pragma unroll
        for (int c = 0; c < NTM_TS; ++c) bs[c] = cj[c] * inv;
#pragma unroll
        for (int r = 0; r < NTM_TS; ++r)
#pragma unroll
            for (int c = 0; c < NTM_TS; ++c) tl.t[r][c] = fma(am[r], bs[c], tl.t[r][c]);
        if (J == K) {
            switch (kc) {
#define NTM_CASE(q) case q: _Pragma("unroll") for (int r = 0; r < NTM_TS; ++r) tl.t[r][q] = ci[r] * sg; break;
                NTM_CASE(0) NTM_CASE(1) NTM_CASE(2) NTM_CASE(3) NTM_CASE(4) NTM_CASE(5) NTM_CASE(6)
#undef NTM_CASE
            }
        }
        if (I == K) {
            switch (kc) {
#define NTM_CASE(q) case q: _Pragma("unroll") for (int c = 0; c < NTM_TS; ++c) tl.t[q][c] = cj[c] * sg; break;
                NTM_CASE(0) NTM_CASE(1) NTM_CASE(2) NTM_CASE(3) NTM_CASE(4) NTM_CASE(5) NTM_CASE(6)
#undef NTM_CASE
            }
        }
    }
    return true;
}

// out_a += sum_b T(a, b) v_b over the whole (symmetric) tableau held in the blocks: every thread multiplies its block
// (and, off the diagonal, its transpose) and adds 7 + 7 partial sums into shared memory.  out must be zeroed, v and out
// hold 7 * nb entries.  Used once or twice per QP (iterative refinement of the border row), so the atomics do not matter.
__device__ __forceinline__ void tile_matvec(const Tile &tl, int I, int J, const double *__restrict__ v, double *out) {
    if (I < 0) return;
    double vi[NTM_TS], vj[NTM_TS];
#pragma unroll
    for (int r = 0; r < NTM_TS; ++r) { vi[r] = v[NTM_TS * I + r]; vj[r] = v[NTM_TS * J + r]; }
#pragma unroll
    for (int r = 0; r < NTM_TS; ++r) {
        double acc = 0.0;
#pragma unroll
        for (int c = 0; c < NTM_TS; ++c) acc = fma(tl.t[r][c], vj[c], acc);
        atomicAdd(out + NTM_TS * I + r, acc);
    }
    if (I != J) {
#pragma unroll
        for (int c = 0; c < NTM_TS; ++c) {
            double acc = 0.0;
#pragma unroll
            for (int r = 0; r < NTM_TS; ++r) acc = fma(tl.t[r][c], vi[r], acc);
            atomicAdd(out + NTM_TS * J + c, acc);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Box QP on the register-resident tableau.  Gy (packed, intact) in w.G.  Same contract as qp_solve.
// Written as ONE loop with a single pivot site, a single block-load site and a single refinement site: the pivot
// routine is ~600 instructions and the block load ~700, and five inlined copies (11.5 k instructions, 184 KB of code)
// did not fit the instruction cache.  Phases:
//   COLD    (first QP of a scenario) every variable is swept once: the clipped unconstrained minimiser joins the
//           start candidates;
//   SELECT  the candidate with the lowest objective (all-lower, all-upper, the two previous solutions) is the start;
//   ENTER   fresh blocks, border row = gradient at the current point, every free variable swept in;
//   ITER    ratio test / multiplier test on the border row, one pivot per pass; when the tableau says "optimal" the
//           exact gradient decides, and if it disagrees the border row is re-derived from it (one step of iterative
//           refinement: the explicit inverse in the tableau is accurate to cond * eps, the refined step to its square).
// ------------------------------------------------------------------------------------------------
template <int GW>
__device__ int qp_solve_tile(int N, int j, const LongWork &w, const TileWork &tw, int I, int J, double Fj, double lbj,
                             double ubj, QpHist &hist, double &Uout, int max_iter, int &iters_out) {
    using Gp = Group<GW>;
    const bool act = j < N;
    const int n1 = N + 1;
    const bool pinned = !(ubj > lbj);
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    const double *__restrict__ Gy = w.G;
    Tile tl;
    int np = 0;
    int status = NTM_SCN_QP_ITER_CAP, it = 0;
    bool broke = false;

    // ---- one pass over Gy: gradient at the candidate points and a fixed gradient scale for this QP
    //      sc_j = |F_j| + sum_k |G_jk| max(|lb_k|, |ub_k|)  (rounding level of any gradient component inside the box)
    const double cu1 = (hist.n >= 1) ? hist.u1 : lbj, cu2 = (hist.n >= 2) ? hist.u2 : lbj;
    if (act) {
        w.cand[2 * j] = make_double2(lbj, ubj);
        w.cand[2 * j + 1] = make_double2(cu2, cu1);
    }
    Gp::sync();
    double g0 = 0.0, g1 = 0.0, g2 = 0.0, g3 = 0.0, sc = 0.0;
    if (act) {
        const double *row = Gy + tri_off(j);
        for (int k = 0; k < N; ++k) {
            const double gk = (k <= j) ? row[k] : Gy[tri_off(k) + j];
            const double2 ca = w.cand[2 * k], cb = w.cand[2 * k + 1];
            g0 = fma(gk, ca.x, g0); g1 = fma(gk, ca.y, g1);
            g2 = fma(gk, cb.x, g2); g3 = fma(gk, cb.y, g3);
            sc = fma(fabs(gk), fmax(fabs(ca.x), fabs(ca.y)), sc);
        }
        sc += fabs(Fj);
    }

    enum { PH_COLD = 0, PH_SELECT = 1, PH_ENTER = 2, PH_ITER = 3 };
    int phase = (hist.n == 0) ? PH_COLD : PH_SELECT;
    int kpos = 0;                                        // COLD: next variable; ENTER: next position in the free list
    int nfree0 = 0;
    int nfree = 0;                                       // ITER: number of free variables (uniform)
    int *flist = reinterpret_cast<int *>(w.sol);         // ENTER: free list (w.sol is not used by this solver)
    bool need_load = (phase == PH_COLD);
    int state = -1;
    double u = lbj, g = g0 + Fj;
    double gseed = g;                                    // gradient that seeds the border row at the next block load
    bool stuck = false;                                  // this thread's variable could not be pivoted in: stays on its bound
    int repairs = 0;
    bool have_y = false;                                 // tw.ybuf holds the current border row

    for (;;) {
        int pk = -1, pvar = -1;                          // tableau index / variable of the pivot of this pass (-1: none)
        bool pfwd = true;
        if (phase == PH_SELECT) {
            const double c2v = (hist.n >= 2) ? hist.u2 : lbj, c3v = (hist.n >= 1) ? hist.u1 : lbj;
            const double q0 = Gp::sum(act ? lbj * fma(0.5, g0, Fj) : 0.0, w.red);
            const double q1 = Gp::sum(act ? ubj * fma(0.5, g1, Fj) : 0.0, w.red);
            double qb = q0;
            state = -1; u = lbj; g = g0 + Fj;
            if (q1 < qb) { qb = q1; state = 1; u = ubj; g = g1 + Fj; }
            if (hist.n >= 2) {
                const double q2 = Gp::sum(act ? c2v * fma(0.5, g2, Fj) : 0.0, w.red);
                if (q2 < qb) { qb = q2; state = hist.s2; u = c2v; g = g2 + Fj; }
            }
            if (hist.n >= 1) {
                const double q3 = Gp::sum(act ? c3v * fma(0.5, g3, Fj) : 0.0, w.red);
                if (q3 < qb) { qb = q3; state = hist.s1; u = c3v; g = g3 + Fj; }
            }
            if (pinned) { state = -1; u = lbj; }
            gseed = g; phase = PH_ENTER; kpos = 0; need_load = true;
        }
        if (need_load) {                                 // fresh blocks: Gy with the border row gseed
            if (act) { tw.gbuf[j] = gseed; w.idx[j] = state; }
            if (phase == PH_ENTER) {                     // list of the variables to sweep in (ascending index)
                const int pos = Gp::prefix(act && state == 0, w.ired, nfree0);
                if (act && state == 0) flist[pos] = j;
            }
            Gp::sync();
            tile_load(tl, I, J, n1, Gy, tw.gbuf);
            need_load = false; have_y = false;
        }
        if (phase == PH_COLD) {
            if (kpos < N) { pvar = kpos++; pk = pvar + 1; }
            else {
                if (I >= 0 && J == 0) {
#pragma unroll
                    for (int r = 0; r < NTM_TS; ++r) tw.ybuf[NTM_TS * I + r] = tl.t[r][0];
                }
                Gp::sync();
                const double un = act ? lbj - tw.ybuf[j + 1] : 0.0;     // u0 - inv(G) g(u0), u0 = the lower vertex
                if (!Gp::any(act && !isfinite(un), w.ired)) {
                    hist.u2 = fmin(fmax(un, lbj), ubj);
                    hist.s2 = (un <= lbj) ? -1 : ((un >= ubj) ? 1 : 0);
                    hist.u1 = hist.u2; hist.s1 = hist.s2;
                    hist.n = 2;
                    if (act) w.uv[j] = hist.u2;
                    Gp::sync();
                    const double t = act ? tab_row_dot(N, j, Gy, w.uv) : 0.0;
                    g2 = t; g3 = t;
                }
                Gp::sync();
                phase = PH_SELECT;
                continue;
            }
        } else if (phase == PH_ENTER) {
            if (kpos < nfree0) { pvar = flist[kpos++]; pk = pvar + 1; }   // uniform: same words
            else { phase = PH_ITER; nfree = Gp::count(act && state == 0, w.ired); continue; }
        } else {                                                          // PH_ITER
            if (++it > max_iter) break;
            if (!have_y) {
                if (I >= 0 && J == 0) {
#pragma unroll
                    for (int r = 0; r < NTM_TS; ++r) tw.ybuf[NTM_TS * I + r] = tl.t[r][0];
                }
                Gp::sync();
            }
            have_y = false;
            const bool isfree = act && state == 0;
            const double yj = act ? tw.ybuf[j + 1] : 0.0;
            bool blocked = false;
            int jblk = -1;
            if (nfree > 0) {
                const double pj = -yj;                                    // Newton step to the minimiser on the face
                double aj = INF;
                if (isfree) {
                    if (pj < 0.0) aj = (lbj - u) / pj;
                    else if (pj > 0.0) aj = (ubj - u) / pj;
                }
                const double amin = Gp::argmin(aj, j, w.red, w.ired, jblk);
                blocked = amin < 1.0;
                const double alpha = blocked ? fmax(amin, 0.0) : 1.0;
                if (isfree) u = blocked ? fma(alpha, pj, u) : u + pj;
                // border row: y_F <- (1 - alpha) y_F (0 after a full step), by its owners, before the partition changes
                if (I >= 0 && J == 0) {
                    const double f = blocked ? 1.0 - alpha : 0.0;
#pragma unroll
                    for (int r = 0; r < NTM_TS; ++r) {
                        const int a = NTM_TS * I + r;
                        if (a >= 1 && a < n1 && w.idx[a - 1] == 0) {
                            tl.t[r][0] *= f;
                            if (I == 0) tl.t[0][r] *= f;                   // block (0,0) also holds the mirrored copy T(0, a)
                        }
                    }
                }
                if (blocked) {                                            // a bound blocks: the variable leaves the free set
                    if (j == jblk) { state = (pj < 0.0) ? -1 : 1; u = (pj < 0.0) ? lbj : ubj; }
                    Gp::sync();                                           // everyone has read idx[]
                    if (j == jblk) w.idx[j] = state;
                    pvar = jblk; pk = jblk + 1; pfwd = false;
                }
            }
            if (!blocked) {
                // bound multipliers at the face minimiser, as the tableau sees them
                double lam = INF;
                if (act && !pinned && !stuck) {
                    if (state < 0) lam = yj / sc;
                    else if (state > 0) lam = -yj / sc;
                }
                int jw;
                const double lmin = Gp::argmin(lam, j, w.red, w.ired, jw);
                if (lmin < -NTM_QP_EPS_G) { pvar = jw; pk = jw + 1; pfwd = true; }     // variable jw leaves its bound
                else {
                    // ---- the tableau says optimal: the exact gradient decides
                    if (act) w.uv[j] = u;
                    Gp::sync();
                    const double ge = (act ? tab_row_dot(N, j, Gy, w.uv) : 0.0) + Fj;
                    bool bad = false;
                    if (act && !pinned && !stuck) {
                        if (state == 0) bad = fabs(ge) > NTM_LONG_REFINE_TOL * sc;
                        else bad = ((state < 0) ? ge : -ge) < -NTM_QP_EPS_G * sc;
                    }
                    g = ge;
                    if (!Gp::any(bad, w.ired) || repairs >= NTM_LONG_MAX_REPAIRS) { status = NTM_SCN_OK; break; }
                    ++repairs;
                    if (repairs == NTM_LONG_MAX_REPAIRS - 1) {            // refinement is not converging: fresh blocks
                        gseed = ge; phase = PH_ENTER; kpos = 0; need_load = true;
                        continue;
                    }
                    // border row from the exact gradient: y_F = -T_FF g_F, y_B = g_B - T_BF g_F  (T v with v = g on F, 0 elsewhere)
                    for (int a = j; a < tw.pcn; a += Gp::T) { tw.pcb[a] = 0.0; tw.ybuf[a] = 0.0; }
                    Gp::sync();
                    if (act && state == 0) tw.pcb[j + 1] = ge;
                    Gp::sync();
                    tile_matvec(tl, I, J, tw.pcb, tw.ybuf);
                    Gp::sync();
                    const double ynew = act ? ((state == 0) ? -tw.ybuf[j + 1] : ge - tw.ybuf[j + 1]) : 0.0;
                    Gp::sync();
                    if (act) tw.ybuf[j + 1] = ynew;
                    Gp::sync();
                    if (I >= 0 && J == 0) {
#pragma unroll
                        for (int r = 0; r < NTM_TS; ++r) {
                            const int a = NTM_TS * I + r;
                            if (a >= 1 && a < n1) {
                                tl.t[r][0] = tw.ybuf[a];
                                if (I == 0) tl.t[0][r] = tw.ybuf[a];
                            }
                        }
                    }
                    have_y = true;                                        // ybuf is the border row the next pass reads
                    np = 0;                                               // pcb was used as scratch: restart the double buffer
                    Gp::sync();
                    continue;
                }
            }
        }
        // ---- the one pivot site
        const bool ok = tile_pivot<GW>(tl, I, J, pk, pfwd, tw, np);
        if (phase == PH_COLD) {
            if (!ok) { phase = PH_SELECT; Gp::sync(); }                   // no unconstrained minimiser: start from a vertex
        } else if (phase == PH_ENTER) {
            if (!ok && j == pvar) {                                       // dependent direction: to the nearer bound
                state = (u - lbj <= ubj - u) ? -1 : 1; u = (state < 0) ? lbj : ubj; w.idx[j] = state; stuck = true;
            }
        } else if (pfwd) {
            if (ok) { if (j == pvar) { state = 0; w.idx[j] = 0; } ++nfree; }
            else if (j == pvar) stuck = true;
            Gp::sync();
        } else if (!ok) { broke = true; break; }
        else --nfree;
    }
    if (it > max_iter) it = max_iter;
    // a pinned variable (lbj == ubj) has one value either way; its state is the side the gradient points to, which is
    // what the literal kernels map back to U: b * [umin, umax] can round to one y although umin < umax
    if (pinned) state = (g < 0.0) ? 1 : -1;
    const bool nonfinite = Gp::any(act && !(isfinite(u) && isfinite(g)), w.ired);
    double Uj = (state < 0) ? lbj : ((state > 0) ? ubj : fmin(fmax(u, lbj), ubj));
    if (nonfinite) Uj = nan("");
    if (nonfinite || broke) status = NTM_SCN_NONFINITE;
    hist.u2 = hist.u1; hist.s2 = hist.s1;
    hist.u1 = Uj; hist.s1 = state;
    hist.n = min(hist.n + 1, 2);
    Gp::sync();
    Uout = Uj;
    iters_out = it;
    return status;
}

}  // namespace ntm
