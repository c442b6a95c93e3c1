// ntm_loop.cuh -- the fused persistent closed loop (NTM_MPC_Sim.m:63-73 + 80-131), shared by the translation units that
// instantiate it: ntm_kernels.cu (one-warp groups, dense-Gamma and state-row instantiations) and ntm_loop_long.cu (the
// long-horizon literal instantiations on the sweep tableau of ntm_long.cuh).
#pragma once
#include "ntm_device.cuh"
#include "ntm_kernels.h"
#include "ntm_long.cuh"
#include <type_traits>

namespace ntm {

// NTM_MPC_Sim.m:130: x+ = A(rho(x)) x + B(rho(x)) u  (+C with NTM_PROFILE_PLANT_C); a22 = the (2,2) entry of A.m:2
__device__ __forceinline__ void plant_euler_a22(const Params &P, int flags, double a22, double w, double om, double u,
                                                double &nw, double &nom) {
    double a11, a21, b;
    schedule(P, flags, w, om, a11, a21, b);
    nw = a11 * w + b * u;
    nom = a21 * w + a22 * om;
    if (flags & NTM_PROFILE_PLANT_C) { nw += P.C1; nom += P.C2; }
}
__device__ __forceinline__ void plant_euler(const Params &P, int flags, double w, double om, double u, double &nw,
                                            double &nom) {
    plant_euler_a22(P, flags, P.a22, w, om, u, nw, nom);
}

// NTM_PROFILE_TAUE_W (SURVEY 8f-4; NTM_MPC_Sim.m:14 "tau_E = tau_E0; currently NOT EXACT FORMULA"): (2,2) entry of A.m:2
// with tau_E(w) = tau_E0 * (1 - c_tauE * w); a22n = 1 - Ts/tau_E0 is params[2], ctau = params[15].
__device__ __forceinline__ double a22_taue(double a22n, double ctau, double w) {
    return 1.0 - (1.0 - a22n) / (1.0 - ctau * w);
}

// The cold plant options: NTM_PROFILE_PLANT_RK4 and NTM_PROFILE_TAUE_W (the Euler map with tau_E of the state it is
// evaluated at).  a22n: the NOMINAL (2,2) entry (the fused loop overwrites P.a22 with the value its controller holds).
// RK4: the Euler map is x + g(x,u) with g = Ts * (dx/dt) of the GRE model, so the classical RK4 step over one sample
// needs no extra parameter: k1 = g(x), k2 = g(x + k1/2), k3 = g(x + k2/2), k4 = g(x + k3),
// x+ = x + (k1 + 2 k2 + 2 k3 + k4)/6, summed as ((k1 + 2 k2) + (2 k3 + k4)) / 6 (the order the tests' CPU checker uses).
// The fused kernel carries this code only in its LoopTraits::COLD instantiations: inlined into the literal hot kernel
// it cost 44 bytes of spills at the 96-register budget, out of line 84.
__device__ __forceinline__ void plant_of(const Params &P, int flags, double a22n, double ctau, double w, double om,
                                         double u, double &nw, double &nom) {
    const bool te = (flags & NTM_PROFILE_TAUE_W) != 0;
    auto euler = [&](double zw, double zo, double &ew, double &eo) {
        plant_euler_a22(P, flags, te ? a22_taue(a22n, ctau, zw) : a22n, zw, zo, u, ew, eo);
    };
    if (!(flags & NTM_PROFILE_PLANT_RK4)) { euler(w, om, nw, nom); return; }
    // a ROLLED loop over the four stages (one copy of the scheduling functions and their three divisions, not four)
    double yw = w, yo = om, sw = 0.0, so = 0.0, aw = 0.0, ao = 0.0;
#pragma unroll 1
    for (int st = 0; st < 4; ++st) {
        double e1, e2;
        euler(yw, yo, e1, e2);
        const double kw = e1 - yw, ko = e2 - yo;
        // ((k1 + 2 k2) + (2 k3 + k4)) / 6: first pair in (sw, so), second pair in (aw, ao)
        if (st == 0) { sw = kw; so = ko; }
        else if (st == 1) { sw += 2.0 * kw; so += 2.0 * ko; }
        else if (st == 2) { aw = 2.0 * kw; ao = 2.0 * ko; }
        else { aw += kw; ao += ko; }
        const double h = (st < 2) ? 0.5 : 1.0;
        yw = w + h * kw; yo = om + h * ko;
    }
    nw = w + (sw + aw) / 6.0;
    nom = om + (so + ao) / 6.0;
}

// The plant of ntm_plant_step and of the perturbed fused loop (LoopTraits::PERT), every rounding spelled out.  nvcc
// contracts the products of plant_euler_a22 / plant_of into FMAs differently depending on where they are inlined: every
// fused-loop instantiation evaluates a21 w + a22 om as fma(a22, om, a21 w), the RK4 / tau_E(w) plant kernel evaluated
// it as fma(w, a21, a22 om), and the RK4 stages of the fused loop take w^2 + w_marg^2 (NTM_PROFILE_RHO1_SQ) as one FMA where
// the Euler map rounds w^2 first.  This function is the fused loop's form, so that stepping a controller with
// ntm_plant_step reproduces the fused loop bit for bit under every plant profile, and so that the perturbed loop
// gives ntm_plant_step's bits wherever it is instantiated.  a22n, ctau: as plant_of.
__device__ __forceinline__ void plant_exact(const Params &P, int flags, double a22n, double ctau, double w, double om,
                                            double u, double &nw, double &nom) {
    const bool te = (flags & NTM_PROFILE_TAUE_W) != 0, sq = (flags & NTM_PROFILE_RHO1_SQ) != 0;
    const bool rk4 = (flags & NTM_PROFILE_PLANT_RK4) != 0, pc = (flags & NTM_PROFILE_PLANT_C) != 0;
    auto euler = [&](double zw, double zo, double &ew, double &eo) {
        const double a22 = te ? __dsub_rn(1.0, __ddiv_rn(__dsub_rn(1.0, a22n), __dsub_rn(1.0, __dmul_rn(ctau, zw)))) : a22n;
        const double ww = __dmul_rn(zw, zw);
        const double r1 = __drcp_rn(sq ? (rk4 ? __fma_rn(zw, zw, P.wmarg2) : __dadd_rn(ww, P.wmarg2)) : __dadd_rn(zw, P.wmarg2));
        const double r2 = __ddiv_rn(ww, zo);
        const double ws = __ddiv_rn(zw, P.w_dep), ws2 = __dmul_rn(ws, ws);
        const double den = __fma_rn(__dmul_rn(ws, ws2), 0.64, __fma_rn(ws2, 0.43, __fma_rn(ws, 1.5, 1.0)));
        const double r3 = __ddiv_rn(__fma_rn(ws, 0.24, 0.25), den);
        const double a11 = __fma_rn(P.c_a11, r1, 1.0), a21 = __dmul_rn(P.c_a21, r2), b = __dmul_rn(P.c_b, r3);
        ew = __fma_rn(zw, a11, __dmul_rn(b, u));
        eo = __fma_rn(a22, zo, __dmul_rn(zw, a21));
        if (pc) { ew = __dadd_rn(ew, P.C1); eo = __dadd_rn(eo, P.C2); }
    };
    if (!rk4) { euler(w, om, nw, nom); return; }
    double yw = w, yo = om, sw = 0.0, so = 0.0, aw = 0.0, ao = 0.0;   // ((k1 + 2 k2) + (2 k3 + k4)) / 6, as plant_of
#pragma unroll 1
    for (int st = 0; st < 4; ++st) {
        double e1, e2;
        euler(yw, yo, e1, e2);
        const double kw = __dsub_rn(e1, yw), ko = __dsub_rn(e2, yo);
        if (st == 0) { sw = kw; so = ko; }
        else if (st == 1) { sw = __fma_rn(kw, 2.0, sw); so = __fma_rn(ko, 2.0, so); }
        else if (st == 2) { aw = __dadd_rn(kw, kw); ao = __dadd_rn(ko, ko); }
        else { aw = __dadd_rn(aw, kw); ao = __dadd_rn(ao, ko); }
        const double h = (st < 2) ? 0.5 : 1.0;
        yw = __fma_rn(h, kw, w); yo = __fma_rn(h, ko, om);
    }
    nw = __dadd_rn(w, __ddiv_rn(__dadd_rn(sw, aw), 6.0));
    nom = __dadd_rn(om, __ddiv_rn(__dadd_rn(so, ao), 6.0));
}

// =================================================================================================
// fused persistent closed loop
// =================================================================================================
// Inclusive composition of the stage maps up to this thread's stage j (cold path of the state rows):
// (pa, pc) = first column of Phi's block j, s22 = its (2,2) entry a22^(j+1), (k1, k2) = Lambda's block j
// (Rho_to_PhiGammaLambda.m:17-23,47-52), so that Phi_j*x + Lambda_j = (pa*x1 + k1, pc*x1 + s22*x2 + k2).
template <int GW>
__device__ void stage_prefix(int N, int j, const Work &w, const Params &P, double a11, double a21, double &pa,
                             double &pc, double &s22, double &k1, double &k2) {
    const bool act = j < N;
    if constexpr (GW == 1) {
        Aff m;
        m.a = act ? a11 : 1.0; m.c = act ? a21 : 0.0;
        m.k1 = act ? P.C1 : 0.0; m.k2 = act ? P.C2 : 0.0;
        const Aff inc = aff_scan(m, j, N, P.a22);
        pa = inc.a; pc = inc.c; k1 = inc.k1; k2 = inc.k2;
        s22 = 1.0;
        for (int t = 0; t <= j && t < N; ++t) s22 *= P.a22;
    } else {
        double p1 = 1.0, p2 = 0.0, v1 = 0.0, v2 = 0.0, s = 1.0;
        pa = 1.0; pc = 0.0; k1 = 0.0; k2 = 0.0; s22 = 1.0;
        for (int d = 0; d < N; ++d) {
            const double a = w.a11s[d], c = w.a21s[d];
            const double nv1 = fma(a, v1, P.C1);
            const double nv2 = fma(P.a22, v2, fma(c, v1, P.C2));
            v1 = nv1; v2 = nv2;
            const double np1 = a * p1;
            const double np2 = fma(c, p1, P.a22 * p2);
            p1 = np1; p2 = np2;
            s *= P.a22;
            if (d == j) { pa = p1; pc = p2; k1 = v1; k2 = v2; s22 = s; }
        }
    }
}

// What the instantiation closed_loop_kernel<GW, DENSE, EXT, LV, CTL> carries.  EXT (EXT_* in ntm_kernels.h) is only the
// key: run_scenario and closed_loop_kernel test these members, never EXT itself.  (They are read through a type alias:
// function-scope constexpr locals for the same conditions changed the register assignment of the literal state-row
// kernels.)  CTL: the controller-step instantiation (ntm_mpc_step, ntm_mpc_step_sc) of a box instantiation with
// multi-warp groups or of a state-row one; the one-warp box instantiations run controller steps as a runtime mode
// (LoopArgs::ctl) at unchanged register counts, in the multi-warp ones that mode cost 2 registers, and 228 bytes of
// spill stores in closed_loop_kernel<4, false, 0, 0>; the state-row ones sit at their register caps (DESIGN section 4.8).
template <int GW, bool DENSE, int EXT, bool CTL = false>
struct LoopTraits {
    static constexpr bool ROWS = (EXT == 2 || EXT == 4);   // getWLc's state rows
    static constexpr bool PERT = (EXT == 3 || EXT == 4);   // the perturbed plant (LoopArgs::pp: its own parameters and
                                                           // profile bits, d_k and v_k)
    static constexpr bool COLD = (EXT == 1 || EXT == 2);   // the controller's plant with the RK4 / tau_E(w) options, and
                                                           // the controller-side tau_E(w)
    // long horizons, literal Gamma, box QP: the QP runs on the packed sweep tableau of ntm_long.cuh
    static constexpr bool LONG = (GW > 1) && !DENSE && !ROWS;
    static constexpr bool CTL_MODE = (GW == 1 && EXT == 0);   // LoopArgs::ctl selects the controller step at run time
    // the record code (NTM_CTRL_DOUBLES): controller steps and the two-phase launch
    static constexpr bool REC = (EXT == 0 && (GW == 1 || CTL)) || (EXT == 2 && CTL);
    static constexpr bool REGEN = ROWS && CTL;   // a resumed frozen record rebuilds its rows (they are not stored)
    // two-phase launch (headline instantiation only): a launch runs the time steps [k_begin, k_end) of the scenario
    static constexpr bool TWOPH = (GW == 1) && !DENSE && (EXT == 0);
    // __launch_bounds__ minimum blocks per SM
    static constexpr int MIN_BLOCKS = GW == 1 ? (EXT == 0 ? 5 : ((EXT == 1 || EXT == 3) ? 4 : 3)) : (LONG ? 3 : 1);
    using WorkT = typename std::conditional<LONG, LongWork, Work>::type;
};

// getWLc's frozen rows (NTM_MPC_Sim.m:74, rho(x0) on every stage), kept at the offline build: Phi0, Lam0 from
// stage_prefix, and the Gamma tile the Hessian build left in shared memory (dense Gamma, to Gam0) or P12 (literal),
// and b0 = b of this build
template <bool DENSE>
__device__ __forceinline__ void freeze_rows(int N, int j, const Work &w, const ExtWork &xw, double *Gam0, double pa,
                                            double pc, double k1, double k2, double bb, double &b0) {
    if (j < N) {
        xw.Phi0[j] = make_double2(pa, pc); xw.Lam0[j] = make_double2(k1, k2);
        if constexpr (DENSE) {
            const double2 *src = reinterpret_cast<const double2 *>(w.GamS + (size_t)j * w.ldgam);
            double2 *dst = reinterpret_cast<double2 *>(Gam0 + (size_t)j * w.ldgam);
            for (int i = 0; i < N; ++i) dst[i] = src[i];
        } else {
            xw.P0[j] = w.P12[j];
        }
    }
    b0 = bb;
}

// The state rows of the QP at hand: the free response fs = Phi x + Lam of this stage, from the G, F just built
// (srows = 1) or from the frozen rows, built at the first QP (srows = 2; literal Gamma: + the column scale cs = b0 / b)
template <int GW, bool DENSE>
__device__ __forceinline__ void state_rows_setup(int N, int j, const Work &w, const Params &P, const ExtWork &xw,
                                                 double *Gam0, bool frozen, bool &built, double a11, double a21,
                                                 double bb, double x1, double x2, double &s22, double &b0) {
    const bool act = j < N;
    if (!frozen || !built) {
        double pa, pc, k1, k2;
        stage_prefix<GW>(N, j, w, P, a11, a21, pa, pc, s22, k1, k2);
        if (frozen) freeze_rows<DENSE>(N, j, w, xw, Gam0, pa, pc, k1, k2, bb, b0);
        else if (act) xw.fs[j] = make_double2(fma(pa, x1, k1), fma(pc, x1, fma(s22, x2, k2)));
        built = true;
    }
    if (frozen && act) {
        const double2 ph = xw.Phi0[j], lm = xw.Lam0[j];
        xw.fs[j] = make_double2(fma(ph.x, x1, lm.x), fma(ph.y, x1, fma(s22, x2, lm.y)));
        if constexpr (!DENSE) xw.cs[j] = b0 / bb;
    }
}

// LV (LONG only): 0 = tableau in registers (N + 1 <= 7 * 10 / 7 * 15 for 2 / 4 warps), 1 = tableau in shared memory
template <int GW, bool DENSE, int EXT, int LV = 0, bool CTL = false>
__device__ void run_scenario(const LoopArgs &a, int s, int j, const typename LoopTraits<GW, DENSE, EXT, CTL>::WorkT &w,
                             unsigned char *gbase, int tI = -1, int tJ = -1) {
    using Gp = Group<GW>;
    using LT = LoopTraits<GW, DENSE, EXT, CTL>;
    const int N = a.N, S = a.S, flags = a.flags, layout = a.layout;
    const bool act = j < N;
    const bool lead = (j == 0);
    const bool fxk = (flags & NTM_PROFILE_F_XK) != 0;
    constexpr bool dense = DENSE;                        // (flags & (GAMMA_I | DENSE_G)) != 0, resolved by the launcher
    load_params_shared(w.prm, a.params, layout, a.params_count, s, j);
    Gp::sync();
    const Params &P = *w.prm;
    // controller step (ntm_mpc_step[_sc]): a.x0 is the measured state, the loop state comes from the caller's record
    const bool ctl = LT::CTL_MODE ? (a.ctl != 0) : CTL;
    double x01 = __ldg(a.x0 + elem(layout, S, 2, s, 0)), x02 = __ldg(a.x0 + elem(layout, S, 2, s, 1));
    double x1 = x01, x2 = x02;
    // perturbed plant: (x1, x2) is what the controller sees, y_k = x_k + v_k; the offline build (:63-65)
    // and frozen state rows (:74) run from y_0.  The true state x_k lives in xk only (written by the lead, read back by
    // the group after a barrier), so no register carries it across the loop.
    if constexpr (LT::PERT) {
        const PlantIn &pi = a.pp;
        if (pi.noise != nullptr) {
            x01 += __ldg(pi.noise + elem(layout, S, 2 * a.k_sim, s, 0)); x02 += __ldg(pi.noise + elem(layout, S, 2 * a.k_sim, s, 1));
            x1 = x01; x2 = x02;
        }
    }
    // NTM_PROFILE_TAUE_W (COLD only): the shared parameter block carries the a22 the controller holds over
    // the horizon of the current time step, a22(tau_E(xk(1,k))); the nominal value and c_tauE stay in registers
    [[maybe_unused]] double a22n = 0.0, ctau = 0.0;
    [[maybe_unused]] bool taue = false;
    if constexpr (LT::COLD) {
        taue = (flags & NTM_PROFILE_TAUE_W) != 0;
        a22n = P.a22;
        if (taue) {
            const int pss = (a.params_count == 1) ? 0 : s, pSS = (a.params_count == 1) ? 1 : a.params_count;
            ctau = __ldg(a.params + elem(layout, pSS, NTM_NPARAM, pss, 15));
            Gp::sync();                                   // every thread has read the nominal a22
            if (lead) w.prm->a22 = a22_taue(a22n, ctau, x1);
            Gp::sync();
        }
    }
    const int EX = 2 * (a.k_sim + 1);
    // output addressing: three arrays in `layout`, or one packed record of rec_ld doubles per scenario
    const bool rec = a.rec_ld > 0;
    const size_t rbase = (size_t)s * (size_t)a.rec_ld;
    auto xk_at = [&](int e) -> size_t { return rec ? rbase + (size_t)e : elem(layout, S, EX, s, e); };
    auto uk_at = [&](int e) -> size_t { return rec ? rbase + (size_t)e : elem(layout, S, a.k_sim, s, e); };

    // offline build, NTM_MPC_Sim.m:63-65: rho(x0) repeated over the horizon.  This thread's stage entries
    // stay in registers; the shared copies feed the broadcast reads (b everywhere, a11/a21 in the serial paths).
    double a11, a21, bb;
    schedule(P, flags, x1, x2, a11, a21, bb);
    double sE = 1.0;                                     // a22^j: (2,2) entry of the product of the first j stage matrices
    if (GW == 1) { const double a22 = P.a22; for (int t = 0; t < j && t < N; ++t) sE *= a22; }
    if (act) { w.bbs[j] = bb; if (GW > 1 || dense) { w.a11s[j] = a11; w.a21s[j] = a21; } }
    Gp::sync();
    double Uold = 1.0;                                   // :86 (ones; persists across k, D13)
    double Uj = 0.0, cost = 0.0;
    QpHist hist = {0.0, 0.0, -1, -1, 0};                 // previous two QP solutions (warm-start candidates)
    double hU1 = 0.0, hU2 = 0.0;                         // the same in U-space (literal path: the QP runs in y = b .* U)
    [[maybe_unused]] double b0 = bb, s22 = 0.0;          // frozen state rows: b and a22^(j+1) of the offline build
    [[maybe_unused]] bool rows_built = false;
    int hs1 = -1, hs2 = -1;
    bool first_qp = true;
    // state rows, literal Gamma: active sets of the last two state-row QPs of this scenario, offered to the
    // next one as a warm start (per thread: (vst + 1) | mask of this state's four rows << 2), and the "warm start failed,
    // run this QP again cold" flag
    [[maybe_unused]] int hw1 = 0, hw2 = 0, hwn = 0;
    [[maybe_unused]] bool retry = false;
    [[maybe_unused]] bool regen_rows = false;            // REGEN: rebuild the frozen rows of a resumed record first
    int status = 0, inner = 0, qpit = 0, k = 0, it = 0;
    const int qp_cap = 10 * N + 20;
    [[maybe_unused]] int nslow = 0, nqpit = 0;
    bool resumed = false;
    if constexpr (LT::REC) {
        // The loop state a record carries across a time step (layout: NTM_CTRL_DOUBLES in include/ntm_mpc.h), restored
        // for phase B of a two-phase launch and for a controller step whose record has run before.  G and F for the first
        // QP are rebuilt at the top of the loop from the same stage entries and from x0 or (NTM_PROFILE_F_XK) the last
        // state the record saw: bit-identical to one launch.
        const int N7 = 7 * N;
        const double *sv = a.sv + (size_t)s * NTM_CTRL_DOUBLES(N);
        if (a.sv != nullptr && (ctl ? sv[N7 + 6] != 0.0 : a.k_begin > 0)) {
            resumed = true;
            if (act) {
                a11 = sv[j]; a21 = sv[N + j]; bb = sv[2 * N + j]; Uold = sv[3 * N + j];
                const int pk = (int)sv[6 * N + j];
                if (dense) {                                     // the QP runs in U itself: its own history
                    hist.u1 = sv[4 * N + j]; hist.u2 = sv[5 * N + j]; hist.s1 = (pk & 3) - 1; hist.s2 = ((pk >> 2) & 3) - 1;
                } else {
                    hU1 = sv[4 * N + j]; hU2 = sv[5 * N + j]; hs1 = (pk & 3) - 1; hs2 = ((pk >> 2) & 3) - 1;
                    if constexpr (LT::ROWS) { hw1 = (pk >> 4) & 63; hw2 = (pk >> 10) & 63; }
                }
            }
            x1 = sv[N7]; x2 = sv[N7 + 1]; x01 = sv[N7 + 2]; x02 = sv[N7 + 3]; cost = sv[N7 + 4];
            const int fl = (int)sv[N7 + 5];
            status = ctl ? 0 : (fl & 3); first_qp = ((fl >> 2) & 1) != 0; hist.n = (fl >> 3) & 3;
            k = ctl ? 0 : a.k_begin;
            if constexpr (LT::REGEN) {
                hwn = (fl >> 5) & 3;
                // Frozen rows (:74) are a function of x0 alone and are not stored: the first pass of the loop builds
                // G, F from rho(x0) on every stage, exactly as the offline build did, copies the rows out and then
                // reloads the record's stage entries (below, after build_GF).
                if (a.srows == 2) {
                    regen_rows = true;
                    schedule(P, flags, x01, x02, a11, a21, bb);
                }
            }
            Gp::sync();
            if (act) { w.bbs[j] = bb; if (GW > 1 || dense) { w.a11s[j] = a11; w.a21s[j] = a21; } }
            Gp::sync();
        }
    }
    if constexpr (LT::PERT) {
        if (lead) { a.xk[xk_at(0)] = __ldg(a.x0 + elem(layout, S, 2, s, 0)); a.xk[xk_at(1)] = __ldg(a.x0 + elem(layout, S, 2, s, 1)); }
    } else {
        if (lead && !resumed && !ctl) { a.xk[xk_at(0)] = x1; a.xk[xk_at(1)] = x2; }
    }

    // One pass of this loop = [re-]condense (:66,:72-73 / :119-121), the stop rule of the iteration that just
    // finished (:123-127) and, at the end of a time step, the plant (:130); then the next QP + rollout (:97-117).
    // Written as a single loop so that build_GF and qp_solve are instantiated once (instruction-cache footprint).
    for (;;) {
        double Fj;
        if constexpr (LT::LONG) Fj = build_GF_toeplitz_packed<GW>(N, j, w, P, fxk ? x1 : x01, fxk ? x2 : x02);
        else Fj = build_GF<GW, DENSE>(N, j, w, P, flags, a11, a21, sE, fxk ? x1 : x01, fxk ? x2 : x02);
        if constexpr (LT::REGEN) {
            if (regen_rows) {                            // the offline build of a resumed frozen record: keep its rows
                double pa, pc, k1, k2;
                stage_prefix<GW>(N, j, w, P, a11, a21, pa, pc, s22, k1, k2);
                freeze_rows<DENSE>(N, j, w, carve_ext(gbase + a.qbytes, N),
                                   reinterpret_cast<double *>(gbase + a.qbytes + ext_bytes(N)), pa, pc, k1, k2, bb, b0);
                rows_built = true; regen_rows = false;
                const double *sv = a.sv + (size_t)s * NTM_CTRL_DOUBLES(N);
                if (act) { a11 = sv[j]; a21 = sv[N + j]; bb = sv[2 * N + j]; }
                Gp::sync();
                if (act) { w.bbs[j] = bb; if (GW > 1 || dense) { w.a11s[j] = a11; w.a21s[j] = a21; } }
                Gp::sync();
                continue;                                // now G, F of the record's stage entries
            }
        }
        if (it > 0 && !retry) {
            inner = it;
            bool brk = false;
            if (!(flags & NTM_PROFILE_INNER_FIXED)) {                               // the fixed policy never looks at |Uold - U|
                const double d = Gp::sum(act ? fabs(Uold - Uj) : 0.0, w.red);      // :123
                brk = d < a.eps;                                                    // :124-125
            }
            const bool stop = brk || it == a.i_sim;                                 // :94
            if (!brk) Uold = Uj;                                                    // :127 (skipped by the break)
            if (stop) {
                const double u0 = Gp::bcast0(Uj, w.red);                            // :107  uk(:,k) = U(1)
                if constexpr (LT::PERT) {
                    // the plant's own block and profile bits, read here (once per time step, no shared copy), then + d_k
                    if (!isfinite(u0)) status = max(status, (int)NTM_SCN_NONFINITE);
                    const PlantIn &pi = a.pp;
                    const Params Q = load_params(pi.pparams, layout, pi.pparams_count, s);
                    const int pf = pi.pflags;
                    const double qtau = (pf & NTM_PROFILE_TAUE_W)
                        ? __ldg(pi.pparams + elem(layout, pi.pparams_count, NTM_NPARAM, pi.pparams_count == 1 ? 0 : s, 15)) : 0.0;
                    const double t1 = a.xk[xk_at(2 * k)], t2 = a.xk[xk_at(2 * k + 1)];   // x_k, written by the lead
                    double nw, nom;
                    plant_exact(Q, pf, Q.a22, qtau, t1, t2, u0, nw, nom);              // = ntm_plant_step
                    if (pi.dist != nullptr) {
                        nw += __ldg(pi.dist + elem(layout, S, 2 * a.k_sim, s, 2 * k));
                        nom += __ldg(pi.dist + elem(layout, S, 2 * a.k_sim, s, 2 * k + 1));
                    }
                    const double e1 = nw - P.r1, e2 = nom - P.r2;                     // judged on the true state
                    cost += e1 * (P.q11 * e1 + P.q12 * e2) + e2 * (P.q12 * e1 + P.q22 * e2);
                    if (lead) {
                        a.xk[xk_at(2 * (k + 1))] = nw;
                        a.xk[xk_at(2 * (k + 1) + 1)] = nom;
                    }
                } else if (ctl) {                                                   // the caller runs the plant
                    if (!isfinite(u0)) status = max(status, (int)NTM_SCN_NONFINITE);
                } else {
                    double nw, nom;
                    if constexpr (LT::COLD) plant_of(P, flags, a22n, ctau, x1, x2, u0, nw, nom);   // :130, or its RK4 / tau_E(w) refinement
                    else plant_euler(P, flags, x1, x2, u0, nw, nom);                // :130
                    x1 = nw; x2 = nom;
                    if constexpr (LT::COLD) {
                        if (taue) {                      // tau_E of the new measured width, held over the next step's horizon
                            Gp::sync();                  // (G, F just built keep the previous value: a workspace assignment)
                            if (lead) w.prm->a22 = a22_taue(a22n, ctau, x1);
                            Gp::sync();
                            if (GW == 1) { const double a22 = P.a22; sE = 1.0; for (int t = 0; t < j && t < N; ++t) sE *= a22; }
                        }
                    }
                    const double e1 = x1 - P.r1, e2 = x2 - P.r2;
                    cost += e1 * (P.q11 * e1 + P.q12 * e2) + e2 * (P.q12 * e1 + P.q22 * e2);
                    if (lead) {
                        a.xk[xk_at(2 * (k + 1))] = x1;
                        a.xk[xk_at(2 * (k + 1) + 1)] = x2;
                    }
                }
                if (lead) {
                    a.uk[uk_at(k)] = u0;
#ifdef NTM_DEBUG_NSLOW
                    if (a.inner) a.inner[elem(layout, S, a.k_sim, s, k)] = nslow;     // cumulative count of active-set QPs
#else
                    if (a.inner) a.inner[elem(layout, S, a.k_sim, s, k)] = inner;
#endif
                    if (a.qpit) a.qpit[elem(layout, S, a.k_sim, s, k)] = qpit;
                }
                ++k; it = 0; qpit = 0;
                if constexpr (LT::REC) {
                    // the record (see the restore above): end of a controller step, or of phase A (then the next scenario)
                    if (a.sv != nullptr && (ctl || (k == a.k_end && k < a.k_sim))) {
                        const int N7 = 7 * N;
                        double *sv = a.sv + (size_t)s * NTM_CTRL_DOUBLES(N);
                        if (act) {
                            sv[j] = a11; sv[N + j] = a21; sv[2 * N + j] = bb; sv[3 * N + j] = Uold;
                            sv[4 * N + j] = dense ? hist.u1 : hU1; sv[5 * N + j] = dense ? hist.u2 : hU2;
                            // + the active sets of the last two state-row QPs (literal Gamma; 0 outside ROWS)
                            sv[6 * N + j] = dense ? (double)((hist.s1 + 1) | ((hist.s2 + 1) << 2))
                                                  : (double)((hs1 + 1) | ((hs2 + 1) << 2) | (hw1 << 4) | (hw2 << 10));
                        }
                        if (lead) {
                            sv[N7] = x1; sv[N7 + 1] = x2; sv[N7 + 2] = x01; sv[N7 + 3] = x02; sv[N7 + 4] = cost;
                            sv[N7 + 5] = (double)((status & 3) | ((first_qp ? 1 : 0) << 2) | (hist.n << 3) | (hwn << 5));
                            sv[N7 + 6] = ctl ? sv[N7 + 6] + 1.0 : (double)k;
                            if constexpr (LT::TWOPH) {
                                if (!ctl) a.lpt_key[s] = min(12 * min(nslow, 12) + min(nqpit, 11), NTM_LPT_BINS - 1);
                            }
                        }
                        if (!ctl) return;
                    }
                }
            }
        }
        if (k >= a.k_sim) break;
        if constexpr (LT::PERT) {
            if (it == 0) {               // as for a controller step: the measurement y_k = x_k + v_k
                Gp::sync();              // the lead has just written x_k
                x1 = a.xk[xk_at(2 * k)]; x2 = a.xk[xk_at(2 * k + 1)];
                const PlantIn &pi = a.pp;
                if (pi.noise != nullptr) {
                    x1 += __ldg(pi.noise + elem(layout, S, 2 * a.k_sim, s, 2 * k)); x2 += __ldg(pi.noise + elem(layout, S, 2 * a.k_sim, s, 2 * k + 1));
                }
                if (!(isfinite(x1) && isfinite(x2))) status = max(status, (int)NTM_SCN_NONFINITE);
            }
        } else if (ctl && it == 0) {     // G, F on hand are built; the step itself (QP, rollout) starts from the measurement
            x1 = __ldg(a.x0 + elem(layout, S, 2, s, 0)); x2 = __ldg(a.x0 + elem(layout, S, 2, s, 1));
        }
        if (!retry) ++it;
        int nit = 0;
        int st = NTM_SCN_OK;
        // the x_0 block of getWLc.m:30 has no U: it only asks that x_k itself (y_k under a perturbed plant: the state the
        // controller sees) is inside the state box
        [[maybe_unused]] bool x0bad = false;
        if constexpr (LT::ROWS) x0bad = x1 < a.xmin1 || x1 > a.xmax1 || x2 < a.xmin2 || x2 > a.xmax2;
        if constexpr (DENSE) {
            st = qp_solve<GW>(N, j, w, Fj, P.umin, P.umax, hist, Uj, qp_cap, nit);   // :97
            if constexpr (LT::ROWS && GW == 1) {
                if (a.srows != 0) {
                    // NTM_MPC_Sim.m:97 as written, ANY Gamma index: the state rows of getWLc.m:57 (L = Mcal*Gamma + Ecal)
                    // are read from the dense Gamma tile the tensor-core Hessian build left in shared memory (DenseRows);
                    // frozen rows (:74) keep a copy of the offline tile.  QP variables are U itself here.  Every QP starts
                    // cold from the box minimiser: the literal branch's warm start, tried here, moved one scenario of the
                    // parity sample by 2 % in one input on the consistent profile (chaotic at the 1e-4 level).
                    const IneqWork q = carve_ineq(gbase + a.wbytes, N, 4 * N);
                    const ExtWork xw = carve_ext(gbase + a.qbytes, N);
                    double *Gam0 = reinterpret_cast<double *>(gbase + a.qbytes + ext_bytes(N));
                    const bool frozen = a.srows == 2;
                    state_rows_setup<GW, true>(N, j, w, P, xw, Gam0, frozen, rows_built, a11, a21, bb, x1, x2, s22, b0);
                    Gp::sync();
                    if (st == NTM_SCN_OK) {
                        const DenseRows rows = {frozen ? Gam0 : w.GamS, w.ldgam, xw.fs, a.xmin1, a.xmax1, a.xmin2, a.xmax2, N};
                        int vs = 0;
                        const int nit0 = nit;
                        double Uc = Uj;
                        const auto regen = make_regen([&]() {  // Gamma tile and Hessian are rebuilt from the stage entries
                            build_GF<GW, true>(N, j, w, P, flags, a11, a21, sE, fxk ? x1 : x01, fxk ? x2 : x02);
                        });
                        st = x0bad ? (int)NTM_SCN_INFEASIBLE
                                   : qp_ineq_continue<GW>(N, rows, j, w, q, Fj, P.umin, P.umax, Uc, nit + 100 * N + 50, nit,
                                                          &vs, regen);
                        if (st != NTM_SCN_OK || nit != nit0) {
                            Uj = (vs < 0) ? P.umin : ((vs > 0) ? P.umax : fmin(fmax(Uc, P.umin), P.umax));
                            if (!(Uc == Uc)) Uj = Uc;
                        }
                    }
                }
            }
        } else {
            // literal Gamma: the Hessian table is in the variables y = b .* U (build_GF_toeplitz).  Box, warm-start
            // candidates and partition states go to y-space with the current b; the result comes back with its bound
            // components exactly umin / umax (the stop rule :123 compares bits).
            const double yl = bb * P.umin, yh = bb * P.umax;
            const bool neg = bb < 0.0;
            double yj = 0.0;
            // state rows: offer the active set of the QP before last (or the last one) instead of solving the box QP first
            [[maybe_unused]] bool try_warm = false;
            [[maybe_unused]] int wv = 0, wm = -1;
            if constexpr (LT::ROWS) {
                if (a.srows != 0) {
                    if ((a.rows_warm & 1) && !retry && hwn > 0 && !x0bad) {
                        const int hh = (hwn >= 2) ? hw2 : hw1;
                        wv = (hh & 3) - 1; wm = hh >> 2;
                        try_warm = Gp::any(act && wm != 0, w.ired);
                    }
                    if (!try_warm) wm = -1;
                }
                retry = false;
            }
            if (!try_warm) {
                hist.u1 = bb * hU1; hist.u2 = bb * hU2;
                hist.s1 = neg ? -hs1 : hs1; hist.s2 = neg ? -hs2 : hs2;
                if constexpr (LT::LONG && LV == 0) {
                    const TileWork tw = {w.tpcb, w.tybuf, w.tgbuf, w.tpcn};
                    st = qp_solve_tile<GW>(N, j, w, tw, tI, tJ, Fj, fmin(yl, yh), fmax(yl, yh), hist, yj, qp_cap, nit);
                } else if constexpr (LT::LONG) {
                    const auto regen = make_regen([&]() {      // the tableau is rebuilt from the stage entries (same values)
                        build_GF_toeplitz_packed<GW>(N, j, w, P, fxk ? x1 : x01, fxk ? x2 : x02);
                    });
                    st = qp_solve_long<GW>(N, j, w, Fj, fmin(yl, yh), fmax(yl, yh), hist, yj, qp_cap, nit, regen);
                } else {
                    if constexpr (LT::TWOPH) {
                        st = qp_solve<GW>(N, j, w, Fj, fmin(yl, yh), fmax(yl, yh), hist, yj, qp_cap, nit, &nslow);
                        nqpit += nit - 1;
                    } else {
                        st = qp_solve<GW>(N, j, w, Fj, fmin(yl, yh), fmax(yl, yh), hist, yj, qp_cap, nit);
                    }
                }
                const int sy = hist.s1, su = neg ? -sy : sy;
                Uj = (su < 0 || bb == 0.0) ? P.umin : ((su > 0) ? P.umax : fmin(fmax(yj / bb, P.umin), P.umax));
                if (!(yj == yj)) Uj = yj;                                                             // NaN stays NaN
                const int sn = (bb == 0.0) ? -1 : su;
                if (first_qp) { hU2 = Uj; hs2 = sn; first_qp = false; } else { hU2 = hU1; hs2 = hs1; }
                hU1 = Uj; hs1 = sn;
            }
            if constexpr (LT::ROWS) {
                if (a.srows != 0) {
                    // NTM_MPC_Sim.m:97 as written: L*U <= c + W*xk(:,k) with getWLc's state rows kept.  The box
                    // minimiser above is the dual-feasible start of the active-set continuation (qp_ineq_continue).
                    const IneqWork q = carve_ineq(gbase + a.wbytes, N, 4 * N);
                    const ExtWork xw = carve_ext(gbase + a.qbytes, N);
                    const bool frozen = a.srows == 2;
                    state_rows_setup<GW, false>(N, j, w, P, xw, nullptr, frozen, rows_built, a11, a21, bb, x1, x2, s22, b0);
                    Gp::sync();
                    if (st == NTM_SCN_OK) {
                        const StateRows rows = {frozen ? xw.P0 : w.P12, xw.fs, frozen ? xw.cs : nullptr,
                                                a.xmin1, a.xmax1, a.xmin2, a.xmax2, N};
                        int vs = 0;
                        const int nit0 = nit;
                        double yc = yj;
                        const auto regen = make_regen([&]() {  // the Hessian table is rebuilt from the stage entries (same values)
                            build_GF<GW, false>(N, j, w, P, flags, a11, a21, sE, fxk ? x1 : x01, fxk ? x2 : x02);
                        });
                        st = x0bad ? (int)NTM_SCN_INFEASIBLE
                                   : qp_ineq_continue<GW>(N, rows, j, w, q, Fj, fmin(yl, yh), fmax(yl, yh), yc,
                                                          nit + 100 * N + 50, nit, &vs, regen, wv, wm);
                        if (st == NTM_QP_WARM_FAILED) {                // the offered set is not dual feasible here: this QP
                            retry = true;                              // again from the box minimiser (the pass starts over:
                            continue;                                  // build_GF restores the Hessian the attempt overwrote)
                        }
                        if (try_warm || st != NTM_SCN_OK || nit != nit0) {   // a row was violated: the answer moved off the box minimiser
                            const int su2 = neg ? -vs : vs;
                            Uj = (su2 < 0 || bb == 0.0) ? P.umin : ((su2 > 0) ? P.umax : fmin(fmax(yc / bb, P.umin), P.umax));
                            if (!(yc == yc)) Uj = yc;
                        }
                        if (st == NTM_SCN_OK) {                        // remember the active set this QP ended on
                            Gp::sync();
                            int hnew = vs + 1;
                            if (act) {
#pragma unroll
                                for (int qq = 0; qq < 4; ++qq) hnew |= (q.gact[4 * j + qq] ? 1 : 0) << (2 + qq);
                            }
                            hw2 = hw1; hw1 = hnew; hwn = min(hwn + 1, 2);
                        }
                    }
                }
            }
        }
        if constexpr (LT::ROWS) {
            if (st == NTM_SCN_INFEASIBLE) {
                // quadprog exitflag -2 (:100-101) returns no U and the script cannot continue: the scenario ends here,
                // everything it has not produced yet is NaN.  A controller step (k_sim = 1) returns NaN u and U and
                // leaves its record as it was before the step: the save sits on the stop-rule path, not on this one.
                const double nan = __longlong_as_double(0x7ff8000000000000LL);
                status = max(status, st);
                for (int kk = k; kk < a.k_sim; ++kk) {
                    if (lead) {
                        a.uk[uk_at(kk)] = nan;
                        if (!ctl) {                      // a controller step has no xk
                            a.xk[xk_at(2 * (kk + 1))] = nan;
                            a.xk[xk_at(2 * (kk + 1) + 1)] = nan;
                        }
                        if (a.inner) a.inner[elem(layout, S, a.k_sim, s, kk)] = (kk == k) ? it : 0;
                        if (a.qpit) a.qpit[elem(layout, S, a.k_sim, s, kk)] = (kk == k) ? qpit + nit : 0;
                    }
                    if (a.Uk != nullptr && act) a.Uk[elem(layout, S, N * a.k_sim, s, kk * N + j)] = nan;
                }
                cost = nan;
                break;
            }
        }
        status = max(status, st);
        qpit += nit;
        if (a.Uk != nullptr && act) a.Uk[elem(layout, S, N * a.k_sim, s, k * N + j)] = Uj;        // :106
        // rollout with the OLD rho (:110-113), then re-schedule on the predicted states (:114-116)
        double xs1 = 0.0, xs2 = 0.0;
        if constexpr (GW == 1) {
            Aff m;
            m.a = act ? a11 : 1.0; m.c = act ? a21 : 0.0;
            m.k1 = act ? fma(bb, Uj, P.C1) : 0.0; m.k2 = act ? P.C2 : 0.0;
            const Aff exc = aff_exclusive(aff_scan(m, j, N, P.a22), j);
            xs1 = fma(exc.a, x1, exc.k1);
            xs2 = fma(exc.c, x1, fma(sE, x2, exc.k2));
        } else {
            if (act) w.qv[j] = fma(bb, Uj, P.C1);
            Gp::sync();
            double c1 = x1, c2 = x2;
            for (int i = 0; i < N; ++i) {
                if (i == j) { xs1 = c1; xs2 = c2; }
                const double aa = w.a11s[i], cc = w.a21s[i], q = w.qv[i];
                const double n1 = fma(aa, c1, q);
                const double n2 = fma(P.a22, c2, fma(cc, c1, P.C2));
                c1 = n1; c2 = n2;
            }
            Gp::sync();
        }
        if (act) {
            schedule<true>(P, flags, xs1, xs2, a11, a21, bb);
            w.bbs[j] = bb;
            if (GW > 1 || dense) { w.a11s[j] = a11; w.a21s[j] = a21; }
        }
        Gp::sync();
    }
    if (lead) {
        if constexpr (LT::PERT) {
            const double t1 = a.xk[xk_at(2 * a.k_sim)], t2 = a.xk[xk_at(2 * a.k_sim + 1)];
            if (!(isfinite(t1) && isfinite(t2) && isfinite(cost))) status = max(status, (int)NTM_SCN_NONFINITE);
        } else {
            if (!(isfinite(x1) && isfinite(x2) && isfinite(cost))) status = max(status, (int)NTM_SCN_NONFINITE);
        }
        if (a.cost) a.cost[rec ? rbase : (size_t)s] = cost;
        if (a.status) a.status[s] = status;
        if (rec && a.rec_status) a.rec_status[rbase] = (double)status;
    }
}

template <int GW, bool DENSE, int EXT, int LV = 0, bool CTL = false>
__global__ void __launch_bounds__(GW == 1 ? 128 : 32 * GW, (LoopTraits<GW, DENSE, EXT, CTL>::MIN_BLOCKS))
closed_loop_kernel(LoopArgs a, unsigned int gbytes) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using Gp = Group<GW>;
    const int gib = (GW == 1) ? (int)(threadIdx.x >> 5) : 0;
    const int j = (GW == 1) ? (int)(threadIdx.x & 31) : (int)threadIdx.x;
    const int gpb = (GW == 1) ? (int)(blockDim.x >> 5) : 1;
    using LT = LoopTraits<GW, DENSE, EXT, CTL>;
    typename LT::WorkT w;
    if constexpr (LT::LONG) {
        w = carve_long(smem_raw, a.N);
    } else {
        double *hbig = a.hscratch + ((size_t)blockIdx.x * gpb + gib) * a.N * odd_ld(a.N);
        w = carve(smem_raw + (size_t)gib * gbytes, a.N, a.hcap, hbig, a.gam);
    }
    int tI = -1, tJ = -1;
    if constexpr (LT::LONG && LV == 0) tile_coords(j, (a.N + 1 + NTM_TS - 1) / NTM_TS, tI, tJ);
    if (w.GamS) for (int i = j; i < (int)gam_doubles(a.N, a.gam); i += Gp::T) w.GamS[i] = 0.0;
    for (int i = j; i < 2 * a.N; i += Gp::T) { w.QP12[i] = make_double2(0.0, 0.0); w.QE12[i] = make_double2(0.0, 0.0); }
    Gp::sync();
    for (;;) {
        int s = 0;
        if (j == 0) s = (int)atomicAdd(a.counter, 1u);
        s = Gp::bcast0(s, w.ired);
        if (s >= a.S) break;
        if (a.perm != nullptr) s = __ldg(a.perm + s);       // phase B of a two-phase launch: longest first
        run_scenario<GW, DENSE, EXT, LV, CTL>(a, s, j, w, smem_raw + (size_t)gib * gbytes, tI, tJ);
        Gp::sync();
    }
    // the last group to leave re-arms the work queue for the next launch (saves a memset per call: latency)
    if (j == 0) {
        const unsigned int groups = gridDim.x * ((GW == 1) ? (blockDim.x >> 5) : 1);
        __threadfence();
        if (atomicAdd(a.counter + 1, 1u) == groups - 1) { a.counter[0] = 0u; a.counter[1] = 0u; __threadfence(); }
    }
}


}  // namespace ntm
